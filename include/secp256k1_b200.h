/*
 * secp256k1_b200.h -- C ABI of the B200-native batched secp256k1 engine.
 *
 * The reference (gitlab.com/yawning/secp256k1-voi, Go) has no FFI boundary of
 * its own; its exported Go API is the contract.  Each entry point below is the
 * batch form of one reference call and cites it (paths relative to the
 * reference root).  INTEGRATION.md shows the cgo binding a maintainer adds.
 *
 * Conventions (inherited from the reference, SURVEY.md section 8b):
 *   - every encoding is big-endian: scalars / digests / x-coordinates 32 B,
 *     compact signatures r||s 64 B (recoverable r||s||v 65 B), points SEC 1
 *     uncompressed 65 B (04||X||Y);
 *   - n items, row-major, caller owns every buffer; calls are synchronous and
 *     retain no pointer after returning (the cgo pointer rule);
 *   - call-level misuse / CUDA failure: negative int return, never abort;
 *     data-level outcomes: one status byte per item;
 *   - a context is bound to one CUDA device and may be used from any thread
 *     (calls on one context serialise on an internal mutex); use one context
 *     per GPU -- or two, from two host threads, so that one batch's copies
 *     overlap the other's arithmetic -- and one process per GPU for multi-GPU runs;
 *   - there is NO CPU fallback: without a usable CUDA device s256_init fails.
 *
 * The *_dev twins take device pointers and a cudaStream_t (as void*; NULL =
 * default stream), enqueue the work and return without synchronising; they
 * are what bench.py times with inputs resident in HBM.  All calls on one
 * context share its scratch memory, so they are also ordered ON THE DEVICE:
 * the work of a call starts only after the work of the previous call on the
 * same context has finished, whatever streams the two calls used (an event
 * recorded at the end of every call).  Two contexts on one device overlap freely.
 */
#ifndef SECP256K1_B200_H
#define SECP256K1_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library itself is built with -fvisibility=hidden */
#endif

typedef struct s256_ctx s256_ctx;

/* return codes */
#define S256_SUCCESS 0
#define S256_ERR_NO_DEVICE (-1)   /* no CUDA device / wrong architecture */
#define S256_ERR_CUDA (-2)        /* a CUDA runtime call failed (see s256_last_cuda_error) */
#define S256_ERR_ARG (-3)         /* NULL pointer, bad length: the reference panics here */
#define S256_ERR_NOMEM (-4)
#define S256_ERR_UNIMPLEMENTED (-5)
#define S256_ERR_NCCL (-6)

/* per-item status bytes */
#define S256_ST_INVALID 0   /* input rejected (bad point / scalar / signature encoding) */
#define S256_ST_OK 1        /* output is a finite point / verification succeeded */
#define S256_ST_IDENTITY 2  /* result is the point at infinity (output bytes zeroed);
                               the reference encodes it as the single byte 0x00
                               (point_s11n.go:75-77) or returns an error (XBytes, :123-125) */
#define S256_ST_BAD_ALGORITHM 3 /* ParseASN1PublicKey: algorithm is not ecPublicKey (secec/s11n.go:31) */
#define S256_ST_BAD_CURVE 4     /* ParseASN1PublicKey: named curve is not secp256k1 (secec/s11n.go:32) */

/* flags */
#define S256_FLAG_REJECT_MALLEABLE 1u /* ECDSAOptions.RejectMalleable, secec/ecdsa.go:72-75,212 */

/* --- lifecycle ----------------------------------------------------------- */
/* device < 0: use the calling thread's current device.  max_batch = 0 picks
 * the default chunk capacity (2^20 items); larger batches are processed in
 * chunks.  Builds the generator tables on the device (the reference does this
 * at package init, point_mul_table.go:75-100,147-160).  Device memory per
 * context: 1.5 GiB of generator tables plus about 2.6 KB of scratch per item of
 * max_batch (2.7 GB at the default); S256_ERR_NOMEM if that does not fit. */
int s256_init(s256_ctx **ctx, int device, size_t max_batch);
void s256_free(s256_ctx *ctx);
const char *s256_strerror(int code);
const char *s256_last_cuda_error(const s256_ctx *ctx);
int s256_device(const s256_ctx *ctx);

/* --- Point.ScalarBaseMult (point_mul_table.go:168) + UncompressedBytes
 *     (point_s11n.go:66).  Constant time.  k32 is decoded like
 *     NewScalarFromBytes (scalar.go:248: reduced mod n). */
int s256_scalar_base_mult(s256_ctx *ctx, const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status);
int s256_scalar_base_mult_dev(s256_ctx *ctx, const uint8_t *d_k32, size_t n, uint8_t *d_out65, uint8_t *d_status,
                              void *stream);

/* --- Point.ScalarMult (point_mul_glv.go:257) + UncompressedBytes.  Constant
 *     time in the scalar.  pt65 decoded like NewPointFromBytes
 *     (point_s11n.go:234,178). */
int s256_scalar_mult(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *out65,
                     uint8_t *status);
int s256_scalar_mult_dev(s256_ctx *ctx, const uint8_t *d_k32, const uint8_t *d_pt65, size_t n, uint8_t *d_out65,
                         uint8_t *d_status, void *stream);

/* --- PrivateKey.ECDH (secec/secec.go:53): x(k*P), 32 B; identity is an
 *     error (status S256_ST_IDENTITY). */
int s256_ecdh(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *x32, uint8_t *status);
int s256_ecdh_dev(s256_ctx *ctx, const uint8_t *d_k32, const uint8_t *d_pt65, size_t n, uint8_t *d_x32,
                  uint8_t *d_status, void *stream);

/* --- NewPointFromBytes on compressed encodings (point_s11n.go:234,140: 02/03||X,
 *     canonical x, square root, parity select): 33 B -> 65 B + status. */
int s256_point_decompress(s256_ctx *ctx, const uint8_t *pt33, size_t n, uint8_t *out65, uint8_t *status);

/* --- (*Point).CompressedBytes (point_s11n.go:90-117) behind NewPointFromBytes (point_s11n.go:234): validated
 *     uncompressed 65 B -> compressed 33 B (02 | 03 by the parity of y, then X) + status; a row that does not
 *     decode to a point of the curve gives zeros and S256_ST_INVALID. */
int s256_point_compress(s256_ctx *ctx, const uint8_t *pt65, size_t n, uint8_t *out33, uint8_t *status);

/* --- Point.DoubleScalarMultBasepointVartime (point_mul_glv.go:307):
 *     u1*G + u2*P, variable time. */
int s256_double_scalar_mult_basepoint_vartime(s256_ctx *ctx, const uint8_t *u1_32, const uint8_t *u2_32,
                                              const uint8_t *pt65, size_t n, uint8_t *out65, uint8_t *status);
int s256_double_scalar_mult_basepoint_vartime_dev(s256_ctx *ctx, const uint8_t *d_u1_32, const uint8_t *d_u2_32,
                                                  const uint8_t *d_pt65, size_t n, uint8_t *d_out65,
                                                  uint8_t *d_status, void *stream);

/* --- secec.PublicKey.Verify with EncodingCompact (secec/ecdsa.go:171 ->
 *     secec/s11n.go:129 -> verify, ecdsa.go:392).  pk65 is decoded like
 *     secec.NewPublicKey (secec/secec.go:188); digest32 is the leftmost
 *     32 bytes of the digest (ecdsa.go:477).  ok[i] in {0,1}. */
int s256_ecdsa_verify(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig64,
                      uint32_t flags, size_t n, uint8_t *ok);
int s256_ecdsa_verify_dev(s256_ctx *ctx, const uint8_t *d_pk65, const uint8_t *d_digest32, const uint8_t *d_sig64,
                          uint32_t flags, size_t n, uint8_t *d_ok, void *stream);

/* --- host-side codecs in front of the batch (byte parsing only, no arithmetic) ----------------
 * Signatures arrive concatenated in `der`, row i being der[offsets[i] .. offsets[i+1]) (n + 1 offsets).
 *   s256_parse_asn1_signatures: secec.ParseASN1Signature (secec/s11n.go:83): strict DER
 *     SEQUENCE{r,s}, both in [1, n) -> r||s rows; ok[i] = 0 (row zeroed) when rejected.
 *   s256_is_valid_signature_encoding_bip0066: bitcoin.IsValidSignatureEncodingBIP0066
 *     (secec/bitcoin/asn1_shitcoin.go:13), rows INCLUDE the trailing sighash byte.
 *   s256_ecdsa_verify_asn1: PublicKey.Verify with EncodingASN1 (secec/ecdsa.go:171-228).  The rows are
 *     staged to the device and parsed there (the parse of s256_parse_asn1_signatures); S256_ERR_ARG for
 *     decreasing offsets, checked before anything is enqueued.
 *   s256_bitcoin_verify_asn1: bitcoin.VerifyASN1 (secec/bitcoin/ecdsa_shitcoin.go:29): BIP-66
 *     check, sighash byte stripped, s <= n/2 enforced; parsed on the device as above.
 *   s256_parse_asn1_public_keys: secec.ParseASN1PublicKey (secec/s11n.go:38-76) up to the call of
 *     NewPublicKey: strict SubjectPublicKeyInfo with the ecPublicKey / secp256k1 OIDs; yields the
 *     SEC 1 point bytes (row stride 65, left-aligned, point_len[i] in {1, 33, 65}) and a status
 *     (S256_ST_OK / S256_ST_INVALID / S256_ST_BAD_ALGORITHM / S256_ST_BAD_CURVE).  Feed the rows
 *     to s256_new_public_keys for the curve checks.
 *   s256_build_asn1_public_keys: PublicKey.ASN1Bytes (secec/secec.go:109, s11n.go:190): 88 bytes.
 *   s256_build_asn1_signatures: secec.BuildASN1Signature (secec/s11n.go:110): rows of stride 72,
 *     out_len[i] bytes used. */
int s256_parse_asn1_public_keys(const uint8_t *der, const size_t *offsets, size_t n, uint8_t *point65,
                                uint8_t *point_len, uint8_t *status);
int s256_build_asn1_public_keys(const uint8_t *pk65, size_t n, uint8_t *out88);
/* secec.NewPublicKey (secec/secec.go:183-199) over rows of mixed SEC 1 encodings (stride 65, enc_len[i] in
 * {1, 33, 65} bytes used): validated uncompressed bytes out; status S256_ST_OK / S256_ST_INVALID /
 * S256_ST_IDENTITY (a valid encoding, but not a public key: errAIsInfinity). */
int s256_new_public_keys(s256_ctx *ctx, const uint8_t *enc65, const uint8_t *enc_len, size_t n, uint8_t *out65,
                         uint8_t *status);
/* secec.ParseASN1PublicKey end to end: host SPKI parse, then s256_new_public_keys. */
int s256_parse_asn1_public_keys_checked(s256_ctx *ctx, const uint8_t *der, const size_t *offsets, size_t n,
                                        uint8_t *out65, uint8_t *status);
int s256_build_asn1_signatures(const uint8_t *sig64, size_t n, uint8_t *out72, uint8_t *out_len);
int s256_parse_asn1_signatures(const uint8_t *der, const size_t *offsets, size_t n, uint8_t *sig64, uint8_t *ok);
int s256_is_valid_signature_encoding_bip0066(const uint8_t *der, const size_t *offsets, size_t n, uint8_t *ok);
int s256_ecdsa_verify_asn1(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *der,
                           const size_t *offsets, uint32_t flags, size_t n, uint8_t *ok);
int s256_bitcoin_verify_asn1(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *der,
                             const size_t *offsets, size_t n, uint8_t *ok);
/* Device-resident DER signatures.  d_der and d_offsets live in device memory: d_offsets holds n + 1 values relative
 * to d_der (offsets[0] need not be 0), row i being d_der[offsets[i] .. offsets[i+1]).  These forms cannot check the
 * offsets without synchronising, so a row with offsets[i+1] < offsets[i] is invalid and none of its bytes are read
 * (ok[i] = 0, and a zeroed r||s row).  The host forms of all four return S256_ERR_ARG for such offsets instead.  One
 * thread parses one row and reads at most 73 bytes of it: a row longer than that is rejected from its length alone
 * (no strict-DER signature exceeds 72 bytes, and BIP-66 allows at most 73 with the sighash byte), in the host forms
 * too.  No form synchronises; outputs are written on `stream`.
 *   s256_ecdsa_verify_asn1_dev: s256_ecdsa_verify_asn1 (flags as for s256_ecdsa_verify).
 *   s256_bitcoin_verify_asn1_dev: s256_bitcoin_verify_asn1; S256_FLAG_REJECT_MALLEABLE is implied.
 *   s256_parse_asn1_signatures_dev: the sig64 and ok bytes of s256_parse_asn1_signatures.
 *   s256_is_valid_signature_encoding_bip0066_dev: the ok bytes of s256_is_valid_signature_encoding_bip0066. */
int s256_ecdsa_verify_asn1_dev(s256_ctx *ctx, const uint8_t *d_pk65, const uint8_t *d_digest32, const uint8_t *d_der,
                               const size_t *d_offsets, uint32_t flags, size_t n, uint8_t *d_ok, void *stream);
int s256_bitcoin_verify_asn1_dev(s256_ctx *ctx, const uint8_t *d_pk65, const uint8_t *d_digest32, const uint8_t *d_der,
                                 const size_t *d_offsets, size_t n, uint8_t *d_ok, void *stream);
int s256_parse_asn1_signatures_dev(s256_ctx *ctx, const uint8_t *d_der, const size_t *d_offsets, size_t n, uint8_t *d_sig64,
                                   uint8_t *d_ok, void *stream);
int s256_is_valid_signature_encoding_bip0066_dev(s256_ctx *ctx, const uint8_t *d_der, const size_t *d_offsets, size_t n,
                                                 uint8_t *d_ok, void *stream);

/* --- PrivateKey.Sign with RFC6979SHA256() as the entropy source (secec/ecdsa.go:92-135,284-390;
 *     nonce: secec/ecdsa_k_rfc6979.go): deterministic, constant time.  priv32 must be a canonical
 *     non-zero scalar (NewPrivateKey, secec/secec.go:141).  Outputs: compact r||s (low-s normalised),
 *     the recovery id (0..3), status.
 *     Two deliberate differences from the reference, neither observable on valid inputs: (1) a nonce that gives r = 0
 *     or s = 0 (probability ~2^-256) is reported as S256_ST_INVALID where the reference draws the next DRBG output
 *     (secec/ecdsa.go's loop); (2) the reference re-verifies a BIP-340 signature before returning it (schnorr.go:393)
 *     and this library does not -- a caller that wants that fault check runs s256_schnorr_verify / s256_ecdsa_verify on
 *     the batch it just signed (same context, ~2.5x the signing time). */
int s256_ecdsa_sign_rfc6979(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *digest32, size_t n, uint8_t *sig64,
                            uint8_t *recid, uint8_t *status);
int s256_ecdsa_sign_rfc6979_dev(s256_ctx *ctx, const uint8_t *d_priv32, const uint8_t *d_digest32, size_t n,
                                uint8_t *d_sig64, uint8_t *d_recid, uint8_t *d_status, void *stream);

/* --- secec.RecoverPublicKey (secec/ecdsa.go:244) on r||s||v
 *     (secec/s11n.go:156). */
int s256_ecdsa_recover(s256_ctx *ctx, const uint8_t *digest32, const uint8_t *sig65, size_t n, uint8_t *pk65,
                       uint8_t *status);
int s256_ecdsa_recover_dev(s256_ctx *ctx, const uint8_t *d_digest32, const uint8_t *d_sig65, size_t n,
                           uint8_t *d_pk65, uint8_t *d_status, void *stream);

/* --- bitcoin.SchnorrPublicKey.Verify (secec/bitcoin/schnorr.go:221) incl.
 *     NewSchnorrPublicKey / lift_x (:257).  msg is n rows of msg_len bytes. */
int s256_schnorr_verify(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                        const uint8_t *sig64, size_t n, uint8_t *ok);
int s256_schnorr_verify_dev(s256_ctx *ctx, const uint8_t *d_pkx32, const uint8_t *d_msg, size_t msg_len,
                            const uint8_t *d_sig64, size_t n, uint8_t *d_ok, void *stream);

/* BIP-340 batch verification (BIP-340 "Batch Verification"; per item: bitcoin.SchnorrPublicKey.Verify,
 * secec/bitcoin/schnorr.go:221, incl. lift_x :257).  Inputs are laid out as for s256_schnorr_verify.
 * *ok = 1 iff every row would verify; 0 otherwise (except with probability <= 2^-127 per call when
 * some row is invalid).  n == 0 gives 1.  Variable time (public data).
 * One equation, (sum a_i s_i) G = sum a_i R_i + sum (a_i e_i) P_i with R_i = lift_x(r_i), a_0 = 1 and 128-bit a_i
 * derived from a hash tree over all the rows (DESIGN.md), checked by one multi-scalar multiplication.  A row is
 * rejected, and with it the batch, when its key does not lift_x, r >= p, r is not the x-coordinate of a curve point, or
 * s >= n.  To find the invalid rows of a rejected batch, run s256_schnorr_verify on it.  The _dev form writes the
 * verdict byte to device memory and does not synchronise.  S256_ERR_ARG for a context with max_batch < 2. */
int s256_schnorr_batch_verify(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                              const uint8_t *sig64, size_t n, uint8_t *ok);
int s256_schnorr_batch_verify_dev(s256_ctx *ctx, const uint8_t *d_pkx32, const uint8_t *d_msg, size_t msg_len,
                                  const uint8_t *d_sig64, size_t n, uint8_t *d_ok, void *stream);

/* Recoverable ECDSA batch verification (per item: secec.PublicKey.Verify with EncodingCompactRecoverable,
 * secec/ecdsa.go:221-227 -- RecoverPublicKey :244 on r||s||v, then a comparison with the key).  Rows: pk65
 * (uncompressed keys), digest32 (leftmost 32 bytes of the digest, reduced mod n as in s256_ecdsa_verify) and sig65
 * (r||s||v).  flags as for s256_ecdsa_verify (S256_FLAG_REJECT_MALLEABLE: s > n/2 fails).  *ok = 1 iff every row
 * would verify; 0 otherwise (except with probability <= 2^-127 per call when some row is invalid).  n == 0 gives 1.
 * Variable time (public data).
 * One equation, (sum a_i u1_i) G + sum (a_i u2_i) Q_i - sum a_i R_i = O with R_i = RecoverPoint(r_i, v_i),
 * u1_i = e_i / s_i, u2_i = r_i / s_i, a_0 = 1 and 128-bit a_i derived from a hash tree over all the rows (DESIGN.md),
 * checked by one multi-scalar multiplication.  A row is rejected, and with it the batch, when r or s is not in [1, n),
 * v >= 4, r + n >= p with v & 2, r (+ n) is not the x-coordinate of a curve point, the key does not decode as
 * secec.NewPublicKey decodes it (04 || X || Y, canonical, on the curve), or, with S256_FLAG_REJECT_MALLEABLE, s > n/2.
 * To find the invalid rows of a rejected batch, run s256_ecdsa_recover on it and compare each recovered key (status
 * S256_ST_OK) with the row's key.  The _dev form writes the verdict byte to device memory and does not synchronise.
 * S256_ERR_ARG for NULL arguments and for a context with max_batch < 2. */
int s256_ecdsa_recoverable_batch_verify(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65,
                                        uint32_t flags, size_t n, uint8_t *ok);
int s256_ecdsa_recoverable_batch_verify_dev(s256_ctx *ctx, const uint8_t *d_pk65, const uint8_t *d_digest32,
                                            const uint8_t *d_sig65, uint32_t flags, size_t n, uint8_t *d_ok, void *stream);

/* --- bitcoin.SchnorrPrivateKey.Sign (secec/bitcoin/schnorr.go:111-147 -> signSchnorr :322): BIP-340
 *     signing with caller-supplied auxiliary randomness (32 B per row; the reference draws it from
 *     its entropy source, :130-141).  priv32 as for NewPrivateKey; constant time. */
int s256_schnorr_sign(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, size_t msg_len, const uint8_t *aux32,
                      size_t n, uint8_t *sig64, uint8_t *status);
int s256_schnorr_sign_dev(s256_ctx *ctx, const uint8_t *d_priv32, const uint8_t *d_msg, size_t msg_len,
                          const uint8_t *d_aux32, size_t n, uint8_t *d_sig64, uint8_t *d_status, void *stream);

/* --- BIP-340 over messages of different lengths (bitcoin.SchnorrPublicKey.Verify, schnorr.go:221, and
 *     bitcoin.SchnorrPrivateKey.Sign, :111, take a message of any length; BIP-340 allows it since 2022).
 *     Messages arrive concatenated in `msg` as for s256_parse_asn1_signatures: row i is
 *     msg[offsets[i] .. offsets[i+1]), n + 1 offsets (offsets[0] need not be 0); msg may be NULL when every row is
 *     empty (host forms only).  Every other buffer is laid out as for the uniform twin.
 *   s256_schnorr_verify_varlen: ok[i] as s256_schnorr_verify gives it for row i alone.
 *   s256_schnorr_batch_verify_varlen: the verdict of s256_schnorr_batch_verify (the same equation, soundness bound,
 *     rejection rules and max_batch < 2 rule) over these rows.  The randomizers are defined as for the uniform call,
 *     so rows that all have length L give the seed and rows of the uniform call with msg_len = L.
 *   s256_schnorr_sign_varlen: sig64 and status as s256_schnorr_sign gives them for each row.
 *   s256_debug_schnorr_batch_rows_varlen: the outputs of s256_debug_schnorr_batch_rows.
 * The host forms return S256_ERR_ARG for decreasing offsets, checked before anything is enqueued, and S256_ERR_NOMEM
 * when the message bytes of one chunk (max_batch rows) do not fit the device staging.  In the _dev forms offsets is a
 * device array of n + 1 values relative to the device pointer msg; these forms cannot check it without synchronising,
 * so a row with offsets[i+1] < offsets[i] is invalid and none of its message bytes are read: ok[i] = 0, the batch
 * verdict 0, the sign status S256_ST_INVALID (zeroed signature).  One thread hashes one row: a warp waits for its
 * longest message, so a very long message slows the 31 rows beside it. */
int s256_schnorr_verify_varlen(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, const size_t *offsets,
                               const uint8_t *sig64, size_t n, uint8_t *ok);
int s256_schnorr_verify_varlen_dev(s256_ctx *ctx, const uint8_t *d_pkx32, const uint8_t *d_msg, const size_t *d_offsets,
                                   const uint8_t *d_sig64, size_t n, uint8_t *d_ok, void *stream);
int s256_schnorr_batch_verify_varlen(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, const size_t *offsets,
                                     const uint8_t *sig64, size_t n, uint8_t *ok);
int s256_schnorr_batch_verify_varlen_dev(s256_ctx *ctx, const uint8_t *d_pkx32, const uint8_t *d_msg,
                                         const size_t *d_offsets, const uint8_t *d_sig64, size_t n, uint8_t *d_ok,
                                         void *stream);
int s256_schnorr_sign_varlen(s256_ctx *ctx, const uint8_t *priv32, const uint8_t *msg, const size_t *offsets,
                             const uint8_t *aux32, size_t n, uint8_t *sig64, uint8_t *status);
int s256_schnorr_sign_varlen_dev(s256_ctx *ctx, const uint8_t *d_priv32, const uint8_t *d_msg, const size_t *d_offsets,
                                 const uint8_t *d_aux32, size_t n, uint8_t *d_sig64, uint8_t *d_status, void *stream);

/* --- h2c.Secp256k1_XMD_SHA256_SSWU_RO / _NU (secec/h2c/h2c.go:25,49): RFC 9380 hash_to_curve
 *     (random_oracle != 0) or encode_to_curve over n messages of msg_len bytes sharing one domain
 *     separation tag.  dst_len == 0 is an error (errInvalidDomainSep); a DST longer than 255 bytes is
 *     hashed as the RFC prescribes.  Constant time.  status: S256_ST_OK / S256_ST_IDENTITY.
 *     s256_expand_message_xmd exposes expandMessageXMD (h2c_expand_message.go:33) for len_in_bytes <= 96. */
int s256_hash_to_curve(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len, size_t n,
                       int random_oracle, uint8_t *out65, uint8_t *status);
int s256_expand_message_xmd(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                            size_t n, size_t len_in_bytes, uint8_t *out);
/* The same over device-resident rows, and over messages of different lengths.  Row i's out65 and status are those of
 * s256_hash_to_curve on that row alone.  The DST stays a host pointer in every form (one public parameter per call,
 * with the rules above); the _dev forms pass it to the device inside a kernel launch, so they read no host memory of
 * the caller after returning.
 *   s256_hash_to_curve_dev: d_msg, d_out65 and d_status are device pointers (any alignment).
 *   s256_hash_to_curve_varlen: messages concatenated in `msg` as for s256_schnorr_verify_varlen: row i is
 *     msg[offsets[i] .. offsets[i+1]), n + 1 offsets (offsets[0] need not be 0); msg may be NULL when every row is
 *     empty.  S256_ERR_ARG for decreasing offsets, checked before anything is enqueued; S256_ERR_NOMEM when the
 *     message bytes of one chunk (max_batch rows) do not fit the device staging.
 *   s256_hash_to_curve_varlen_dev: d_offsets is a device array of n + 1 values relative to d_msg.  This form cannot
 *     check it without synchronising, so a row with offsets[i+1] < offsets[i] reads none of its bytes and gets
 *     S256_ST_INVALID with 65 zero bytes (a status the uniform forms never return).
 * The _dev forms do not synchronise; outputs are written on `stream`.  Hashing is constant time in the message bytes
 * and the DST, not in the message length (as in the reference, whose SHA-256 also runs longer on longer input): one
 * thread hashes one row, so a warp waits for its longest message and a very long message slows the 31 rows beside it. */
int s256_hash_to_curve_dev(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *d_msg, size_t msg_len,
                           size_t n, int random_oracle, uint8_t *d_out65, uint8_t *d_status, void *stream);
int s256_hash_to_curve_varlen(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *msg,
                              const size_t *offsets, size_t n, int random_oracle, uint8_t *out65, uint8_t *status);
int s256_hash_to_curve_varlen_dev(s256_ctx *ctx, const uint8_t *dst, size_t dst_len, const uint8_t *d_msg,
                                  const size_t *d_offsets, size_t n, int random_oracle, uint8_t *d_out65,
                                  uint8_t *d_status, void *stream);

/* --- Point.MultiScalarMult[Vartime] (point_mul_multi.go:25,73): sum k_i*P_i
 *     over this context's items -> one 65-byte point.  n == 0 gives the
 *     identity.  *status: S256_ST_OK / S256_ST_IDENTITY / S256_ST_INVALID (a
 *     point failed to decode).  s256_msm_partial returns the projective
 *     partial sum (X||Y||Z, 96 B big-endian) for the caller to combine across
 *     GPUs (one small gather), and s256_msm_combine folds m partials. */
int s256_msm(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, uint8_t *out65,
             uint8_t *status);
int s256_msm_partial(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime,
                     uint8_t *partial96, uint8_t *status);
int s256_msm_combine(s256_ctx *ctx, const uint8_t *partials96, size_t m, uint8_t *out65, uint8_t *status);
/* device-resident twin: k32 / pt65 / out65 / status are device pointers, nothing is synchronised */
int s256_msm_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n, int vartime, uint8_t *out65,
                 uint8_t *status, void *stream);

/* --- Point.MultiScalarMult over a batch SHARDED across GPUs (BASELINE.json configs[4]; the operation is
 *     point_mul_multi.go:25-117, the sharding is this engine's).  One process and one context per GPU; rank g
 *     passes its own contiguous slice (n_local items, possibly 0).  Every rank reduces its slice to one projective
 *     partial, ONE ncclAllGather of 112 bytes per rank brings the partials together on every GPU, they are folded
 *     and encoded there: all ranks return the same 65-byte point and status.  The partials never visit the host;
 *     the host-pointer form synchronises once per call, the _dev form not at all.
 *       s256_comm_unique_id : rank 0 calls it and hands the 128 bytes to the other ranks (any channel);
 *       s256_comm_init      : every rank, collectively (ncclCommInitRank on the context's device);
 *       s256_comm_free      : optional, s256_free releases the communicator too.
 *     NCCL is loaded with dlopen on first use (the copy already in the process if there is one); a context without a
 *     communicator, or a communicator of one rank, computes the plain MSM.  S256_ERR_NCCL: library missing or a
 *     collective failed (s256_last_cuda_error has the text). */
int s256_msm_plan(size_t n, int *window_bits, int *windows); /* the Pippenger plan for n points (measurement aid) */
int s256_comm_unique_id(uint8_t id128[128]);
int s256_comm_init(s256_ctx *ctx, const uint8_t id128[128], int rank, int nranks);
int s256_comm_free(s256_ctx *ctx);
int s256_msm_sharded(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n_local, int vartime, uint8_t *out65,
                     uint8_t *status);
int s256_msm_sharded_dev(s256_ctx *ctx, const uint8_t *k32, const uint8_t *pt65, size_t n_local, int vartime,
                         uint8_t *out65, uint8_t *status, void *stream);

/* --- page-locked host buffers.  The host-pointer entry points accept any memory, but copies from and
 *     to pageable memory are staged by the driver at a fraction of the PCIe rate; batch buffers
 *     allocated here (the cgo shim can wrap them as Go slices) move at full speed and let the
 *     sub-chunk pipeline overlap them with the kernels.  NULL on failure. */
void *s256_host_alloc(size_t bytes);
void s256_host_free(void *p);

/* --- measurement / debug hooks (not part of the reference surface) -------- */
/* Regenerates multiples d * 2^(wbits*w) * G, d in [1, 2^wbits), w in [0, nwin)
 * as X||Y (64 B each), window-major: with wbits = 8, nwin = 32 this is byte for
 * byte internal/gentable/point_mul_table.bin. */
int s256_debug_gen_table(s256_ctx *ctx, int wbits, int nwin, uint8_t *out);
/* out32[i] = a32[i] (op) b32[i] in F_p (op 0 mul, 1 add, 2 sub, 3 inv(a), 4 sqrt(a) or zeros, 5 a*21,
 * 6 a^2; 8 + op for the variable-time flavour of mul / add / sub / a*21 / a^2 used by the vartime paths)
 * or Z_n (op 16 mul, 17 add, 18 inv(a)); inputs are reduced like SetBytes. */
int s256_debug_field_op(s256_ctx *ctx, int op, const uint8_t *a32, const uint8_t *b32, size_t n, uint8_t *out32);
/* Integer-multiply peak: runs independent IMAD.WIDE.U32 chains on every SM and
 * returns MAC32 per second (the roofline denominator, SURVEY.md section 8d). */
int s256_microbench_imad(s256_ctx *ctx, int iters, double *mac32_per_s, double *ms);
/* Other probes of the integer pipes (variant ids in csrc/microbench.cuh): carry-chained
 * IMAD.WIDE.X, 32-bit IMAD, IMAD.HI, IADD3.X chains, mixed issue. */
int s256_microbench_variant(s256_ctx *ctx, int variant, int iters, double *ops_per_s, double *ms);
/* Field-multiplication probe: dependent F_p products per second over all SMs.  form 0 = the ladders'
 * out-of-line 8x32-limb IMAD.WIDE multiplier, 1 = the same inlined, 2 = the 5x52-limb FP64-pipe
 * experiment (csrc/fe52.cuh; not used by any entry point). */
int s256_microbench_fe_mul(s256_ctx *ctx, int form, int iters, double *muls_per_s, double *ms);
/* CUDA-event timing of the dominant kernel (the u1*G + u2*P ladder) on the stream
 * it is launched on: enable, run steps, read the summed device time. */
int s256_profile_enable(s256_ctx *ctx, int enable);
int s256_profile_read(s256_ctx *ctx, double *dsm_ms_total, uint64_t *dsm_launches);
/* Number of kernel launches issued through this context so far. */
uint64_t s256_launch_count(const s256_ctx *ctx);
/* MAC32 (32x32->64 multiply-accumulates) executed per item by each path,
 * derived from the modmul counts in DESIGN.md; key is an entry point name. */
double s256_mac32_per_item(const char *entry_point);
/* Measurement aids for the roofline (bench.py): the ladder additions the last verification-type call really executed
 * for the first n items of its last chunk (zero digits are skipped), and the executed MAC32 of one k_dsm item given
 * those counts per item. */
int s256_debug_ladder_add_count(s256_ctx *ctx, size_t n, uint64_t *adds_first_half, uint64_t *adds_lambda_half);
double s256_mac32_k_dsm(double adds_per_item, double beta_muls_per_item);
/* The equation s256_schnorr_batch_verify checks for the same host rows, as its kernels build it (for tests): the
 * 32-byte seed; per row the two MSM scalars a_i and a_i e_i mod n (k64: 2 x 32 B big-endian) and the two points -R_i
 * and -P_i (pts128: 2 x X||Y, 32 B big-endian each; G with scalar 0 for a rejected row); sum32 = sum a_i s_i mod n
 * big-endian; *rejected = 1 if some row was rejected.  Chunks as in the verification.  n >= 1. */
int s256_debug_schnorr_batch_rows(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, size_t msg_len,
                                  const uint8_t *sig64, size_t n, uint8_t *seed32, uint8_t *k64, uint8_t *pts128,
                                  uint8_t *sum32, uint8_t *rejected);
/* The same over messages of different lengths, laid out as for s256_schnorr_batch_verify_varlen. */
int s256_debug_schnorr_batch_rows_varlen(s256_ctx *ctx, const uint8_t *pkx32, const uint8_t *msg, const size_t *offsets,
                                         const uint8_t *sig64, size_t n, uint8_t *seed32, uint8_t *k64, uint8_t *pts128,
                                         uint8_t *sum32, uint8_t *rejected);
/* The same for s256_ecdsa_recoverable_batch_verify: the seed; per row a_i and a_i u2_i mod n (k64) and the points
 * -R_i and Q_i (pts128; G with scalar 0 for a rejected row); sum32 = sum a_i u1_i mod n; *rejected.  n >= 1. */
int s256_debug_ecdsa_batch_rows(s256_ctx *ctx, const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65,
                                uint32_t flags, size_t n, uint8_t *seed32, uint8_t *k64, uint8_t *pts128, uint8_t *sum32,
                                uint8_t *rejected);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* SECP256K1_B200_H */
