// der.cuh -- strict-DER and BIP-66 signature parsing, one row per thread (k_parse_der, k_check_bip66 in api.cu).
//
// The item functions restate the host codecs of codecs.cpp (parse_one, bip66_one) byte for byte, so that the
// device parse and the exported host codecs give the same sig64 and ok bytes; tests/hostsim/der_sim.cpp runs them
// on the CPU against those codecs.
//   der_parse_one  secec.ParseASN1Signature (secec/s11n.go:83-108,203-218): cryptobyte ReadASN1 with a single-byte
//                  tag, minimal definite length (short form below 128, long form of 1-4 octets without a leading zero
//                  octet), no truncation; ReadASN1Integer (non-empty, minimal, non-negative, leading zero stripped);
//                  SEQUENCE { r INTEGER, s INTEGER } with nothing trailing at either level; r, s of at most 32 bytes,
//                  below n and non-zero.
//   der_bip66_one  bitcoin.IsValidSignatureEncodingBIP0066 (secec/bitcoin/asn1_shitcoin.go:13-115), sighash byte
//                  included.
// Row bound: a row der_parse_one accepts is at most 72 bytes.  Each INTEGER's content is at most 33 bytes (a value of
// at most 32 bytes behind at most one leading zero, which minimality allows only before a byte >= 0x80), so its
// length takes the short form (the long form of a length below 128 is not minimal) and its TLV at most 35 bytes; the
// SEQUENCE content is then at most 70 bytes, again in the short form, and nothing may follow it.  der_bip66_one
// rejects every row longer than 73 bytes.  So a row longer than DER_ROW_MAX is rejected from its length alone, in
// both modes, and no thread reads more than 73 bytes of its row.
#pragma once
#include "kernels.cuh"

namespace s256 {

constexpr size_t DER_ROW_MAX = 73;

struct der_span {
    const uint8_t *p;
    size_t n;
};

// cryptobyte String.ReadASN1 with an expected tag; advances `s`, yields the contents
S256_HD bool der_read(der_span &s, uint8_t want_tag, der_span &out) {
    if (s.n < 2) return false;
    const uint8_t tag = s.p[0], len_byte = s.p[1];
    if ((tag & 0x1f) == 0x1f) return false;  // high-tag-number form
    size_t header, length;
    if ((len_byte & 0x80) == 0) {
        header = 2;
        length = len_byte;
    } else {
        const size_t len_len = len_byte & 0x7f;
        if (len_len == 0 || len_len > 4 || s.n < 2 + len_len) return false;
        uint32_t len32 = 0;
        for (size_t i = 0; i < len_len; i++) len32 = (len32 << 8) | s.p[2 + i];
        if (len32 < 128) return false;                        // should have used the short form
        if ((len32 >> ((len_len - 1) * 8)) == 0) return false;  // leading zero octet
        header = 2 + len_len;
        length = len32;
    }
    if (s.n < header || s.n - header < length) return false;
    if (tag != want_tag) return false;
    out.p = s.p + header;
    out.n = length;
    s.p += header + length;
    s.n -= header + length;
    return true;
}

// cryptobyte ReadASN1Integer(*[]byte): minimal, non-negative; leading zero stripped
S256_HD bool der_read_uint(der_span &s, der_span &out) {
    der_span b;
    if (!der_read(s, 0x02, b)) return false;
    if (b.n == 0) return false;
    if (b.n > 1 && ((b.p[0] == 0x00 && (b.p[1] & 0x80) == 0) || (b.p[0] == 0xff && (b.p[1] & 0x80) == 0x80))) return false;
    if (b.p[0] & 0x80) return false;
    while (b.n > 1 && b.p[0] == 0) {
        b.p++;
        b.n--;
    }
    out = b;
    return true;
}

// secec/s11n.go:203-218 bytesToCanonicalScalar + the IsZero checks of :97-105.  The value is right-aligned into eight
// big-endian words (the byte index is a compile-time constant after unrolling, so w stays in registers).
S256_HD bool der_scalar(const der_span &b, uint32_t w[8]) {
    if (b.n == 0 || b.n > 32) return false;
    const size_t lead = 32 - b.n;
#pragma unroll
    for (int k = 0; k < 8; k++) w[k] = 0;
#pragma unroll
    for (int j = 0; j < 32; j++) w[j >> 2] = (w[j >> 2] << 8) | ((size_t)j >= lead ? b.p[j - lead] : 0u);
    const uint32_t N_BE[8] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFEu,
                              0xBAAEDCE6u, 0xAF48A03Bu, 0xBFD25E8Cu, 0xD0364141u};
    bool below = false, decided = false;
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        acc |= w[k];
        if (!decided && w[k] != N_BE[k]) {
            below = w[k] < N_BE[k];
            decided = true;
        }
    }
    return below && acc != 0;
}

// codecs.cpp parse_one: r||s as sixteen big-endian words when accepted (rs is undefined otherwise)
S256_HD bool der_parse_one(const uint8_t *der, size_t len, uint32_t rs[16]) {
    der_span in{der, len}, inner, r, s;
    if (!der_read(in, 0x30, inner) || in.n != 0) return false;
    if (!der_read_uint(inner, r) || !der_read_uint(inner, s) || inner.n != 0) return false;
    return der_scalar(r, rs) && der_scalar(s, rs + 8);
}

// codecs.cpp bip66_one
S256_HD bool der_bip66_one(const uint8_t *data, size_t len_sig) {
    if (len_sig < 9 || len_sig > 73) return false;
    if (data[0] != 0x30) return false;
    if ((size_t)data[1] != len_sig - 3) return false;
    const size_t len_r = data[3];
    if (5 + len_r >= len_sig) return false;
    const size_t len_s = data[5 + len_r];
    if (len_r + len_s + 7 != len_sig) return false;
    if (data[2] != 0x02) return false;
    if (len_r == 0) return false;
    if (data[4] & 0x80) return false;
    if (len_r > 1 && data[4] == 0x00 && (data[5] & 0x80) == 0) return false;
    if (data[len_r + 4] != 0x02) return false;
    if (len_s == 0) return false;
    if (data[len_r + 6] & 0x80) return false;
    if (len_s > 1 && data[len_r + 6] == 0x00 && (data[len_r + 7] & 0x80) == 0) return false;
    return true;
}

// One row of k_parse_der.  Strict DER: the row is the signature.  BIP66: the row carries the sighash byte and passes
// when der_bip66_one accepts it and der_parse_one accepts it without its last byte (bitcoin.VerifyASN1,
// secec/bitcoin/ecdsa_shitcoin.go:29-35).  A row that cannot be read (decreasing offsets) or is longer than
// DER_ROW_MAX is rejected before any of its bytes is read.  rs: r||s as big-endian words, all zero when rejected.
template <bool BIP66, class M>
S256_HD uint32_t item_parse_der(size_t i, const M &rows, uint32_t rs[16]) {
    const uint8_t *p;
    size_t len;
    bool ok = rows.row(i, p, len) && len <= DER_ROW_MAX;
    if (BIP66) {
        ok = ok && der_bip66_one(p, len);
        if (ok) len--;  // the sighash byte
    }
    ok = ok && der_parse_one(p, len, rs);
    if (!ok) {
#pragma unroll
        for (int k = 0; k < 16; k++) rs[k] = 0;
    }
    return ok ? 1u : 0u;
}

// One row of k_check_bip66: s256_is_valid_signature_encoding_bip0066 on the device
template <class M>
S256_HD uint32_t item_check_bip66(size_t i, const M &rows) {
    const uint8_t *p;
    size_t len;
    return (rows.row(i, p, len) && len <= DER_ROW_MAX && der_bip66_one(p, len)) ? 1u : 0u;
}

// Writes the 64 bytes of r||s; with 16-byte stores where the row is 16-byte aligned (the verification scratch is).
S256_HD void der_store_sig64(uint8_t *out, const uint32_t rs[16]) {
#if defined(__CUDA_ARCH__)
    if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        uint4 *q = reinterpret_cast<uint4 *>(out);
#pragma unroll
        for (int g = 0; g < 4; g++)
            q[g] = make_uint4(__byte_perm(rs[4 * g], 0, 0x0123), __byte_perm(rs[4 * g + 1], 0, 0x0123),
                              __byte_perm(rs[4 * g + 2], 0, 0x0123), __byte_perm(rs[4 * g + 3], 0, 0x0123));
        return;
    }
#endif
#pragma unroll
    for (int k = 0; k < 16; k++) {
        out[4 * k] = (uint8_t)(rs[k] >> 24);
        out[4 * k + 1] = (uint8_t)(rs[k] >> 16);
        out[4 * k + 2] = (uint8_t)(rs[k] >> 8);
        out[4 * k + 3] = (uint8_t)rs[k];
    }
}

}  // namespace s256
