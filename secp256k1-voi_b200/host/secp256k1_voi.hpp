// secp256k1_voi.hpp -- host-side mirror of the reference's Go API over the C ABI.
//
// The reference is Go and there is no Go toolchain in this image, so the host
// layer above include/secp256k1_b200.h is C++ with the SAME type / method names,
// argument meaning and error behaviour as the Go packages it mirrors:
//   secp256k1.Scalar  (scalar.go:52-261)      -> secp256k1::Scalar
//   secp256k1.Point   (point.go:42-224, point_s11n.go, point_mul_*.go) -> secp256k1::Point
//   secec.PublicKey.Verify (all three encodings) / RecoverPublicKey / PrivateKey.ECDH / PrivateKey.Sign with
//   RFC6979SHA256() / ParseASN1PublicKey / ASN1Bytes / Parse- and BuildASN1Signature (secec/*.go)
//   bitcoin.SchnorrPublicKey.Verify, SchnorrPrivateKey.Sign, VerifyASN1 (secec/bitcoin/*.go)
//   h2c.Secp256k1_XMD_SHA256_SSWU_RO / _NU (secec/h2c/h2c.go)
// plus the batch entry points the engine adds (…Batch).  Single-item methods are
// batches of one: correct, but the GPU only pays off on the batch forms.
// Misuse that panics in Go throws std::logic_error; data errors that return
// `error` in Go throw secp256k1::Error or return false exactly where Go does.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/secp256k1_b200.h"

namespace secp256k1 {

constexpr size_t ScalarSize = 32, CoordSize = 32, CompressedPointSize = 33, UncompressedPointSize = 65,
                 IdentityPointSize = 1;

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// One engine context per process/GPU (the reference builds its tables at package init).
class Engine {
  public:
    static Engine &Default() {
        static Engine e(-1, 0);
        return e;
    }
    Engine(int device, size_t max_batch) {
        int rc = s256_init(&ctx_, device, max_batch);
        if (rc != S256_SUCCESS) throw Error(std::string("s256_init: ") + s256_strerror(rc));
    }
    ~Engine() { s256_free(ctx_); }
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;
    s256_ctx *ctx() const { return ctx_; }
    void check(int rc, const char *what) const {
        if (rc != S256_SUCCESS)
            throw Error(std::string(what) + ": " + s256_strerror(rc) + " " + s256_last_cuda_error(ctx_));
    }

  private:
    s256_ctx *ctx_ = nullptr;
};

namespace detail {
static const uint8_t N_BE[32] = {0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFE,
                                 0xBA, 0xAE, 0xDC, 0xE6, 0xAF, 0x48, 0xA0, 0x3B, 0xBF, 0xD2, 0x5E, 0x8C, 0xD0, 0x36, 0x41, 0x41};
static const uint8_t P_BE[32] = {0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF,
                                 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFE, 0xFF, 0xFF, 0xFC, 0x2F};
inline int cmp_be(const uint8_t *a, const uint8_t *b) { return std::memcmp(a, b, 32); }
inline void sub_be(uint8_t *r, const uint8_t *a, const uint8_t *b) {
    int borrow = 0;
    for (int i = 31; i >= 0; i--) {
        int d = (int)a[i] - (int)b[i] - borrow;
        borrow = d < 0;
        r[i] = (uint8_t)(d + (borrow << 8));
    }
}
}  // namespace detail

// scalar.go: an integer mod n.  Decode / encode / range predicates / negation / selection are byte
// operations on the host; products, sums and inverses mod n happen on the GPU.
class Scalar {
  public:
    Scalar() { b_.fill(0); }  // NewScalar(): zero
    // scalar.go:123 SetBytes: reduces once, returns didReduce
    uint64_t SetBytes(const uint8_t src[32]) {
        if (detail::cmp_be(src, detail::N_BE) >= 0) {
            detail::sub_be(b_.data(), src, detail::N_BE);
            return 1;
        }
        std::memcpy(b_.data(), src, 32);
        return 0;
    }
    // scalar.go:136 SetCanonicalBytes: error if >= n, receiver unchanged
    void SetCanonicalBytes(const uint8_t src[32]) {
        if (detail::cmp_be(src, detail::N_BE) >= 0) throw Error("secp256k1: scalar value out of range");
        std::memcpy(b_.data(), src, 32);
    }
    static Scalar NewScalarFromBytes(const uint8_t src[32]) {
        Scalar s;
        s.SetBytes(src);
        return s;
    }
    static Scalar NewScalarFromCanonicalBytes(const uint8_t src[32]) {
        Scalar s;
        s.SetCanonicalBytes(src);
        return s;
    }
    static Scalar NewScalarFromUint64(uint64_t v) {
        Scalar s;
        for (int i = 0; i < 8; i++) s.b_[31 - i] = (uint8_t)(v >> (8 * i));
        return s;
    }
    const std::array<uint8_t, 32> &Bytes() const { return b_; }  // scalar.go:148, canonical big-endian
    // scalar.go:52-121 and scalar_invert.go:11 -- receiver = result, arguments may alias the receiver.
    // The mod-n products, sums and inverses run on the device (the Z_n kernels of the verification path,
    // through s256_debug_field_op); negation and selection are byte operations on canonical values.
    Scalar &Zero() { b_.fill(0); return *this; }
    Scalar &One() { b_.fill(0); b_[31] = 1; return *this; }
    Scalar &Set(const Scalar &a) { b_ = a.b_; return *this; }
    Scalar &Add(const Scalar &a, const Scalar &b, Engine &e = Engine::Default()) { return devOp(17, a, b, e); }
    Scalar &Multiply(const Scalar &a, const Scalar &b, Engine &e = Engine::Default()) { return devOp(16, a, b, e); }
    Scalar &Square(const Scalar &a, Engine &e = Engine::Default()) { return devOp(16, a, a, e); }
    Scalar &Invert(const Scalar &a, Engine &e = Engine::Default()) { return devOp(18, a, a, e); }  // Invert(0) = 0
    Scalar &Negate(const Scalar &a) {
        if (a.IsZero()) return Zero();
        std::array<uint8_t, 32> t;
        detail::sub_be(t.data(), detail::N_BE, a.b_.data());
        b_ = t;
        return *this;
    }
    Scalar &Subtract(const Scalar &a, const Scalar &b, Engine &e = Engine::Default()) {
        Scalar nb;
        nb.Negate(b);
        return Add(a, nb, e);
    }
    template <class It>
    Scalar &Sum(It first, It last, Engine &e = Engine::Default()) {  // scalar.go:96
        Scalar acc;
        for (; first != last; ++first) acc.Add(acc, *first, e);
        return Set(acc);
    }
    template <class It>
    Scalar &Product(It first, It last, Engine &e = Engine::Default()) {  // scalar.go:106
        Scalar acc;
        acc.One();
        for (; first != last; ++first) acc.Multiply(acc, *first, e);
        return Set(acc);
    }
    Scalar &ConditionalNegate(const Scalar &a, uint64_t ctrl) {  // scalar.go:162
        Scalar n;
        n.Negate(a);
        return ConditionalSelect(a, n, ctrl);
    }
    Scalar &ConditionalSelect(const Scalar &a, const Scalar &b, uint64_t ctrl) {  // scalar.go:170: a iff ctrl == 0
        const uint8_t m = (uint8_t)(0 - (uint8_t)(ctrl != 0));
        for (int i = 0; i < 32; i++) b_[i] = (uint8_t)((a.b_[i] & ~m) | (b.b_[i] & m));
        return *this;
    }
    uint64_t IsZero() const {
        uint8_t acc = 0;
        for (uint8_t x : b_) acc |= x;
        return acc == 0;
    }
    uint64_t Equal(const Scalar &o) const { return b_ == o.b_; }
    // scalar.go:190
    uint64_t IsGreaterThanHalfN() const {
        static const uint8_t HALF[32] = {0x7F, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF, 0xFF,
                                         0x5D, 0x57, 0x6E, 0x73, 0x57, 0xA4, 0x50, 0x1D, 0xDF, 0xE9, 0x2F, 0x46, 0x68, 0x1B, 0x20, 0xA0};
        return detail::cmp_be(b_.data(), HALF) > 0;
    }

  private:
    Scalar &devOp(int op, const Scalar &a, const Scalar &b, Engine &e) {
        std::array<uint8_t, 32> out;
        e.check(s256_debug_field_op(e.ctx(), op, a.b_.data(), b.b_.data(), 1, out.data()), "Scalar arithmetic");
        b_ = out;
        return *this;
    }
    std::array<uint8_t, 32> b_;
};

// point.go: a curve point or the point at infinity.  Only the affine value is
// observable in the reference (point_test.go:359-390), so the mirror stores it.
class Point {
  public:
    Point() = default;  // the zero value is NOT valid (point.go:24-26)
    static Point NewIdentityPoint() {
        Point p;
        p.valid_ = true;
        p.identity_ = true;
        return p;
    }
    static Point NewGeneratorPoint() {
        static const uint8_t G[65] = {
            0x04, 0x79, 0xBE, 0x66, 0x7E, 0xF9, 0xDC, 0xBB, 0xAC, 0x55, 0xA0, 0x62, 0x95, 0xCE, 0x87, 0x0B, 0x07,
            0x02, 0x9B, 0xFC, 0xDB, 0x2D, 0xCE, 0x28, 0xD9, 0x59, 0xF2, 0x81, 0x5B, 0x16, 0xF8, 0x17, 0x98, 0x48,
            0x3A, 0xDA, 0x77, 0x26, 0xA3, 0xC4, 0x65, 0x5D, 0xA4, 0xFB, 0xFC, 0x0E, 0x11, 0x08, 0xA8, 0xFD, 0x17,
            0xB4, 0x48, 0xA6, 0x85, 0x54, 0x19, 0x9C, 0x47, 0xD0, 0x8F, 0xFB, 0x10, 0xD4, 0xB8};
        Point p;
        p.valid_ = true;
        std::memcpy(p.enc_.data(), G, 65);
        return p;
    }
    // point_s11n.go:218-241 SetBytes / NewPointFromBytes: 1, 33 or 65 bytes
    static Point NewPointFromBytes(const uint8_t *src, size_t len, Engine &e = Engine::Default()) {
        Point p;
        if (len == IdentityPointSize) {
            if (src[0] != 0x00) throw Error("secp256k1: invalid encoded point prefix");
            return NewIdentityPoint();
        }
        uint8_t st = 0;
        if (len == CompressedPointSize) {
            e.check(s256_point_decompress(e.ctx(), src, 1, p.enc_.data(), &st), "point_decompress");
        } else if (len == UncompressedPointSize) {
            // validate by a 1*P constant-time multiplication-free path: decode happens inside every
            // entry point; use u1 = 0, u2 = 1 so the result is P itself
            uint8_t zero[32] = {0}, one[32] = {0};
            one[31] = 1;
            e.check(s256_double_scalar_mult_basepoint_vartime(e.ctx(), zero, one, src, 1, p.enc_.data(), &st), "decode");
        } else {
            throw Error("secp256k1: invalid encoded point");
        }
        if (st != S256_ST_OK) throw Error("secp256k1: point not on curve / invalid encoding");
        p.valid_ = true;
        return p;
    }
    uint64_t IsIdentity() const {
        assertValid();
        return identity_;
    }
    uint64_t IsYOdd() const {  // point.go:155
        assertValid();
        return identity_ ? 0 : (enc_[64] & 1);
    }
    uint64_t Equal(const Point &o) const {
        assertValid();
        o.assertValid();
        return identity_ == o.identity_ && (identity_ || enc_ == o.enc_);
    }
    // point_s11n.go:66-134
    std::vector<uint8_t> UncompressedBytes() const {
        assertValid();
        if (identity_) return {0x00};
        return std::vector<uint8_t>(enc_.begin(), enc_.end());
    }
    std::vector<uint8_t> CompressedBytes() const {
        assertValid();
        if (identity_) return {0x00};
        std::vector<uint8_t> o(33);
        o[0] = (uint8_t)(2 + (enc_[64] & 1));
        std::memcpy(o.data() + 1, enc_.data() + 1, 32);
        return o;
    }
    std::vector<uint8_t> XBytes() const {
        assertValid();
        if (identity_) throw Error("secp256k1: point not on curve");  // point_s11n.go:123-125
        return std::vector<uint8_t>(enc_.begin() + 1, enc_.begin() + 33);
    }

    // point_mul_table.go:168 -- v = s * G (constant time)
    Point &ScalarBaseMult(const Scalar &s, Engine &e = Engine::Default()) {
        uint8_t st = 0;
        e.check(s256_scalar_base_mult(e.ctx(), s.Bytes().data(), 1, enc_.data(), &st), "ScalarBaseMult");
        return set(st);
    }
    // point_mul_glv.go:257 -- v = s * p (constant time)
    Point &ScalarMult(const Scalar &s, const Point &p, Engine &e = Engine::Default()) {
        p.assertValid();
        if (p.identity_) return *this = NewIdentityPoint();
        uint8_t st = 0;
        std::array<uint8_t, 65> in = p.enc_;
        e.check(s256_scalar_mult(e.ctx(), s.Bytes().data(), in.data(), 1, enc_.data(), &st), "ScalarMult");
        return set(st);
    }
    // point_mul_glv.go:307 -- v = u1 * G + u2 * p (variable time)
    Point &DoubleScalarMultBasepointVartime(const Scalar &u1, const Scalar &u2, const Point &p,
                                            Engine &e = Engine::Default()) {
        p.assertValid();
        if (p.identity_) return ScalarBaseMult(u1, e);
        uint8_t st = 0;
        std::array<uint8_t, 65> in = p.enc_;
        e.check(s256_double_scalar_mult_basepoint_vartime(e.ctx(), u1.Bytes().data(), u2.Bytes().data(), in.data(), 1,
                                                          enc_.data(), &st),
                "DoubleScalarMultBasepointVartime");
        return set(st);
    }
    // point_mul_multi.go:25,73 -- v = sum scalars[i] * points[i]; length mismatch panics
    Point &MultiScalarMult(const std::vector<Scalar> &scalars, const std::vector<Point> &points, bool vartime = false,
                           Engine &e = Engine::Default()) {
        if (scalars.size() != points.size()) throw std::logic_error("secp256k1: len(scalars) != len(points)");
        std::vector<uint8_t> k, p;
        for (size_t i = 0; i < scalars.size(); i++) {
            points[i].assertValid();
            if (points[i].identity_) continue;  // contributes nothing
            k.insert(k.end(), scalars[i].Bytes().begin(), scalars[i].Bytes().end());
            p.insert(p.end(), points[i].enc_.begin(), points[i].enc_.end());
        }
        uint8_t st = 0;
        e.check(s256_msm(e.ctx(), k.data(), p.data(), k.size() / 32, vartime ? 1 : 0, enc_.data(), &st), "MultiScalarMult");
        return set(st);
    }
    Point &MultiScalarMultVartime(const std::vector<Scalar> &s, const std::vector<Point> &p, Engine &e = Engine::Default()) {
        return MultiScalarMult(s, p, true, e);
    }
    // point.go:62 -- v = p + q, through the engine's projective combine
    Point &Add(const Point &p, const Point &q, Engine &e = Engine::Default()) {
        p.assertValid();
        q.assertValid();
        uint8_t parts[2 * 96], st = 0;
        p.toPartial(parts);
        q.toPartial(parts + 96);
        e.check(s256_msm_combine(e.ctx(), parts, 2, enc_.data(), &st), "Add");
        return set(st);
    }
    // point.go:42-59,73-131,164-224
    Point &Identity() { return Set(NewIdentityPoint()); }
    Point &Generator() { return Set(NewGeneratorPoint()); }
    Point &Set(const Point &p) {
        p.assertValid();
        enc_ = p.enc_;
        valid_ = true;
        identity_ = p.identity_;
        return *this;
    }
    static Point NewPointFrom(const Point &p) {
        Point r;
        r.Set(p);
        return r;
    }
    // point.go:203 -- (x, y) big-endian; rejects non-canonical coordinates and points off the curve
    static Point NewPointFromCoords(const uint8_t x[32], const uint8_t y[32], Engine &e = Engine::Default()) {
        uint8_t buf[65];
        buf[0] = 0x04;
        std::memcpy(buf + 1, x, 32);
        std::memcpy(buf + 33, y, 32);
        return NewPointFromBytes(buf, 65, e);
    }
    Point &Double(const Point &p, Engine &e = Engine::Default()) { return Add(p, p, e); }  // the combine's addition is complete
    Point &Negate(const Point &p) {  // (x, y) -> (x, p - y); y is never 0 on this curve (no points of order 2)
        Set(p);
        if (!identity_) detail::sub_be(enc_.data() + 33, detail::P_BE, enc_.data() + 33);
        return *this;
    }
    Point &Subtract(const Point &p, const Point &q, Engine &e = Engine::Default()) {
        Point nq;
        nq.Negate(q);
        return Add(p, nq, e);
    }
    Point &ConditionalNegate(const Point &p, uint64_t ctrl) {
        Point n;
        n.Negate(p);
        return ConditionalSelect(p, n, ctrl);
    }
    Point &ConditionalSelect(const Point &a, const Point &b, uint64_t ctrl) {  // point.go:116: a iff ctrl == 0
        a.assertValid();
        b.assertValid();
        return Set(ctrl != 0 ? b : a);
    }
    const std::array<uint8_t, 65> &raw() const { return enc_; }

  private:
    void assertValid() const {
        if (!valid_) throw std::logic_error("secp256k1: use of uninitialized Point");  // point.go:227-233
    }
    Point &set(uint8_t st) {
        if (st == S256_ST_INVALID) throw Error("secp256k1: invalid input");
        valid_ = true;
        identity_ = st == S256_ST_IDENTITY;
        return *this;
    }
    void toPartial(uint8_t out[96]) const {
        std::memset(out, 0, 96);
        if (identity_) {
            out[63] = 1;  // (0 : 1 : 0)
        } else {
            std::memcpy(out, enc_.data() + 1, 64);
            out[95] = 1;
        }
    }
    std::array<uint8_t, 65> enc_{};
    bool valid_ = false, identity_ = false;
};

// ---- batch entry points the engine adds next to the Go API --------------------------------------
inline void ScalarBaseMultBatch(const uint8_t *k32, size_t n, uint8_t *out65, uint8_t *status, Engine &e = Engine::Default()) {
    e.check(s256_scalar_base_mult(e.ctx(), k32, n, out65, status), "ScalarBaseMultBatch");
}
inline void ScalarMultBatch(const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *out65, uint8_t *status,
                            Engine &e = Engine::Default()) {
    e.check(s256_scalar_mult(e.ctx(), k32, pt65, n, out65, status), "ScalarMultBatch");
}
inline void DoubleScalarMultBasepointVartimeBatch(const uint8_t *u1, const uint8_t *u2, const uint8_t *pt65, size_t n,
                                                  uint8_t *out65, uint8_t *status, Engine &e = Engine::Default()) {
    e.check(s256_double_scalar_mult_basepoint_vartime(e.ctx(), u1, u2, pt65, n, out65, status), "DoubleScalarMultBatch");
}

namespace secec {

// secec/ecdsa.go:38-50
enum SignatureEncoding { EncodingASN1 = 0, EncodingCompact = 1, EncodingCompactRecoverable = 2 };
// secec/ecdsa.go:52-77.  Go's `Hash crypto.Hash` only validates the digest length; here it is that length
// in bytes (0: SHA-256, 32).
struct ECDSAOptions {
    size_t HashSize = 0;
    SignatureEncoding Encoding = EncodingASN1;
    bool SelfVerify = false;
    bool RejectMalleable = false;
};
constexpr size_t CompactSignatureSize = 64, CompactRecoverableSignatureSize = 65;

// secec/s11n.go:83 ParseASN1Signature: strict DER SEQUENCE { r, s }, both in [1, n) -> r || s
inline std::array<uint8_t, 64> ParseASN1Signature(const uint8_t *data, size_t len) {
    std::array<uint8_t, 64> sig{};
    size_t offs[2] = {0, len};
    uint8_t ok = 0, dummy = 0;
    if (s256_parse_asn1_signatures(len ? data : &dummy, offs, 1, sig.data(), &ok) != S256_SUCCESS || !ok)
        throw Error("secp256k1/secec: invalid ASN.1 signature");
    return sig;
}
// secec/s11n.go:112 BuildASN1Signature
inline std::vector<uint8_t> BuildASN1Signature(const uint8_t sig64[64]) {
    uint8_t out[72], n = 0;
    if (s256_build_asn1_signatures(sig64, 1, out, &n) != S256_SUCCESS) throw Error("BuildASN1Signature");
    return std::vector<uint8_t>(out, out + n);
}

// secec/s11n.go:129-176 -- compact [R | S] and recoverable [R | S | V] signatures: r, s in [1, n)
struct RawSignature {
    Scalar r, s;
    uint8_t v = 0;
};
inline RawSignature ParseCompactSignature(const uint8_t *data, size_t len) {
    if (len != CompactSignatureSize) throw Error("secp256k1/secec: invalid compact signature");
    RawSignature sig;
    try {
        sig.r.SetCanonicalBytes(data);
        sig.s.SetCanonicalBytes(data + 32);
    } catch (const Error &) {
        throw Error("secp256k1/secec: invalid scalar");
    }
    if (sig.r.IsZero() || sig.s.IsZero()) throw Error("secp256k1/secec: invalid scalar");
    return sig;
}
inline std::vector<uint8_t> BuildCompactSignature(const Scalar &r, const Scalar &s) {
    std::vector<uint8_t> out(r.Bytes().begin(), r.Bytes().end());
    out.insert(out.end(), s.Bytes().begin(), s.Bytes().end());
    return out;
}
inline RawSignature ParseCompactRecoverableSignature(const uint8_t *data, size_t len) {
    if (len != CompactRecoverableSignatureSize) throw Error("secp256k1/secec: invalid compact signature");
    RawSignature sig = ParseCompactSignature(data, CompactSignatureSize);
    sig.v = data[64];  // not range-checked here, as in the reference: RecoverPublicKey refuses v > 3
    return sig;
}
inline std::vector<uint8_t> BuildCompactRecoverableSignature(const Scalar &r, const Scalar &s, uint8_t v) {
    std::vector<uint8_t> out = BuildCompactSignature(r, s);
    out.push_back(v);
    return out;
}

class PublicKey {
  public:
    // secec/secec.go:188 NewPublicKey: any SEC 1 encoding, identity rejected
    static PublicKey NewPublicKey(const uint8_t *key, size_t len, Engine &e = Engine::Default()) {
        Point p = Point::NewPointFromBytes(key, len, e);
        if (p.IsIdentity()) throw Error("secp256k1/secec: public key is the point at infinity");
        PublicKey k;
        k.point_ = p;
        return k;
    }
    // secec/s11n.go:45 ParseASN1PublicKey: SubjectPublicKeyInfo, named curve only
    static PublicKey ParseASN1PublicKey(const uint8_t *data, size_t len, Engine &e = Engine::Default()) {
        size_t offs[2] = {0, len};
        uint8_t pt[65], plen = 0, st = 0, dummy = 0;
        if (s256_parse_asn1_public_keys(len ? data : &dummy, offs, 1, pt, &plen, &st) != S256_SUCCESS)
            throw Error("ParseASN1PublicKey");
        if (st == S256_ST_BAD_ALGORITHM) throw Error("secp256k1/secec: algorithm is not ecPublicKey");
        if (st == S256_ST_BAD_CURVE) throw Error("secp256k1/secec: named curve is not secp256k1");
        if (st != S256_ST_OK) throw Error("secp256k1/secec: invalid ASN.1 Subject Public Key Info");
        return NewPublicKey(pt, plen, e);
    }
    const Point &point() const { return point_; }
    std::vector<uint8_t> Bytes() const { return point_.UncompressedBytes(); }
    // secec/secec.go:109 ASN1Bytes
    std::vector<uint8_t> ASN1Bytes() const {
        std::vector<uint8_t> out(88);
        if (s256_build_asn1_public_keys(point_.raw().data(), 1, out.data()) != S256_SUCCESS) throw Error("ASN1Bytes");
        return out;
    }
    // secec/ecdsa.go:171 Verify.  opts == nullptr: EncodingASN1, any s in [1, n), digest of any length >= 32
    // (the leftmost 32 bytes are used, ecdsa.go:477).
    bool Verify(const uint8_t *digest, size_t digest_len, const uint8_t *sig, size_t sig_len, const ECDSAOptions *opts = nullptr,
                Engine &e = Engine::Default()) const {
        SignatureEncoding enc = EncodingASN1;
        uint32_t flags = 0;
        if (opts) {
            enc = opts->Encoding;
            if (opts->RejectMalleable) flags = S256_FLAG_REJECT_MALLEABLE;
            if (digest_len != (opts->HashSize ? opts->HashSize : 32)) return false;
        }
        if (digest_len < 32) return false;
        uint8_t ok = 0, dummy = 0;
        switch (enc) {
        case EncodingASN1: {
            size_t offs[2] = {0, sig_len};
            e.check(s256_ecdsa_verify_asn1(e.ctx(), point_.raw().data(), digest, sig_len ? sig : &dummy, offs, flags, 1, &ok),
                    "Verify");
            return ok == 1;
        }
        case EncodingCompact:
            if (sig_len != CompactSignatureSize) return false;
            e.check(s256_ecdsa_verify(e.ctx(), point_.raw().data(), digest, sig, flags, 1, &ok), "Verify");
            return ok == 1;
        case EncodingCompactRecoverable: {
            // ecdsa.go:221-227: recover with (r, s, v) and compare keys
            if (sig_len != CompactRecoverableSignatureSize) return false;
            if (flags && Scalar::NewScalarFromBytes(sig + 32).IsGreaterThanHalfN()) return false;
            uint8_t pk[65], st = 0;
            e.check(s256_ecdsa_recover(e.ctx(), digest, sig, 1, pk, &st), "Verify");
            return st == S256_ST_OK && std::memcmp(pk, point_.raw().data(), 65) == 0;
        }
        }
        return false;  // errInvalidEncoding
    }
    bool Equal(const PublicKey &o) const { return point_.Equal(o.point_); }
    // secec/secec.go:98,114,202
    std::vector<uint8_t> CompressedBytes() const { return point_.CompressedBytes(); }
    Point PointCopy() const { return Point::NewPointFrom(point_); }  // Go: Point() returns a copy
    uint64_t IsYOdd() const { return point_.IsYOdd(); }
    static PublicKey NewPublicKeyFromPoint(const Point &p) {
        if (p.IsIdentity()) throw Error("secp256k1/secec: public key is the point at infinity");
        PublicKey k;
        k.point_ = Point::NewPointFrom(p);
        return k;
    }
    // secec/ecdsa.go:234 VerifyRaw: (r, s) as scalars; zero r or s fails inside the kernel as in verify()
    bool VerifyRaw(const uint8_t *digest, size_t digest_len, const Scalar &r, const Scalar &s, Engine &e = Engine::Default()) const {
        if (digest_len < 32) return false;
        uint8_t sig[64], ok = 0;
        std::memcpy(sig, r.Bytes().data(), 32);
        std::memcpy(sig + 32, s.Bytes().data(), 32);
        e.check(s256_ecdsa_verify(e.ctx(), point_.raw().data(), digest, sig, 0, 1, &ok), "VerifyRaw");
        return ok == 1;
    }

  private:
    Point point_;
};

// secec/secec.go:149 NewPrivateKey + Sign with RFC6979SHA256() as the entropy source (secec/ecdsa.go:92,
// ecdsa_k_rfc6979.go:38).  The engine implements the deterministic path only; randomised nonces with the
// reference's TupleHash hardening stay on the host library.
class PrivateKey {
  public:
    static PrivateKey NewPrivateKey(const uint8_t *key, size_t len, Engine &e = Engine::Default()) {
        if (len != ScalarSize) throw Error("secp256k1/secec: invalid private key");
        if (std::memcmp(key, detail::N_BE, 32) >= 0) throw Error("secp256k1/secec: invalid private key");
        uint8_t acc = 0;
        for (size_t i = 0; i < 32; i++) acc |= key[i];
        if (!acc) throw Error("secp256k1/secec: invalid private key");
        PrivateKey k;
        std::memcpy(k.d_.data(), key, 32);
        uint8_t pk[65], st = 0;
        e.check(s256_scalar_base_mult(e.ctx(), key, 1, pk, &st), "NewPrivateKey");
        k.pub_ = PublicKey::NewPublicKey(pk, 65, e);
        return k;
    }
    const std::array<uint8_t, 32> &Bytes() const { return d_; }
    const PublicKey &PublicKeyRef() const { return pub_; }
    // secec/secec.go:45,53,61,75,164
    // (Go: Scalar() and PublicKey(); a C++ member cannot share its name with the type it returns)
    secp256k1::Scalar ScalarCopy() const { return secp256k1::Scalar::NewScalarFromCanonicalBytes(d_.data()); }
    bool Equal(const PrivateKey &o) const {
        uint8_t acc = 0;
        for (size_t i = 0; i < 32; i++) acc |= (uint8_t)(d_[i] ^ o.d_[i]);
        return acc == 0;
    }
    static PrivateKey NewPrivateKeyFromScalar(const secp256k1::Scalar &s, Engine &e = Engine::Default()) {
        return NewPrivateKey(s.Bytes().data(), ScalarSize, e);  // zero is refused there
    }
    std::array<uint8_t, 32> ECDH(const PublicKey &remote, Engine &e = Engine::Default()) const {
        std::array<uint8_t, 32> x;
        uint8_t st = 0;
        e.check(s256_ecdh(e.ctx(), d_.data(), remote.point().raw().data(), 1, x.data(), &st), "ECDH");
        if (st != S256_ST_OK) throw Error("secp256k1/secec: ECDH failed");
        return x;
    }
    // secec/ecdsa.go:161 SignRaw with RFC6979SHA256(): (r, s, recovery id)
    RawSignature SignRaw(const uint8_t *digest, size_t digest_len, Engine &e = Engine::Default()) const {
        ECDSAOptions o;
        o.Encoding = EncodingCompactRecoverable;
        o.HashSize = digest_len;
        std::vector<uint8_t> sig = Sign(digest, digest_len, &o, e);
        return ParseCompactRecoverableSignature(sig.data(), sig.size());
    }
    // Sign(RFC6979SHA256(), digest, opts): opts == nullptr -> EncodingASN1, digest of any length >= 32
    std::vector<uint8_t> Sign(const uint8_t *digest, size_t digest_len, const ECDSAOptions *opts = nullptr,
                              Engine &e = Engine::Default()) const {
        SignatureEncoding enc = opts ? opts->Encoding : EncodingASN1;
        if (opts && digest_len != (opts->HashSize ? opts->HashSize : 32)) throw Error("secp256k1/secec: invalid digest");
        if (digest_len < 32) throw Error("secp256k1/secec: invalid digest");
        uint8_t sig[65], st = 0;
        e.check(s256_ecdsa_sign_rfc6979(e.ctx(), d_.data(), digest, 1, sig, sig + 64, &st), "Sign");
        if (st != S256_ST_OK) throw Error("secp256k1/secec: signing failed");
        if (opts && opts->SelfVerify) {
            ECDSAOptions v;
            v.Encoding = EncodingCompact;
            v.HashSize = digest_len;
            if (!pub_.Verify(digest, digest_len, sig, 64, &v, e) || (sig[64] & 3) != sig[64])
                throw Error("secp256k1/secec: failed to verify freshly generated signature");
        }
        switch (enc) {
        case EncodingASN1: return BuildASN1Signature(sig);
        case EncodingCompact: return std::vector<uint8_t>(sig, sig + 64);
        case EncodingCompactRecoverable: return std::vector<uint8_t>(sig, sig + 65);
        }
        throw Error("secp256k1/secec: invalid signature encoding");
    }

  private:
    std::array<uint8_t, 32> d_{};
    PublicKey pub_;
};
// batch forms of the above
inline void SignRFC6979Batch(const uint8_t *priv32, const uint8_t *digest32, size_t n, uint8_t *sig64, uint8_t *recid,
                             uint8_t *status, Engine &e = Engine::Default()) {
    e.check(s256_ecdsa_sign_rfc6979(e.ctx(), priv32, digest32, n, sig64, recid, status), "SignRFC6979Batch");
}
inline void VerifyASN1Batch(const uint8_t *pk65, const uint8_t *digest32, const uint8_t *der, const size_t *offsets, size_t n,
                            bool reject_malleable, uint8_t *ok, Engine &e = Engine::Default()) {
    e.check(s256_ecdsa_verify_asn1(e.ctx(), pk65, digest32, der, offsets, reject_malleable ? S256_FLAG_REJECT_MALLEABLE : 0u, n, ok),
            "VerifyASN1Batch");
}
inline void ParseASN1PublicKeyBatch(const uint8_t *der, const size_t *offsets, size_t n, uint8_t *pk65, uint8_t *status,
                                    Engine &e = Engine::Default()) {
    e.check(s256_parse_asn1_public_keys_checked(e.ctx(), der, offsets, n, pk65, status), "ParseASN1PublicKeyBatch");
}

// secec/ecdsa.go:244 RecoverPublicKey on r || s || v
inline PublicKey RecoverPublicKey(const uint8_t digest32[32], const uint8_t sig65[65], Engine &e);
// secec/ecdsa.go:244 RecoverPublicKey(digest, r, s, recoveryID)
inline PublicKey RecoverPublicKey(const uint8_t digest32[32], const Scalar &r, const Scalar &s, uint8_t recoveryID,
                                  Engine &e = Engine::Default()) {
    std::vector<uint8_t> sig = BuildCompactRecoverableSignature(r, s, recoveryID);
    return RecoverPublicKey(digest32, sig.data(), e);
}
inline PublicKey RecoverPublicKey(const uint8_t digest32[32], const uint8_t sig65[65], Engine &e = Engine::Default()) {
    uint8_t pk[65], st = 0;
    e.check(s256_ecdsa_recover(e.ctx(), digest32, sig65, 1, pk, &st), "RecoverPublicKey");
    if (st != S256_ST_OK) throw Error("secp256k1/secec: public key recovery failed");
    return PublicKey::NewPublicKey(pk, 65, e);
}
// secec/secec.go:53 PrivateKey.ECDH: x(k * P)
inline std::array<uint8_t, 32> ECDH(const Scalar &priv, const PublicKey &remote, Engine &e = Engine::Default()) {
    std::array<uint8_t, 32> x{};
    uint8_t st = 0;
    e.check(s256_ecdh(e.ctx(), priv.Bytes().data(), remote.point().raw().data(), 1, x.data(), &st), "ECDH");
    if (st != S256_ST_OK) throw Error("secp256k1/secec: ECDH result is the point at infinity");
    return x;
}
// batch forms
inline void VerifyBatch(const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig64, size_t n, bool reject_malleable,
                        uint8_t *ok, Engine &e = Engine::Default()) {
    e.check(s256_ecdsa_verify(e.ctx(), pk65, digest32, sig64, reject_malleable ? S256_FLAG_REJECT_MALLEABLE : 0u, n, ok), "VerifyBatch");
}
inline void RecoverPublicKeyBatch(const uint8_t *digest32, const uint8_t *sig65, size_t n, uint8_t *pk65, uint8_t *status,
                                  Engine &e = Engine::Default()) {
    e.check(s256_ecdsa_recover(e.ctx(), digest32, sig65, n, pk65, status), "RecoverPublicKeyBatch");
}
// Recoverable ECDSA batch verification: true iff every row would pass PublicKey::Verify with
// EncodingCompactRecoverable (ecdsa.go:221-227; reject_malleable as ECDSAOptions::RejectMalleable), from one randomized
// multi-scalar multiplication; a batch with an invalid row passes with probability <= 2^-127.  RecoverPublicKeyBatch
// and a comparison with the keys find the bad rows.
inline bool RecoverableBatchVerify(const uint8_t *pk65, const uint8_t *digest32, const uint8_t *sig65, size_t n,
                                   bool reject_malleable = false, Engine &e = Engine::Default()) {
    uint8_t ok = 0;
    e.check(s256_ecdsa_recoverable_batch_verify(e.ctx(), pk65, digest32, sig65,
                                                reject_malleable ? S256_FLAG_REJECT_MALLEABLE : 0u, n, &ok),
            "RecoverableBatchVerify");
    return ok == 1;
}
inline void ECDHBatch(const uint8_t *k32, const uint8_t *pt65, size_t n, uint8_t *x32, uint8_t *status, Engine &e = Engine::Default()) {
    e.check(s256_ecdh(e.ctx(), k32, pt65, n, x32, status), "ECDHBatch");
}

namespace bitcoin {
constexpr size_t SchnorrPublicKeySize = 32, SchnorrSignatureSize = 64;
// secec/bitcoin/schnorr.go:56 PreHashSchnorrMessage: SHA-256(SHA-256(name) || SHA-256(name) || msg), the tagged
// hash of BIP-340 with the caller's domain separator.  `name` must be non-empty valid UTF-8 (Go refuses a string
// that strings.ToValidUTF8 would change).  Message pre-hashing is byte hashing on the host, as in the reference
// (Go's crypto/sha256); the challenge / nonce / aux hashes of signing and verification run on the device.
namespace hashing {
inline void sha256_block(uint32_t h[8], const uint8_t *p) {
    static const uint32_t K[64] = {
        0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01, 0x243185be,
        0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa,
        0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85,
        0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3,
        0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f,
        0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};
    auto rotr = [](uint32_t x, int n) { return (x >> n) | (x << (32 - n)); };
    uint32_t w[64];
    for (int i = 0; i < 16; i++) w[i] = (uint32_t)p[4 * i] << 24 | (uint32_t)p[4 * i + 1] << 16 | (uint32_t)p[4 * i + 2] << 8 | p[4 * i + 3];
    for (int i = 16; i < 64; i++) {
        uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
        uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
        w[i] = w[i - 16] + s0 + w[i - 7] + s1;
    }
    uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
    for (int i = 0; i < 64; i++) {
        uint32_t t1 = hh + (rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25)) + ((e & f) ^ (~e & g)) + K[i] + w[i];
        uint32_t t2 = (rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22)) + ((a & b) ^ (a & c) ^ (b & c));
        hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
    }
    h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
}
inline std::array<uint8_t, 32> sha256(const std::vector<uint8_t> &m) {
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    std::vector<uint8_t> p(m);
    p.push_back(0x80);
    while (p.size() % 64 != 56) p.push_back(0);
    const uint64_t bits = (uint64_t)m.size() * 8;
    for (int i = 7; i >= 0; i--) p.push_back((uint8_t)(bits >> (8 * i)));
    for (size_t o = 0; o < p.size(); o += 64) sha256_block(h, p.data() + o);
    std::array<uint8_t, 32> out;
    for (int i = 0; i < 8; i++)
        for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(h[i] >> (24 - 8 * j));
    return out;
}
// RFC 3629 well-formedness as Go's utf8 package decides it: no overlongs, no surrogates, nothing above U+10FFFF
inline bool valid_utf8(const std::string &s) {
    size_t i = 0, n = s.size();
    while (i < n) {
        const uint8_t c = (uint8_t)s[i];
        size_t len;
        uint8_t lo = 0x80, hi = 0xBF;
        if (c < 0x80) { i++; continue; }
        else if (c >= 0xC2 && c <= 0xDF) len = 2;
        else if (c == 0xE0) { len = 3; lo = 0xA0; }
        else if (c == 0xED) { len = 3; hi = 0x9F; }
        else if (c >= 0xE1 && c <= 0xEF) len = 3;
        else if (c == 0xF0) { len = 4; lo = 0x90; }
        else if (c >= 0xF1 && c <= 0xF3) len = 4;
        else if (c == 0xF4) { len = 4; hi = 0x8F; }
        else return false;
        if (i + len > n) return false;
        const uint8_t c1 = (uint8_t)s[i + 1];
        if (c1 < lo || c1 > hi) return false;
        for (size_t k = 2; k < len; k++)
            if (((uint8_t)s[i + k] & 0xC0) != 0x80) return false;
        i += len;
    }
    return true;
}
}  // namespace hashing
inline std::array<uint8_t, 32> PreHashSchnorrMessage(const std::string &name, const uint8_t *msg, size_t msg_len) {
    if (name.empty() || !hashing::valid_utf8(name)) throw Error("secp256k1/secec/bitcoin: invalid domain separator");
    const std::array<uint8_t, 32> tag = hashing::sha256(std::vector<uint8_t>(name.begin(), name.end()));
    std::vector<uint8_t> buf(tag.begin(), tag.end());
    buf.insert(buf.end(), tag.begin(), tag.end());
    buf.insert(buf.end(), msg, msg + msg_len);
    return hashing::sha256(buf);
}

class SchnorrPublicKey {
  public:
    // secec/bitcoin/schnorr.go:257 NewSchnorrPublicKey (lift_x is validated here, as in Go)
    static SchnorrPublicKey NewSchnorrPublicKey(const uint8_t *key, size_t len, Engine &e = Engine::Default()) {
        if (len != SchnorrPublicKeySize) throw Error("secp256k1/secec/bitcoin: invalid public key");
        uint8_t cp[33];
        cp[0] = 0x02;  // lift_x: the point with even y
        std::memcpy(cp + 1, key, 32);
        SchnorrPublicKey k;
        try {
            k.point_ = Point::NewPointFromBytes(cp, 33, e);
        } catch (const Error &) {
            throw Error("secp256k1/secec/bitcoin: failed to decompress public key");
        }
        std::memcpy(k.x_.data(), key, 32);
        return k;
    }
    // secec/bitcoin/schnorr.go:282 -- any point but the identity; the y coordinate is made even
    static SchnorrPublicKey NewSchnorrPublicKeyFromPoint(const Point &point) {
        if (point.IsIdentity()) throw Error("secp256k1/secec/bitcoin: public key is the point at infinity");
        SchnorrPublicKey k;
        k.point_.ConditionalNegate(point, point.IsYOdd());
        std::vector<uint8_t> x = k.point_.XBytes();
        std::memcpy(k.x_.data(), x.data(), 32);
        return k;
    }
    // secec/bitcoin/schnorr.go:303
    static SchnorrPublicKey NewSchnorrPublicKeyFromECDSA(const PublicKey &pk) { return NewSchnorrPublicKeyFromPoint(pk.point()); }
    Point PointCopy() const { return Point::NewPointFrom(point_); }  // Go: Point() returns a copy
    bool Equal(const SchnorrPublicKey &o) const { return x_ == o.x_; }
    // secec/bitcoin/schnorr.go:221 Verify
    bool Verify(const uint8_t *msg, size_t msg_len, const uint8_t *sig, size_t sig_len, Engine &e = Engine::Default()) const {
        if (sig_len != SchnorrSignatureSize) return false;
        uint8_t ok = 0;
        e.check(s256_schnorr_verify(e.ctx(), x_.data(), msg, msg_len, sig, 1, &ok), "SchnorrPublicKey.Verify");
        return ok == 1;
    }
    const std::array<uint8_t, 32> &Bytes() const { return x_; }

  private:
    Point point_;  // never the identity, y even
    std::array<uint8_t, 32> x_{};
};
// secec/bitcoin/ecdsa_shitcoin.go:29 VerifyASN1: BIP-66 syntax, trailing sighash byte, s <= n/2
inline bool VerifyASN1(const PublicKey &k, const uint8_t *digest, size_t digest_len, const uint8_t *sig, size_t sig_len,
                       Engine &e = Engine::Default()) {
    if (digest_len != 32) return false;
    size_t offs[2] = {0, sig_len};
    uint8_t ok = 0, dummy = 0;
    e.check(s256_bitcoin_verify_asn1(e.ctx(), k.point().raw().data(), digest, sig_len ? sig : &dummy, offs, 1, &ok), "VerifyASN1");
    return ok == 1;
}
// secec/bitcoin/asn1_shitcoin.go:13
inline bool IsValidSignatureEncodingBIP0066(const uint8_t *data, size_t len) {
    size_t offs[2] = {0, len};
    uint8_t ok = 0, dummy = 0;
    return s256_is_valid_signature_encoding_bip0066(len ? data : &dummy, offs, 1, &ok) == S256_SUCCESS && ok == 1;
}
// secec/bitcoin/schnorr.go:140 NewSchnorrPrivateKey + :111 Sign with caller-supplied auxiliary randomness
class SchnorrPrivateKey {
  public:
    static SchnorrPrivateKey NewSchnorrPrivateKey(const uint8_t *key, size_t len, Engine &e = Engine::Default()) {
        try {
            return NewSchnorrPrivateKeyFromECDSA(PrivateKey::NewPrivateKey(key, len, e));
        } catch (const Error &) {
            throw Error("secp256k1/secec/bitcoin: invalid private key");
        }
    }
    // secec/bitcoin/schnorr.go:162
    static SchnorrPrivateKey NewSchnorrPrivateKeyFromECDSA(const PrivateKey &sk) {
        SchnorrPrivateKey k;
        k.d_ = sk.Bytes();
        k.pub_ = SchnorrPublicKey::NewSchnorrPublicKeyFromECDSA(sk.PublicKeyRef());
        return k;
    }
    const std::array<uint8_t, 32> &Bytes() const { return d_; }  // d', the scalar as given (schnorr.go:76)
    secp256k1::Scalar ScalarCopy() const { return secp256k1::Scalar::NewScalarFromCanonicalBytes(d_.data()); }
    const SchnorrPublicKey &PublicKeyRef() const { return pub_; }
    bool Equal(const SchnorrPrivateKey &o) const {
        uint8_t acc = 0;
        for (size_t i = 0; i < 32; i++) acc |= (uint8_t)(d_[i] ^ o.d_[i]);
        return acc == 0;
    }
    std::array<uint8_t, 64> Sign(const uint8_t aux32[32], const uint8_t *msg, size_t msg_len, Engine &e = Engine::Default()) const {
        std::array<uint8_t, 64> sig{};
        uint8_t st = 0, dummy = 0;
        e.check(s256_schnorr_sign(e.ctx(), d_.data(), msg_len ? msg : &dummy, msg_len, aux32, 1, sig.data(), &st), "SchnorrPrivateKey.Sign");
        if (st != S256_ST_OK) throw Error("secp256k1/secec/bitcoin: signing failed");
        return sig;
    }

  private:
    std::array<uint8_t, 32> d_{};
    SchnorrPublicKey pub_;
};
inline void SchnorrVerifyBatch(const uint8_t *pkx32, const uint8_t *msg, size_t msg_len, const uint8_t *sig64, size_t n,
                               uint8_t *ok, Engine &e = Engine::Default()) {
    e.check(s256_schnorr_verify(e.ctx(), pkx32, msg, msg_len, sig64, n, ok), "SchnorrVerifyBatch");
}
// BIP-340 batch verification: true iff every row would pass SchnorrPublicKey.Verify (one randomized multi-scalar
// multiplication; a batch with an invalid row passes with probability <= 2^-127).  SchnorrVerifyBatch finds the bad rows.
inline bool SchnorrBatchVerify(const uint8_t *pkx32, const uint8_t *msg, size_t msg_len, const uint8_t *sig64, size_t n,
                               Engine &e = Engine::Default()) {
    uint8_t ok = 0;
    e.check(s256_schnorr_batch_verify(e.ctx(), pkx32, msg, msg_len, sig64, n, &ok), "SchnorrBatchVerify");
    return ok == 1;
}
// The same over messages of any length, one per row (msgs.size() rows): flattened with n + 1 offsets for the
// *_varlen entry points.
namespace detail {
struct RaggedRows {
    std::vector<uint8_t> flat;
    std::vector<size_t> offsets{0};
    explicit RaggedRows(const std::vector<std::vector<uint8_t>> &msgs) {
        for (const auto &m : msgs) {
            flat.insert(flat.end(), m.begin(), m.end());
            offsets.push_back(flat.size());
        }
    }
    const uint8_t *data() const { return flat.empty() ? nullptr : flat.data(); }
};
}  // namespace detail
inline void SchnorrVerifyBatch(const uint8_t *pkx32, const std::vector<std::vector<uint8_t>> &msgs, const uint8_t *sig64,
                               uint8_t *ok, Engine &e = Engine::Default()) {
    detail::RaggedRows r(msgs);
    e.check(s256_schnorr_verify_varlen(e.ctx(), pkx32, r.data(), r.offsets.data(), sig64, msgs.size(), ok), "SchnorrVerifyBatch");
}
inline bool SchnorrBatchVerify(const uint8_t *pkx32, const std::vector<std::vector<uint8_t>> &msgs, const uint8_t *sig64,
                               Engine &e = Engine::Default()) {
    detail::RaggedRows r(msgs);
    uint8_t ok = 0;
    e.check(s256_schnorr_batch_verify_varlen(e.ctx(), pkx32, r.data(), r.offsets.data(), sig64, msgs.size(), &ok),
            "SchnorrBatchVerify");
    return ok == 1;
}
// SchnorrPrivateKey.Sign over rows: priv32 (d' as for NewSchnorrPrivateKey), one message of any length and 32 bytes
// of auxiliary randomness per row -> sig64 and a status byte per row (S256_ST_OK or S256_ST_INVALID).
inline void SchnorrSignBatch(const uint8_t *priv32, const std::vector<std::vector<uint8_t>> &msgs, const uint8_t *aux32,
                             uint8_t *sig64, uint8_t *status, Engine &e = Engine::Default()) {
    detail::RaggedRows r(msgs);
    e.check(s256_schnorr_sign_varlen(e.ctx(), priv32, r.data(), r.offsets.data(), aux32, msgs.size(), sig64, status),
            "SchnorrSignBatch");
}
}  // namespace bitcoin

namespace h2c {
// secec/h2c/h2c.go:25,49: RFC 9380 secp256k1_XMD:SHA-256_SSWU_RO_ / _NU_
inline Point Secp256k1_XMD_SHA256_SSWU(bool random_oracle, const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                                       Engine &e) {
    if (dst_len == 0) throw Error("secp256k1/secec/h2c: invalid domain separator");
    uint8_t out[65], st = 0, dummy = 0;
    e.check(s256_hash_to_curve(e.ctx(), dst, dst_len, msg_len ? msg : &dummy, msg_len, 1, random_oracle ? 1 : 0, out, &st),
            "hash_to_curve");
    if (st == S256_ST_IDENTITY) return Point::NewIdentityPoint();
    return Point::NewPointFromBytes(out, 65, e);
}
inline Point Secp256k1_XMD_SHA256_SSWU_RO(const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                                          Engine &e = Engine::Default()) {
    return Secp256k1_XMD_SHA256_SSWU(true, dst, dst_len, msg, msg_len, e);
}
inline Point Secp256k1_XMD_SHA256_SSWU_NU(const uint8_t *dst, size_t dst_len, const uint8_t *msg, size_t msg_len,
                                          Engine &e = Engine::Default()) {
    return Secp256k1_XMD_SHA256_SSWU(false, dst, dst_len, msg, msg_len, e);
}
// Secp256k1_XMD_SHA256_SSWU_RO (random_oracle) or _NU over messages of any length, one per row (msgs.size() rows)
// under one DST: out65 gets the uncompressed point of each row and status S256_ST_OK, or 65 zero bytes and
// S256_ST_IDENTITY where the per-item call returns the identity.
inline void HashToCurveBatch(const std::vector<uint8_t> &dst, const std::vector<std::vector<uint8_t>> &msgs, bool random_oracle,
                             uint8_t *out65, uint8_t *status, Engine &e = Engine::Default()) {
    if (dst.empty()) throw Error("secp256k1/secec/h2c: invalid domain separator");
    bitcoin::detail::RaggedRows r(msgs);
    e.check(s256_hash_to_curve_varlen(e.ctx(), dst.data(), dst.size(), r.data(), r.offsets.data(), msgs.size(),
                                      random_oracle ? 1 : 0, out65, status),
            "HashToCurveBatch");
}
}  // namespace h2c
}  // namespace secec
}  // namespace secp256k1
