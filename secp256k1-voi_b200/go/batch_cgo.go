// Package secp256k1b200 is the reference-side binding of the B200 engine: the
// cgo shim a maintainer of gitlab.com/yawning/secp256k1-voi adds next to the
// existing API.  It keeps the reference's types (secp256k1.Point / Scalar,
// secec.PublicKey, bitcoin.SchnorrPublicKey) and adds batch entry points that
// call the C ABI (include/secp256k1_b200.h).
//
// NOTE: there is no Go toolchain in the build image, so this file is reviewed,
// not compiled, there; the identical C ABI is exercised from C++
// (host/secp256k1_voi.hpp, tests/cpp) and Python (ctypes).
//
// cgo rules honoured: every call is synchronous, C keeps no Go pointer after
// returning, slices are passed as pointers to their first element only.
package secp256k1b200

/*
#cgo CFLAGS: -I${SRCDIR}/../../include
#cgo LDFLAGS: -L${SRCDIR}/../lib -lsecp256k1_b200 -Wl,-rpath,${SRCDIR}/../lib
#include <stdlib.h>
#include "secp256k1_b200.h"
*/
import "C"

import (
	"errors"
	"fmt"
	"runtime"
	"unsafe"

	"gitlab.com/yawning/secp256k1-voi"
	"gitlab.com/yawning/secp256k1-voi/secec"
)

// Engine owns one context on one GPU (s256_init).  Safe for concurrent use.
type Engine struct{ ctx *C.s256_ctx }

// NewEngine binds to `device` (-1: current) with chunk capacity maxBatch (0: 2^20).
func NewEngine(device int, maxBatch int) (*Engine, error) {
	e := &Engine{}
	if rc := C.s256_init(&e.ctx, C.int(device), C.size_t(maxBatch)); rc != 0 {
		return nil, fmt.Errorf("secp256k1b200: %s", C.GoString(C.s256_strerror(rc)))
	}
	runtime.SetFinalizer(e, func(e *Engine) { C.s256_free(e.ctx) })
	return e, nil
}

func (e *Engine) err(rc C.int) error {
	if rc == 0 {
		return nil
	}
	return fmt.Errorf("secp256k1b200: %s %s", C.GoString(C.s256_strerror(rc)), C.GoString(C.s256_last_cuda_error(e.ctx)))
}

func ptr(b []byte) *C.uint8_t {
	if len(b) == 0 {
		return nil
	}
	return (*C.uint8_t)(unsafe.Pointer(&b[0]))
}

// VerifyBatch is secec.PublicKey.Verify (EncodingCompact) over n rows:
// pk 65 B uncompressed, digest 32 B, sig r||s 64 B.  ok[i] mirrors the bool.
func (e *Engine) VerifyBatch(pk65, digest32, sig64 []byte, opts *secec.ECDSAOptions) ([]bool, error) {
	n := len(digest32) / 32
	if len(pk65) != 65*n || len(sig64) != 64*n {
		panic("secp256k1b200: VerifyBatch: length mismatch") // misuse panics, as in the reference
	}
	var flags C.uint32_t
	if opts != nil && opts.RejectMalleable {
		flags |= C.S256_FLAG_REJECT_MALLEABLE
	}
	ok := make([]byte, n)
	if err := e.err(C.s256_ecdsa_verify(e.ctx, ptr(pk65), ptr(digest32), ptr(sig64), flags, C.size_t(n), ptr(ok))); err != nil {
		return nil, err
	}
	out := make([]bool, n)
	for i, v := range ok {
		out[i] = v == 1
	}
	return out, nil
}

// RecoverPublicKeyBatch is secec.RecoverPublicKey over rows of digest (32 B) and r||s||v (65 B).
func (e *Engine) RecoverPublicKeyBatch(digest32, sig65 []byte) (pk65 []byte, status []byte, err error) {
	n := len(digest32) / 32
	if len(sig65) != 65*n {
		panic("secp256k1b200: RecoverPublicKeyBatch: length mismatch")
	}
	pk65, status = make([]byte, 65*n), make([]byte, n)
	err = e.err(C.s256_ecdsa_recover(e.ctx, ptr(digest32), ptr(sig65), C.size_t(n), ptr(pk65), ptr(status)))
	return
}

// ECDSARecoverableBatchVerify is recoverable ECDSA batch verification: true iff every row of uncompressed key (65 B),
// digest (32 B) and r||s||v (65 B) would pass secec.PublicKey.Verify with EncodingCompactRecoverable
// (secec/ecdsa.go:221-227), from one randomized multi-scalar multiplication; a batch with an invalid row passes with
// probability <= 2^-127.  rejectMalleable is ECDSAOptions.RejectMalleable.  RecoverPublicKeyBatch and a comparison
// with the keys find the bad rows of a rejected batch.
func (e *Engine) ECDSARecoverableBatchVerify(pk65, digest32, sig65 []byte, rejectMalleable bool) (bool, error) {
	n := len(pk65) / 65
	if len(pk65) != 65*n || len(digest32) != 32*n || len(sig65) != 65*n {
		panic("secp256k1b200: ECDSARecoverableBatchVerify: length mismatch")
	}
	var flags C.uint32_t
	if rejectMalleable {
		flags = C.S256_FLAG_REJECT_MALLEABLE
	}
	var ok C.uint8_t
	if err := e.err(C.s256_ecdsa_recoverable_batch_verify(e.ctx, ptr(pk65), ptr(digest32), ptr(sig65), flags, C.size_t(n), &ok)); err != nil {
		return false, err
	}
	return ok == 1, nil
}

// SignRFC6979Batch is PrivateKey.Sign(secec.RFC6979SHA256(), digest, EncodingCompactRecoverable) over rows of
// private scalars (32 B) and digests (32 B): returns r||s rows (low-s), recovery ids and per-row status.
func (e *Engine) SignRFC6979Batch(priv32, digest32 []byte) (sig64, recid, status []byte, err error) {
	n := len(priv32) / 32
	if len(digest32) != 32*n {
		panic("secp256k1b200: SignRFC6979Batch: length mismatch")
	}
	sig64, recid, status = make([]byte, 64*n), make([]byte, n), make([]byte, n)
	err = e.err(C.s256_ecdsa_sign_rfc6979(e.ctx, ptr(priv32), ptr(digest32), C.size_t(n), ptr(sig64), ptr(recid), ptr(status)))
	return
}

// SchnorrVerifyBatch is bitcoin.SchnorrPublicKey.Verify (incl. lift_x) over x-only keys.
func (e *Engine) SchnorrVerifyBatch(pkx32, msgs []byte, msgLen int, sig64 []byte) ([]bool, error) {
	n := len(pkx32) / 32
	if len(msgs) != msgLen*n || len(sig64) != 64*n {
		panic("secp256k1b200: SchnorrVerifyBatch: length mismatch")
	}
	ok := make([]byte, n)
	if err := e.err(C.s256_schnorr_verify(e.ctx, ptr(pkx32), ptr(msgs), C.size_t(msgLen), ptr(sig64), C.size_t(n), ptr(ok))); err != nil {
		return nil, err
	}
	out := make([]bool, n)
	for i, v := range ok {
		out[i] = v == 1
	}
	return out, nil
}

// SchnorrBatchVerify is BIP-340 batch verification: true iff every row would pass bitcoin.SchnorrPublicKey.Verify
// (one randomized multi-scalar multiplication; a batch with an invalid row passes with probability <= 2^-127).
// SchnorrVerifyBatch finds the bad rows of a rejected batch.
func (e *Engine) SchnorrBatchVerify(pkx32, msgs []byte, msgLen int, sig64 []byte) (bool, error) {
	n := len(pkx32) / 32
	if len(pkx32) != 32*n || len(msgs) != msgLen*n || len(sig64) != 64*n {
		panic("secp256k1b200: SchnorrBatchVerify: length mismatch")
	}
	var ok C.uint8_t
	if err := e.err(C.s256_schnorr_batch_verify(e.ctx, ptr(pkx32), ptr(msgs), C.size_t(msgLen), ptr(sig64), C.size_t(n), &ok)); err != nil {
		return false, err
	}
	return ok == 1, nil
}

// raggedRows flattens messages of any length into one buffer and the n + 1 offsets the *_varlen entry points take
// (row i = flat[offsets[i]:offsets[i+1]]).  Neither holds a Go pointer, so both may be passed to C.
func raggedRows(msgs [][]byte) (flat []byte, offsets []C.size_t) {
	total := 0
	for _, m := range msgs {
		total += len(m)
	}
	flat = make([]byte, 0, total)
	offsets = make([]C.size_t, len(msgs)+1)
	for i, m := range msgs {
		flat = append(flat, m...)
		offsets[i+1] = C.size_t(len(flat))
	}
	return flat, offsets
}

// SchnorrVerifyBatchVarlen is SchnorrVerifyBatch over messages of any length, one per row.
func (e *Engine) SchnorrVerifyBatchVarlen(pkx32 []byte, msgs [][]byte, sig64 []byte) ([]bool, error) {
	n := len(msgs)
	if len(pkx32) != 32*n || len(sig64) != 64*n {
		panic("secp256k1b200: SchnorrVerifyBatchVarlen: length mismatch")
	}
	flat, offs := raggedRows(msgs)
	ok := make([]byte, n)
	if err := e.err(C.s256_schnorr_verify_varlen(e.ctx, ptr(pkx32), ptr(flat), &offs[0], ptr(sig64), C.size_t(n), ptr(ok))); err != nil {
		return nil, err
	}
	out := make([]bool, n)
	for i, v := range ok {
		out[i] = v == 1
	}
	return out, nil
}

// SchnorrBatchVerifyVarlen is SchnorrBatchVerify over messages of any length, one per row.
func (e *Engine) SchnorrBatchVerifyVarlen(pkx32 []byte, msgs [][]byte, sig64 []byte) (bool, error) {
	n := len(msgs)
	if len(pkx32) != 32*n || len(sig64) != 64*n {
		panic("secp256k1b200: SchnorrBatchVerifyVarlen: length mismatch")
	}
	flat, offs := raggedRows(msgs)
	var ok C.uint8_t
	if err := e.err(C.s256_schnorr_batch_verify_varlen(e.ctx, ptr(pkx32), ptr(flat), &offs[0], ptr(sig64), C.size_t(n), &ok)); err != nil {
		return false, err
	}
	return ok == 1, nil
}

// SchnorrSignBatchVarlen is bitcoin.SchnorrPrivateKey.Sign over rows of priv32 (d'), one message of any length and
// 32 bytes of auxiliary randomness each: sig64 and a status byte per row (S256_ST_OK / S256_ST_INVALID).
func (e *Engine) SchnorrSignBatchVarlen(priv32 []byte, msgs [][]byte, aux32 []byte) (sig64, status []byte, err error) {
	n := len(msgs)
	if len(priv32) != 32*n || len(aux32) != 32*n {
		panic("secp256k1b200: SchnorrSignBatchVarlen: length mismatch")
	}
	flat, offs := raggedRows(msgs)
	sig64, status = make([]byte, 64*n), make([]byte, n)
	if err := e.err(C.s256_schnorr_sign_varlen(e.ctx, ptr(priv32), ptr(flat), &offs[0], ptr(aux32), C.size_t(n), ptr(sig64), ptr(status))); err != nil {
		return nil, nil, err
	}
	return sig64, status, nil
}

// HashToCurveBatch is h2c.Secp256k1_XMD_SHA256_SSWU_RO (randomOracle) or _NU over messages of any length, one per
// row, under one domain separation tag: 65 bytes per row (the uncompressed point) and a status byte per row
// (S256_ST_OK, or S256_ST_IDENTITY with zeroed bytes where the per-item call returns the identity).  An empty dst is
// an error (errInvalidDomainSep).
func (e *Engine) HashToCurveBatch(dst []byte, msgs [][]byte, randomOracle bool) ([]byte, []byte, error) {
	if len(dst) == 0 {
		return nil, nil, errors.New("secp256k1/secec/h2c: invalid domain separator")
	}
	n := len(msgs)
	flat, offs := raggedRows(msgs)
	ro := C.int(0)
	if randomOracle {
		ro = 1
	}
	out65, status := make([]byte, 65*n), make([]byte, n)
	if err := e.err(C.s256_hash_to_curve_varlen(e.ctx, ptr(dst), C.size_t(len(dst)), ptr(flat), &offs[0], C.size_t(n), ro,
		ptr(out65), ptr(status))); err != nil {
		return nil, nil, err
	}
	return out65, status, nil
}

// ScalarBaseMultBatch is Point.ScalarBaseMult + UncompressedBytes (constant time).
func (e *Engine) ScalarBaseMultBatch(scalars []*secp256k1.Scalar) ([]*secp256k1.Point, error) {
	n := len(scalars)
	k := make([]byte, 0, 32*n)
	for _, s := range scalars {
		k = append(k, s.Bytes()...)
	}
	out, st := make([]byte, 65*n), make([]byte, n)
	if err := e.err(C.s256_scalar_base_mult(e.ctx, ptr(k), C.size_t(n), ptr(out), ptr(st))); err != nil {
		return nil, err
	}
	return decodePoints(out, st)
}

// ScalarMultBatch is Point.ScalarMult (constant time) over (scalar, point) pairs.
func (e *Engine) ScalarMultBatch(scalars []*secp256k1.Scalar, points []*secp256k1.Point) ([]*secp256k1.Point, error) {
	if len(scalars) != len(points) {
		panic("secp256k1: len(scalars) != len(points)")
	}
	n := len(scalars)
	// The identity has a 1-byte encoding (point_s11n.go:73-76), the C ABI takes 65-byte rows: identity operands are
	// answered here (k * identity = identity, as Point.ScalarMult does) and only the other rows travel.
	k, p := make([]byte, 0, 32*n), make([]byte, 0, 65*n)
	rows := make([]int, 0, n)
	for i := range scalars {
		if points[i].IsIdentity() == 1 {
			continue
		}
		k = append(k, scalars[i].Bytes()...)
		p = appendPoint65(p, points[i])
		rows = append(rows, i)
	}
	m := len(rows)
	out, st := make([]byte, 65*m), make([]byte, m)
	if err := e.err(C.s256_scalar_mult(e.ctx, ptr(k), ptr(p), C.size_t(m), ptr(out), ptr(st))); err != nil {
		return nil, err
	}
	return scatterPoints(n, rows, out, st, nil)
}

// DoubleScalarMultBasepointVartimeBatch is Point.DoubleScalarMultBasepointVartime.
func (e *Engine) DoubleScalarMultBasepointVartimeBatch(u1, u2 []*secp256k1.Scalar, points []*secp256k1.Point) ([]*secp256k1.Point, error) {
	n := len(u1)
	if len(u2) != n || len(points) != n {
		panic("secp256k1: length mismatch")
	}
	// u1*G + u2*identity = u1*G: identity rows go through ScalarBaseMultBatch (the reference accepts them,
	// point_mul_glv.go:307-317), the others through the ladder.
	a, b, p := make([]byte, 0, 32*n), make([]byte, 0, 32*n), make([]byte, 0, 65*n)
	rows, idRows := make([]int, 0, n), make([]int, 0)
	idScalars := make([]*secp256k1.Scalar, 0)
	for i := 0; i < n; i++ {
		if points[i].IsIdentity() == 1 {
			idRows = append(idRows, i)
			idScalars = append(idScalars, u1[i])
			continue
		}
		a = append(a, u1[i].Bytes()...)
		b = append(b, u2[i].Bytes()...)
		p = appendPoint65(p, points[i])
		rows = append(rows, i)
	}
	m := len(rows)
	out, st := make([]byte, 65*m), make([]byte, m)
	if err := e.err(C.s256_double_scalar_mult_basepoint_vartime(e.ctx, ptr(a), ptr(b), ptr(p), C.size_t(m), ptr(out), ptr(st))); err != nil {
		return nil, err
	}
	var idPts []*secp256k1.Point
	if len(idRows) > 0 {
		var err error
		if idPts, err = e.ScalarBaseMultBatch(idScalars); err != nil {
			return nil, err
		}
	}
	res, err := scatterPoints(n, rows, out, st, nil)
	if err != nil {
		return nil, err
	}
	for j, i := range idRows {
		res[i] = idPts[j]
	}
	return res, nil
}

// MultiScalarMult is Point.MultiScalarMult[Vartime]: sum scalars[i] * points[i].
func (e *Engine) MultiScalarMult(scalars []*secp256k1.Scalar, points []*secp256k1.Point, vartime bool) (*secp256k1.Point, error) {
	if len(scalars) != len(points) {
		panic("secp256k1: len(scalars) != len(points)")
	}
	n := 0
	k, p := make([]byte, 0, 32*len(scalars)), make([]byte, 0, 65*len(scalars))
	for i := range scalars {
		if points[i].IsIdentity() == 1 { // contributes nothing to the sum (point_mul_multi.go accepts it)
			continue
		}
		k = append(k, scalars[i].Bytes()...)
		p = appendPoint65(p, points[i])
		n++
	}
	out := make([]byte, 65)
	var st C.uint8_t
	vt := C.int(0)
	if vartime {
		vt = 1
	}
	if err := e.err(C.s256_msm(e.ctx, ptr(k), ptr(p), C.size_t(n), vt, ptr(out), &st)); err != nil {
		return nil, err
	}
	pts, err := decodePoints(out, []byte{byte(st)})
	if err != nil {
		return nil, err
	}
	return pts[0], nil
}

// ECDHBatch is secec.PrivateKey.ECDH: x(k*P), 32 bytes per row.
func (e *Engine) ECDHBatch(k32, pt65 []byte) (x32 []byte, status []byte, err error) {
	n := len(k32) / 32
	if len(pt65) != 65*n {
		panic("secp256k1b200: ECDHBatch: length mismatch")
	}
	x32, status = make([]byte, 32*n), make([]byte, n)
	err = e.err(C.s256_ecdh(e.ctx, ptr(k32), ptr(pt65), C.size_t(n), ptr(x32), ptr(status)))
	return
}

// CompressedBytesBatch is NewPointFromBytes + (*Point).CompressedBytes over rows of 65 bytes: 33 bytes per row
// (02 | 03, X); status 0 marks a row that is not a point of the curve.
func (e *Engine) CompressedBytesBatch(pt65 []byte) (pt33 []byte, status []byte, err error) {
	if len(pt65)%65 != 0 {
		panic("secp256k1b200: CompressedBytesBatch: length is not a multiple of 65")
	}
	n := len(pt65) / 65
	pt33, status = make([]byte, 33*n), make([]byte, n)
	err = e.err(C.s256_point_compress(e.ctx, ptr(pt65), C.size_t(n), ptr(pt33), ptr(status)))
	return
}

// PinnedBytes returns a page-locked byte slice of length n for batch inputs / outputs: copies from and to
// such memory run at PCIe speed and overlap the kernels, while ordinary Go heap memory is staged by the
// driver.  The slice is C memory (not moved or freed by the Go GC); release it with FreePinned.
func PinnedBytes(n int) []byte {
	p := C.s256_host_alloc(C.size_t(n))
	if p == nil {
		return nil
	}
	return unsafe.Slice((*byte)(p), n)
}

// FreePinned releases a slice obtained from PinnedBytes.
func FreePinned(b []byte) {
	if len(b) > 0 {
		C.s256_host_free(unsafe.Pointer(&b[0]))
	}
}

// packRows concatenates variable-length rows and returns the n + 1 offsets the C ABI expects.
func packRows(rows [][]byte) ([]byte, []C.size_t) {
	offs := make([]C.size_t, len(rows)+1)
	var data []byte
	for i, r := range rows {
		data = append(data, r...)
		offs[i+1] = C.size_t(len(data))
	}
	if len(data) == 0 {
		data = []byte{0}
	}
	return data, offs
}

// ParseASN1PublicKeyBatch is secec.ParseASN1PublicKey over DER SubjectPublicKeyInfo blobs: the strict
// SPKI parse runs on the host, NewPublicKey's curve checks on the GPU.  status[i] is S256_ST_OK or the
// reason (invalid / not ecPublicKey / not secp256k1 / identity); accepted rows hold the 65-byte key.
func (e *Engine) ParseASN1PublicKeyBatch(der [][]byte) (pk65 []byte, status []byte, err error) {
	n := len(der)
	data, offs := packRows(der)
	pk65, status = make([]byte, 65*n), make([]byte, n)
	err = e.err(C.s256_parse_asn1_public_keys_checked(e.ctx, ptr(data), &offs[0], C.size_t(n), ptr(pk65), ptr(status)))
	return
}

// VerifyASN1Batch is secec.PublicKey.Verify with EncodingASN1 (the default encoding) over n rows.
func (e *Engine) VerifyASN1Batch(pk65, digest32 []byte, sigs [][]byte, opts *secec.ECDSAOptions) ([]bool, error) {
	n := len(sigs)
	if len(pk65) != 65*n || len(digest32) != 32*n {
		panic("secp256k1b200: VerifyASN1Batch: length mismatch")
	}
	var flags C.uint32_t
	if opts != nil && opts.RejectMalleable {
		flags = C.S256_FLAG_REJECT_MALLEABLE
	}
	data, offs := packRows(sigs)
	ok := make([]byte, n)
	if err := e.err(C.s256_ecdsa_verify_asn1(e.ctx, ptr(pk65), ptr(digest32), ptr(data), &offs[0], flags, C.size_t(n), ptr(ok))); err != nil {
		return nil, err
	}
	res := make([]bool, n)
	for i, b := range ok {
		res[i] = b == 1
	}
	return res, nil
}

var errInvalid = errors.New("secp256k1b200: invalid input row")

// decodePoints rebuilds reference Points from the engine's rows; the identity comes back as the
// status byte because the reference's identity encoding is the 1-byte 0x00 (point_s11n.go:75-77).
// appendPoint65 appends the 65-byte SEC 1 encoding of a non-identity point; anything else would shift every later
// row of the batch and make the C side read past the slice, so it panics instead.
func appendPoint65(dst []byte, p *secp256k1.Point) []byte {
	enc := p.UncompressedBytes()
	if len(enc) != 65 {
		panic("secp256k1b200: point without a 65-byte encoding in a batch row")
	}
	return append(dst, enc...)
}

// scatterPoints decodes the m computed rows into a result of n points; rows[j] is the position of computed row j, every
// other position is the identity (fill == nil) .
func scatterPoints(n int, rows []int, out, st []byte, fill *secp256k1.Point) ([]*secp256k1.Point, error) {
	got, err := decodePoints(out, st)
	if err != nil {
		return nil, err
	}
	res := make([]*secp256k1.Point, n)
	for i := range res {
		if fill != nil {
			res[i] = fill
		} else {
			res[i] = secp256k1.NewIdentityPoint()
		}
	}
	for j, i := range rows {
		res[i] = got[j]
	}
	return res, nil
}

func decodePoints(out, st []byte) ([]*secp256k1.Point, error) {
	pts := make([]*secp256k1.Point, len(st))
	for i, s := range st {
		switch s {
		case C.S256_ST_OK:
			p, err := secp256k1.NewPointFromBytes(out[65*i : 65*i+65])
			if err != nil {
				return nil, err
			}
			pts[i] = p
		case C.S256_ST_IDENTITY:
			pts[i] = secp256k1.NewIdentityPoint()
		default:
			return nil, errInvalid
		}
	}
	return pts, nil
}
