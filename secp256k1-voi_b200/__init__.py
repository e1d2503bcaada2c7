"""B200-native batched secp256k1 engine: Python view of the C ABI.

Everything here is a thin ctypes layer over `lib/libsecp256k1_b200.so`
(include/secp256k1_b200.h); the names follow the reference's Go API
(secp256k1.Point.ScalarBaseMult, .ScalarMult, .DoubleScalarMultBasepointVartime,
.MultiScalarMult, secec.PublicKey.Verify, secec.RecoverPublicKey,
secec.PrivateKey.ECDH, bitcoin.SchnorrPublicKey.Verify) in batch form.

There is no CPU path: importing works anywhere (so the symbol table can be
checked), but creating an Engine without a CUDA device raises.

Inputs are either host arrays (numpy uint8 / bytes; the library copies in and
out) or CUDA torch tensors (uint8, contiguous; the `_dev` entry points run on
torch's current stream and return torch tensors without synchronising).
"""
import ctypes as C
import os

import numpy as np

from . import build as _build
from . import parallel  # noqa: F401  (re-exported)
from . import synth  # noqa: F401  (re-exported)

ST_INVALID, ST_OK, ST_IDENTITY = 0, 1, 2
FLAG_REJECT_MALLEABLE = 1

EXPORTED_SYMBOLS = [
    "s256_init", "s256_free", "s256_strerror", "s256_last_cuda_error", "s256_device",
    "s256_scalar_base_mult", "s256_scalar_base_mult_dev",
    "s256_scalar_mult", "s256_scalar_mult_dev",
    "s256_ecdh", "s256_ecdh_dev", "s256_point_decompress", "s256_point_compress",
    "s256_double_scalar_mult_basepoint_vartime", "s256_double_scalar_mult_basepoint_vartime_dev",
    "s256_ecdsa_verify", "s256_ecdsa_verify_dev",
    "s256_parse_asn1_signatures", "s256_is_valid_signature_encoding_bip0066",
    "s256_parse_asn1_public_keys", "s256_build_asn1_public_keys", "s256_build_asn1_signatures",
    "s256_new_public_keys", "s256_parse_asn1_public_keys_checked",
    "s256_ecdsa_verify_asn1", "s256_bitcoin_verify_asn1",
    "s256_ecdsa_recover", "s256_ecdsa_recover_dev",
    "s256_ecdsa_sign_rfc6979", "s256_ecdsa_sign_rfc6979_dev",
    "s256_schnorr_verify", "s256_schnorr_verify_dev", "s256_schnorr_sign", "s256_schnorr_sign_dev",
    "s256_schnorr_batch_verify", "s256_schnorr_batch_verify_dev",
    "s256_msm", "s256_msm_partial", "s256_msm_combine", "s256_msm_dev", "s256_msm_sharded", "s256_msm_sharded_dev",
    "s256_comm_unique_id", "s256_comm_init", "s256_comm_free", "s256_msm_plan", "s256_hash_to_curve", "s256_expand_message_xmd",
    "s256_debug_ladder_add_count", "s256_mac32_k_dsm",
    "s256_debug_gen_table", "s256_debug_field_op", "s256_debug_schnorr_batch_rows", "s256_microbench_imad",
    "s256_microbench_variant", "s256_microbench_fe_mul", "s256_profile_enable", "s256_profile_read",
    "s256_launch_count", "s256_mac32_per_item", "s256_host_alloc", "s256_host_free",
]

_lib = None


class S256Error(RuntimeError):
    pass


def library_path():
    return _build.LIB


def load_library():
    """Loads (building first if stale and nvcc is present) the C-ABI library."""
    global _lib
    if _lib is not None:
        return _lib
    try:
        _build.build()
    except FileNotFoundError:
        pass  # no nvcc on this box: use the prebuilt library shipped in-tree
    if not os.path.exists(_build.LIB):
        raise S256Error(f"{_build.LIB} is missing: run `python -m __graft_entry__` / build() where nvcc exists; "
                        "there is no fallback implementation")
    lib = C.CDLL(_build.LIB)
    lib.s256_strerror.restype = C.c_char_p
    lib.s256_last_cuda_error.restype = C.c_char_p
    lib.s256_last_cuda_error.argtypes = [C.c_void_p]
    lib.s256_launch_count.restype = C.c_uint64
    lib.s256_launch_count.argtypes = [C.c_void_p]
    lib.s256_mac32_per_item.restype = C.c_double
    lib.s256_mac32_per_item.argtypes = [C.c_char_p]
    lib.s256_mac32_k_dsm.restype = C.c_double
    lib.s256_mac32_k_dsm.argtypes = [C.c_double, C.c_double]
    lib.s256_free.argtypes = [C.c_void_p]
    lib.s256_free.restype = None
    lib.s256_host_alloc.restype = C.c_void_p
    lib.s256_host_alloc.argtypes = [C.c_size_t]
    lib.s256_host_free.argtypes = [C.c_void_p]
    lib.s256_host_free.restype = None
    _lib = lib
    return lib


def msm_plan(n):
    """(window bits, windows) of the Pippenger plan for n points on one GPU."""
    c, w = C.c_int(0), C.c_int(0)
    load_library().s256_msm_plan(C.c_size_t(n), C.byref(c), C.byref(w))
    return c.value, w.value


def mac32_per_item(entry_point):
    return load_library().s256_mac32_per_item(entry_point.encode())


def _pack_rows(rows):
    """list of byte strings -> (concatenated uint8 array, size_t offsets array)"""
    rows = [bytes(r) for r in rows]
    offs = np.zeros(len(rows) + 1, dtype=np.uintp)
    np.cumsum([len(r) for r in rows], out=offs[1:])
    data = np.frombuffer(b"".join(rows) or b"\x00", dtype=np.uint8).copy()
    return data, offs


def parse_asn1_signatures(rows):
    """secec.ParseASN1Signature over a list of DER signatures -> (sig64 rows, ok). Host-side, no GPU needed."""
    lib = load_library()
    data, offs = _pack_rows(rows)
    n = len(rows)
    sig = np.zeros((n, 64), np.uint8)
    ok = np.zeros(n, np.uint8)
    rc = lib.s256_parse_asn1_signatures(data.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p), C.c_size_t(n),
                                        sig.ctypes.data_as(C.c_void_p), ok.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise S256Error(f"parse_asn1_signatures rc={rc}")
    return sig, ok


def parse_asn1_public_keys(rows):
    """secec.ParseASN1PublicKey up to NewPublicKey, over a list of DER SubjectPublicKeyInfo blobs ->
    (point rows of stride 65, point_len, status).  Host-side, no GPU needed; feed Engine.new_public_keys."""
    lib = load_library()
    data, offs = _pack_rows(rows)
    n = len(rows)
    pts = np.zeros((n, 65), np.uint8)
    ln = np.zeros(n, np.uint8)
    st = np.zeros(n, np.uint8)
    rc = lib.s256_parse_asn1_public_keys(data.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p), C.c_size_t(n),
                                         pts.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p),
                                         st.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise S256Error(f"parse_asn1_public_keys rc={rc}")
    return pts, ln, st


def build_asn1_public_keys(pk65):
    """PublicKey.ASN1Bytes over validated uncompressed keys -> (n, 88) rows."""
    lib = load_library()
    p = _host(pk65, 65)
    out = np.zeros((len(p), 88), np.uint8)
    rc = lib.s256_build_asn1_public_keys(p.ctypes.data_as(C.c_void_p), C.c_size_t(len(p)), out.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise S256Error(f"build_asn1_public_keys rc={rc}")
    return out


def build_asn1_signatures(sig64):
    """secec.BuildASN1Signature over compact r||s rows -> list of DER byte strings."""
    lib = load_library()
    g = _host(sig64, 64)
    out = np.zeros((len(g), 72), np.uint8)
    ln = np.zeros(len(g), np.uint8)
    rc = lib.s256_build_asn1_signatures(g.ctypes.data_as(C.c_void_p), C.c_size_t(len(g)), out.ctypes.data_as(C.c_void_p),
                                        ln.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise S256Error(f"build_asn1_signatures rc={rc}")
    return [out[i, :ln[i]].tobytes() for i in range(len(g))]


def is_valid_signature_encoding_bip0066(rows):
    """bitcoin.IsValidSignatureEncodingBIP0066 over a list of signatures (with the sighash byte)."""
    lib = load_library()
    data, offs = _pack_rows(rows)
    n = len(rows)
    ok = np.zeros(n, np.uint8)
    rc = lib.s256_is_valid_signature_encoding_bip0066(data.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p),
                                                      C.c_size_t(n), ok.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise S256Error(f"is_valid_signature_encoding_bip0066 rc={rc}")
    return ok


def _is_torch_cuda(x):
    return hasattr(x, "is_cuda") and x.is_cuda


def _host(x, width):
    if isinstance(x, (bytes, bytearray, memoryview)):
        x = np.frombuffer(bytes(x), dtype=np.uint8)
    a = np.ascontiguousarray(x, dtype=np.uint8)
    if width:
        a = a.reshape(-1, width)
    return a


class Engine:
    """One context on one GPU (s256_init).  Use one Engine per process/GPU."""

    def __init__(self, device=-1, max_batch=0, pinned_outputs=False):
        """pinned_outputs=True: host results are returned as views into page-locked buffers owned by the
        engine (s256_host_alloc) -- D2H at full PCIe speed instead of a staged copy into pageable
        memory -- and stay valid only until the next call of the same method."""
        self._pinned = bool(pinned_outputs)
        self._pool = {}
        self._lib = load_library()
        self._ctx = C.c_void_p()
        rc = self._lib.s256_init(C.byref(self._ctx), int(device), C.c_size_t(max_batch))
        if rc != 0:
            self._ctx = C.c_void_p()
            raise S256Error(f"s256_init failed: {self._lib.s256_strerror(rc).decode()} (rc={rc})")

    # -- plumbing -----------------------------------------------------------
    def close(self):
        for ptr, _ in getattr(self, "_pool", {}).values():
            self._lib.s256_host_free(C.c_void_p(ptr))
        self._pool = {}
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.s256_free(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            detail = self._lib.s256_last_cuda_error(self._ctx).decode()
            raise S256Error(f"{what}: {self._lib.s256_strerror(rc).decode()} (rc={rc}) {detail}")

    @property
    def device(self):
        return self._lib.s256_device(self._ctx)

    @property
    def launch_count(self):
        return int(self._lib.s256_launch_count(self._ctx))

    def _out(self, key, shape):
        if isinstance(shape, int):
            shape = (shape,)
        if not self._pinned:
            return np.zeros(shape, np.uint8)
        size = int(np.prod(shape))
        ent = self._pool.get(key)
        if ent is None or ent[1] < size:
            if ent is not None:
                self._lib.s256_host_free(C.c_void_p(ent[0]))
            cap = max(size, 1)
            ptr = self._lib.s256_host_alloc(C.c_size_t(cap))
            if not ptr:
                raise S256Error("s256_host_alloc failed")
            ent = (ptr, cap)
            self._pool[key] = ent
        arr = np.ctypeslib.as_array((C.c_uint8 * ent[1]).from_address(ent[0]))
        return arr[:size].reshape(shape)

    def pinned_empty(self, shape):
        """A page-locked uint8 array for INPUT batches (freed with the engine)."""
        self._pin_seq = getattr(self, "_pin_seq", 0) + 1
        keep, self._pinned = self._pinned, True
        try:
            return self._out(("in", self._pin_seq), shape)
        finally:
            self._pinned = keep

    @staticmethod
    def _hp(a):
        return a.ctypes.data_as(C.c_void_p)

    @staticmethod
    def _dev_args(*tensors):
        import torch
        for t in tensors:
            if t.dtype != torch.uint8 or not t.is_contiguous():
                raise S256Error("device inputs must be contiguous uint8 CUDA tensors")
        return [C.c_void_p(t.data_ptr()) for t in tensors]

    @staticmethod
    def _stream():
        import torch
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    # -- Point.ScalarBaseMult (point_mul_table.go:168) ------------------------
    def scalar_base_mult(self, k32):
        if _is_torch_cuda(k32):
            import torch
            n = k32.numel() // 32
            out = torch.empty((n, 65), dtype=torch.uint8, device=k32.device)
            st = torch.empty(n, dtype=torch.uint8, device=k32.device)
            a = self._dev_args(k32, out, st)
            self._check(self._lib.s256_scalar_base_mult_dev(self._ctx, a[0], C.c_size_t(n), a[1], a[2], self._stream()),
                        "scalar_base_mult_dev")
            return out, st
        k = _host(k32, 32)
        n = len(k)
        out = self._out(1, (n, 65))
        st = self._out(2, n)
        self._check(self._lib.s256_scalar_base_mult(self._ctx, self._hp(k), C.c_size_t(n), self._hp(out), self._hp(st)),
                    "scalar_base_mult")
        return out, st

    # -- Point.ScalarMult (point_mul_glv.go:257), constant time ---------------
    def scalar_mult(self, k32, pt65):
        if _is_torch_cuda(k32):
            import torch
            n = k32.numel() // 32
            out = torch.empty((n, 65), dtype=torch.uint8, device=k32.device)
            st = torch.empty(n, dtype=torch.uint8, device=k32.device)
            a = self._dev_args(k32, pt65, out, st)
            self._check(self._lib.s256_scalar_mult_dev(self._ctx, a[0], a[1], C.c_size_t(n), a[2], a[3], self._stream()),
                        "scalar_mult_dev")
            return out, st
        k, p = _host(k32, 32), _host(pt65, 65)
        n = len(k)
        if len(p) != n:
            raise ValueError("len(scalars) != len(points)")
        out = self._out(3, (n, 65))
        st = self._out(4, n)
        self._check(self._lib.s256_scalar_mult(self._ctx, self._hp(k), self._hp(p), C.c_size_t(n), self._hp(out), self._hp(st)),
                    "scalar_mult")
        return out, st

    # -- PrivateKey.ECDH (secec/secec.go:53) ----------------------------------
    def ecdh(self, k32, pt65):
        if _is_torch_cuda(k32):
            import torch
            n = k32.numel() // 32
            out = torch.empty((n, 32), dtype=torch.uint8, device=k32.device)
            st = torch.empty(n, dtype=torch.uint8, device=k32.device)
            a = self._dev_args(k32, pt65, out, st)
            self._check(self._lib.s256_ecdh_dev(self._ctx, a[0], a[1], C.c_size_t(n), a[2], a[3], self._stream()), "ecdh_dev")
            return out, st
        k, p = _host(k32, 32), _host(pt65, 65)
        n = len(k)
        if len(p) != n:
            raise ValueError("len(scalars) != len(points)")
        out = self._out(5, (n, 32))
        st = self._out(6, n)
        self._check(self._lib.s256_ecdh(self._ctx, self._hp(k), self._hp(p), C.c_size_t(n), self._hp(out), self._hp(st)), "ecdh")
        return out, st

    # -- NewPointFromBytes, compressed form (point_s11n.go:140) ---------------
    def point_decompress(self, pt33):
        p = _host(pt33, 33)
        n = len(p)
        out = self._out(7, (n, 65))
        st = self._out(8, n)
        self._check(self._lib.s256_point_decompress(self._ctx, self._hp(p), C.c_size_t(n), self._hp(out), self._hp(st)),
                    "point_decompress")
        return out, st

    def point_compress(self, pt65):
        """(*Point).CompressedBytes behind NewPointFromBytes: 65 B -> 33 B + status (point_s11n.go:90-117,234)."""
        p = _host(pt65, 65)
        n = len(p)
        out = self._out(7, (n, 33))
        st = self._out(8, n)
        self._check(self._lib.s256_point_compress(self._ctx, self._hp(p), C.c_size_t(n), self._hp(out), self._hp(st)),
                    "point_compress")
        return out, st

    # -- secec.NewPublicKey / ParseASN1PublicKey (secec/secec.go:183, secec/s11n.go:38) ----
    def new_public_keys(self, enc, enc_len=None):
        """Rows of SEC 1 encodings: a list of byte strings of mixed length, or (stride-65 rows, lengths)."""
        if enc_len is None:
            rows = [bytes(r) for r in enc]
            enc_len = np.array([len(r) if len(r) <= 65 else 0 for r in rows], np.uint8)
            enc = self._out(9, (len(rows), 65))
            for i, r in enumerate(rows):
                if len(r) <= 65:
                    enc[i, :len(r)] = np.frombuffer(r, np.uint8)
        e, ln = _host(enc, 65), _host(enc_len, 0).reshape(-1)
        n = len(e)
        out = self._out(10, (n, 65))
        st = self._out(11, n)
        self._check(self._lib.s256_new_public_keys(self._ctx, self._hp(e), self._hp(ln), C.c_size_t(n), self._hp(out),
                                                   self._hp(st)), "new_public_keys")
        return out, st

    def parse_asn1_public_keys(self, rows):
        data, offs = _pack_rows(rows)
        n = len(rows)
        out = self._out(12, (n, 65))
        st = self._out(13, n)
        self._check(self._lib.s256_parse_asn1_public_keys_checked(self._ctx, self._hp(data), offs.ctypes.data_as(C.c_void_p),
                                                                  C.c_size_t(n), self._hp(out), self._hp(st)),
                    "parse_asn1_public_keys")
        return out, st

    # -- Point.DoubleScalarMultBasepointVartime (point_mul_glv.go:307) --------
    def double_scalar_mult_basepoint_vartime(self, u1, u2, pt65):
        if _is_torch_cuda(u1):
            import torch
            n = u1.numel() // 32
            out = torch.empty((n, 65), dtype=torch.uint8, device=u1.device)
            st = torch.empty(n, dtype=torch.uint8, device=u1.device)
            a = self._dev_args(u1, u2, pt65, out, st)
            self._check(self._lib.s256_double_scalar_mult_basepoint_vartime_dev(
                self._ctx, a[0], a[1], a[2], C.c_size_t(n), a[3], a[4], self._stream()), "double_scalar_mult_dev")
            return out, st
        a1, a2, p = _host(u1, 32), _host(u2, 32), _host(pt65, 65)
        n = len(a1)
        if len(a2) != n or len(p) != n:
            raise ValueError("length mismatch")
        out = self._out(14, (n, 65))
        st = self._out(15, n)
        self._check(self._lib.s256_double_scalar_mult_basepoint_vartime(
            self._ctx, self._hp(a1), self._hp(a2), self._hp(p), C.c_size_t(n), self._hp(out), self._hp(st)),
            "double_scalar_mult_basepoint_vartime")
        return out, st

    # -- secec.PublicKey.Verify, EncodingCompact (secec/ecdsa.go:171) ---------
    def ecdsa_verify(self, pk65, digest32, sig64, flags=0):
        if _is_torch_cuda(pk65):
            import torch
            n = pk65.numel() // 65
            ok = torch.empty(n, dtype=torch.uint8, device=pk65.device)
            a = self._dev_args(pk65, digest32, sig64, ok)
            self._check(self._lib.s256_ecdsa_verify_dev(self._ctx, a[0], a[1], a[2], C.c_uint32(flags), C.c_size_t(n), a[3],
                                                        self._stream()), "ecdsa_verify_dev")
            return ok
        pk, dg, sg = _host(pk65, 65), _host(digest32, 32), _host(sig64, 64)
        n = len(pk)
        if len(dg) != n or len(sg) != n:
            raise ValueError("length mismatch")
        ok = self._out(16, n)
        self._check(self._lib.s256_ecdsa_verify(self._ctx, self._hp(pk), self._hp(dg), self._hp(sg), C.c_uint32(flags),
                                                C.c_size_t(n), self._hp(ok)), "ecdsa_verify")
        return ok

    # -- PublicKey.Verify, EncodingASN1 (secec/ecdsa.go:171) and bitcoin.VerifyASN1 ----------
    def ecdsa_verify_asn1(self, pk65, digest32, der_rows, flags=0):
        pk, dg = _host(pk65, 65), _host(digest32, 32)
        data, offs = _pack_rows(der_rows)
        n = len(der_rows)
        if len(pk) != n or len(dg) != n:
            raise ValueError("length mismatch")
        ok = self._out(17, n)
        self._check(self._lib.s256_ecdsa_verify_asn1(self._ctx, self._hp(pk), self._hp(dg), self._hp(data), self._hp(offs),
                                                     C.c_uint32(flags), C.c_size_t(n), self._hp(ok)), "ecdsa_verify_asn1")
        return ok

    def bitcoin_verify_asn1(self, pk65, digest32, der_rows_with_sighash):
        pk, dg = _host(pk65, 65), _host(digest32, 32)
        data, offs = _pack_rows(der_rows_with_sighash)
        n = len(der_rows_with_sighash)
        if len(pk) != n or len(dg) != n:
            raise ValueError("length mismatch")
        ok = self._out(18, n)
        self._check(self._lib.s256_bitcoin_verify_asn1(self._ctx, self._hp(pk), self._hp(dg), self._hp(data), self._hp(offs),
                                                       C.c_size_t(n), self._hp(ok)), "bitcoin_verify_asn1")
        return ok

    # -- PrivateKey.Sign(RFC6979SHA256(), digest) (secec/ecdsa.go:92,284) -------------------
    def ecdsa_sign_rfc6979(self, priv32, digest32):
        """-> (sig64 rows r||s low-s, recovery ids, status)"""
        if _is_torch_cuda(priv32):
            import torch
            n = priv32.numel() // 32
            sig = torch.empty((n, 64), dtype=torch.uint8, device=priv32.device)
            rec = torch.empty(n, dtype=torch.uint8, device=priv32.device)
            st = torch.empty(n, dtype=torch.uint8, device=priv32.device)
            a = self._dev_args(priv32, digest32, sig, rec, st)
            self._check(self._lib.s256_ecdsa_sign_rfc6979_dev(self._ctx, a[0], a[1], C.c_size_t(n), a[2], a[3], a[4],
                                                              self._stream()), "ecdsa_sign_rfc6979_dev")
            return sig, rec, st
        d, dg = _host(priv32, 32), _host(digest32, 32)
        n = len(d)
        if len(dg) != n:
            raise ValueError("length mismatch")
        sig = self._out(19, (n, 64))
        rec = self._out(20, n)
        st = self._out(21, n)
        self._check(self._lib.s256_ecdsa_sign_rfc6979(self._ctx, self._hp(d), self._hp(dg), C.c_size_t(n), self._hp(sig),
                                                      self._hp(rec), self._hp(st)), "ecdsa_sign_rfc6979")
        return sig, rec, st

    # -- secec.RecoverPublicKey (secec/ecdsa.go:244) ---------------------------
    def ecdsa_recover(self, digest32, sig65):
        if _is_torch_cuda(digest32):
            import torch
            n = digest32.numel() // 32
            out = torch.empty((n, 65), dtype=torch.uint8, device=digest32.device)
            st = torch.empty(n, dtype=torch.uint8, device=digest32.device)
            a = self._dev_args(digest32, sig65, out, st)
            self._check(self._lib.s256_ecdsa_recover_dev(self._ctx, a[0], a[1], C.c_size_t(n), a[2], a[3], self._stream()),
                        "ecdsa_recover_dev")
            return out, st
        dg, sg = _host(digest32, 32), _host(sig65, 65)
        n = len(dg)
        if len(sg) != n:
            raise ValueError("length mismatch")
        out = self._out(22, (n, 65))
        st = self._out(23, n)
        self._check(self._lib.s256_ecdsa_recover(self._ctx, self._hp(dg), self._hp(sg), C.c_size_t(n), self._hp(out), self._hp(st)),
                    "ecdsa_recover")
        return out, st

    # -- bitcoin.SchnorrPublicKey.Verify (secec/bitcoin/schnorr.go:221) --------
    def schnorr_verify(self, pkx32, msg, sig64):
        if _is_torch_cuda(pkx32):
            import torch
            n = pkx32.numel() // 32
            msg_len = msg.numel() // n if n else 0
            ok = torch.empty(n, dtype=torch.uint8, device=pkx32.device)
            a = self._dev_args(pkx32, msg, sig64, ok)
            self._check(self._lib.s256_schnorr_verify_dev(self._ctx, a[0], a[1], C.c_size_t(msg_len), a[2], C.c_size_t(n), a[3],
                                                          self._stream()), "schnorr_verify_dev")
            return ok
        pk, sg = _host(pkx32, 32), _host(sig64, 64)
        n = len(pk)
        m = _host(msg, 0).reshape(n, -1) if n else np.zeros((0, 0), np.uint8)
        if len(sg) != n:
            raise ValueError("length mismatch")
        ok = self._out(24, n)
        self._check(self._lib.s256_schnorr_verify(self._ctx, self._hp(pk), self._hp(m), C.c_size_t(m.shape[1] if n else 0),
                                                  self._hp(sg), C.c_size_t(n), self._hp(ok)), "schnorr_verify")
        return ok

    # -- BIP-340 batch verification: one verdict for the whole batch ----------------------------
    def schnorr_batch_verify(self, pkx32, msg, sig64):
        """True iff every row would pass schnorr_verify (one randomized multi-scalar multiplication; a batch with an
        invalid row is accepted with probability <= 2^-127).  With CUDA tensors: a (1,) uint8 tensor, not synchronised."""
        if _is_torch_cuda(pkx32):
            import torch
            n = pkx32.numel() // 32
            msg_len = msg.numel() // n if n else 0
            if sig64.numel() != 64 * n or msg.numel() != msg_len * n:
                raise ValueError("length mismatch")
            ok = torch.empty(1, dtype=torch.uint8, device=pkx32.device)
            a = self._dev_args(pkx32, msg, sig64, ok)
            self._check(self._lib.s256_schnorr_batch_verify_dev(self._ctx, a[0], a[1], C.c_size_t(msg_len), a[2], C.c_size_t(n),
                                                                a[3], self._stream()), "schnorr_batch_verify_dev")
            return ok
        pk, sg = _host(pkx32, 32), _host(sig64, 64)
        n = len(pk)
        m = _host(msg, 0)
        msg_len = m.size // n if n else 0
        if len(sg) != n or m.size != msg_len * n:
            raise ValueError("length mismatch")
        m = m.reshape(n, msg_len)
        ok = C.c_uint8(0)
        self._check(self._lib.s256_schnorr_batch_verify(self._ctx, self._hp(pk), self._hp(m), C.c_size_t(msg_len), self._hp(sg),
                                                        C.c_size_t(n), C.byref(ok)), "schnorr_batch_verify")
        return bool(ok.value)

    # -- bitcoin.SchnorrPrivateKey.Sign (secec/bitcoin/schnorr.go:111,322) ---------------------
    def schnorr_sign(self, priv32, msg, aux32):
        if _is_torch_cuda(priv32):
            import torch
            n = priv32.numel() // 32
            msg_len = msg.numel() // n if n else 0
            sig = torch.empty((n, 64), dtype=torch.uint8, device=priv32.device)
            st = torch.empty(n, dtype=torch.uint8, device=priv32.device)
            a = self._dev_args(priv32, msg, aux32, sig, st)
            self._check(self._lib.s256_schnorr_sign_dev(self._ctx, a[0], a[1], C.c_size_t(msg_len), a[2], C.c_size_t(n),
                                                        a[3], a[4], self._stream()), "schnorr_sign_dev")
            return sig, st
        d, ax = _host(priv32, 32), _host(aux32, 32)
        n = len(d)
        m = _host(msg, 0).reshape(n, -1) if n else np.zeros((0, 0), np.uint8)
        if len(ax) != n:
            raise ValueError("length mismatch")
        sig = self._out(25, (n, 64))
        st = self._out(26, n)
        self._check(self._lib.s256_schnorr_sign(self._ctx, self._hp(d), self._hp(m), C.c_size_t(m.shape[1] if n else 0),
                                                self._hp(ax), C.c_size_t(n), self._hp(sig), self._hp(st)), "schnorr_sign")
        return sig, st

    # -- h2c.Secp256k1_XMD_SHA256_SSWU_RO / _NU (secec/h2c/h2c.go:25,49) ------------------------
    def hash_to_curve(self, dst, msgs, random_oracle=True):
        """msgs: (n, msg_len) uint8 rows (equal length).  -> (out65, status)"""
        dst = bytes(dst)
        m = np.ascontiguousarray(msgs, dtype=np.uint8)
        if m.ndim != 2:
            raise ValueError("msgs must be a 2-D array of equal-length rows")
        n, msg_len = m.shape
        out = self._out(27, (n, 65))
        st = self._out(28, n)
        self._check(self._lib.s256_hash_to_curve(self._ctx, dst, C.c_size_t(len(dst)), self._hp(m), C.c_size_t(msg_len),
                                                 C.c_size_t(n), int(bool(random_oracle)), self._hp(out), self._hp(st)),
                    "hash_to_curve")
        return out, st

    def expand_message_xmd(self, dst, msgs, length):
        dst = bytes(dst)
        m = np.ascontiguousarray(msgs, dtype=np.uint8)
        n, msg_len = m.shape
        out = self._out(29, (n, length))
        self._check(self._lib.s256_expand_message_xmd(self._ctx, dst, C.c_size_t(len(dst)), self._hp(m), C.c_size_t(msg_len),
                                                      C.c_size_t(n), C.c_size_t(length), self._hp(out)), "expand_message_xmd")
        return out

    # -- Point.MultiScalarMult[Vartime] (point_mul_multi.go:25,73) -------------
    def msm(self, k32, pt65, vartime=True):
        if _is_torch_cuda(k32):  # device-resident: (65,) and (1,) uint8 tensors, nothing synchronised
            import torch
            n = k32.numel() // 32
            if pt65.numel() // 65 != n:
                raise ValueError("secp256k1: len(scalars) != len(points)")
            out = torch.empty(65, dtype=torch.uint8, device=k32.device)
            st = torch.empty(1, dtype=torch.uint8, device=k32.device)
            a = self._dev_args(k32, pt65, out, st)
            self._check(self._lib.s256_msm_dev(self._ctx, a[0], a[1], C.c_size_t(n), int(vartime), a[2], a[3], self._stream()),
                        "msm_dev")
            return out, st
        k, p = _host(k32, 32), _host(pt65, 65)
        n = len(k)
        if len(p) != n:
            # the reference panics: point_mul_multi.go:27-29
            raise ValueError("secp256k1: len(scalars) != len(points)")
        out = self._out(30, 65)
        st = C.c_uint8(0)
        self._check(self._lib.s256_msm(self._ctx, self._hp(k), self._hp(p), C.c_size_t(n), int(vartime), self._hp(out),
                                       C.byref(st)), "msm")
        return out, st.value

    # -- the same product over a batch sharded across GPUs (BASELINE configs[4]) ------------
    @staticmethod
    def comm_unique_id():
        """Rank 0: the 128 bytes (ncclUniqueId) every rank passes to comm_init."""
        buf = (C.c_uint8 * 128)()
        rc = load_library().s256_comm_unique_id(buf)
        if rc != 0:
            raise S256Error(f"comm_unique_id: {load_library().s256_strerror(rc).decode()} (rc={rc})")
        return bytes(buf)

    def comm_init(self, unique_id, rank, nranks):
        """Collective: builds this context's NCCL communicator (one rank per GPU)."""
        if len(unique_id) != 128:
            raise ValueError("unique id must be 128 bytes")
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(unique_id))
        self._check(self._lib.s256_comm_init(self._ctx, buf, int(rank), int(nranks)), "comm_init")
        self.comm_size = int(nranks)

    def comm_free(self):
        self._check(self._lib.s256_comm_free(self._ctx), "comm_free")
        self.comm_size = 0

    def msm_sharded(self, k32_local, pt65_local, vartime=True):
        """This rank's slice in, the whole product out (on every rank): local Pippenger, ONE ncclAllGather of 112 bytes
        per rank inside the library, fold, encode.  Device tensors: nothing is synchronised; host arrays: one sync."""
        if _is_torch_cuda(k32_local):
            import torch
            n = k32_local.numel() // 32
            if pt65_local.numel() // 65 != n:
                raise ValueError("secp256k1: len(scalars) != len(points)")
            out = torch.empty(65, dtype=torch.uint8, device=k32_local.device)
            st = torch.empty(1, dtype=torch.uint8, device=k32_local.device)
            a = self._dev_args(k32_local, pt65_local, out, st)
            self._check(self._lib.s256_msm_sharded_dev(self._ctx, a[0], a[1], C.c_size_t(n), int(vartime), a[2], a[3],
                                                       self._stream()), "msm_sharded_dev")
            return out, st
        k, p = _host(k32_local, 32), _host(pt65_local, 65)
        n = len(k)
        if len(p) != n:
            raise ValueError("secp256k1: len(scalars) != len(points)")
        out = self._out(34, 65)
        st = C.c_uint8(0)
        self._check(self._lib.s256_msm_sharded(self._ctx, self._hp(k), self._hp(p), C.c_size_t(n), int(vartime),
                                               self._hp(out), C.byref(st)), "msm_sharded")
        return out, st.value

    def ladder_add_count(self, n):
        """(additions of the first half, of the lambda half) the last verification-type call executed for its first n items."""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._check(self._lib.s256_debug_ladder_add_count(self._ctx, C.c_size_t(n), C.byref(a), C.byref(b)), "ladder_add_count")
        return a.value, b.value

    def msm_partial(self, k32, pt65, vartime=True):
        k, p = _host(k32, 32), _host(pt65, 65)
        n = len(k)
        if len(p) != n:
            raise ValueError("secp256k1: len(scalars) != len(points)")
        out = self._out(31, 96)
        st = C.c_uint8(0)
        self._check(self._lib.s256_msm_partial(self._ctx, self._hp(k), self._hp(p), C.c_size_t(n), int(vartime),
                                               self._hp(out), C.byref(st)), "msm_partial")
        return out, st.value

    def msm_combine(self, partials96):
        p = _host(partials96, 96)
        out = self._out(32, 65)
        st = C.c_uint8(0)
        self._check(self._lib.s256_msm_combine(self._ctx, self._hp(p), C.c_size_t(len(p)), self._hp(out), C.byref(st)),
                    "msm_combine")
        return out, st.value

    # -- measurement / debug ----------------------------------------------------
    def debug_gen_table(self, wbits, nwin):
        out = self._out(33, ((2 ** wbits - 1) * nwin, 64))
        self._check(self._lib.s256_debug_gen_table(self._ctx, int(wbits), int(nwin), self._hp(out)), "debug_gen_table")
        return out

    def debug_field_op(self, op, a32, b32):
        a, b = _host(a32, 32), _host(b32, 32)
        out = self._out(34, (len(a), 32))
        self._check(self._lib.s256_debug_field_op(self._ctx, int(op), self._hp(a), self._hp(b), C.c_size_t(len(a)),
                                                  self._hp(out)), "debug_field_op")
        return out

    def debug_schnorr_batch_rows(self, pkx32, msg, sig64):
        """What schnorr_batch_verify checks for these host rows: (seed (32,), k (n, 2, 32) = a_i and a_i e_i mod n,
        pts (n, 2, 64) = -R_i and -P_i as X||Y (G for a rejected row), sum (32,) = sum a_i s_i mod n, rejected),
        all big-endian bytes."""
        pk, sg = _host(pkx32, 32), _host(sig64, 64)
        n = len(pk)
        m = _host(msg, 0)
        msg_len = m.size // n if n else 0
        if n == 0 or len(sg) != n or m.size != msg_len * n:
            raise ValueError("length mismatch or empty batch")
        seed, k, pts, ssum, rej = (np.zeros(32, np.uint8), np.zeros((n, 2, 32), np.uint8), np.zeros((n, 2, 64), np.uint8),
                                   np.zeros(32, np.uint8), C.c_uint8(0))
        self._check(self._lib.s256_debug_schnorr_batch_rows(self._ctx, self._hp(pk), self._hp(m), C.c_size_t(msg_len),
                                                            self._hp(sg), C.c_size_t(n), self._hp(seed), self._hp(k),
                                                            self._hp(pts), self._hp(ssum), C.byref(rej)),
                    "debug_schnorr_batch_rows")
        return seed.tobytes(), k, pts, ssum.tobytes(), bool(rej.value)

    def profile_enable(self, on=True):
        self._check(self._lib.s256_profile_enable(self._ctx, int(bool(on))), "profile_enable")

    def profile_read(self):
        """(summed device ms of the ladder kernel, number of its launches) since profile_enable."""
        ms, cnt = C.c_double(0), C.c_uint64(0)
        self._check(self._lib.s256_profile_read(self._ctx, C.byref(ms), C.byref(cnt)), "profile_read")
        return ms.value, int(cnt.value)

    def microbench_variant(self, variant, iters=4096):
        rate, ms = C.c_double(0), C.c_double(0)
        self._check(self._lib.s256_microbench_variant(self._ctx, int(variant), int(iters), C.byref(rate), C.byref(ms)),
                    "microbench_variant")
        return rate.value, ms.value

    def microbench_fe_mul(self, form, iters=2048):
        rate, ms = C.c_double(), C.c_double()
        self._check(self._lib.s256_microbench_fe_mul(self._ctx, int(form), int(iters), C.byref(rate), C.byref(ms)),
                    "microbench_fe_mul")
        return rate.value, ms.value

    def microbench_imad(self, iters=4096):
        rate, ms = C.c_double(0), C.c_double(0)
        self._check(self._lib.s256_microbench_imad(self._ctx, int(iters), C.byref(rate), C.byref(ms)), "microbench_imad")
        return rate.value, ms.value
