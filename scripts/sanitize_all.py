"""Every entry point once at small sizes (driven under compute-sanitizer)."""
import importlib, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
pkg = importlib.import_module("secp256k1-voi_b200")
eng = pkg.Engine(device=0, max_batch=4096)
for n in (1, 33, 1500):
    ks = pkg.synth.base_mult_scalars(n)
    pk, st = eng.scalar_base_mult(ks)
    w = pkg.synth.ecdsa_batch(n, eng.scalar_base_mult)
    assert np.array_equal(eng.ecdsa_verify(w["pk65"], w["digest32"], w["sig64"]), w["expected"])
    sig65 = np.concatenate([w["sig64"], np.zeros((n, 1), np.uint8)], axis=1)
    eng.ecdsa_recover(w["digest32"], sig65)
    ws = pkg.synth.schnorr_batch(n, eng.scalar_base_mult)
    assert np.array_equal(eng.schnorr_verify(ws["pkx32"], ws["msg"], ws["sig64"]), ws["expected"])
    we = pkg.synth.ecdh_batch(n, eng.scalar_base_mult)
    eng.scalar_mult(we["k32"], we["pt65"]); eng.ecdh(we["k32"], we["pt65"])
    eng.double_scalar_mult_basepoint_vartime(we["k32"], ks, we["pt65"])
    for vt in (True, False):
        eng.msm(we["k32"], we["pt65"], vartime=vt)
    comp = np.concatenate([2 + (we["pt65"][:, 64:] & 1), we["pt65"][:, 1:33]], axis=1)
    eng.point_decompress(comp)
    eng.point_compress(we["pt65"])
    priv = ks.copy(); priv[:, 0] &= 0x7F; priv[:, 31] |= 1
    sig, rec, st = eng.ecdsa_sign_rfc6979(priv, w["digest32"])
    eng.schnorr_sign(priv, w["digest32"], ks)
    eng.hash_to_curve(b"QUUX-V01-CS02-with-secp256k1_XMD:SHA-256_SSWU_RO_", w["digest32"], random_oracle=True)
    eng.new_public_keys([bytes(r) for r in pk[:8]] + [b"\x00", b"\x02" + bytes(pk[-1][1:33])])
    der = pkg.build_asn1_signatures(w["sig64"])
    eng.ecdsa_verify_asn1(w["pk65"], w["digest32"], der)
    eng.bitcoin_verify_asn1(w["pk65"], w["digest32"], [r + b"\x01" for r in der])
# the sort / slice / super-slice / window stages of the MSM: random scalars, then one heavy bucket per window
wm = pkg.synth.msm_batch(6000, eng.scalar_base_mult)
eng.msm(wm["k32"], wm["pt65"])
eng.msm(np.tile(wm["k32"][:1], (6000, 1)), wm["pt65"])
# round 2: the device-resident and sharded MSM entry points (a one-rank communicator still runs pack -> ncclAllGather ->
# fold), a mid-size MSM (short slices + the parallel bucket fold), back-to-back calls on two streams
import torch
dk, dp = torch.from_numpy(wm["k32"]).cuda(), torch.from_numpy(wm["pt65"]).cuda()
eng.msm(dk, dp)
eng.comm_init(pkg.Engine.comm_unique_id(), 0, 1)
eng.msm_sharded(wm["k32"], wm["pt65"]); eng.msm_sharded(dk, dp)
eng.comm_free()
s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
d = [torch.from_numpy(w[k]).cuda() for k in ("pk65", "digest32", "sig64")]
with torch.cuda.stream(s1):
    a = eng.ecdsa_verify(*d)
with torch.cuda.stream(s2):
    b = eng.ecdsa_verify(*d)
torch.cuda.synchronize()
assert np.array_equal(a.cpu().numpy(), w["expected"]) and np.array_equal(b.cpu().numpy(), w["expected"])
# the device-resident DER entry points (misaligned rows: the parse reads byte by byte)
for rows in (pkg.build_asn1_signatures(w["sig64"]), [r + b"\x01" for r in pkg.build_asn1_signatures(w["sig64"])]):
    flat, offs = pkg.ragged_rows(rows)
    dflat = torch.zeros(len(flat) + 1, dtype=torch.uint8, device="cuda")
    dflat[1:] = torch.from_numpy(flat.copy()).cuda()
    dd = (dflat, torch.from_numpy(offs.astype(np.int64) + 1).cuda())
    eng.ecdsa_verify_asn1(d[0], d[1], dd)
    eng.bitcoin_verify_asn1(d[0], d[1], dd)
    eng.parse_asn1_signatures_dev(dd)
    eng.is_valid_signature_encoding_bip0066_dev(dd)
torch.cuda.synchronize()
eng.close()
mid = pkg.Engine(device=0, max_batch=1 << 16)
wmid = pkg.synth.msm_batch(1 << 16, mid.scalar_base_mult)
mid.msm(wmid["k32"], wmid["pt65"])
mid.close()
if os.environ.get("SANITIZE_BIG", "1") == "1":
    # the three-part host pipeline of ecdsa_verify and the four-part one of the other entry points
    n = 1 << 18
    big = pkg.Engine(device=0, max_batch=n)
    w = pkg.synth.ecdsa_batch(n, big.scalar_base_mult)
    assert np.array_equal(big.ecdsa_verify(w["pk65"], w["digest32"], w["sig64"]), w["expected"])
    big.close()
print("sanitize_all ok")
