// jac.cuh -- Jacobian-coordinate group law (x = X / Z^2, y = Y / Z^3) for the VARIABLE-TIME ladders only.
//
// Every function is a template over the field-operation set F, passed as an object (fe_ops<VT> of fe_vt.cuh).
//
// The reference runs every path on the Renes-Costello-Batina complete formulas (point_projective.go:24-273), and so do
// the constant-time kernels and the Point API here (point.cuh).  The verification ladder
// (DoubleScalarMultBasepointVartime, point_mul_glv.go:307-317) handles public data, is variable time in the reference
// too, and only its affine result is observable -- so its 125 doublings may use the a = 0 Jacobian doubling
// (2 M + 5 S = 371 MAC32 against 519 for Algorithm 9) and its additions the mixed Jacobian addition against an AFFINE
// per-item table (6 M + 3 S + one fused pair = 710 against 849 for Algorithm 7).  These formulas are incomplete; the
// exceptional cases the complete formulas absorb are handled explicitly, by branches (public data):
//   * accumulator at infinity          -> a flag kept by the caller; the addition becomes an assignment
//   * addend == accumulator (H = R = 0) -> the doubling
//   * addend == -accumulator (H = 0)    -> the flag is set
//   * doubling of a point with Y = 0    -> cannot occur (no 2-torsion on a prime-order curve)
// SURVEY.md section 6 names the Wycheproof groups that exercise them (PointDuplication, EdgeCaseShamirMultiplication,
// ArithmeticError); tests/parity_suites.py runs them plus crafted u1 G = +-u2 P rows against the oracle.
#pragma once
#include "point.cuh"

namespace s256 {

// v = 2p (a = 0).  p must not be at infinity for the result to mean anything; (0, 0, 0) maps to itself.
template <class F>
S256_HD void jac_double(F &fo, pt &v, const pt &p) {
    fe a, b, c, d, e, f, t, z3;
    fo.sqr(a, p.x);
    fo.sqr(b, p.y);
    fo.sqr(c, b);
#ifndef S256_JDBL_3M4S
    fo.add(t, p.x, b);  // D = 2 ((X + B)^2 - A - C)
    fo.sqr(t, t);
    fo.sub(t, t, a);
    fo.sub(t, t, c);
    fo.mul2(d, t);
#else
    fo.mul(t, p.x, b);  // D = 4 X B
    fo.mul2(t, t);
    fo.mul2(d, t);
#endif
    fo.mul3(e, a);  // E = 3 A
    fo.sqr(f, e);
    fo.mul(z3, p.y, p.z);
    fo.mul2(v.z, z3);
    fo.sub2(t, f, d);  // X3 = F - 2 D
    v.x = t;
    fo.sub(t, d, t);
    fo.mul(f, e, t);  // Y3 = E (D - X3) - 8 C
    fo.submul8(v.y, f, c);
}
// v = p + (x2, y2) for a finite p whose sum with the addend is known not to be exceptional (the constant-time
// fixed-base accumulation, whose argument is given where it is used).
template <class F>
S256_HD void jac_add_mixed_nocheck(F &fo, pt &v, const pt &p, const fe &x2, const fe &y2) {
    fe zz, u2, s2, h, r, hh, hhh, w, t, x3;
    fo.sqr(zz, p.z);
    fo.mul(u2, x2, zz);
    fo.mul(s2, y2, p.z);
    fo.mul(s2, s2, zz);
    fo.sub(h, u2, p.x);
    fo.sub(r, s2, p.y);
    fo.sqr(hh, h);
    fo.mul(hhh, h, hh);
    fo.mul(w, p.x, hh);
    fo.mul(v.z, p.z, h);
    fo.sqr(x3, r);
    fo.sub(x3, x3, hhh);
    fo.sub2(x3, x3, w);
    fo.sub(t, w, x3);
    fo.mul2sub(v.y, r, t, p.y, hhh);
    v.x = x3;
}

// Co-Z formulas (Meloni 2007; Goundar, Joye, Miyaji 2011) for chains of consecutive multiples: two points kept at ONE
// shared Z, which neither formula computes -- the caller follows it through the returned ratio.
//
// DBLU from an affine point P = (x, y): (x2, y2) = 2P at Z = 2y, and (x1, y1) = P at that same Z, (4 x y^2, 8 y^4),
// which the doubling produces on the way: 1 M + 5 S.  2y != 0: there is no 2-torsion on a curve of prime order.
template <class F>
S256_HD void jac_dblu(F &fo, fe &x2, fe &y2, fe &x1, fe &y1, const fe &x, const fe &y) {
    fe a, b, c, d, e, t;
    fo.sqr(a, x);
    fo.sqr(b, y);
    fo.sqr(c, b);
    fo.add(t, x, b);  // D = 2 ((x + B)^2 - A - C) = 4 x B
    fo.sqr(t, t);
    fo.sub(t, t, a);
    fo.sub(t, t, c);
    fo.mul2(d, t);
    fo.mul3(e, a);  // E = 3 A
    fo.sqr(t, e);
    fo.sub2(x2, t, d);  // X = E^2 - 2 D
    fo.sub(t, d, x2);
    fo.mul(a, e, t);
    fo.submul8(y2, a, c);  // Y = E (D - X) - 8 C
    x1 = d;
    fo.mul8(y1, c);
}
// ZADDU: for P = (x1, y1) and Q = (x2, y2) at one shared Z, Q becomes P + Q and P becomes P again, both at the Z of the
// sum, which is Z u with u = x1 - x2 (returned): 4 M + 2 S.  Not for P = +-Q (u = 0) nor for either at infinity.
template <class F>
S256_HD void jac_zaddu(F &fo, fe &x1, fe &y1, fe &x2, fe &y2, fe &u) {
    fe c, w1, w2, r, t;
    fo.sub(u, x1, x2);
    fo.sqr(c, u);
    fo.mul(w1, x1, c);  // W1 = X1 C
    fo.mul(w2, x2, c);  // W2 = X2 C
    fo.sub(r, y1, y2);
    fo.sub(t, w1, w2);
    fo.mul(y1, y1, t);  // A1 = Y1 (W1 - W2)
    fo.sqr(t, r);
    fo.sub(t, t, w1);
    fo.sub(x2, t, w2);  // X3 = (Y1 - Y2)^2 - W1 - W2
    fo.sub(t, w1, x2);
    fo.mul(c, r, t);
    fo.sub(y2, c, y1);  // Y3 = (Y1 - Y2) (W1 - X3) - A1
    x1 = w1;
}

// acc += (x2, y2), every case handled; inf is the caller's "accumulator is the identity" flag.
template <class F>
S256_HD void jac_add_mixed_var(F &fo, pt &acc, uint32_t &inf, const fe &x2, const fe &y2) {
    if (inf) {
        acc.x = x2;
        acc.y = y2;
        acc.z = fe_one();
        inf = 0u;
        return;
    }
    fe zz, u2, s2, h, r, hh, hhh, w, t, x3;
    fo.sqr(zz, acc.z);
    fo.mul(u2, x2, zz);
    fo.mul(s2, y2, acc.z);
    fo.mul(s2, s2, zz);
    fo.sub(h, u2, acc.x);
    fo.sub(r, s2, acc.y);
    if (fe_is_zero(h)) {
        if (!fe_is_zero(r)) {
            inf = 1u;
            acc.x = acc.y = acc.z = fe_zero();  // (see item_dsm_ladder: zero coordinates under the flag)
        } else {
            jac_double(fo, acc, acc);
        }
        return;
    }
    fo.sqr(hh, h);
    fo.mul(hhh, h, hh);
    fo.mul(w, acc.x, hh);
    fo.mul(acc.z, acc.z, h);
    fo.sqr(x3, r);
    fo.sub(x3, x3, hhh);
    fo.sub2(x3, x3, w);
    fo.sub(t, w, x3);
    fo.mul2sub(acc.y, r, t, acc.y, hhh);
    acc.x = x3;
}

// Jacobian -> the homogeneous projective form every consumer of the ladder's result expects: (X Z : Y : Z^3)
template <class F>
S256_HD void jac_to_projective(F &fo, pt &v, const pt &p, uint32_t inf) {
    if (inf) {
        pt_set_identity(v);
        return;
    }
    fe zz;
    fo.sqr(zz, p.z);
    fo.mul(v.x, p.x, p.z);
    v.y = p.y;
    fo.mul(v.z, zz, p.z);
}

}  // namespace s256
