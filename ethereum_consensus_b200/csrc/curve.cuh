// Short-Weierstrass (a = 0) point arithmetic in Jacobian coordinates, generic over the coordinate field:
// F = Fp gives E(Fp): y^2 = x^3 + 4 (G1, public keys); F = Fp2 gives the twist E'(Fp2): y^2 = x^3 + 4(1+u)
// (G2, signatures and hashed messages).  Infinity <=> Z == 0.
#pragma once
#include "fp2.cuh"

namespace b200 {

// uniform names over Fp / Fp2
B200_HD void f_add(Fp& r, const Fp& a, const Fp& b) { fp_add(r, a, b); }
B200_HD void f_sub(Fp& r, const Fp& a, const Fp& b) { fp_sub(r, a, b); }
B200_HD void f_mul(Fp& r, const Fp& a, const Fp& b) { fp_mul(r, a, b); }
B200_HD void f_sqr(Fp& r, const Fp& a) { fp_sqr(r, a); }
B200_HD void f_neg(Fp& r, const Fp& a) { fp_neg(r, a); }
B200_HD void f_dbl(Fp& r, const Fp& a) { fp_dbl(r, a); }
B200_HD void f_inv(Fp& r, const Fp& a) { fp_inv(r, a); }
B200_HD bool f_is_zero(const Fp& a) { return fp_is_zero(a); }
B200_HD bool f_eq(const Fp& a, const Fp& b) { return fp_eq(a, b); }
B200_HD void f_add(Fp2& r, const Fp2& a, const Fp2& b) { fp2_add(r, a, b); }
B200_HD void f_sub(Fp2& r, const Fp2& a, const Fp2& b) { fp2_sub(r, a, b); }
B200_HD void f_mul(Fp2& r, const Fp2& a, const Fp2& b) { fp2_mul(r, a, b); }
B200_HD void f_sqr(Fp2& r, const Fp2& a) { fp2_sqr(r, a); }
B200_HD void f_neg(Fp2& r, const Fp2& a) { fp2_neg(r, a); }
B200_HD void f_dbl(Fp2& r, const Fp2& a) { fp2_dbl(r, a); }
B200_HD void f_inv(Fp2& r, const Fp2& a) { fp2_inv(r, a); }
B200_HD bool f_is_zero(const Fp2& a) { return fp2_is_zero(a); }
B200_HD bool f_eq(const Fp2& a, const Fp2& b) { return fp2_eq(a, b); }
template <class F> B200_HD F f_one();
template <> B200_HD Fp f_one<Fp>() { return fp_one(); }
template <> B200_HD Fp2 f_one<Fp2>() { return fp2_one(); }
template <class F> B200_HD F f_zero();
template <> B200_HD Fp f_zero<Fp>() { return fp_zero(); }
template <> B200_HD Fp2 f_zero<Fp2>() { return fp2_zero(); }
template <class F> B200_HD F curve_b();
template <> B200_HD Fp curve_b<Fp>() { Fp b = B200_FP_B_G1; return b; }
template <> B200_HD Fp2 curve_b<Fp2>() { Fp2 b = B200_FP2_B_G2; return b; }

template <class F>
struct Aff {
    F x, y;
    uint32_t inf;  // 1 = point at infinity (x, y ignored)
};
template <class F>
struct Jac {
    F x, y, z;
};

template <class F> B200_HD bool jac_is_inf(const Jac<F>& p) { return f_is_zero(p.z); }
template <class F> B200_HD void jac_set_inf(Jac<F>& p) { p.x = f_one<F>(); p.y = f_one<F>(); p.z = f_zero<F>(); }
template <class F> B200_HD void jac_from_aff(Jac<F>& p, const Aff<F>& a) {
    if (a.inf) { jac_set_inf(p); return; }
    p.x = a.x; p.y = a.y; p.z = f_one<F>();
}
template <class F> B200_HD void jac_neg(Jac<F>& r, const Jac<F>& p) { r.x = p.x; f_neg(r.y, p.y); r.z = p.z; }

// y^2 == x^3 + b
template <class F> B200_HD bool aff_on_curve(const F& x, const F& y) {
    F l, r;
    f_sqr(l, y);
    f_sqr(r, x);
    f_mul(r, r, x);
    const F b = curve_b<F>();
    f_add(r, r, b);
    return f_eq(l, r);
}

// dbl-2009-l (a = 0): 2M + 5S
template <class F> B200_BIG void jac_double(Jac<F>& r, const Jac<F>& p) {
    F A, B, C, D, E, Fq, t;
    f_sqr(A, p.x);
    f_sqr(B, p.y);
    f_sqr(C, B);
    f_add(t, p.x, B);
    f_sqr(t, t);
    f_sub(t, t, A);
    f_sub(t, t, C);
    f_dbl(D, t);
    f_dbl(E, A);
    f_add(E, E, A);
    f_sqr(Fq, E);
    F z3;
    f_mul(z3, p.y, p.z);
    f_dbl(z3, z3);
    F x3;
    f_dbl(t, D);
    f_sub(x3, Fq, t);
    f_sub(t, D, x3);
    f_mul(t, E, t);
    f_dbl(C, C); f_dbl(C, C); f_dbl(C, C);
    f_sub(r.y, t, C);
    r.x = x3;
    r.z = z3;
}

// r = p + q, q affine and not infinity.  Handles p = inf, p = q (doubling) and p = -q.
// Optionally returns the pieces the Miller loop needs: Rr = y2*Z^3 - Y and the new Z (= Z*H), see pairing.cuh.
template <class F> B200_BIG void jac_add_mixed(Jac<F>& r, const Jac<F>& p, const F& qx, const F& qy) {
    if (jac_is_inf(p)) { r.x = qx; r.y = qy; r.z = f_one<F>(); return; }
    F zz, zzz, u2, s2, h, rr;
    f_sqr(zz, p.z);
    f_mul(zzz, zz, p.z);
    f_mul(u2, qx, zz);
    f_mul(s2, qy, zzz);
    f_sub(h, u2, p.x);
    f_sub(rr, s2, p.y);
    if (f_is_zero(h)) {
        if (f_is_zero(rr)) { Jac<F> t; t.x = qx; t.y = qy; t.z = f_one<F>(); jac_double(r, t); }
        else jac_set_inf(r);
        return;
    }
    F hh, hhh, v, x3, t;
    f_sqr(hh, h);
    f_mul(hhh, hh, h);
    f_mul(v, p.x, hh);
    f_sqr(x3, rr);
    f_sub(x3, x3, hhh);
    f_dbl(t, v);
    f_sub(x3, x3, t);
    f_sub(t, v, x3);
    f_mul(t, rr, t);
    F y1h;
    f_mul(y1h, p.y, hhh);
    f_sub(r.y, t, y1h);
    f_mul(r.z, p.z, h);
    r.x = x3;
}

// general Jacobian addition (handles infinity, doubling, inverse)
template <class F> B200_BIG void jac_add(Jac<F>& r, const Jac<F>& p, const Jac<F>& q) {
    if (jac_is_inf(p)) { r = q; return; }
    if (jac_is_inf(q)) { r = p; return; }
    F z1z1, z2z2, u1, u2, s1, s2, h, rr, t;
    f_sqr(z1z1, p.z);
    f_sqr(z2z2, q.z);
    f_mul(u1, p.x, z2z2);
    f_mul(u2, q.x, z1z1);
    f_mul(t, q.z, z2z2);
    f_mul(s1, p.y, t);
    f_mul(t, p.z, z1z1);
    f_mul(s2, q.y, t);
    f_sub(h, u2, u1);
    f_sub(rr, s2, s1);
    if (f_is_zero(h)) {
        if (f_is_zero(rr)) jac_double(r, p); else jac_set_inf(r);
        return;
    }
    F hh, hhh, v, x3;
    f_sqr(hh, h);
    f_mul(hhh, hh, h);
    f_mul(v, u1, hh);
    f_sqr(x3, rr);
    f_sub(x3, x3, hhh);
    f_dbl(t, v);
    f_sub(x3, x3, t);
    f_sub(t, v, x3);
    f_mul(t, rr, t);
    f_mul(s1, s1, hhh);
    f_sub(r.y, t, s1);
    f_mul(t, p.z, q.z);
    f_mul(r.z, t, h);
    r.x = x3;
}

template <class F> B200_BIG void jac_to_aff(Aff<F>& a, const Jac<F>& p) {
    if (jac_is_inf(p)) { a.inf = 1; a.x = f_zero<F>(); a.y = f_zero<F>(); return; }
    F zi, zi2, zi3;
    f_inv(zi, p.z);
    f_sqr(zi2, zi);
    f_mul(zi3, zi2, zi);
    f_mul(a.x, p.x, zi2);
    f_mul(a.y, p.y, zi3);
    a.inf = 0;
}

// equality of a Jacobian point with an affine one (neither at infinity unless flagged)
template <class F> B200_HD bool jac_eq_aff(const Jac<F>& p, const F& qx, const F& qy) {
    if (jac_is_inf(p)) return false;
    F zz, zzz, a, b;
    f_sqr(zz, p.z);
    f_mul(zzz, zz, p.z);
    f_mul(a, qx, zz);
    f_mul(b, qy, zzz);
    return f_eq(a, p.x) && f_eq(b, p.y);
}

// r = [k] * (qx, qy) for a 64-bit scalar, left-to-right double-and-add (k != 0)
template <class F> B200_BIG void jac_mul_u64(Jac<F>& r, const F& qx, const F& qy, uint64_t k) {
    Jac<F> acc;
    jac_set_inf(acc);
    bool started = false;
#pragma unroll 1
    for (int bit = 63; bit >= 0; bit--) {
        if (started) jac_double(acc, acc);
        if ((k >> bit) & 1) {
            jac_add_mixed(acc, acc, qx, qy);
            started = true;
        }
    }
    r = acc;
}
// r = [k] * (qx, qy) for a 256-bit scalar given as 8 little-endian 32-bit limbs, left-to-right double-and-add over all
// 256 bits (k = 0 gives infinity; doubling infinity keeps Z = 0).  The scalar is shifted out of the top limb, so it stays
// in registers (no dynamically indexed limb array).
template <class F> B200_BIG void jac_mul_u256(Jac<F>& r, const F& qx, const F& qy, const uint32_t k_in[8]) {
    uint32_t k[8];
#pragma unroll
    for (int i = 0; i < 8; i++) k[i] = k_in[i];
    Jac<F> acc;
    jac_set_inf(acc);
#pragma unroll 1
    for (int bit = 0; bit < 256; bit++) {
        jac_double(acc, acc);
        if (k[7] >> 31) jac_add_mixed(acc, acc, qx, qy);
#pragma unroll
        for (int i = 7; i > 0; i--) k[i] = (k[i] << 1) | (k[i - 1] >> 31);
        k[0] <<= 1;
    }
    r = acc;
}
// same for a Jacobian base point
template <class F> B200_BIG void jac_mul_u64_jac(Jac<F>& r, const Jac<F>& q, uint64_t k) {
    Jac<F> acc;
    jac_set_inf(acc);
    bool started = false;
#pragma unroll 1
    for (int bit = 63; bit >= 0; bit--) {
        if (started) jac_double(acc, acc);
        if ((k >> bit) & 1) {
            jac_add(acc, acc, q);
            started = true;
        }
    }
    r = acc;
}

}  // namespace b200
