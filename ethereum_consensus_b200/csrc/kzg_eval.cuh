// evaluate_polynomial_in_evaluation_form as fraction folding (host + device; the CTA layout is in kzg.cu).
//
//   y = (z^N - 1) / N * sum_i f_i w_i / (z - w_i)      (w_i: the N = 4 096 roots of unity, bit-reversed order)
//
// The terms are summed as one fraction num / den: a term a / d folds in as num <- num d + a den, den <- den d (three
// products, no inverse), two partial fractions the same way.  Over the whole domain den = prod_i (z - w_i) = z^N - 1, which
// cancels the spec's factor: y = num / N.  A term with z == w_i is the spec's in-domain branch (y = f_i) and is not folded.
#pragma once
#include "fr.cuh"

namespace b200 {

constexpr uint32_t kBlobElems = 4096;

struct Frac {
    Fr n, d;
};
B200_HD Frac frac_zero() { Frac r; r.n = fr_zero(); r.d = fr_one(); return r; }
B200_HD void frac_add(Frac& a, const Frac& b) {
    Fr t0, t1;
    fr_mul(t0, a.n, b.d);
    fr_mul(t1, b.n, a.d);
    fr_add(a.n, t0, t1);
    fr_mul(a.d, a.d, b.d);
}
// folds f w / (z - w) into acc; false (nothing folded) when z == w
B200_HD bool frac_push(Frac& acc, const Fr& f, const Fr& w, const Fr& z) {
    Fr d, a, t0;
    fr_sub(d, z, w);
    if (fr_is_zero(d)) return false;
    fr_mul(a, f, w);
    fr_mul(t0, acc.n, d);
    fr_mul(a, a, acc.d);
    fr_add(acc.n, t0, a);
    fr_mul(acc.d, acc.d, d);
    return true;
}
// y from the fraction over the whole domain
B200_HD Fr kzg_eval_finish(const Frac& acc) {
    const Fr inv_n = B200_FR_INV_4096;
    Fr y;
    fr_mul(y, acc.n, inv_n);
    return y;
}
// w^brp(i): the i-th entry of the bit-reversed domain
B200_HD Fr kzg_root_brp(uint32_t i) {
    uint32_t rev = 0;
    for (int b = 0; b < 12; b++) rev |= ((i >> b) & 1u) << (11 - b);
    Fr e = fr_zero();
    e.l[0] = rev;
    const Fr w = B200_FR_OMEGA_4096;
    Fr r;
    fr_pow(r, w, e);
    return r;
}

}  // namespace b200
