// The KZG quotient in evaluation form (compute_kzg_proof_impl of the deneb polynomial-commitments spec), host + device
// (the CTA layout is in kzg_prove.cu; tests/host_math/host_kzg_prover.cpp runs the same functions on the host):
//
//   q_i = (f_i - y) / (w_i - z)                               for w_i != z
//   q_m = sum_(i != m) (f_i - y) w_i / (z (z - w_i))          for w_m == z  (compute_quotient_eval_within_domain)
//       = -(1/z) sum_(i != m) q_i w_i
//
// The 4 096 denominators are inverted together (Montgomery's trick): each thread walks its elements once forward, storing
// the running product of the denominators before each element in q[i] and returning the thread's product; the CTA inverts
// the product of all of them with one fr_inv and hands each thread the inverse of its own product; the backward walk then
// peels one inverse per element off it.  1/z on the domain is itself a root of unity: w^-j = w^(4096 - j).
#pragma once
#include "kzg_eval.cuh"

namespace b200 {

B200_HD uint32_t kzg_brp12(uint32_t i) {
    uint32_t rev = 0;
    for (int b = 0; b < 12; b++) rev |= ((i >> b) & 1u) << (11 - b);
    return rev;
}
// the bit-reversed index of 1 / w_m (w_m the m-th entry of the bit-reversed domain)
B200_HD uint32_t kzg_inv_root_index(uint32_t m) { return kzg_brp12((kBlobElems - kzg_brp12(m)) & (kBlobElems - 1)); }

// Forward walk over i = first + k * stride, k < cnt: q[i] = prod of the earlier denominators (Montgomery form); returns the
// product of all of them.  The denominator w_i - z is zero at most once per blob (z on the domain): it counts as one and
// its index goes to dom.
B200_HD Fr quot_prefix(Fr* q, const Fr* roots, const Fr& z, uint32_t first, uint32_t stride, uint32_t cnt, int32_t& dom) {
    Fr acc = fr_one();
    for (uint32_t k = 0; k < cnt; k++) {
        const uint32_t i = first + k * stride;
        Fr d;
        fr_sub(d, roots[i], z);
        q[i] = acc;
        if (fr_is_zero(d)) dom = int32_t(i);
        else fr_mul(acc, acc, d);
    }
    return acc;
}

// Backward walk over the same elements with inv = 1 / (the forward walk's product): q[i] = q_i as canonical limbs (the MSM's
// scalars), q[dom] = 0 for now.  f_i are read from the blob (32 big-endian bytes each, already checked < r).  With
// in_domain, returns sum q_i w_i over these elements (Montgomery form), else zero.
B200_HD Fr quot_finish(Fr* q, const uint8_t* blob, const Fr* roots, const Fr& z, const Fr& y, Fr inv, uint32_t first,
                       uint32_t stride, uint32_t cnt, bool in_domain) {
    Fr sum = fr_zero();
    for (uint32_t k = cnt; k-- > 0;) {
        const uint32_t i = first + k * stride;
        Fr d;
        fr_sub(d, roots[i], z);
        if (fr_is_zero(d)) { q[i] = fr_zero(); continue; }
        Fr inv_d, raw, f, qi;
        fr_mul(inv_d, inv, q[i]);
        fr_mul(inv, inv, d);
        fr_from_be32_raw(raw, blob + 32 * size_t(i));
        fr_to_mont(f, raw);
        fr_sub(f, f, y);
        fr_mul(qi, f, inv_d);
        if (in_domain) {
            Fr t;
            fr_mul(t, qi, roots[i]);
            fr_add(sum, sum, t);
        }
        fr_from_mont(q[i], qi);
    }
    return sum;
}

// q_m from sum_(i != m) q_i w_i, as canonical limbs
B200_HD Fr quot_within_domain(const Fr& sum_qw, const Fr* roots, uint32_t m) {
    Fr t, out;
    fr_mul(t, sum_qw, roots[kzg_inv_root_index(m)]);
    fr_neg(t, t);
    fr_from_mont(out, t);
    return out;
}

}  // namespace b200
