// Host build of the prover's scalar code (kzg_quotient.cuh: the quotient with its batch inversion and in-domain branch;
// msm.cuh: the signed-digit recoding) for tests/test_kzg_prover_host.py: the same source the kernels compile, checked
// against Python ints.  Field elements cross the boundary as 32-byte big-endian canonical integers.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../ethereum_consensus_b200/csrc/kzg_quotient.cuh"
#include "../../ethereum_consensus_b200/csrc/msm.cuh"

using namespace b200;

#define HK_API extern "C" __attribute__((visibility("default")))

static Fr in_mont(const uint8_t* be) {
    Fr raw, m;
    fr_from_be32_raw(raw, be);
    fr_to_mont(m, raw);
    return m;
}
static void out_canon(uint8_t* be, const Fr& raw) {   // canonical limbs -> 32 big-endian bytes
    for (int i = 0; i < 8; i++) {
        uint8_t* p = be + 28 - 4 * i;
        p[0] = uint8_t(raw.l[i] >> 24); p[1] = uint8_t(raw.l[i] >> 16); p[2] = uint8_t(raw.l[i] >> 8); p[3] = uint8_t(raw.l[i]);
    }
}

// The quotient of a 131 072-byte blob at z with y = p(z) given, split over `parts` interleaved threads (element i to
// thread i % parts) exactly as k_kzg_quotient splits it over its CTA; q_out: 4 096 x 32 big-endian bytes.
HK_API void hk_quotient(const uint8_t* blob, const uint8_t* z_be, const uint8_t* y_be, uint32_t parts, uint8_t* q_out) {
    const Fr z = in_mont(z_be), y = in_mont(y_be);
    std::vector<Fr> roots(kBlobElems), q(kBlobElems), prod(parts), inv(parts);
    for (uint32_t i = 0; i < kBlobElems; i++) roots[i] = kzg_root_brp(i);
    int32_t dom = -1;
    const uint32_t cnt = kBlobElems / parts;
    for (uint32_t t = 0; t < parts; t++) prod[t] = quot_prefix(q.data(), roots.data(), z, t, parts, cnt, dom);
    // the CTA's step: one inversion of the product of all, then each thread's inverse from the others' products
    Fr all = fr_one(), inv_all;
    for (uint32_t t = 0; t < parts; t++) fr_mul(all, all, prod[t]);
    fr_inv(inv_all, all);
    for (uint32_t t = 0; t < parts; t++) {
        inv[t] = inv_all;
        for (uint32_t u = 0; u < parts; u++)
            if (u != t) fr_mul(inv[t], inv[t], prod[u]);
    }
    Fr sum = fr_zero();
    for (uint32_t t = 0; t < parts; t++) {
        const Fr s = quot_finish(q.data(), blob, roots.data(), z, y, inv[t], t, parts, cnt, dom >= 0);
        fr_add(sum, sum, s);
    }
    if (dom >= 0) q[dom] = quot_within_domain(sum, roots.data(), uint32_t(dom));
    for (uint32_t i = 0; i < kBlobElems; i++) out_canon(q_out + 32 * i, q[i]);
}

HK_API uint32_t hk_inv_root_index(uint32_t m) { return kzg_inv_root_index(m); }

// the signed digits of a canonical scalar (32 big-endian bytes), kMsmWindows of them; returns the final carry
HK_API uint32_t hk_digits(const uint8_t* s_be, int32_t* digits) {
    Fr raw;
    fr_from_be32_raw(raw, s_be);
    uint32_t k[8], carry = 0;
    for (int j = 0; j < 8; j++) k[j] = raw.l[j];
    for (int w = 0; w < kMsmWindows; w++) digits[w] = msm_next_digit(k, carry);
    return carry;
}

HK_API int hk_msm_params(int32_t* out) {
    out[0] = kMsmC; out[1] = kMsmWindows; out[2] = kMsmMaxDigit; out[3] = kMsmGroups;
    return 4;
}
