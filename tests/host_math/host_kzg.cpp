// Host build of the KZG scalar-field code (fr.cuh, kzg_eval.cuh) for tests/test_kzg_host.py: the same source the kernels
// compile, checked against Python ints.  Field elements cross the boundary as 32-byte big-endian canonical integers.
#include <cstdint>
#include <cstring>

#include "../../ethereum_consensus_b200/csrc/kzg_eval.cuh"

using namespace b200;

#define HK_API extern "C" __attribute__((visibility("default")))

static Fr in_mont(const uint8_t* be) {
    Fr raw, m;
    fr_from_be32_raw(raw, be);
    fr_to_mont(m, raw);
    return m;
}

// op: 0 a*b, 1 a^2, 2 a^-1, 3 a+b, 4 a-b, 5 -a; inputs must be < r
HK_API void hk_fr_op(int op, const uint8_t* a_be, const uint8_t* b_be, uint8_t* out_be) {
    const Fr a = in_mont(a_be), b = in_mont(b_be);
    Fr r;
    switch (op) {
    case 0: fr_mul(r, a, b); break;
    case 1: fr_sqr(r, a); break;
    case 2: fr_inv(r, a); break;
    case 3: fr_add(r, a, b); break;
    case 4: fr_sub(r, a, b); break;
    default: fr_neg(r, a); break;
    }
    fr_to_be32(out_be, r);
}

// bytes_to_bls_field: 1 if the 32 big-endian bytes are < r (out = the same value after a Montgomery round trip)
HK_API int hk_fr_from_be32(const uint8_t* be, uint8_t* out_be) {
    Fr m;
    if (!fr_from_be32(m, be)) return 0;
    fr_to_be32(out_be, m);
    return 1;
}

// hash_to_bls_field of a digest: the 256-bit big-endian integer mod r
HK_API void hk_fr_reduce(const uint8_t* be, uint8_t* out_be) {
    Fr raw, m;
    fr_from_be32_raw(raw, be);
    fr_from_u256_reduce(m, raw);
    fr_to_be32(out_be, m);
}

HK_API void hk_root_brp(uint32_t i, uint8_t* out_be) { fr_to_be32(out_be, kzg_root_brp(i)); }

// evaluate_polynomial_in_evaluation_form over a 131 072-byte blob at z, with the fraction folding of the CTA kernel done in
// `parts` interleaved partial fractions (thread i % parts) and then folded together, as the kernel does; 17 on an element >= r
HK_API int hk_eval(const uint8_t* blob, const uint8_t* z_be, uint32_t parts, uint8_t* y_out) {
    const Fr z = in_mont(z_be);
    Frac acc[256];
    for (uint32_t p = 0; p < parts; p++) acc[p] = frac_zero();
    int dom = -1;
    Fr fdom = fr_zero();
    for (uint32_t i = 0; i < kBlobElems; i++) {
        Fr f;
        if (!fr_from_be32(f, blob + 32 * i)) return 17;
        if (!frac_push(acc[i % parts], f, kzg_root_brp(i), z)) { dom = int(i); fdom = f; }
    }
    for (uint32_t p = 1; p < parts; p++) frac_add(acc[0], acc[p]);
    fr_to_be32(y_out, dom >= 0 ? fdom : kzg_eval_finish(acc[0]));
    return 0;
}
