// The device-resident KZG settings and the pieces of the verification pipeline (kzg.cu) that the prover (kzg_prove.cu)
// runs unchanged.  Internal to the library.
#pragma once
#include <cuda_runtime.h>

#include "bls_kernels.cuh"
#include "engine.h"
#include "kzg_eval.cuh"

namespace b200 {
struct MsmAff;   // msm.cuh
}

struct b200_kzg_settings {
    b200::G2Aff* d_g2 = nullptr;   // [0] = -G2 (the generator, negated), [1] = [tau]G2 = g2_monomial[1]
    b200::Fr* d_roots = nullptr;   // the 4 096 roots of unity in bit-reversed order, Montgomery form
    // the prover's fixed bases (msm.cuh): entry (w, i, j) = [(j + 1) 2^(c w)] g1_lagrange[reverse_bits(i)], affine
    b200::MsmAff* d_table = nullptr;
    uint8_t* d_base_inf = nullptr;   // [i] = 1 when g1_lagrange[reverse_bits(i)] is the point at infinity
};

namespace b200 {

// kzg.cu: z = compute_challenge(blob, C) per blob (one thread per blob)
void launch_kzg_challenge(const uint8_t* blobs, const uint8_t* comms, uint32_t n, Fr* z, cudaStream_t s);
// kzg.cu: y = p(z) per blob (one CTA per blob); codes[b] = B200_KZG_BAD_ARGS for an element >= r, else 0
void launch_kzg_eval(const uint8_t* blobs, const Fr* zs, const Fr* roots, Fr* ys, int32_t* codes, uint32_t n, cudaStream_t s);
// kzg_prove.cu: builds the MSM table of a settings object from the decoded g1_lagrange points (natural order) and their
// K1 codes; synchronous
int32_t kzg_prover_settings_build(Engine& e, b200_kzg_settings* st, const G1Aff* g1, const int32_t* g1_codes);

}  // namespace b200
