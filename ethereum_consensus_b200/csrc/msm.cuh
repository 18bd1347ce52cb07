// Fixed-base multi-scalar multiplication over G1: sum_i [s_i] B_i for the 4 096 KZG bases (the prover's hot path,
// kzg_prove.cu).
//
// Signed-digit comb over a table built once per settings object (k_msm_table, at load time):
//   s = sum_w d_w 2^(c w),  d_w in [-2^(c-1), 2^(c-1)]  (c = 5: 52 windows cover s < 2^255 plus the recoding carry)
//   sum_i [s_i] B_i = sum_i sum_w [d_(i,w)] T_(w,i),   T_(w,i) = [2^(c w)] B_i
// With [j] T_(w,i) for j = 1..16 resident as affine points, every term is one table lookup (y negated for d < 0) and one
// mixed addition: no doublings and no buckets, so the work spreads over any number of threads with nothing to sort.
// Per blob the kernel runs 4 096 x kMsmGroups threads (base i, a contiguous group of windows); each folds its terms with
// jac_add_mixed, and the partial sums are reduced by CTA trees (jac_add).  Both formulas handle the point at infinity,
// P + P and P + (-P), so the sum is exact for every input; an infinite base is skipped (its flag in base_inf).
//
// Work per blob, uniform scalars: 4 096 x 51 x 31/32 + 4 096 x 1/32 ~ 203 k mixed additions (11 Fp products each) and
// 8 191 + 63 Jacobian additions (16 each) in the trees: ~2.37 M Fp products (tools/bench_kzg.py computes the exact count).
// Table: 52 x 4 096 x 16 affine points x 96 bytes = 327 MB per settings object.
//
// The digit recoding is host + device (tests/host_math/host_kzg_prover.cpp checks it); the kernels are device only.
#pragma once
#include "fr.cuh"
#include "groups.cuh"

namespace b200 {

constexpr uint32_t kMsmBases = 4096;
constexpr int kMsmC = 5;                       // window width in bits
constexpr int kMsmWindows = 52;                // ceil(256 / 5): s < 2^255 and the final carry fit
constexpr int kMsmMaxDigit = 1 << (kMsmC - 1); // 16: table entries per (window, base)
constexpr int kMsmGroups = 2;                  // window groups per base: threads per blob = 4 096 x 2
constexpr int kMsmThreads = 128;               // threads per CTA of k_msm_partial
constexpr int kMsmCtasPerBlob = int(kMsmBases) * kMsmGroups / kMsmThreads;   // 64 partial sums per blob
constexpr int kMsmWindowsPerGroup = kMsmWindows / kMsmGroups;
static_assert(kMsmWindows % kMsmGroups == 0, "window groups must split the windows evenly");

struct alignas(16) MsmAff {
    Fp x, y;
};

// The next signed digit of k (little-endian canonical limbs), shifted out of k: raw = low c bits + carry; raw > 2^(c-1)
// becomes raw - 2^c with a carry into the next window.  Digits lie in [-(2^(c-1) - 1), 2^(c-1)]; the limbs stay in registers
// (constant indices only).
B200_HD int32_t msm_next_digit(uint32_t k[8], uint32_t& carry) {
    const uint32_t raw = (k[0] & ((1u << kMsmC) - 1)) + carry;
#pragma unroll
    for (int j = 0; j < 7; j++) k[j] = (k[j] >> kMsmC) | (k[j + 1] << (32 - kMsmC));
    k[7] >>= kMsmC;
    carry = raw > uint32_t(kMsmMaxDigit) ? 1u : 0u;
    return int32_t(raw) - int32_t(carry << kMsmC);
}

#if defined(__CUDACC__)

__device__ __forceinline__ uint32_t brp12(uint32_t i) { return __brev(i) >> 20; }

// Sum of one G1Jac per thread over a CTA of T threads (shared-memory tree); the result is valid in thread 0.
template <int T>
__device__ __forceinline__ G1Jac msm_cta_sum(G1Jac acc, G1Jac* sh) {
    const uint32_t tid = threadIdx.x;
    sh[tid] = acc;
    __syncthreads();
#pragma unroll 1
    for (uint32_t s = T / 2; s > 0; s >>= 1) {
        if (tid < s) {
            G1Jac a = sh[tid];
            const G1Jac b = sh[tid + s];
            jac_add(a, a, b);
            sh[tid] = a;
        }
        __syncthreads();
    }
    return sh[0];
}

// Load time, one thread per (window w, base i): T = [2^(c w)] B_i by c w doublings, then [j] T for j = 1..16 by additions,
// each normalised to affine.  B_i = g1[reverse_bits(i)] (g1 in natural order; the bit reversal is the spec's).
__global__ void __launch_bounds__(128) k_msm_table(const G1Aff* __restrict__ g1, const int32_t* __restrict__ g1_codes,
                                                   MsmAff* __restrict__ table, uint8_t* __restrict__ base_inf) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= kMsmWindows * kMsmBases) return;
    const uint32_t w = t / kMsmBases, i = t % kMsmBases, src = brp12(i);
    const bool inf = g1_codes[src] == BLS_PK_IS_INFINITY;   // K1 writes the point only for BLS_SUCCESS
    if (w == 0) base_inf[i] = inf ? 1 : 0;
    MsmAff* out = table + (size_t(w) * kMsmBases + i) * kMsmMaxDigit;
    if (inf) {
        for (int j = 0; j < kMsmMaxDigit; j++) { out[j].x = fp_zero(); out[j].y = fp_zero(); }
        return;
    }
    const G1Aff b = g1[src];
    G1Jac p;
    jac_from_aff(p, b);
#pragma unroll 1
    for (uint32_t s = 0; s < uint32_t(kMsmC) * w; s++) jac_double(p, p);
    G1Jac acc = p;
#pragma unroll 1
    for (int j = 0; j < kMsmMaxDigit; j++) {
        G1Aff a;
        jac_to_aff(a, acc);   // never infinity: (j + 1) 2^(c w) is not a multiple of the prime r
        out[j].x = a.x;
        out[j].y = a.y;
        jac_add(acc, acc, p);
    }
}

// Partial sums: grid (kMsmCtasPerBlob, blobs).  Thread t of a blob takes base i = t % 4 096 and windows
// [g W/G, (g + 1) W/G), g = t / 4 096.  scalars: canonical little-endian limbs, 4 096 per blob; a blob whose code is
// non-zero contributes nothing.
__global__ void __launch_bounds__(kMsmThreads) k_msm_partial(const Fr* __restrict__ scalars, const int32_t* __restrict__ codes,
                                                             const MsmAff* __restrict__ table, const uint8_t* __restrict__ base_inf,
                                                             G1Jac* __restrict__ partials) {
    __shared__ G1Jac sh[kMsmThreads];
    const uint32_t b = blockIdx.y;
    const uint32_t t = blockIdx.x * kMsmThreads + threadIdx.x;
    const uint32_t i = t % kMsmBases, g = t / kMsmBases;
    G1Jac acc;
    jac_set_inf(acc);
    if (codes[b] == 0 && !base_inf[i]) {
        uint32_t k[8];
        const Fr s = scalars[size_t(b) * kMsmBases + i];
#pragma unroll
        for (int j = 0; j < 8; j++) k[j] = s.l[j];
        const uint32_t w0 = g * kMsmWindowsPerGroup, w1 = w0 + kMsmWindowsPerGroup;
        uint32_t carry = 0;
#pragma unroll 1
        for (uint32_t w = 0; w < w1; w++) {
            const int32_t d = msm_next_digit(k, carry);
            if (w < w0 || d == 0) continue;
            const uint32_t m = uint32_t(d < 0 ? -d : d);
            const MsmAff e = table[(size_t(w) * kMsmBases + i) * kMsmMaxDigit + (m - 1)];
            Fp y = e.y;
            if (d < 0) fp_neg(y, y);
            jac_add_mixed(acc, acc, e.x, y);
        }
    }
    const G1Jac sum = msm_cta_sum<kMsmThreads>(acc, sh);
    if (threadIdx.x == 0) partials[size_t(b) * kMsmCtasPerBlob + blockIdx.x] = sum;
}

// One CTA of kMsmCtasPerBlob threads per blob: the partial sums -> one point -> 48 compressed bytes (zeros for a failed
// blob).  With ys, also y as 32 big-endian bytes (zeros for a failed blob).
__global__ void __launch_bounds__(kMsmCtasPerBlob) k_msm_final(const G1Jac* __restrict__ partials, const int32_t* __restrict__ codes,
                                                               const Fr* __restrict__ ys, uint8_t* __restrict__ out48,
                                                               uint8_t* __restrict__ out_y) {
    __shared__ G1Jac sh[kMsmCtasPerBlob];
    const uint32_t b = blockIdx.x;
    const G1Jac sum = msm_cta_sum<kMsmCtasPerBlob>(partials[size_t(b) * kMsmCtasPerBlob + threadIdx.x], sh);
    if (threadIdx.x != 0) return;
    const int32_t code = codes[b];
    uint8_t* o = out48 + size_t(b) * 48;
    if (code) {
        for (int j = 0; j < 48; j++) o[j] = 0;
    } else {
        G1Aff a;
        jac_to_aff(a, sum);
        g1_compress(o, a);
    }
    if (out_y) {
        uint8_t* oy = out_y + size_t(b) * 32;
        if (code) {
            for (int j = 0; j < 32; j++) oy[j] = 0;
        } else {
            fr_to_be32(oy, ys[b]);
        }
    }
}

#endif  // __CUDACC__

}  // namespace b200
