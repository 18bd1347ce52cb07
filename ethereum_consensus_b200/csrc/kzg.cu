// KZG blob-proof verification (deneb polynomial-commitments, the verification half of
// ethereum_consensus::crypto::kzg) on the device, and the extern "C" entry points of include/b200_consensus.h that
// drive it.
//
// Per blob b (commitment C, proof pi, 4 096 field elements f_i):
//   decode        K1 (bls_g1.cu, unchanged) on C and pi: decompression + subgroup check; its PK_IS_INFINITY is exactly
//                 the canonical infinity encoding, which KZG accepts (the zero polynomial); 1 / 2 / 3 -> B200_KZG_BAD_ARGS
//   challenge     z = SHA-256("FSBLOBVERIFY_V1_" || be128(4096) || blob || C) mod r: 2 050 dependent compressions,
//                 one thread per blob (k_kzg_challenge)
//   evaluation    y = p(z) in evaluation form, one CTA per blob (k_kzg_eval)
//   combination   P = C - [y]G1 + [z]pi (k_kzg_combine)
//   pairing       e(P, -G2) * e(pi, [tau]G2) == 1 on the lane-parallel Miller / final-exponentiation kernels (bls_vm.cu)
// verify_blob_kzg_proof_batch is the per-blob check reduced to one code (see b200_verify_blob_kzg_proof_batch).
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "bls_kernels.cuh"
#include "engine.h"
#include "kzg_eval.cuh"
#include "kzg_settings.h"
#include "sha256.cuh"

namespace b200 {
namespace {

constexpr size_t kBlobBytes = size_t(kBlobElems) * 32;
constexpr uint32_t kEvalThreads = 256;   // 16 elements per thread
constexpr int32_t KZG_BAD_ARGS = B200_KZG_BAD_ARGS;

// K1 code -> KZG code (0 = valid point, infinity included)
__device__ __forceinline__ int32_t kzg_point_code(int32_t k1) {
    return (k1 == BLS_SUCCESS || k1 == BLS_PK_IS_INFINITY) ? 0 : KZG_BAD_ARGS;
}

// a decoded point: K1 writes the affine point only for BLS_SUCCESS, so its PK_IS_INFINITY becomes the point at infinity here
__device__ __forceinline__ G1Aff kzg_point(const G1Aff* pts, const int32_t* pt_code, uint32_t i) {
    G1Aff a;
    if (pt_code[i] == BLS_PK_IS_INFINITY) { a.inf = 1; a.x = fp_zero(); a.y = fp_zero(); }
    else a = pts[i];
    return a;
}

__device__ __forceinline__ void load_words(uint32_t* w, const uint4* src, int n_uint4) {
#pragma unroll
    for (int k = 0; k < n_uint4; k++) {
        const uint4 v = src[k];
        w[4 * k] = bswap32(v.x); w[4 * k + 1] = bswap32(v.y); w[4 * k + 2] = bswap32(v.z); w[4 * k + 3] = bswap32(v.w);
    }
}

// big-endian state words of a digest -> Fr (hash_to_bls_field: the digest as a big-endian integer mod r)
__device__ __forceinline__ Fr fr_from_digest(const uint32_t h[8]) {
    Fr raw, r;
#pragma unroll
    for (int i = 0; i < 8; i++) raw.l[i] = h[7 - i];
    fr_from_u256_reduce(r, raw);
    return r;
}

__global__ void k_kzg_roots(Fr* __restrict__ roots) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kBlobElems) roots[i] = kzg_root_brp(i);
}

// compute_challenge: one thread per blob.  The message is 32 + 131 072 + 48 = 131 152 bytes = 2 049.25 blocks; every
// piece is a whole number of 16-byte vectors, and a blob block straddles two 64-byte windows of the blob (offset 32), so
// block k >= 1 is blob bytes [64k - 32, 64k + 32).  The next block's loads are issued before the current compression.
__global__ void __launch_bounds__(32) k_kzg_challenge(const uint8_t* __restrict__ blobs, const uint8_t* __restrict__ comms, uint32_t n,
                                                      Fr* __restrict__ z) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint4* blob = reinterpret_cast<const uint4*>(blobs + size_t(t) * kBlobBytes);
    const uint4* comm = reinterpret_cast<const uint4*>(comms + size_t(t) * 48);
    uint32_t h[8], w[16];
    sha256_init(h);
    // "FSBLOBVERIFY_V1_" || be128(4096) || blob[0..32)
    w[0] = 0x4653424cu; w[1] = 0x4f425645u; w[2] = 0x52494659u; w[3] = 0x5f56315fu;
    w[4] = 0; w[5] = 0; w[6] = 0; w[7] = kBlobElems;
    load_words(w + 8, blob, 2);
    uint4 nx[4];
#pragma unroll
    for (int k = 0; k < 4; k++) nx[k] = blob[2 + k];
    sha256_compress(h, w);
#pragma unroll 1
    for (uint32_t b = 1; b < 2048; b++) {
#pragma unroll
        for (int k = 0; k < 4; k++) {
            w[4 * k] = bswap32(nx[k].x); w[4 * k + 1] = bswap32(nx[k].y); w[4 * k + 2] = bswap32(nx[k].z); w[4 * k + 3] = bswap32(nx[k].w);
        }
        if (b + 1 < 2048) {
#pragma unroll
            for (int k = 0; k < 4; k++) nx[k] = blob[4 * b + 2 + k];
        }
        sha256_compress(h, w);
    }
    // blob[131 040..131 072) || C[0..32)
    load_words(w, blob + 8190, 2);
    load_words(w + 8, comm, 2);
    sha256_compress(h, w);
    // C[32..48) || padding || bit length
    load_words(w, comm + 2, 1);
    w[4] = 0x80000000u;
#pragma unroll
    for (int k = 5; k < 15; k++) w[k] = 0;
    w[15] = uint32_t((32 + kBlobBytes + 48) * 8);
    sha256_compress(h, w);
    z[t] = fr_from_digest(h);
}

// evaluate_polynomial_in_evaluation_form (kzg_eval.cuh), one CTA per blob: each thread folds its 16 terms into one
// fraction, the CTA folds the fractions (warp shuffles, then one warp over shared memory).  Any element >= r sets
// B200_KZG_BAD_ARGS.
__device__ __forceinline__ void shfl_frac(Frac& dst, const Frac& src, int delta) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(&src);
    uint32_t* d = reinterpret_cast<uint32_t*>(&dst);
#pragma unroll
    for (int k = 0; k < 16; k++) d[k] = __shfl_down_sync(0xffffffffu, s[k], delta);
}

__global__ void __launch_bounds__(kEvalThreads) k_kzg_eval(const uint8_t* __restrict__ blobs, const Fr* __restrict__ zs,
                                                           const Fr* __restrict__ roots, Fr* __restrict__ ys, int32_t* __restrict__ codes) {
    __shared__ Frac s_part[kEvalThreads / 32];
    __shared__ int s_bad, s_dom;
    __shared__ Fr s_fdom;
    const uint32_t b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { s_bad = 0; s_dom = -1; }
    __syncthreads();
    const Fr z = zs[b];
    const uint4* blob = reinterpret_cast<const uint4*>(blobs + size_t(b) * kBlobBytes);
    Frac acc = frac_zero();
    bool bad = false;
#pragma unroll 1
    for (uint32_t k = 0; k < kBlobElems / kEvalThreads; k++) {
        const uint32_t i = k * kEvalThreads + tid;
        uint32_t wds[8];
        load_words(wds, blob + 2 * i, 2);
        Fr raw, f;
#pragma unroll
        for (int j = 0; j < 8; j++) raw.l[j] = wds[7 - j];
        bad = bad || !fr_is_canonical(raw);
        fr_to_mont(f, raw);
        if (!frac_push(acc, f, roots[i], z)) {   // z is the i-th domain point (at most one i per blob)
            s_dom = int(i);
            s_fdom = f;
        }
    }
    if (bad) s_bad = 1;
#pragma unroll 1
    for (int s = 16; s > 0; s >>= 1) {
        Frac o;
        shfl_frac(o, acc, s);
        if (lane < uint32_t(s)) frac_add(acc, o);
    }
    if (lane == 0) s_part[warp] = acc;
    __syncthreads();
    if (warp != 0) return;
    acc = frac_zero();
    if (lane < kEvalThreads / 32) acc = s_part[lane];
#pragma unroll 1
    for (int s = 4; s > 0; s >>= 1) {
        Frac o;
        shfl_frac(o, acc, s);
        if (lane < uint32_t(s)) frac_add(acc, o);
    }
    if (lane == 0) {
        Fr y = fr_zero();
        int32_t code = 0;
        if (s_bad) code = KZG_BAD_ARGS;
        else if (s_dom >= 0) y = s_fdom;
        else y = kzg_eval_finish(acc);
        ys[b] = y;
        codes[b] = code;
    }
}

// verify_kzg_proof inputs: z and y as 32-byte big-endian field elements
__global__ void k_kzg_zy(const uint8_t* __restrict__ zy, uint32_t n, Fr* __restrict__ zs, Fr* __restrict__ ys, int32_t* __restrict__ codes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    Fr z, y;
    const bool ok = fr_from_be32(z, zy + 64 * size_t(t)) & fr_from_be32(y, zy + 64 * size_t(t) + 32);
    zs[t] = ok ? z : fr_zero();
    ys[t] = ok ? y : fr_zero();
    codes[t] = ok ? 0 : KZG_BAD_ARGS;
}

__device__ __forceinline__ void canon_limbs(uint32_t out[8], const Fr& a) {
    Fr raw;
    fr_from_mont(raw, a);
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = raw.l[i];
}
__device__ __forceinline__ G1Pre pre_from_jac(const G1Jac& p) {
    G1Pre o;
    o.inf = jac_is_inf(p) ? 1u : 0u;
    Fp zz;
    fp_sqr(zz, p.z);
    fp_mul(o.z3, zz, p.z);
    fp_mul(o.xz, p.x, p.z);
    o.y = p.y;
    return o;
}
__device__ __forceinline__ G1Pre pre_from_aff(const G1Aff& a) {
    G1Pre o;
    o.xz = a.x; o.y = a.y; o.z3 = fp_one(); o.inf = a.inf;
    return o;
}
__device__ __forceinline__ void jac_add_aff(G1Jac& acc, const G1Aff& a) {
    if (!a.inf) jac_add_mixed(acc, acc, a.x, a.y);
}
// acc += [k](qx, qy) for a Montgomery-form scalar.  A real call: the double-and-add loop is the largest code in the
// combination kernel, which needs two of them.
__device__ __noinline__ void jac_add_mul(G1Jac& acc, const Fp& qx, const Fp& qy, const Fr& k) {
    uint32_t kl[8];
    canon_limbs(kl, k);
    G1Jac t;
    jac_mul_u256(t, qx, qy, kl);
    jac_add(acc, acc, t);
}

// Per blob: the merged code (decode, evaluation) and, for a live blob, the VM operands of the tuple
// (C - [y]G1 + [z]pi, -G2), (pi, [tau]G2) at pairs 2t, 2t + 1.  A failed blob's code goes to the VM as its pk_code, which
// skips its Miller loops and returns the code unchanged.
__global__ void __launch_bounds__(64) k_kzg_combine(const G1Aff* __restrict__ pts, const int32_t* __restrict__ pt_code,
                                                    const Fr* __restrict__ zs, const Fr* __restrict__ ys, uint32_t n,
                                                    int32_t* __restrict__ codes, G1Pre* __restrict__ g1, uint32_t* __restrict__ g1_idx,
                                                    uint32_t* __restrict__ g2_idx, uint32_t* __restrict__ pair_tuple,
                                                    uint32_t* __restrict__ pair_off) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    int32_t code = codes[t];
    if (kzg_point_code(pt_code[t]) || kzg_point_code(pt_code[n + t])) code = KZG_BAD_ARGS;
    codes[t] = code;
    g1_idx[2 * t] = 2 * t; g1_idx[2 * t + 1] = 2 * t + 1;
    g2_idx[2 * t] = 0; g2_idx[2 * t + 1] = 1;
    pair_tuple[2 * t] = t; pair_tuple[2 * t + 1] = t;
    pair_off[t] = 2 * t;
    if (code) return;
    const G1Aff c = kzg_point(pts, pt_code, t), pi = kzg_point(pts, pt_code, n + t);
    G1Jac acc;
    jac_set_inf(acc);
    if (!pi.inf) jac_add_mul(acc, pi.x, pi.y, zs[t]);
    const Fp gx = B200_FP_G1_X, ngy = B200_FP_G1_NEG_Y;
    jac_add_mul(acc, gx, ngy, ys[t]);
    jac_add_aff(acc, c);
    g1[2 * t] = pre_from_jac(acc);
    g1[2 * t + 1] = pre_from_aff(pi);
}

// ---- host orchestration -----------------------------------------------------------------------------------------------
struct KzgState {
    DevBuf blobs, pts48, aff, pcode, zy, z, y, code, zeros, g1pre, idx, f, out;
    PinnedBuf host;
    cudaEvent_t ev[8] = {nullptr};
    bool trace = false;   // B200_KZG_TRACE=1: per-stage CUDA-event timings on stderr
};
KzgState* g_kzg = nullptr;

int32_t kzg_ready(Engine& e, KzgState** out) {
    if (!e.ready) { e.last_error = "b200_init has not been called (or failed)"; return B200_ERR_NOT_INITIALIZED; }
    cudaError_t ce = cudaSetDevice(e.device);
    if (ce != cudaSuccess) { e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    if (!g_kzg) {
        KzgState* s = new KzgState();
        if (const char* v = getenv("B200_KZG_TRACE")) s->trace = atoi(v) != 0;
        for (auto& ev : s->ev) B200_CUDA_TRY(cudaEventCreate(&ev));
        if (vm_init(e.stream) != 0) { e.last_error = "pairing VM initialisation failed"; return B200_ERR_CUDA; }
        g_kzg = s;
    }
    *out = g_kzg;
    return B200_SUCCESS;
}

enum KzgMode { KZG_POINT = 0, KZG_BLOB = 1 };

// n tuples -> out_codes[n].  KZG_POINT: commitments, zy (n x 64 bytes: z || y), proofs.  KZG_BLOB: blobs, commitments, proofs.
int32_t kzg_run(Engine& e, KzgState& s, const b200_kzg_settings* st, KzgMode mode, uint32_t n, const uint8_t* blobs,
                const uint8_t* comms, const uint8_t* zy, const uint8_t* proofs, int32_t* out_codes) {
    cudaStream_t sa = e.stream;
    B200_CUDA_TRY(s.pts48.reserve(size_t(96) * n));
    B200_CUDA_TRY(s.aff.reserve(sizeof(G1Aff) * 2 * n));
    B200_CUDA_TRY(s.pcode.reserve(sizeof(int32_t) * 2 * n));
    B200_CUDA_TRY(s.z.reserve(sizeof(Fr) * n));
    B200_CUDA_TRY(s.y.reserve(sizeof(Fr) * n));
    B200_CUDA_TRY(s.code.reserve(sizeof(int32_t) * n));
    B200_CUDA_TRY(s.zeros.reserve(sizeof(int32_t) * n));
    B200_CUDA_TRY(s.g1pre.reserve(sizeof(G1Pre) * 2 * n));
    B200_CUDA_TRY(s.idx.reserve(sizeof(uint32_t) * 7 * n));
    B200_CUDA_TRY(s.f.reserve(sizeof(Fp12) * 2 * n));
    B200_CUDA_TRY(s.out.reserve(sizeof(int32_t) * n));
    B200_CUDA_TRY(s.host.reserve(sizeof(int32_t) * n));
    if (mode == KZG_POINT) B200_CUDA_TRY(s.zy.reserve(size_t(64) * n));
    else B200_CUDA_TRY(s.blobs.reserve(kBlobBytes * n));
    uint8_t* d_pts48 = static_cast<uint8_t*>(s.pts48.p);
    G1Aff* d_aff = static_cast<G1Aff*>(s.aff.p);
    int32_t* d_pcode = static_cast<int32_t*>(s.pcode.p);
    Fr* d_z = static_cast<Fr*>(s.z.p);
    Fr* d_y = static_cast<Fr*>(s.y.p);
    int32_t* d_code = static_cast<int32_t*>(s.code.p);
    uint32_t* d_zeros = static_cast<uint32_t*>(s.zeros.p);
    G1Pre* d_g1 = static_cast<G1Pre*>(s.g1pre.p);
    uint32_t* d_idx = static_cast<uint32_t*>(s.idx.p);
    int32_t* d_out = static_cast<int32_t*>(s.out.p);

    B200_CUDA_TRY(cudaEventRecord(s.ev[0], sa));
    B200_CUDA_TRY(cudaMemcpyAsync(d_pts48, comms, size_t(48) * n, cudaMemcpyHostToDevice, sa));
    B200_CUDA_TRY(cudaMemcpyAsync(d_pts48 + size_t(48) * n, proofs, size_t(48) * n, cudaMemcpyHostToDevice, sa));
    if (mode == KZG_POINT) B200_CUDA_TRY(cudaMemcpyAsync(s.zy.p, zy, size_t(64) * n, cudaMemcpyHostToDevice, sa));
    else B200_CUDA_TRY(cudaMemcpyAsync(s.blobs.p, blobs, kBlobBytes * n, cudaMemcpyHostToDevice, sa));
    B200_CUDA_TRY(cudaMemsetAsync(d_zeros, 0, sizeof(int32_t) * n, sa));
    B200_CUDA_TRY(cudaEventRecord(s.ev[1], sa));
    launch_g1_validate(d_pts48, 2 * n, d_aff, d_pcode, sa);
    e.launches++;
    B200_CUDA_TRY(cudaEventRecord(s.ev[2], sa));
    if (mode == KZG_POINT) {
        k_kzg_zy<<<(n + 63) / 64, 64, 0, sa>>>(static_cast<const uint8_t*>(s.zy.p), n, d_z, d_y, d_code);
        B200_CUDA_TRY(cudaEventRecord(s.ev[3], sa));
        e.launches++;
    } else {
        k_kzg_challenge<<<(n + 31) / 32, 32, 0, sa>>>(static_cast<const uint8_t*>(s.blobs.p), d_pts48, n, d_z);
        B200_CUDA_TRY(cudaEventRecord(s.ev[3], sa));
        k_kzg_eval<<<n, kEvalThreads, 0, sa>>>(static_cast<const uint8_t*>(s.blobs.p), d_z, st->d_roots, d_y, d_code);
        e.launches += 2;
    }
    B200_CUDA_TRY(cudaEventRecord(s.ev[4], sa));
    uint32_t *g1_idx = d_idx, *g2_idx = d_idx + 2 * n, *pair_tuple = d_idx + 4 * n, *pair_off = d_idx + 6 * n;
    k_kzg_combine<<<(n + 63) / 64, 64, 0, sa>>>(d_aff, d_pcode, d_z, d_y, n, d_code, d_g1, g1_idx, g2_idx, pair_tuple, pair_off);
    e.launches++;
    B200_CUDA_TRY(cudaEventRecord(s.ev[5], sa));
    launch_vm_miller(d_g1, g1_idx, st->d_g2, g2_idx, pair_tuple, d_code, d_zeros, reinterpret_cast<const int32_t*>(d_zeros),
                     2 * n, static_cast<Fp12*>(s.f.p), sa);
    B200_CUDA_TRY(cudaEventRecord(s.ev[6], sa));
    launch_vm_final(static_cast<const Fp12*>(s.f.p), pair_off, d_code, d_zeros, reinterpret_cast<const int32_t*>(d_zeros), n,
                    d_out, sa);
    e.launches += 2;
    B200_CUDA_TRY(cudaEventRecord(s.ev[7], sa));
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(s.host.p, d_out, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    B200_CUDA_TRY(cudaEventElapsedTime(&e.last_kernel_ms, s.ev[1], s.ev[7]));
    if (s.trace) {
        float t[7];
        for (int k = 0; k < 7; k++) cudaEventElapsedTime(&t[k], s.ev[k], s.ev[k + 1]);
        fprintf(stderr, "[b200 kzg] %s n=%u | h2d %.3f | decode %.3f | %s %.3f | eval %.3f | combine %.3f | miller %.3f | final %.3f | "
                        "kernels %.3f ms\n", mode == KZG_POINT ? "verify_kzg_proof" : "verify_blob_kzg_proofs", n, t[0], t[1],
                mode == KZG_POINT ? "zy" : "challenge", t[2], t[3], t[4], t[5], t[6], e.last_kernel_ms);
    }
    memcpy(out_codes, s.host.p, sizeof(int32_t) * n);
    return B200_SUCCESS;
}

}  // namespace

// the prover (kzg_prove.cu) runs the challenge and the evaluation as they are
void launch_kzg_challenge(const uint8_t* blobs, const uint8_t* comms, uint32_t n, Fr* z, cudaStream_t s) {
    k_kzg_challenge<<<(n + 31) / 32, 32, 0, s>>>(blobs, comms, n, z);
}
void launch_kzg_eval(const uint8_t* blobs, const Fr* zs, const Fr* roots, Fr* ys, int32_t* codes, uint32_t n, cudaStream_t s) {
    k_kzg_eval<<<n, kEvalThreads, 0, s>>>(blobs, zs, roots, ys, codes);
}

}  // namespace b200

using namespace b200;

namespace {
// the compressed encoding of -G2 (the negated generator): appended to the setup's G2 points and decoded with them
const uint8_t kNegG2[96] = {
    0xb3, 0xe0, 0x2b, 0x60, 0x52, 0x71, 0x9f, 0x60, 0x7d, 0xac, 0xd3, 0xa0, 0x88, 0x27, 0x4f, 0x65, 0x59, 0x6b, 0xd0, 0xd0,
    0x99, 0x20, 0xb6, 0x1a, 0xb5, 0xda, 0x61, 0xbb, 0xdc, 0x7f, 0x50, 0x49, 0x33, 0x4c, 0xf1, 0x12, 0x13, 0x94, 0x5d, 0x57,
    0xe5, 0xac, 0x7d, 0x05, 0x5d, 0x04, 0x2b, 0x7e, 0x02, 0x4a, 0xa2, 0xb2, 0xf0, 0x8f, 0x0a, 0x91, 0x26, 0x08, 0x05, 0x27,
    0x2d, 0xc5, 0x10, 0x51, 0xc6, 0xe4, 0x7a, 0xd4, 0xfa, 0x40, 0x3b, 0x02, 0xb4, 0x51, 0x0b, 0x64, 0x7a, 0xe3, 0xd1, 0x77,
    0x0b, 0xac, 0x03, 0x26, 0xa8, 0x05, 0xbb, 0xef, 0xd4, 0x80, 0x56, 0xc8, 0xc1, 0x21, 0xbd, 0xb8};

int32_t settings_load(Engine& e, const uint8_t* g1, size_t n_g1, const uint8_t* g2, size_t n_g2, b200_kzg_settings** out) {
    cudaStream_t sa = e.stream;
    const size_t n2 = n_g2 + 1;
    uint8_t *d_g1b = nullptr, *d_g2b = nullptr;
    G1Aff* d_g1a = nullptr;
    G2Aff* d_g2a = nullptr;
    int32_t* d_codes = nullptr;
    int32_t rc = B200_SUCCESS;
    std::vector<int32_t> codes(n_g1 + n2);
    std::vector<uint8_t> g2b(96 * n2);
    memcpy(g2b.data(), g2, 96 * n_g2);
    memcpy(g2b.data() + 96 * n_g2, kNegG2, 96);
    b200_kzg_settings* st = new b200_kzg_settings();
    auto fail = [&](int32_t code, const char* what) {
        if (code >= 0x100) e.last_error = std::string("b200_kzg_settings_load: ") + what;
        rc = code;
    };
    do {
        if (cudaMalloc(&d_g1b, 48 * n_g1) || cudaMalloc(&d_g2b, 96 * n2) || cudaMalloc(&d_g1a, sizeof(G1Aff) * n_g1) ||
            cudaMalloc(&d_g2a, sizeof(G2Aff) * n2) || cudaMalloc(&d_codes, sizeof(int32_t) * (n_g1 + n2)) ||
            cudaMalloc(&st->d_g2, sizeof(G2Aff) * 2) || cudaMalloc(&st->d_roots, sizeof(Fr) * kBlobElems)) { fail(B200_ERR_CUDA, "cudaMalloc"); break; }
        cudaMemcpyAsync(d_g1b, g1, 48 * n_g1, cudaMemcpyHostToDevice, sa);
        cudaMemcpyAsync(d_g2b, g2b.data(), 96 * n2, cudaMemcpyHostToDevice, sa);
        launch_g1_validate(d_g1b, uint32_t(n_g1), d_g1a, d_codes, sa);
        launch_g2_sig_decode(d_g2b, uint32_t(n2), d_g2a, d_codes + n_g1, sa);
        k_kzg_roots<<<kBlobElems / 128, 128, 0, sa>>>(st->d_roots);
        cudaMemcpyAsync(st->d_g2, d_g2a + n_g2, sizeof(G2Aff), cudaMemcpyDeviceToDevice, sa);
        cudaMemcpyAsync(st->d_g2 + 1, d_g2a + 1, sizeof(G2Aff), cudaMemcpyDeviceToDevice, sa);
        cudaMemcpyAsync(codes.data(), d_codes, sizeof(int32_t) * codes.size(), cudaMemcpyDeviceToHost, sa);
        e.launches += 3;
        const cudaError_t ce = cudaStreamSynchronize(sa);
        if (ce != cudaSuccess || cudaGetLastError() != cudaSuccess) { fail(B200_ERR_CUDA, cudaGetErrorString(ce)); break; }
        for (size_t i = 0; i < n_g1 && !rc; i++)   // infinity is a point of G1 (K1 reports it as PK_IS_INFINITY)
            if (codes[i] != BLS_SUCCESS && codes[i] != BLS_PK_IS_INFINITY) rc = B200_KZG_BAD_ARGS;
        for (size_t i = 0; i < n2 && !rc; i++)
            if (codes[n_g1 + i] != SIG_OK) rc = B200_KZG_BAD_ARGS;
        if (!rc) rc = kzg_prover_settings_build(e, st, d_g1a, d_codes);   // the prover's bases, from the decoded points
    } while (0);
    cudaFree(d_g1b); cudaFree(d_g2b); cudaFree(d_g1a); cudaFree(d_g2a); cudaFree(d_codes);
    if (rc) { b200_kzg_settings_free(st); return rc; }
    *out = st;
    return B200_SUCCESS;
}

int32_t kzg_entry(const b200_kzg_settings* st, KzgMode mode, size_t n, const uint8_t* blobs, const uint8_t* comms, const uint8_t* zy,
                  const uint8_t* proofs, int32_t* out_codes) {
    Engine& e = engine();
    std::lock_guard<std::mutex> g(e.mu);
    KzgState* s;
    int32_t rc = kzg_ready(e, &s);
    if (rc) return rc;
    if (!st || !out_codes || n > B200_KZG_MAX_BLOBS) return B200_ERR_BAD_ARG;
    if (n == 0) return B200_SUCCESS;
    if (!comms || !proofs || (mode == KZG_POINT ? !zy : !blobs)) return B200_ERR_BAD_ARG;
    return kzg_run(e, *s, st, mode, uint32_t(n), blobs, comms, zy, proofs, out_codes);
}
}  // namespace

extern "C" {

int32_t b200_kzg_settings_load(const uint8_t* g1_lagrange, size_t n_g1, const uint8_t* g2_monomial, size_t n_g2,
                               b200_kzg_settings** out) {
    if (!out) return B200_ERR_BAD_ARG;
    *out = nullptr;
    if (n_g1 != kBlobElems || n_g2 < 2) return B200_KZG_BAD_ARGS;
    if (!g1_lagrange || !g2_monomial) return B200_ERR_BAD_ARG;
    Engine& e = engine();
    std::lock_guard<std::mutex> g(e.mu);
    KzgState* s;
    int32_t rc = kzg_ready(e, &s);
    if (rc) return rc;
    return settings_load(e, g1_lagrange, n_g1, g2_monomial, n_g2, out);
}

void b200_kzg_settings_free(b200_kzg_settings* st) {
    if (!st) return;
    cudaFree(st->d_g2);
    cudaFree(st->d_roots);
    cudaFree(st->d_table);
    cudaFree(st->d_base_inf);
    delete st;
}

int32_t b200_verify_kzg_proof(const b200_kzg_settings* st, const uint8_t commitment[48], const uint8_t z[32], const uint8_t y[32],
                              const uint8_t proof[48]) {
    if (!z || !y) return B200_ERR_BAD_ARG;
    uint8_t zy[64];
    memcpy(zy, z, 32);
    memcpy(zy + 32, y, 32);
    int32_t code = 0;
    const int32_t rc = kzg_entry(st, KZG_POINT, 1, nullptr, commitment, zy, proof, &code);
    return rc ? rc : code;
}

int32_t b200_verify_blob_kzg_proofs(const b200_kzg_settings* st, const uint8_t* blobs, const uint8_t* commitments,
                                    const uint8_t* proofs, size_t n, int32_t* out_codes) {
    return kzg_entry(st, KZG_BLOB, n, blobs, commitments, nullptr, proofs, out_codes);
}

int32_t b200_verify_blob_kzg_proof(const b200_kzg_settings* st, const uint8_t* blob, const uint8_t commitment[48],
                                   const uint8_t proof[48]) {
    int32_t code = 0;
    const int32_t rc = kzg_entry(st, KZG_BLOB, 1, blob, commitment, nullptr, proof, &code);
    return rc ? rc : code;
}

// Every blob is checked on its own and the codes reduce to one: any malformed input -> B200_KZG_BAD_ARGS (c-kzg validates
// every input before it checks any proof), else any failed proof -> B200_VERIFY_FAIL, else 0.  The spec's random linear
// combination accepts a batch with an invalid proof with probability <= n / r (~2^-241) and otherwise agrees with this
// conjunction; on the device the separate checks are also the faster form (one tuple per blob fills the machine, the
// combination's transcript hash and three scalar multiplications per blob do not), so the combination is not run.
int32_t b200_verify_blob_kzg_proof_batch(const b200_kzg_settings* st, const uint8_t* blobs, const uint8_t* commitments,
                                         const uint8_t* proofs, size_t n) {
    if (n > B200_KZG_MAX_BLOBS) return B200_ERR_BAD_ARG;
    std::vector<int32_t> codes(n + 1);   // never empty: n = 0 still reaches the argument checks with a valid pointer
    const int32_t rc = kzg_entry(st, KZG_BLOB, n, blobs, commitments, nullptr, proofs, codes.data());
    codes.pop_back();
    if (rc) return rc;
    int32_t out = B200_SUCCESS;
    for (int32_t c : codes) {
        if (c == B200_KZG_BAD_ARGS) return c;
        if (c != B200_SUCCESS) out = c;
    }
    return out;
}

}  // extern "C"
