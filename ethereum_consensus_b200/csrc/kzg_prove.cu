// KZG proof generation (deneb polynomial-commitments, the prover half of ethereum_consensus::crypto::kzg) on the device,
// and the extern "C" entry points of include/b200_consensus.h that drive it.
//
// Per blob, in chunks of kChunk blobs, every stage on the engine stream with no host round trip in between:
//   commitment    elements checked and unpacked to canonical limbs (k_commit_scalars), then the MSM over the bases
//   proof         K1 (bls_g1.cu, unchanged) on C; z = compute_challenge(blob, C) and y = p(z) (k_kzg_challenge and
//                 k_kzg_eval of kzg.cu, unchanged) -- or z supplied by the caller (compute_kzg_proof); the quotient
//                 (k_kzg_quotient, kzg_quotient.cuh); the MSM over its 4 096 values
//   MSM           k_msm_partial + k_msm_final (msm.cuh): the fixed-base comb over the settings' table, then jac_to_aff and
//                 g1_compress
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "kzg_quotient.cuh"
#include "kzg_settings.h"
#include "msm.cuh"

namespace b200 {
namespace {

constexpr size_t kBlobBytes = size_t(kBlobElems) * 32;
constexpr uint32_t kChunk = 1024;          // blobs per pass: bounds the device scratch whatever n is
constexpr uint32_t kQuotThreads = 256;     // 16 elements per thread
constexpr int32_t KZG_BAD_ARGS = B200_KZG_BAD_ARGS;

// blob elements -> canonical little-endian limbs; any element >= r sets the blob's code (codes zeroed beforehand).
// grid (4 096 / 256, n)
__global__ void __launch_bounds__(256) k_commit_scalars(const uint8_t* __restrict__ blobs, Fr* __restrict__ scalars,
                                                        int32_t* __restrict__ codes) {
    const uint32_t b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint4* src = reinterpret_cast<const uint4*>(blobs + size_t(b) * kBlobBytes + 32 * size_t(i));
    const uint4 v0 = src[0], v1 = src[1];
    const uint32_t w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
    Fr raw;
#pragma unroll
    for (int j = 0; j < 8; j++) raw.l[j] = __byte_perm(w[7 - j], 0, 0x0123);
    if (!fr_is_canonical(raw)) codes[b] = KZG_BAD_ARGS;
    scalars[size_t(b) * kBlobElems + i] = raw;
}

// compute_kzg_proof's z: 32 big-endian bytes -> Montgomery Fr; z >= r -> B200_KZG_BAD_ARGS (and z = 0 for the stages after)
__global__ void k_prove_z(const uint8_t* __restrict__ zb, uint32_t n, Fr* __restrict__ zs, int32_t* __restrict__ codes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    Fr z;
    const bool ok = fr_from_be32(z, zb + 32 * size_t(t));
    zs[t] = ok ? z : fr_zero();
    codes[t] = ok ? 0 : KZG_BAD_ARGS;
}

// K1 code of a commitment -> KZG code (infinity is a valid commitment)
__global__ void k_prove_point_codes(const int32_t* __restrict__ pcode, uint32_t n, int32_t* __restrict__ codes) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    codes[t] = (pcode[t] == BLS_SUCCESS || pcode[t] == BLS_PK_IS_INFINITY) ? 0 : KZG_BAD_ARGS;
}

// The quotient of one blob per CTA (kzg_quotient.cuh): element i goes to thread i % 256.  The merged code (evaluation's
// element check, then the z / commitment code) goes to out_codes; a failed blob writes no scalars (the MSM skips it).
__global__ void __launch_bounds__(kQuotThreads) k_kzg_quotient(const uint8_t* __restrict__ blobs, const Fr* __restrict__ zs,
                                                               const Fr* __restrict__ ys, const Fr* __restrict__ roots,
                                                               const int32_t* __restrict__ eval_codes,
                                                               const int32_t* __restrict__ in_codes, Fr* __restrict__ q_all,
                                                               int32_t* __restrict__ out_codes) {
    __shared__ Fr s_pre[kQuotThreads], s_suf[kQuotThreads];
    __shared__ Fr s_inv;
    __shared__ int32_t s_dom;
    const uint32_t b = blockIdx.x, tid = threadIdx.x;
    const int32_t code = eval_codes[b] ? eval_codes[b] : in_codes[b];
    if (tid == 0) { out_codes[b] = code; s_dom = -1; }
    if (code) return;   // uniform over the CTA
    const Fr z = zs[b], y = ys[b];
    Fr* q = q_all + size_t(b) * kBlobElems;
    const uint8_t* blob = blobs + size_t(b) * kBlobBytes;
    int32_t dom = -1;
    const Fr prod = quot_prefix(q, roots, z, tid, kQuotThreads, kBlobElems / kQuotThreads, dom);
    // inclusive prefix and suffix products of the threads' products (Hillis-Steele)
    s_pre[tid] = prod;
    s_suf[tid] = prod;
    __syncthreads();
    if (dom >= 0) s_dom = dom;
#pragma unroll 1
    for (uint32_t off = 1; off < kQuotThreads; off <<= 1) {
        Fr a = s_pre[tid], c = s_suf[tid];
        if (tid >= off) fr_mul(a, a, s_pre[tid - off]);
        if (tid + off < kQuotThreads) fr_mul(c, c, s_suf[tid + off]);
        __syncthreads();
        s_pre[tid] = a;
        s_suf[tid] = c;
        __syncthreads();
    }
    if (tid == 0) fr_inv(s_inv, s_pre[kQuotThreads - 1]);
    __syncthreads();
    // 1 / prod = (1 / all) * (product of every other thread's)
    Fr inv = s_inv;
    if (tid > 0) fr_mul(inv, inv, s_pre[tid - 1]);
    if (tid + 1 < kQuotThreads) fr_mul(inv, inv, s_suf[tid + 1]);
    const int32_t m = s_dom;
    const Fr sum = quot_finish(q, blob, roots, z, y, inv, tid, kQuotThreads, kBlobElems / kQuotThreads, m >= 0);
    if (m < 0) return;   // uniform
    __syncthreads();     // s_pre is reused for the sum of q_i w_i
    s_pre[tid] = sum;
    __syncthreads();
#pragma unroll 1
    for (uint32_t s = kQuotThreads / 2; s > 0; s >>= 1) {
        if (tid < s) fr_add(s_pre[tid], s_pre[tid], s_pre[tid + s]);
        __syncthreads();
    }
    if (tid == 0) q[m] = quot_within_domain(s_pre[0], roots, uint32_t(m));
}

// ---- host orchestration -----------------------------------------------------------------------------------------------
enum ProveMode { PROVE_COMMIT = 0, PROVE_POINT = 1, PROVE_BLOB = 2 };
const char* const kEntry[3] = {"blob_to_kzg_commitments", "compute_kzg_proof", "compute_blob_kzg_proofs"};

// stage boundaries recorded per chunk: ev[k] -> ev[k + 1] is stage k ("none": an empty stage of that mode)
constexpr int kStages[3] = {5, 8, 8};
const char* const kStageNames[3][8] = {{"h2d", "check", "msm", "final", "d2h"},
                                       {"h2d", "z", "none", "eval", "quotient", "msm", "final", "d2h"},
                                       {"h2d", "decode", "challenge", "eval", "quotient", "msm", "final", "d2h"}};

struct ProveState {
    DevBuf blobs, aux, aff, pcode, z, y, code, code2, code3, scal, part, out48, outy;
    PinnedBuf host;
    std::vector<cudaEvent_t> ev;
    bool trace = false;   // B200_KZG_TRACE=1: per-stage CUDA-event timings on stderr
};
ProveState* g_prove = nullptr;

int32_t prove_ready(Engine& e, ProveState** out) {
    if (!e.ready) { e.last_error = "b200_init has not been called (or failed)"; return B200_ERR_NOT_INITIALIZED; }
    cudaError_t ce = cudaSetDevice(e.device);
    if (ce != cudaSuccess) { e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    if (!g_prove) {
        ProveState* s = new ProveState();
        if (const char* v = getenv("B200_KZG_TRACE")) s->trace = atoi(v) != 0;
        g_prove = s;
    }
    *out = g_prove;
    return B200_SUCCESS;
}

// n blobs -> out48 (n x 48), out_y (PROVE_POINT: n x 32), out_codes[n].  aux: PROVE_POINT z (n x 32), PROVE_BLOB
// commitments (n x 48).
int32_t prove_run(Engine& e, ProveState& s, const b200_kzg_settings* st, ProveMode mode, uint32_t n, const uint8_t* blobs,
                  const uint8_t* aux, uint8_t* out48, uint8_t* out_y, int32_t* out_codes) {
    cudaStream_t sa = e.stream;
    const uint32_t cmax = n < kChunk ? n : kChunk;
    const uint32_t n_chunks = (n + kChunk - 1) / kChunk;
    const int n_ev = kStages[mode] + 1;
    B200_CUDA_TRY(s.blobs.reserve(kBlobBytes * cmax));
    B200_CUDA_TRY(s.aux.reserve(size_t(48) * cmax));
    B200_CUDA_TRY(s.aff.reserve(sizeof(G1Aff) * cmax));
    B200_CUDA_TRY(s.pcode.reserve(sizeof(int32_t) * cmax));
    B200_CUDA_TRY(s.z.reserve(sizeof(Fr) * cmax));
    B200_CUDA_TRY(s.y.reserve(sizeof(Fr) * cmax));
    B200_CUDA_TRY(s.code.reserve(sizeof(int32_t) * cmax));
    B200_CUDA_TRY(s.code2.reserve(sizeof(int32_t) * cmax));
    B200_CUDA_TRY(s.code3.reserve(sizeof(int32_t) * cmax));
    B200_CUDA_TRY(s.scal.reserve(sizeof(Fr) * kBlobElems * cmax));
    B200_CUDA_TRY(s.part.reserve(sizeof(G1Jac) * kMsmCtasPerBlob * cmax));
    B200_CUDA_TRY(s.out48.reserve(size_t(48) * cmax));
    B200_CUDA_TRY(s.outy.reserve(size_t(32) * cmax));
    const size_t host_bytes = size_t(n) * (48 + 32 + sizeof(int32_t));
    B200_CUDA_TRY(s.host.reserve(host_bytes));
    while (s.ev.size() < size_t(n_ev) * n_chunks) {
        cudaEvent_t ev;
        B200_CUDA_TRY(cudaEventCreate(&ev));
        s.ev.push_back(ev);
    }
    uint8_t* d_blobs = static_cast<uint8_t*>(s.blobs.p);
    uint8_t* d_aux = static_cast<uint8_t*>(s.aux.p);
    G1Aff* d_aff = static_cast<G1Aff*>(s.aff.p);
    int32_t* d_pcode = static_cast<int32_t*>(s.pcode.p);
    Fr* d_z = static_cast<Fr*>(s.z.p);
    Fr* d_y = static_cast<Fr*>(s.y.p);
    int32_t* d_code = static_cast<int32_t*>(s.code.p);    // the final per-blob code
    int32_t* d_code2 = static_cast<int32_t*>(s.code2.p);  // evaluation's element check
    int32_t* d_code3 = static_cast<int32_t*>(s.code3.p);  // z / commitment
    Fr* d_scal = static_cast<Fr*>(s.scal.p);
    G1Jac* d_part = static_cast<G1Jac*>(s.part.p);
    uint8_t* d_out48 = static_cast<uint8_t*>(s.out48.p);
    uint8_t* d_outy = static_cast<uint8_t*>(s.outy.p);
    uint8_t* h_out48 = static_cast<uint8_t*>(s.host.p);
    uint8_t* h_outy = h_out48 + size_t(48) * n;
    int32_t* h_code = reinterpret_cast<int32_t*>(h_outy + size_t(32) * n);

    for (uint32_t c = 0; c < n_chunks; c++) {
        const uint32_t b0 = c * kChunk, m = (n - b0) < kChunk ? (n - b0) : kChunk;
        cudaEvent_t* ev = s.ev.data() + size_t(c) * n_ev;
        int k = 0;
        B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
        B200_CUDA_TRY(cudaMemcpyAsync(d_blobs, blobs + kBlobBytes * b0, kBlobBytes * m, cudaMemcpyHostToDevice, sa));
        if (mode == PROVE_POINT) B200_CUDA_TRY(cudaMemcpyAsync(d_aux, aux + size_t(32) * b0, size_t(32) * m, cudaMemcpyHostToDevice, sa));
        if (mode == PROVE_BLOB) B200_CUDA_TRY(cudaMemcpyAsync(d_aux, aux + size_t(48) * b0, size_t(48) * m, cudaMemcpyHostToDevice, sa));
        B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
        if (mode == PROVE_COMMIT) {
            B200_CUDA_TRY(cudaMemsetAsync(d_code, 0, sizeof(int32_t) * m, sa));
            k_commit_scalars<<<dim3(kBlobElems / 256, m), 256, 0, sa>>>(d_blobs, d_scal, d_code);
            e.launches++;
            B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
        } else {
            if (mode == PROVE_POINT) {
                k_prove_z<<<(m + 63) / 64, 64, 0, sa>>>(d_aux, m, d_z, d_code3);
                B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
                B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));   // no challenge: z is given
                e.launches++;
            } else {
                launch_g1_validate(d_aux, m, d_aff, d_pcode, sa);
                k_prove_point_codes<<<(m + 63) / 64, 64, 0, sa>>>(d_pcode, m, d_code3);
                B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
                launch_kzg_challenge(d_blobs, d_aux, m, d_z, sa);
                B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
                e.launches += 3;
            }
            launch_kzg_eval(d_blobs, d_z, st->d_roots, d_y, d_code2, m, sa);
            B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
            k_kzg_quotient<<<m, kQuotThreads, 0, sa>>>(d_blobs, d_z, d_y, st->d_roots, d_code2, d_code3, d_scal, d_code);
            B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
            e.launches += 2;
        }
        k_msm_partial<<<dim3(kMsmCtasPerBlob, m), kMsmThreads, 0, sa>>>(d_scal, d_code, st->d_table, st->d_base_inf, d_part);
        B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
        k_msm_final<<<m, kMsmCtasPerBlob, 0, sa>>>(d_part, d_code, d_y, d_out48, mode == PROVE_POINT ? d_outy : nullptr);
        B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
        e.launches += 2;
        B200_CUDA_TRY(cudaGetLastError());
        B200_CUDA_TRY(cudaMemcpyAsync(h_out48 + size_t(48) * b0, d_out48, size_t(48) * m, cudaMemcpyDeviceToHost, sa));
        if (mode == PROVE_POINT)
            B200_CUDA_TRY(cudaMemcpyAsync(h_outy + size_t(32) * b0, d_outy, size_t(32) * m, cudaMemcpyDeviceToHost, sa));
        B200_CUDA_TRY(cudaMemcpyAsync(h_code + b0, d_code, sizeof(int32_t) * m, cudaMemcpyDeviceToHost, sa));
        B200_CUDA_TRY(cudaEventRecord(ev[k++], sa));
    }
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    // kernel time: from after each chunk's upload to its last kernel, summed over the chunks
    float kernels = 0.f, st_ms[8] = {0.f};
    const int n_st = kStages[mode];
    for (uint32_t c = 0; c < n_chunks; c++) {
        cudaEvent_t* ev = s.ev.data() + size_t(c) * n_ev;
        float t;
        B200_CUDA_TRY(cudaEventElapsedTime(&t, ev[1], ev[n_ev - 2]));
        kernels += t;
        for (int k = 0; k < n_st; k++) {
            B200_CUDA_TRY(cudaEventElapsedTime(&t, ev[k], ev[k + 1]));
            st_ms[k] += t;
        }
    }
    e.last_kernel_ms = kernels;
    if (s.trace) {
        char line[512];
        int len = snprintf(line, sizeof line, "[b200 kzg] %s n=%u", kEntry[mode], n);
        for (int k = 0; k < n_st; k++)
            if (strcmp(kStageNames[mode][k], "none") != 0)
                len += snprintf(line + len, sizeof line - len, " | %s %.3f", kStageNames[mode][k], st_ms[k]);
        fprintf(stderr, "%s | kernels %.3f ms\n", line, kernels);
    }
    memcpy(out48, h_out48, size_t(48) * n);
    if (mode == PROVE_POINT) memcpy(out_y, h_outy, size_t(32) * n);
    memcpy(out_codes, h_code, sizeof(int32_t) * n);
    return B200_SUCCESS;
}

int32_t prove_entry(const b200_kzg_settings* st, ProveMode mode, size_t n, const uint8_t* blobs, const uint8_t* aux,
                    uint8_t* out48, uint8_t* out_y, int32_t* out_codes) {
    Engine& e = engine();
    std::lock_guard<std::mutex> g(e.mu);
    ProveState* s;
    int32_t rc = prove_ready(e, &s);
    if (rc) return rc;
    if (!st || n > B200_KZG_MAX_BLOBS) return B200_ERR_BAD_ARG;
    if (n == 0) return B200_SUCCESS;
    if (!blobs || !out48 || !out_codes || (mode != PROVE_COMMIT && !aux) || (mode == PROVE_POINT && !out_y)) return B200_ERR_BAD_ARG;
    return prove_run(e, *s, st, mode, uint32_t(n), blobs, aux, out48, out_y, out_codes);
}

}  // namespace

int32_t kzg_prover_settings_build(Engine& e, b200_kzg_settings* st, const G1Aff* g1, const int32_t* g1_codes) {
    cudaStream_t sa = e.stream;
    const size_t entries = size_t(kMsmWindows) * kMsmBases * kMsmMaxDigit;
    if (cudaMalloc(&st->d_table, sizeof(MsmAff) * entries) != cudaSuccess || cudaMalloc(&st->d_base_inf, kMsmBases) != cudaSuccess) {
        e.last_error = "b200_kzg_settings_load: cudaMalloc (prover table)";
        return B200_ERR_CUDA;
    }
    const uint32_t threads = kMsmWindows * kMsmBases;
    k_msm_table<<<(threads + 127) / 128, 128, 0, sa>>>(g1, g1_codes, st->d_table, st->d_base_inf);
    e.launches++;
    cudaError_t ce = cudaGetLastError();
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(sa);
    if (ce != cudaSuccess) {
        e.last_error = std::string("b200_kzg_settings_load: ") + cudaGetErrorString(ce);
        return B200_ERR_CUDA;
    }
    return B200_SUCCESS;
}

}  // namespace b200

using namespace b200;

extern "C" {

int32_t b200_blob_to_kzg_commitments(const b200_kzg_settings* st, const uint8_t* blobs, size_t n, uint8_t* out_commitments,
                                     int32_t* out_codes) {
    return prove_entry(st, PROVE_COMMIT, n, blobs, nullptr, out_commitments, nullptr, out_codes);
}

int32_t b200_compute_blob_kzg_proofs(const b200_kzg_settings* st, const uint8_t* blobs, const uint8_t* commitments, size_t n,
                                     uint8_t* out_proofs, int32_t* out_codes) {
    return prove_entry(st, PROVE_BLOB, n, blobs, commitments, out_proofs, nullptr, out_codes);
}

int32_t b200_blob_to_kzg_commitment(const b200_kzg_settings* st, const uint8_t* blob, uint8_t out_commitment[48]) {
    int32_t code = 0;
    const int32_t rc = prove_entry(st, PROVE_COMMIT, 1, blob, nullptr, out_commitment, nullptr, &code);
    return rc ? rc : code;
}

int32_t b200_compute_kzg_proof(const b200_kzg_settings* st, const uint8_t* blob, const uint8_t z[32], uint8_t out_proof[48],
                               uint8_t out_y[32]) {
    int32_t code = 0;
    const int32_t rc = prove_entry(st, PROVE_POINT, 1, blob, z, out_proof, out_y, &code);
    return rc ? rc : code;
}

int32_t b200_compute_blob_kzg_proof(const b200_kzg_settings* st, const uint8_t* blob, const uint8_t commitment[48],
                                    uint8_t out_proof[48]) {
    int32_t code = 0;
    const int32_t rc = prove_entry(st, PROVE_BLOB, 1, blob, commitment, out_proof, nullptr, &code);
    return rc ? rc : code;
}

}  // extern "C"
