// extern "C" entry points — the BLS half of include/b200_consensus.h — and the host orchestration of the batch
// pipeline.  Every function below is a drop-in for one body in
// /root/reference/ethereum-consensus/src/crypto/bls.rs (line ranges in the header); all curve arithmetic runs in
// the kernels of bls_g1.cu / bls_g2.cu / bls_pairing.cu.  The host only stages bytes and index arrays.
//
// Flow for T tuples with NK public keys in total (strict mode):
//   stream A: H2D offsets, keys (100 MB) ........ wait(B,C) | K1 key_validate (NK threads) | K2 per-tuple aggregate
//   stream B: H2D sigs | K3 sig decompress + subgroup check (T threads)   } under the key copy, before K1
//   stream C: H2D msgs | K4 hash_to_G2 (2T + T threads)                   }
//   stream A: K5 Miller loops (2T teams of 8 lanes) | K6 Gt product + final exponentiation (T teams) | D2H codes
// Registry mode skips K1: validated affine keys stay resident in HBM and K2 gathers them by validator index.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "bls_kernels.cuh"
#include "comm.h"
#include "engine.h"
#include "state_handle.h"

namespace b200 {

struct BlsState {
    cudaStream_t sb = nullptr, sc = nullptr;  // signatures / messages: run under the per-key kernel
    // Chunked strict batches (OFF by default): the per-key kernel goes out in `chunks` key ranges on the engine stream, and
    // each range's aggregate -> Miller loops -> final exponentiation chain runs on `sd` UNDER the next range's per-key
    // kernel (B200_BLS_CHUNKS, 1 = one range; B200_BLS_CHUNK_MIN_TUPLES; B200_BLS_CHUNK_K1_CTA = 128 | 384).
    // Measured on B200, T = 4096 x K = 512 (profiles/r2_ab_variants.txt, call 15): one range 130.2 ms; 2 ranges 137.3;
    // 4 ranges 144.4 (138.8 with 384-thread K1 CTAs); 8 ranges 158.1.  The pairing chain does not fit under the per-key
    // kernel: its CTAs need the registers / shared memory of a retiring per-key CTA, both kernels then run at reduced
    // occupancy, and the per-key kernel loses more (114 -> 129 ms) than the 14 ms chain it hides.
    static constexpr uint32_t kMaxChunks = 16;
    cudaStream_t sd = nullptr, se = nullptr;   // se: odd key ranges, so that range c+1's CTAs fill range c's draining tail
    cudaEvent_t ev_ck[kMaxChunks] = {nullptr}, ev_join = nullptr;
    uint32_t chunks = 1, chunk_min_tuples = 2048;
    int chunk_k1_cta = 128;
    bool chunk_alt = true;
    bool key_split = true;   // B200_BLS_KEY_SPLIT / b200_tune("bls_key_split")
    // CTA size of the first (4-wave) per-key launch of a split batch, the one the signature / message kernels run under: as three
    // 128-thread CTAs per SM a side kernel's CTA displaces a third of an SM's per-key work instead of all of it
    // (T = 4096: 116.84 -> 116.43 ms per step, profiles/r2_ab_variants.txt call 32)
    int k1_first_cta = 128;
    cudaEvent_t ev_in = nullptr, ev_b = nullptr, ev_c = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_d0 = nullptr, ev_d1 = nullptr;
    DevBuf keys, key_aff, key_code, g1pts, g1pre, pk_code, flags, sigs, g2pts, sig_code, msgs, small, f, out, h2c_tmp, gath;
    // RLC whole-batch check (bls_rlc.cu): Jacobian aggregates, scaled points, reduction ping-pong, zeros, indices, exchange
    DevBuf rlc_jac, rlc_g1, rlc_q, rlc_fa, rlc_fb, rlc_qa, rlc_qb, rlc_zero, rlc_idx, rlc_misc, rlc_xch;
    PinnedBuf stage;
    G1Aff* d_negg1 = nullptr;
    G1Pre* d_negg1_pre = nullptr;
    // registry (validated keys resident on the device)
    DevBuf reg_aff, reg_code;
    size_t reg_n = 0;
    float last_dominant_ms = 0.f;
    bool trace = false;          // B200_BLS_TRACE=1: per-phase CUDA-event timings on stderr
    cudaEvent_t ev_t[8] = {nullptr};
    // B200_SMALL_ORDER: where the signature / message kernels go relative to the per-key kernel K1: 0 (default) under it on
    // high-priority streams, 1 before it, 2 after it.  Round 1 measured 211 / 199 / 201 ms per step (T=4096, K=512) and ran
    // them first; with round 2's K1 (call-based products: a fifth of the code, 12 warps/SM) the overlap wins:
    // 130.9 / 136.2 ms at T=4096 with 128-thread CTAs, 18.2 / 25.2 ms at T=256 with 32-thread CTAs
    // (profiles/r2_ab_variants.txt).  B200_SMALL_CTA overrides the CTA size (default: 32 up to 1 024 tuples, else 128).
    int small_order = 0;
    int small_cta_override = 0;
    bool use_vm = true;  // lane-parallel pairing kernels (B200_PAIRING_VM=0 selects the one-thread-per-pair kernels)
};

static int32_t bls_state(Engine& e, BlsState** out) {
    if (!e.bls) {
        BlsState* s = new BlsState();
        if (const char* v = getenv("B200_G1_VARIANT")) set_g1_variant(atoi(v));
        if (const char* v = getenv("B200_G1_SMALL_N")) set_g1_small_n(uint32_t(atol(v)));
        if (const char* v = getenv("B200_PAIRING_VM")) s->use_vm = atoi(v) != 0;
        if (const char* v = getenv("B200_BLS_TRACE")) s->trace = atoi(v) != 0;
        if (const char* v = getenv("B200_SMALL_ORDER")) s->small_order = atoi(v);
        if (const char* v = getenv("B200_SMALL_CTA")) s->small_cta_override = atoi(v);
        for (auto& ev : s->ev_t) B200_CUDA_TRY(cudaEventCreate(&ev));
        // High priority only matters for B200_SMALL_ORDER=0 (dispatch under the per-key kernel as its CTAs retire).
        int prio_lo = 0, prio = 0;
        B200_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio));          // highest priority
        if (const char* v = getenv("B200_SMALL_STREAM_PRIORITY")) prio = atoi(v);  // A/B knob
        B200_CUDA_TRY(cudaStreamCreateWithPriority(&s->sb, cudaStreamNonBlocking, prio));
        B200_CUDA_TRY(cudaStreamCreateWithPriority(&s->sc, cudaStreamNonBlocking, prio));
        if (const char* v = getenv("B200_BLS_CHUNKS")) s->chunks = uint32_t(std::max(1, atoi(v)));
        if (const char* v = getenv("B200_BLS_CHUNK_MIN_TUPLES")) s->chunk_min_tuples = uint32_t(std::max(2, atoi(v)));
        if (const char* v = getenv("B200_BLS_CHUNK_K1_CTA")) s->chunk_k1_cta = atoi(v);
        if (const char* v = getenv("B200_BLS_CHUNK_ALT")) s->chunk_alt = atoi(v) != 0;
        if (const char* v = getenv("B200_BLS_KEY_SPLIT")) s->key_split = atoi(v) != 0;
        if (const char* v = getenv("B200_BLS_K1_FIRST_CTA")) s->k1_first_cta = atoi(v) == 384 ? 384 : 128;
        if (const char* v = getenv("B200_BLS_SMALL_CTA")) s->small_cta_override = atoi(v);
        int prio_d = prio;
        if (const char* v = getenv("B200_PAIR_STREAM_PRIORITY")) prio_d = atoi(v);
        B200_CUDA_TRY(cudaStreamCreateWithPriority(&s->sd, cudaStreamNonBlocking, prio_d));
        B200_CUDA_TRY(cudaStreamCreateWithPriority(&s->se, cudaStreamNonBlocking, prio_lo));
        for (auto& ev : s->ev_ck) B200_CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        B200_CUDA_TRY(cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming));
        B200_CUDA_TRY(cudaEventCreateWithFlags(&s->ev_c, cudaEventDisableTiming));
        B200_CUDA_TRY(cudaEventCreateWithFlags(&s->ev_in, cudaEventDisableTiming));
        B200_CUDA_TRY(cudaEventCreateWithFlags(&s->ev_b, cudaEventDisableTiming));
        B200_CUDA_TRY(cudaEventCreate(&s->ev_k0));
        B200_CUDA_TRY(cudaEventCreate(&s->ev_k1));
        B200_CUDA_TRY(cudaEventCreate(&s->ev_d0));
        B200_CUDA_TRY(cudaEventCreate(&s->ev_d1));
        B200_CUDA_TRY(cudaMalloc(&s->d_negg1, sizeof(G1Aff)));
        B200_CUDA_TRY(cudaMalloc(&s->d_negg1_pre, sizeof(G1Pre)));
        launch_neg_g1(s->d_negg1, s->d_negg1_pre, e.stream);
        e.launches++;
        if (vm_init(e.stream) != 0) { e.last_error = "pairing VM initialisation failed"; return B200_ERR_CUDA; }
        e.launches++;
        B200_CUDA_TRY(cudaGetLastError());
        B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
        e.bls = s;
    }
    *out = static_cast<BlsState*>(e.bls);
    return B200_SUCCESS;
}

struct Guard {
    std::unique_lock<std::mutex> lk;
    explicit Guard(Engine& e) : lk(e.mu) {}
};
static int32_t check_ready(Engine& e) {
    if (!e.ready) { e.last_error = "b200_init has not been called (or failed)"; return B200_ERR_NOT_INITIALIZED; }
    cudaError_t ce = cudaSetDevice(e.device);
    if (ce != cudaSuccess) { e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    return B200_SUCCESS;
}

enum PairMode { MODE_FAST_AGGREGATE = 0, MODE_AGGREGATE = 1 };
// message offsets travel as uint32 (32 bytes per tuple on the batch paths): 32 * T must not wrap
constexpr size_t kMaxBatchTuples = size_t(1) << 26;
// keys a `..._batch_mixed` call may bring along (a block carries <= 16 deposits + 16 bls-to-execution changes)
constexpr size_t kRegistryExtraKeys = size_t(1) << 16;

// Core: `n_tuples` tuples.  MODE_FAST_AGGREGATE: tuple t sums keys [key_off[t], key_off[t+1]) and checks
// e(sum, H(msg_t)) e(-g1, sig_t) == 1.  MODE_AGGREGATE: one tuple, pairs (key_i, H(msg_i)) + (-g1, sig).
// keys: host bytes (strict) or nullptr with `index` (registry gather).  msgs: host bytes + offsets (n_msgs + 1).
// whole-batch RLC request: when passed, the pairing phase answers ONE boolean for all tuples instead of T codes
struct RlcReq {
    const uint8_t* seed32;  // scalars r_t = H(seed || t0 + t)
    uint64_t t0;            // global index of this call's first tuple (sharded batches)
    bool exchange;          // all-gather the per-rank (Gt, G2) partials over the library's communicator
    int32_t all_ok;         // out
};
static int32_t run_verify_impl(Engine& e, BlsState& s, PairMode mode, const uint8_t* keys, uint32_t n_keys,
                               const uint32_t* index, uint32_t n_index, const uint32_t* key_off, const uint8_t* msgs,
                               const uint32_t* msg_off, uint32_t n_msgs, const uint8_t* sigs, uint32_t n_tuples,
                               bool force_fail_shape, int32_t* out_codes, RlcReq* rlc);
// An early error return must not leave work queued on the side streams (they read the caller's host buffers and the
// engine's grow-only device buffers): drain all three before handing the error back.
static int32_t run_verify(Engine& e, BlsState& s, PairMode mode, const uint8_t* keys, uint32_t n_keys,
                          const uint32_t* index, uint32_t n_index, const uint32_t* key_off, const uint8_t* msgs,
                          const uint32_t* msg_off, uint32_t n_msgs, const uint8_t* sigs, uint32_t n_tuples,
                          bool force_fail_shape, int32_t* out_codes, RlcReq* rlc = nullptr) {
    const int32_t rc = run_verify_impl(e, s, mode, keys, n_keys, index, n_index, key_off, msgs, msg_off, n_msgs, sigs,
                                       n_tuples, force_fail_shape, out_codes, rlc);
    if (rc != B200_SUCCESS) {
        cudaStreamSynchronize(e.stream);
        cudaStreamSynchronize(s.sb);
        cudaStreamSynchronize(s.sc);
        cudaStreamSynchronize(s.sd);
        cudaStreamSynchronize(s.se);
        cudaGetLastError();
    }
    return rc;
}
static int32_t run_verify_impl(Engine& e, BlsState& s, PairMode mode, const uint8_t* keys, uint32_t n_keys,
                               const uint32_t* index, uint32_t n_index, const uint32_t* key_off, const uint8_t* msgs,
                               const uint32_t* msg_off, uint32_t n_msgs, const uint8_t* sigs, uint32_t n_tuples,
                               bool force_fail_shape, int32_t* out_codes, RlcReq* rlc) {
    if (rlc && (mode != MODE_FAST_AGGREGATE || !s.use_vm)) return B200_ERR_BAD_ARG;
    // registry gather; with `keys` as well: `n_keys` EXTRA keys (deposits, bls-to-execution changes) validated by this call into
    // the registry arrays' spare tail, named by indices reg_n + j
    const bool registry = index != nullptr;
    const uint32_t T = n_tuples;
    const uint32_t n_g1 = (mode == MODE_FAST_AGGREGATE ? T : n_keys) + 1;  // + (-g1)
    const uint32_t n_pairs = (mode == MODE_FAST_AGGREGATE) ? 2 * T : (force_fail_shape ? 0 : n_msgs + 1);
    const uint32_t n_g2 = n_msgs + T;
    const uint32_t msg_bytes = msg_off[n_msgs];

    // ---- device buffers
    B200_CUDA_TRY(s.keys.reserve(size_t(n_keys) * 48 + 64));
    B200_CUDA_TRY(s.key_aff.reserve(size_t(n_keys + 1) * sizeof(G1Aff)));
    B200_CUDA_TRY(s.key_code.reserve(size_t(n_keys + 1) * 4));
    B200_CUDA_TRY(s.g1pts.reserve(size_t(n_g1) * sizeof(G1Aff)));
    B200_CUDA_TRY(s.g1pre.reserve(size_t(n_g1) * sizeof(G1Pre)));
    B200_CUDA_TRY(s.pk_code.reserve(size_t(T + 1) * 4));
    B200_CUDA_TRY(s.flags.reserve(size_t(T + 1) * 4));
    B200_CUDA_TRY(s.sigs.reserve(size_t(T) * 96 + 64));
    B200_CUDA_TRY(s.g2pts.reserve(size_t(n_g2 + 1) * sizeof(G2Aff)));
    B200_CUDA_TRY(s.sig_code.reserve(size_t(T + 1) * 4));
    B200_CUDA_TRY(s.msgs.reserve(size_t(msg_bytes) + 64));
    B200_CUDA_TRY(s.f.reserve(size_t(n_pairs + 1) * sizeof(Fp12)));
    B200_CUDA_TRY(s.out.reserve(size_t(T + 1) * 4));
    B200_CUDA_TRY(s.h2c_tmp.reserve(size_t(2 * n_msgs + 2) * sizeof(G2Jac)));
    const uint32_t rlc_world = rlc && rlc->exchange ? uint32_t(comm().world) : 1u;
    const uint32_t rlc_part = (T + 31) / 32 + rlc_world + 2;   // capacity of one reduction level (+ gathered partials)
    if (rlc) {
        B200_CUDA_TRY(s.rlc_jac.reserve(size_t(T + 1) * sizeof(G1Jac)));
        B200_CUDA_TRY(s.rlc_g1.reserve(size_t(T + 2) * sizeof(G1Pre)));
        B200_CUDA_TRY(s.rlc_q.reserve(size_t(T + 1) * sizeof(G2Jac)));
        B200_CUDA_TRY(s.rlc_fa.reserve(size_t(rlc_part) * sizeof(Fp12)));
        B200_CUDA_TRY(s.rlc_fb.reserve(size_t(rlc_part) * sizeof(Fp12)));
        B200_CUDA_TRY(s.rlc_qa.reserve(size_t(rlc_part) * sizeof(G2Jac)));
        B200_CUDA_TRY(s.rlc_qb.reserve(size_t(rlc_part) * sizeof(G2Jac)));
        B200_CUDA_TRY(s.rlc_zero.reserve(size_t(T + 8) * 4));
        B200_CUDA_TRY(s.rlc_idx.reserve(size_t(2 * (T + 1)) * 4));
        B200_CUDA_TRY(s.rlc_misc.reserve(256));
        B200_CUDA_TRY(s.rlc_xch.reserve(size_t(rlc_world + 1) * (sizeof(Fp12) + sizeof(G2Jac) + 16)));
    }

    // ---- small host-built arrays, one staged copy: [key_off | index | msg_off | g1_idx | g2_idx | pair_tuple | pair_off]
    const uint32_t n_koff = (mode == MODE_FAST_AGGREGATE) ? T + 1 : 2;
    std::vector<uint32_t> small;
    small.reserve(size_t(n_koff) + n_index + n_msgs + 1 + 3 * size_t(n_pairs) + T + 1 + 8);
    const size_t o_koff = small.size();
    if (mode == MODE_FAST_AGGREGATE) small.insert(small.end(), key_off, key_off + T + 1);
    else { small.push_back(0); small.push_back(n_keys); }
    const size_t o_index = small.size();
    if (registry) small.insert(small.end(), index, index + n_index);
    const size_t o_moff = small.size();
    small.insert(small.end(), msg_off, msg_off + n_msgs + 1);
    const size_t o_g1i = small.size();
    small.resize(small.size() + 3 * size_t(n_pairs) + T + 1);
    uint32_t* g1i = small.data() + o_g1i;
    uint32_t* g2i = g1i + n_pairs;
    uint32_t* ptu = g2i + n_pairs;
    uint32_t* poff = ptu + n_pairs;
    if (mode == MODE_FAST_AGGREGATE) {
        for (uint32_t t = 0; t < T; t++) {
            g1i[2 * t] = t;          g2i[2 * t] = t;          // (agg_t, H(msg_t))
            g1i[2 * t + 1] = T;      g2i[2 * t + 1] = n_msgs + t;  // (-g1, sig_t)
            ptu[2 * t] = ptu[2 * t + 1] = t;
            poff[t] = 2 * t;
        }
        poff[T] = 2 * T;
    } else {
        for (uint32_t i = 0; i + 1 < n_pairs; i++) { g1i[i] = i; g2i[i] = i; ptu[i] = 0; }
        if (n_pairs) { g1i[n_pairs - 1] = n_keys; g2i[n_pairs - 1] = n_msgs; ptu[n_pairs - 1] = 0; }
        poff[0] = 0; poff[1] = n_pairs;
    }
    const size_t small_bytes = small.size() * 4;
    const size_t kRlcPart = sizeof(Fp12) + sizeof(G2Jac) + 16;   // one rank's exchanged partial: Gt | G2 | bad flag
    B200_CUDA_TRY(s.stage.reserve(small_bytes + size_t(T + 1) * 4 + 64 +
                                  (rlc ? 256 + size_t(rlc_world) * kRlcPart + size_t(8 + 2 * (T + 1)) * 4 : 0)));
    B200_CUDA_TRY(s.small.reserve(small_bytes + 64));
    memcpy(s.stage.p, small.data(), small_bytes);
    int32_t* h_out = reinterpret_cast<int32_t*>(static_cast<uint8_t*>(s.stage.p) + ((small_bytes + 15) & ~size_t(15)));

    cudaStream_t sa = e.stream, sb = s.sb, sc = s.sc;
    uint32_t* d_small = static_cast<uint32_t*>(s.small.p);
    G1Aff* d_g1 = static_cast<G1Aff*>(s.g1pts.p);
    G2Aff* d_g2 = static_cast<G2Aff*>(s.g2pts.p);
    const G1Aff* key_aff = registry ? static_cast<const G1Aff*>(s.reg_aff.p) : static_cast<const G1Aff*>(s.key_aff.p);
    const int32_t* key_code = registry ? static_cast<const int32_t*>(s.reg_code.p) : static_cast<const int32_t*>(s.key_code.p);
    // where the per-key kernel writes: the call's own arrays, or (registry + extra keys) the tail behind the reg_n resident keys
    G1Aff* k1_aff = registry ? static_cast<G1Aff*>(s.reg_aff.p) + s.reg_n : static_cast<G1Aff*>(s.key_aff.p);
    int32_t* k1_code = registry ? static_cast<int32_t*>(s.reg_code.p) + s.reg_n : static_cast<int32_t*>(s.key_code.p);

    // ---- small arrays + keys (stream A); signatures / messages on streams B, C (they overlap the 100 MB key copy)
    B200_CUDA_TRY(cudaMemcpyAsync(d_small, s.stage.p, small_bytes, cudaMemcpyHostToDevice, sa));
    B200_CUDA_TRY(cudaEventRecord(s.ev_in, sa));
    const bool have_k1 = n_keys != 0;
    const uint32_t n_chunks = (mode == MODE_FAST_AGGREGATE && !rlc && s.use_vm && have_k1 && !registry && s.small_order == 0 && !force_fail_shape &&
                               s.chunks > 1 && T >= s.chunk_min_tuples) ? std::min(s.chunks, BlsState::kMaxChunks) : 1u;
    // Big strict batches: the first kSplitWaves full waves of the per-key kernel start as soon as THEIR keys have arrived; the rest of
    // the key bytes (~90 MB at T = 4096) cross PCIe on stream E under that first launch, and the second launch follows them there
    // (two streams, so its CTAs fill the first launch's draining tail).  b200_tune("bls_key_split", 0) restores the single copy.
    constexpr uint32_t kSplitWaves = 4, kSplitKeys = kSplitWaves * 148u * 384u;
    const uint32_t k_split = (s.key_split && have_k1 && !registry && n_chunks == 1 && s.small_order == 0 && n_keys >= 4u * kSplitKeys)
                                 ? kSplitKeys : n_keys;
    if (n_keys) B200_CUDA_TRY(cudaMemcpyAsync(s.keys.p, keys, size_t(k_split) * 48, cudaMemcpyHostToDevice, sa));
    B200_CUDA_TRY(cudaEventRecord(s.ev_k0, sa));
    auto launch_small = [&]() -> int32_t {
        B200_CUDA_TRY(cudaStreamWaitEvent(sb, s.ev_in, 0));
        B200_CUDA_TRY(cudaStreamWaitEvent(sc, s.ev_in, 0));
        if (T) B200_CUDA_TRY(cudaMemcpyAsync(s.sigs.p, sigs, size_t(T) * 96, cudaMemcpyHostToDevice, sb));
        if (msg_bytes) B200_CUDA_TRY(cudaMemcpyAsync(s.msgs.p, msgs, msg_bytes, cudaMemcpyHostToDevice, sc));
        launch_g2_sig_decode(static_cast<const uint8_t*>(s.sigs.p), T, d_g2 + n_msgs, static_cast<int32_t*>(s.sig_code.p), sb);
        launch_hash_to_g2(static_cast<const uint8_t*>(s.msgs.p), d_small + o_moff, n_msgs, d_g2, s.h2c_tmp.p, sc);
        e.launches += (T ? 1 : 0) + (n_msgs ? 2 : 0);
        B200_CUDA_TRY(cudaEventRecord(s.ev_b, sb));
        B200_CUDA_TRY(cudaEventRecord(s.ev_c, sc));
        return B200_SUCCESS;
    };
    // packed CTAs only when there is a big per-key kernel to run under; alone (registry mode, small batches) they spread
    set_small_cta(s.small_cta_override ? s.small_cta_override : ((have_k1 && n_keys >= 148u * 384u && s.small_order == 0 && T > 1024) ? 128 : 32));
    if (have_k1 && s.small_order == 1) {   // signatures / messages first, the per-key kernel only afterwards
        int32_t rc = launch_small();
        if (rc) return rc;
        B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_b, 0));
        B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_c, 0));
    }
    // ---- stream A: public keys
    B200_CUDA_TRY(cudaEventRecord(s.ev_d0, sa));
    const uint32_t* d_g1i = nullptr; const uint32_t* d_g2i = nullptr; const uint32_t* d_ptu = nullptr; const uint32_t* d_poff = nullptr;
    bool chunked = false;
    const G1Aff* pair_g1 = d_g1;
    if (n_chunks > 1) {
        // Chunked strict batch: tuple range c's keys are validated on stream A while range c-1's aggregate -> Miller ->
        // final-exponentiation chain (latency-bound: ~1/3 of the IMAD pipe when alone) runs on stream D in the slots the
        // per-key kernel's retiring 128-thread CTAs leave.  Same kernels, same per-tuple arithmetic, same code vector.
        chunked = true;
        cudaStream_t sd = s.sd;
        d_g1i = d_small + o_g1i; d_g2i = d_g1i + n_pairs; d_ptu = d_g2i + n_pairs; d_poff = d_ptu + n_pairs;
        uint32_t tb[BlsState::kMaxChunks + 1];
        for (uint32_t c = 0; c <= n_chunks; c++) tb[c] = uint32_t(uint64_t(T) * c / n_chunks);
        B200_CUDA_TRY(cudaStreamWaitEvent(s.se, s.ev_k0, 0));   // the key bytes
        for (uint32_t c = 0; c < n_chunks; c++) {
            const uint32_t k0 = key_off[tb[c]], k1 = key_off[tb[c + 1]];
            cudaStream_t sk = ((c & 1u) && s.chunk_alt) ? s.se : sa;
            launch_g1_validate(static_cast<const uint8_t*>(s.keys.p) + size_t(k0) * 48, k1 - k0, static_cast<G1Aff*>(s.key_aff.p) + k0,
                               static_cast<int32_t*>(s.key_code.p) + k0, sk, s.chunk_k1_cta);
            if (k1 > k0) e.launches++;
            B200_CUDA_TRY(cudaEventRecord(s.ev_ck[c], sk));
            if (c == 0) {   // signature / message kernels right behind the first range, as in the one-range flow
                int32_t rc = launch_small();
                if (rc) return rc;
            }
        }
        if (s.chunk_alt)
            for (uint32_t c = 1; c < n_chunks; c += 2) B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_ck[c], 0));
        B200_CUDA_TRY(cudaEventRecord(s.ev_d1, sa));
        B200_CUDA_TRY(cudaStreamWaitEvent(sd, s.ev_in, 0));   // the small index arrays
        B200_CUDA_TRY(cudaStreamWaitEvent(sd, s.ev_b, 0));
        B200_CUDA_TRY(cudaStreamWaitEvent(sd, s.ev_c, 0));
        B200_CUDA_TRY(cudaMemcpyAsync(static_cast<G1Pre*>(s.g1pre.p) + T, s.d_negg1_pre, sizeof(G1Pre), cudaMemcpyDeviceToDevice, sd));
        int32_t* d_pk = static_cast<int32_t*>(s.pk_code.p);
        uint32_t* d_fl = static_cast<uint32_t*>(s.flags.p);
        const int32_t* d_sc = static_cast<const int32_t*>(s.sig_code.p);
        for (uint32_t c = 0; c < n_chunks; c++) {
            const uint32_t t0 = tb[c], nt = tb[c + 1] - tb[c];
            if (!nt) continue;
            B200_CUDA_TRY(cudaStreamWaitEvent(sd, s.ev_ck[c], 0));
            launch_g1_aggregate(key_aff, key_code, nullptr, d_small + o_koff + t0, nt, nullptr, static_cast<G1Pre*>(s.g1pre.p) + t0,
                                d_pk + t0, d_fl + t0, 0u, sd, nullptr);
            // pair-indexed arrays start at 2 t0 (values are absolute); tuple-indexed code arrays are read through pair_tuple
            launch_vm_miller(static_cast<const G1Pre*>(s.g1pre.p), d_g1i + 2 * t0, d_g2, d_g2i + 2 * t0, d_ptu + 2 * t0, d_pk, d_fl, d_sc,
                             2 * nt, static_cast<Fp12*>(s.f.p) + 2 * size_t(t0), sd);
            // f BASE + absolute pair offsets; tuple-indexed arrays start at t0
            launch_vm_final(static_cast<const Fp12*>(s.f.p), d_poff + t0, d_pk + t0, d_fl + t0, d_sc + t0, nt,
                            static_cast<int32_t*>(s.out.p) + t0, sd);
            e.launches += 3;
        }
        B200_CUDA_TRY(cudaEventRecord(s.ev_join, sd));
        B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_join, 0));
        if (s.trace) { cudaEventRecord(s.ev_t[0], sa); cudaEventRecord(s.ev_t[1], sa); cudaEventRecord(s.ev_t[2], sa); cudaEventRecord(s.ev_t[3], sa); }
    }
    if (!chunked) {
        if (have_k1) {
            launch_g1_validate(static_cast<const uint8_t*>(s.keys.p), k_split, k1_aff, k1_code, sa, k_split < n_keys ? s.k1_first_cta : 0);
            e.launches++;
        }
        if (!(have_k1 && s.small_order == 1)) {
            if (have_k1 && s.small_order == 2) {  // strictly after the per-key kernel
                B200_CUDA_TRY(cudaEventRecord(s.ev_in, sa));
            }
            int32_t rc = launch_small();
            if (rc) return rc;
        }
        if (k_split < n_keys) {   // the remaining keys: copy strictly after the first part's (one PCIe link), then their launch
            B200_CUDA_TRY(cudaStreamWaitEvent(s.se, s.ev_k0, 0));
            B200_CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(s.keys.p) + size_t(k_split) * 48, keys + size_t(k_split) * 48,
                                          size_t(n_keys - k_split) * 48, cudaMemcpyHostToDevice, s.se));
            launch_g1_validate(static_cast<const uint8_t*>(s.keys.p) + size_t(k_split) * 48, n_keys - k_split, k1_aff + k_split,
                               k1_code + k_split, s.se, 384);
            e.launches++;
            B200_CUDA_TRY(cudaEventRecord(s.ev_ck[0], s.se));
            B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_ck[0], 0));
        }
        B200_CUDA_TRY(cudaEventRecord(s.ev_d1, sa));
        if (s.trace) cudaEventRecord(s.ev_t[0], sa);
        const uint32_t n_agg_tuples = (mode == MODE_FAST_AGGREGATE) ? T : 1;
        launch_g1_aggregate(key_aff, key_code, registry ? d_small + o_index : nullptr, d_small + o_koff, n_agg_tuples,
                            (mode == MODE_FAST_AGGREGATE && !s.use_vm) ? d_g1 : nullptr,
                            (mode == MODE_FAST_AGGREGATE && s.use_vm) ? static_cast<G1Pre*>(s.g1pre.p) : nullptr,
                            static_cast<int32_t*>(s.pk_code.p), static_cast<uint32_t*>(s.flags.p),
                            force_fail_shape ? uint32_t(TUPLE_FLAG_EMPTY) : 0u, sa,
                            rlc ? static_cast<G1Jac*>(s.rlc_jac.p) : nullptr);
        e.launches++;
        if (mode == MODE_FAST_AGGREGATE) {
            B200_CUDA_TRY(cudaMemcpyAsync(d_g1 + T, s.d_negg1, sizeof(G1Aff), cudaMemcpyDeviceToDevice, sa));
            B200_CUDA_TRY(cudaMemcpyAsync(static_cast<G1Pre*>(s.g1pre.p) + T, s.d_negg1_pre, sizeof(G1Pre), cudaMemcpyDeviceToDevice, sa));
        } else {
            G1Aff* ka = static_cast<G1Aff*>(s.key_aff.p);
            B200_CUDA_TRY(cudaMemcpyAsync(ka + n_keys, s.d_negg1, sizeof(G1Aff), cudaMemcpyDeviceToDevice, sa));
            pair_g1 = ka;  // len(msgs) != len(pks) or no keys: flagged EMPTY above -> VERIFY_FAIL after the decoding checks
        }
        // ---- join, pairing
        if (s.trace) cudaEventRecord(s.ev_t[1], sa);
        B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_b, 0));
        B200_CUDA_TRY(cudaStreamWaitEvent(sa, s.ev_c, 0));
        if (s.trace) cudaEventRecord(s.ev_t[2], sa);
    }
    d_g1i = d_small + o_g1i;
    d_g2i = d_g1i + n_pairs;
    d_ptu = d_g2i + n_pairs;
    d_poff = d_ptu + n_pairs;
    if (rlc) {
        // ---- RLC whole-batch check (bls_rlc.cu): T Miller loops + ONE final exponentiation
        const size_t kPart = kRlcPart;
        uint8_t* h_x = reinterpret_cast<uint8_t*>(h_out + 16);                    // gathered partials (their bad flags are read on the host)
        uint32_t* d_zero = static_cast<uint32_t*>(s.rlc_zero.p);  // "every tuple alive" code arrays for the VM kernels
        uint32_t* d_idx = static_cast<uint32_t*>(s.rlc_idx.p);   // [0..T] identity (g1 / tuple index) | [0..T-1, n_g2] (H_t, then S)
        uint8_t* d_misc = static_cast<uint8_t*>(s.rlc_misc.p);    // [0,32) seed words | [32,36) bad flag | [64,68) final code
        G1Pre* d_rg1 = static_cast<G1Pre*>(s.rlc_g1.p);
        G2Jac* d_rq = static_cast<G2Jac*>(s.rlc_q.p);
        B200_CUDA_TRY(cudaMemsetAsync(d_zero, 0, size_t(T + 8) * 4, sa));
        B200_CUDA_TRY(cudaMemsetAsync(d_misc + 32, 0, 96, sa));
        {   // seed words + index arrays through the pinned staging area (behind the small arrays and the code slots)
            uint32_t* h = reinterpret_cast<uint32_t*>(h_x + ((size_t(rlc_world) * kPart + 63) & ~size_t(63)));
            for (int i = 0; i < 8; i++)
                h[i] = (uint32_t(rlc->seed32[4 * i]) << 24) | (uint32_t(rlc->seed32[4 * i + 1]) << 16) | (uint32_t(rlc->seed32[4 * i + 2]) << 8) | rlc->seed32[4 * i + 3];
            uint32_t* hi = h + 8;
            for (uint32_t t = 0; t <= T; t++) { hi[t] = t; hi[T + 1 + t] = t < T ? t : n_g2; }
            B200_CUDA_TRY(cudaMemcpyAsync(d_misc, h, 32, cudaMemcpyHostToDevice, sa));
            B200_CUDA_TRY(cudaMemcpyAsync(d_idx, hi, size_t(2 * (T + 1)) * 4, cudaMemcpyHostToDevice, sa));
        }
        launch_rlc_scale(static_cast<const G1Jac*>(s.rlc_jac.p), d_g2 + n_msgs, static_cast<const int32_t*>(s.pk_code.p),
                         static_cast<const uint32_t*>(s.flags.p), static_cast<const int32_t*>(s.sig_code.p),
                         reinterpret_cast<const uint32_t*>(d_misc), rlc->t0, T, d_rg1, d_rq, reinterpret_cast<int32_t*>(d_misc + 32), sa);
        B200_CUDA_TRY(cudaMemcpyAsync(d_rg1 + T, s.d_negg1_pre, sizeof(G1Pre), cudaMemcpyDeviceToDevice, sa));
        if (s.trace) cudaEventRecord(s.ev_t[3], sa);
        Fp12* fbuf[2] = {static_cast<Fp12*>(s.rlc_fa.p), static_cast<Fp12*>(s.rlc_fb.p)};
        G2Jac* qbuf[2] = {static_cast<G2Jac*>(s.rlc_qa.p), static_cast<G2Jac*>(s.rlc_qb.p)};
        // S = sum_t r_t sig_t first (warp-shuffle folds T -> T/32 -> ... -> 1): its pair (-g1, S) then rides in the SAME
        // Miller launch as the T tuple pairs instead of costing a second, latency-bound launch of one team
        const G2Jac* qi = d_rq;
        uint32_t n_cur = T;
        int pp = 0;
        do {
            n_cur = launch_rlc_reduce(nullptr, qi, n_cur, nullptr, qbuf[pp], sa);
            e.launches++;
            qi = qbuf[pp]; pp ^= 1;
        } while (n_cur > 1);
        launch_rlc_finish(qi, d_g2 + n_g2, sa);
        // T + 1 Miller loops on the lane-parallel VM: (r_t agg_t, H_t) for every tuple and (-g1, S)
        launch_vm_miller(d_rg1, d_idx, d_g2, d_idx + T + 1, d_zero, reinterpret_cast<const int32_t*>(d_zero), d_zero,
                         reinterpret_cast<const int32_t*>(d_zero), T + 1, static_cast<Fp12*>(s.f.p), sa);
        // Gt product of the T + 1 Miller values, again by warp-shuffle folds
        const Fp12* fi = static_cast<const Fp12*>(s.f.p);
        n_cur = T + 1;
        pp = 0;
        do {
            n_cur = launch_rlc_reduce(fi, nullptr, n_cur, fbuf[pp], nullptr, sa);
            e.launches++;
            fi = fbuf[pp]; pp ^= 1;
        } while (n_cur > 1);
        if (rlc->exchange && rlc_world > 1) {
            // the path's one exchange step: e(-g1, sum over ranks) = product over ranks, so every rank has already paired
            // its own partial sum and only the Gt partial (576 B) and the bad flag travel; then the same fold on all ranks
            uint8_t* x = static_cast<uint8_t*>(s.rlc_xch.p);
            B200_CUDA_TRY(cudaMemcpyAsync(x, fi, sizeof(Fp12), cudaMemcpyDeviceToDevice, sa));
            B200_CUDA_TRY(cudaMemcpyAsync(x + sizeof(Fp12) + sizeof(G2Jac), d_misc + 32, 16, cudaMemcpyDeviceToDevice, sa));
            int32_t rcx = comm_all_gather(e, x, x + kPart, kPart, sa);
            if (rcx) return rcx;
            for (uint32_t r = 0; r < rlc_world; r++)   // unpack into the fold's input array (world <= a few dozen)
                B200_CUDA_TRY(cudaMemcpyAsync(fbuf[pp] + r, x + kPart * (1 + r), sizeof(Fp12), cudaMemcpyDeviceToDevice, sa));
            B200_CUDA_TRY(cudaMemcpyAsync(h_x, x + kPart, size_t(rlc_world) * kPart, cudaMemcpyDeviceToHost, sa));   // for the ranks' bad flags
            fi = fbuf[pp]; pp ^= 1;
            n_cur = rlc_world;
            do {
                n_cur = launch_rlc_reduce(fi, nullptr, n_cur, fbuf[pp], nullptr, sa);
                e.launches++;
                fi = fbuf[pp]; pp ^= 1;
            } while (n_cur > 1);
        }
        // the single final exponentiation: (Gt product) * 1
        Fp12* d_fin = fbuf[pp];
        B200_CUDA_TRY(cudaMemcpyAsync(d_fin, fi, sizeof(Fp12), cudaMemcpyDeviceToDevice, sa));
        launch_fp12_one(d_fin + 1, sa);
        launch_vm_final(d_fin, d_zero, reinterpret_cast<const int32_t*>(d_zero), d_zero, reinterpret_cast<const int32_t*>(d_zero), 1,
                        reinterpret_cast<int32_t*>(d_misc + 64), sa);
        e.launches += 5;
        B200_CUDA_TRY(cudaEventRecord(s.ev_k1, sa));
        B200_CUDA_TRY(cudaGetLastError());
        B200_CUDA_TRY(cudaMemcpyAsync(h_out, d_misc + 32, 64, cudaMemcpyDeviceToHost, sa));   // [0] bad, [8] final code
        B200_CUDA_TRY(cudaStreamSynchronize(sa));
        B200_CUDA_TRY(cudaStreamSynchronize(sb));
        B200_CUDA_TRY(cudaStreamSynchronize(sc));
        B200_CUDA_TRY(cudaEventElapsedTime(&e.last_kernel_ms, s.ev_k0, s.ev_k1));
        B200_CUDA_TRY(cudaEventElapsedTime(&s.last_dominant_ms, s.ev_d0, s.ev_d1));
        bool bad = h_out[0] != 0;
        if (rlc->exchange && rlc_world > 1)
            for (uint32_t r = 0; r < rlc_world; r++) {
                int32_t flag;
                memcpy(&flag, h_x + size_t(r) * kPart + sizeof(Fp12) + sizeof(G2Jac), 4);
                bad = bad || flag != 0;
            }
        rlc->all_ok = (!bad && h_out[8] == BLS_SUCCESS) ? 1 : 0;
        if (s.trace) {
            float a = 0, g2 = 0;
            cudaEventElapsedTime(&a, s.ev_t[2], s.ev_k1); cudaEventElapsedTime(&g2, s.ev_k0, s.ev_k1);
            fprintf(stderr, "[b200 bls rlc] K1 %.2f | scale + T Miller loops + folds + 1 final exponentiation %.2f | total %.2f ms\n",
                    s.last_dominant_ms, a, g2);
        }
        return B200_SUCCESS;
    }
    if (chunked) {
        // every range's Miller loops and final exponentiations are already queued on stream D (joined above)
    } else if (mode == MODE_FAST_AGGREGATE && s.use_vm) {
        launch_vm_miller(static_cast<const G1Pre*>(s.g1pre.p), d_g1i, d_g2, d_g2i, d_ptu, static_cast<const int32_t*>(s.pk_code.p),
                         static_cast<const uint32_t*>(s.flags.p), static_cast<const int32_t*>(s.sig_code.p), n_pairs,
                         static_cast<Fp12*>(s.f.p), sa);
        if (s.trace) cudaEventRecord(s.ev_t[3], sa);
        launch_vm_final(static_cast<const Fp12*>(s.f.p), d_poff, static_cast<const int32_t*>(s.pk_code.p),
                        static_cast<const uint32_t*>(s.flags.p), static_cast<const int32_t*>(s.sig_code.p), T,
                        static_cast<int32_t*>(s.out.p), sa);
    } else {
        launch_miller(pair_g1, d_g1i, d_g2, d_g2i, d_ptu, static_cast<const int32_t*>(s.pk_code.p),
                      static_cast<const uint32_t*>(s.flags.p), static_cast<const int32_t*>(s.sig_code.p), n_pairs,
                      static_cast<Fp12*>(s.f.p), sa);
        launch_final(static_cast<const Fp12*>(s.f.p), d_poff, static_cast<const int32_t*>(s.pk_code.p),
                     static_cast<const uint32_t*>(s.flags.p), static_cast<const int32_t*>(s.sig_code.p), T,
                     static_cast<int32_t*>(s.out.p), sa);
    }
    if (!chunked) e.launches += (n_pairs ? 1 : 0) + (T ? 1 : 0);
    B200_CUDA_TRY(cudaEventRecord(s.ev_k1, sa));
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(h_out + 4, s.out.p, size_t(T) * 4, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sb));
    B200_CUDA_TRY(cudaStreamSynchronize(sc));
    if (chunked) B200_CUDA_TRY(cudaStreamSynchronize(s.sd));
    B200_CUDA_TRY(cudaEventElapsedTime(&e.last_kernel_ms, s.ev_k0, s.ev_k1));
    B200_CUDA_TRY(cudaEventElapsedTime(&s.last_dominant_ms, s.ev_d0, s.ev_d1));
    if (s.trace) {
        float a = 0, b = 0, c = 0, d = 0, f2 = 0, g2 = 0;
        cudaEventElapsedTime(&a, s.ev_k0, s.ev_d0); cudaEventElapsedTime(&b, s.ev_t[0], s.ev_t[1]);
        cudaEventElapsedTime(&c, s.ev_t[1], s.ev_t[2]); cudaEventElapsedTime(&d, s.ev_t[2], s.ev_t[3]);
        cudaEventElapsedTime(&f2, s.ev_t[3], s.ev_k1); cudaEventElapsedTime(&g2, s.ev_k0, s.ev_k1);
        fprintf(stderr, "[b200 bls] pre-K1 %.2f | K1 %.2f | K2 %.2f | wait(streamB) %.2f | miller %.2f | final %.2f | total %.2f ms\n",
                a, s.last_dominant_ms, b, c, d, f2, g2);
    }
    for (uint32_t t = 0; t < T; t++) out_codes[t] = h_out[4 + t];
    return B200_SUCCESS;
}

}  // namespace b200

using namespace b200;

extern "C" {

int32_t b200_tune(const char* knob, int64_t value) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    if (!knob) return B200_ERR_BAD_ARG;
    const std::string k(knob);
    if (k == "bls_chunks") s->chunks = uint32_t(std::max<int64_t>(1, value));
    else if (k == "bls_chunk_min_tuples") s->chunk_min_tuples = uint32_t(std::max<int64_t>(2, value));
    else if (k == "bls_chunk_k1_cta") s->chunk_k1_cta = int(value);
    else if (k == "bls_chunk_alt") s->chunk_alt = value != 0;
    else if (k == "bls_key_split") s->key_split = value != 0;
    else if (k == "bls_k1_first_cta") s->k1_first_cta = (value == 128) ? 128 : 384;
    else if (k == "bls_small_cta") s->small_cta_override = int(value);
    else if (k == "vm_team16_max") set_vm_team16_max(uint32_t(std::max<int64_t>(0, value)));
    else if (k == "vm_cta") set_vm_cta(int(value));
    else return B200_ERR_BAD_ARG;
    return B200_SUCCESS;
}

int32_t b200_vm_load_programs(const uint32_t* blob, size_t n_words) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    if (vm_load_programs(blob, n_words, e.stream) != 0) { e.last_error = "malformed pairing-VM program blob"; return B200_ERR_BAD_ARG; }
    return B200_SUCCESS;
}

float b200_last_dominant_kernel_ms(void) {
    Engine& e = engine();
    return e.bls ? static_cast<BlsState*>(e.bls)->last_dominant_ms : 0.f;
}

int32_t b200_fp_selftest(uint32_t n, uint32_t seed, uint32_t* mismatches) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!mismatches) return B200_ERR_BAD_ARG;
    uint32_t* d = nullptr;
    B200_CUDA_TRY(cudaMalloc(&d, 4));
    B200_CUDA_TRY(cudaMemsetAsync(d, 0, 4, e.stream));
    launch_fp_selftest(n, seed, d, e.stream);
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(mismatches, d, 4, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    cudaFree(d);
    return B200_SUCCESS;
}

int32_t b200_fast_aggregate_verify_batch(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                         const uint8_t* sigs, size_t n_tuples, int32_t* out_codes) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (n_tuples == 0) return B200_SUCCESS;
    if (!pk_offsets || !msgs32 || !sigs || !out_codes || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    for (size_t t = 0; t < n_tuples; t++)
        if (pk_offsets[t] > pk_offsets[t + 1]) return B200_ERR_BAD_ARG;
    const uint32_t nk = pk_offsets[n_tuples];
    if (nk && !pks_flat) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    std::vector<uint32_t> moff(n_tuples + 1);
    for (size_t t = 0; t <= n_tuples; t++) moff[t] = uint32_t(32 * t);
    return run_verify(e, *s, MODE_FAST_AGGREGATE, pks_flat, nk, nullptr, 0, pk_offsets, msgs32, moff.data(),
                      uint32_t(n_tuples), sigs, uint32_t(n_tuples), false, out_codes);
}

// BASELINE configs[4]: the batch sharded over the communicator's ranks; verdicts exchanged with one ncclAllGather.
int32_t b200_fast_aggregate_verify_batch_sharded(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                                 const uint8_t* sigs, size_t n_tuples, int32_t* out_codes) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    const Comm& c = comm();
    if (!c.ready) { e.last_error = "b200_comm_init has not been called"; return B200_ERR_NOT_INITIALIZED; }
    if (n_tuples == 0) return B200_SUCCESS;
    if (!pk_offsets || !msgs32 || !sigs || !out_codes || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    for (size_t t = 0; t < n_tuples; t++)
        if (pk_offsets[t] > pk_offsets[t + 1]) return B200_ERR_BAD_ARG;
    if (pk_offsets[n_tuples] && !pks_flat) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    // contiguous block of tuples per rank, balanced to within one (parallel.tuple_shard in the Python mirror)
    const size_t world = size_t(c.world), rank = size_t(c.rank);
    const size_t base = n_tuples / world, rem = n_tuples % world;
    const size_t lo = rank * base + std::min(rank, rem), cnt = base + (rank < rem ? 1 : 0);
    const size_t per = base + (rem ? 1 : 0);  // padded shard length: equal contributions to the all-gather
    B200_CUDA_TRY(s->out.reserve((per + 1) * 4));
    B200_CUDA_TRY(s->gath.reserve(world * per * 4 + 16));
    if (cnt) {
        std::vector<uint32_t> koff(cnt + 1), moff(cnt + 1);
        for (size_t t = 0; t <= cnt; t++) { koff[t] = pk_offsets[lo + t] - pk_offsets[lo]; moff[t] = uint32_t(32 * t); }
        std::vector<int32_t> local(cnt);
        rc = run_verify(e, *s, MODE_FAST_AGGREGATE, pks_flat ? pks_flat + size_t(pk_offsets[lo]) * 48 : nullptr, koff[cnt], nullptr, 0,
                        koff.data(), msgs32 + 32 * lo, moff.data(), uint32_t(cnt), sigs + 96 * lo, uint32_t(cnt), false,
                        local.data());
        if (rc) return rc;
    }
    cudaStream_t sa = e.stream;
    int32_t* d_out = static_cast<int32_t*>(s->out.p);
    if (per > cnt) B200_CUDA_TRY(cudaMemsetAsync(d_out + cnt, 0xff, (per - cnt) * 4, sa));
    rc = comm_all_gather(e, d_out, s->gath.p, per * 4, sa);   // the path's one exchange step
    if (rc) return rc;
    B200_CUDA_TRY(s->stage.reserve(world * per * 4 + 64));
    B200_CUDA_TRY(cudaMemcpyAsync(s->stage.p, s->gath.p, world * per * 4, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    const int32_t* h = static_cast<const int32_t*>(s->stage.p);
    for (size_t r = 0; r < world; r++) {
        const size_t rlo = r * base + std::min(r, rem), rcnt = base + (r < rem ? 1 : 0);
        memcpy(out_codes + rlo, h + r * per, rcnt * 4);
    }
    return B200_SUCCESS;
}

// ---- RLC whole-batch entry points (bls_rlc.cu) --------------------------------------------------------------------
static void rlc_seed(const uint8_t* seed32, uint8_t out[32]) {
    if (seed32) { memcpy(out, seed32, 32); return; }
    std::random_device rd;   // the scalars must be unpredictable to whoever produced the signatures
    for (int i = 0; i < 8; i++) { const uint32_t v = rd(); memcpy(out + 4 * i, &v, 4); }
}

int32_t b200_fast_aggregate_verify_batch_all(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                             const uint8_t* sigs, size_t n_tuples, const uint8_t* seed32, int32_t* all_ok) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!all_ok) return B200_ERR_BAD_ARG;
    if (n_tuples == 0) { *all_ok = 1; return B200_SUCCESS; }
    if (!pk_offsets || !msgs32 || !sigs || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    for (size_t t = 0; t < n_tuples; t++)
        if (pk_offsets[t] > pk_offsets[t + 1]) return B200_ERR_BAD_ARG;
    const uint32_t nk = pk_offsets[n_tuples];
    if (nk && !pks_flat) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    std::vector<uint32_t> moff(n_tuples + 1);
    for (size_t t = 0; t <= n_tuples; t++) moff[t] = uint32_t(32 * t);
    uint8_t seed[32];
    rlc_seed(seed32, seed);
    RlcReq req{seed, 0, false, 0};
    rc = run_verify(e, *s, MODE_FAST_AGGREGATE, pks_flat, nk, nullptr, 0, pk_offsets, msgs32, moff.data(), uint32_t(n_tuples), sigs,
                    uint32_t(n_tuples), false, nullptr, &req);
    if (rc) return rc;
    *all_ok = req.all_ok;
    return B200_SUCCESS;
}

int32_t b200_fast_aggregate_verify_batch_indexed_all(const uint32_t* indices, const uint32_t* offsets, const uint8_t* msgs32,
                                                     const uint8_t* sigs, size_t n_tuples, const uint8_t* seed32, int32_t* all_ok) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!all_ok) return B200_ERR_BAD_ARG;
    if (n_tuples == 0) { *all_ok = 1; return B200_SUCCESS; }
    if (!offsets || !msgs32 || !sigs || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    for (size_t t = 0; t < n_tuples; t++)
        if (offsets[t] > offsets[t + 1]) return B200_ERR_BAD_ARG;
    const uint32_t ni = offsets[n_tuples];
    if (ni && !indices) return B200_ERR_BAD_ARG;
    for (uint32_t i = 0; i < ni; i++)
        if (indices[i] >= s->reg_n) { e.last_error = "validator index outside the loaded registry"; return B200_ERR_BAD_ARG; }
    std::vector<uint32_t> moff(n_tuples + 1);
    for (size_t t = 0; t <= n_tuples; t++) moff[t] = uint32_t(32 * t);
    static const uint32_t dummy = 0;
    uint8_t seed[32];
    rlc_seed(seed32, seed);
    RlcReq req{seed, 0, false, 0};
    rc = run_verify(e, *s, MODE_FAST_AGGREGATE, nullptr, 0, indices ? indices : &dummy, ni, offsets, msgs32, moff.data(),
                    uint32_t(n_tuples), sigs, uint32_t(n_tuples), false, nullptr, &req);
    if (rc) return rc;
    *all_ok = req.all_ok;
    return B200_SUCCESS;
}

// every rank passes the same batch AND the same seed; each verifies its block, the (Gt, G2) partials are all-gathered and
// every rank finishes the same single final exponentiation
int32_t b200_fast_aggregate_verify_batch_all_sharded(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                                     const uint8_t* sigs, size_t n_tuples, const uint8_t seed32[32], int32_t* all_ok) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    const Comm& c = comm();
    if (!c.ready) { e.last_error = "b200_comm_init has not been called"; return B200_ERR_NOT_INITIALIZED; }
    if (!all_ok || !seed32) return B200_ERR_BAD_ARG;   // the ranks must agree on the scalars: the caller supplies the seed
    if (n_tuples == 0) { *all_ok = 1; return B200_SUCCESS; }
    if (!pk_offsets || !msgs32 || !sigs || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    if (n_tuples < size_t(c.world)) { e.last_error = "fewer tuples than ranks"; return B200_ERR_BAD_ARG; }
    for (size_t t = 0; t < n_tuples; t++)
        if (pk_offsets[t] > pk_offsets[t + 1]) return B200_ERR_BAD_ARG;
    if (pk_offsets[n_tuples] && !pks_flat) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    const size_t world = size_t(c.world), rank = size_t(c.rank);
    const size_t base = n_tuples / world, rem = n_tuples % world;
    const size_t lo = rank * base + std::min(rank, rem), cnt = base + (rank < rem ? 1 : 0);
    std::vector<uint32_t> koff(cnt + 1), moff(cnt + 1);
    for (size_t t = 0; t <= cnt; t++) { koff[t] = pk_offsets[lo + t] - pk_offsets[lo]; moff[t] = uint32_t(32 * t); }
    RlcReq req{seed32, uint64_t(lo), true, 0};
    rc = run_verify(e, *s, MODE_FAST_AGGREGATE, pks_flat ? pks_flat + size_t(pk_offsets[lo]) * 48 : nullptr, koff[cnt], nullptr, 0,
                    koff.data(), msgs32 + 32 * lo, moff.data(), uint32_t(cnt), sigs + 96 * lo, uint32_t(cnt), false, nullptr, &req);
    if (rc) return rc;
    *all_ok = req.all_ok;
    return B200_SUCCESS;
}

int32_t b200_registry_load(const uint8_t* pks_flat, size_t n) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if ((!pks_flat && n) || n > 0x7fffffffu) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    B200_CUDA_TRY(s->keys.reserve(n * 48 + 64));
    B200_CUDA_TRY(s->reg_aff.reserve((n + kRegistryExtraKeys + 1) * sizeof(G1Aff)));   // + the tail `..._batch_mixed` validates into
    B200_CUDA_TRY(s->reg_code.reserve((n + kRegistryExtraKeys + 1) * 4));
    if (n) B200_CUDA_TRY(cudaMemcpyAsync(s->keys.p, pks_flat, n * 48, cudaMemcpyHostToDevice, e.stream));
    B200_CUDA_TRY(cudaEventRecord(s->ev_k0, e.stream));
    launch_g1_validate(static_cast<const uint8_t*>(s->keys.p), uint32_t(n), static_cast<G1Aff*>(s->reg_aff.p),
                       static_cast<int32_t*>(s->reg_code.p), e.stream);
    e.launches += n ? 1 : 0;
    B200_CUDA_TRY(cudaEventRecord(s->ev_k1, e.stream));
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    B200_CUDA_TRY(cudaEventElapsedTime(&e.last_kernel_ms, s->ev_k0, s->ev_k1));
    s->last_dominant_ms = e.last_kernel_ms;
    s->reg_n = n;
    return B200_SUCCESS;
}

int32_t b200_registry_key_codes(int32_t* out_codes, size_t n) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    if (!out_codes || n > s->reg_n) return B200_ERR_BAD_ARG;
    if (n) B200_CUDA_TRY(cudaMemcpy(out_codes, s->reg_code.p, n * 4, cudaMemcpyDeviceToHost));
    return B200_SUCCESS;
}

static int32_t verify_batch_indexed(const uint8_t* extra_pks, size_t n_extra, const uint32_t* indices, const uint32_t* offsets,
                                    const uint8_t* msgs32, const uint8_t* sigs, size_t n_tuples, int32_t* out_codes) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (n_tuples == 0) return B200_SUCCESS;
    if (!offsets || !msgs32 || !sigs || !out_codes || n_tuples > kMaxBatchTuples) return B200_ERR_BAD_ARG;
    if ((n_extra && !extra_pks) || n_extra > kRegistryExtraKeys) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    if (n_extra && !s->reg_aff.p) { e.last_error = "no registry loaded"; return B200_ERR_BAD_ARG; }
    for (size_t t = 0; t < n_tuples; t++)
        if (offsets[t] > offsets[t + 1]) return B200_ERR_BAD_ARG;
    const uint32_t ni = offsets[n_tuples];
    if (ni && !indices) return B200_ERR_BAD_ARG;
    for (uint32_t i = 0; i < ni; i++)
        if (indices[i] >= s->reg_n + n_extra) { e.last_error = "validator index outside the loaded registry (+ extra keys)"; return B200_ERR_BAD_ARG; }
    std::vector<uint32_t> moff(n_tuples + 1);
    for (size_t t = 0; t <= n_tuples; t++) moff[t] = uint32_t(32 * t);
    static const uint32_t dummy = 0;
    return run_verify(e, *s, MODE_FAST_AGGREGATE, n_extra ? extra_pks : nullptr, uint32_t(n_extra), indices ? indices : &dummy, ni, offsets,
                      msgs32, moff.data(), uint32_t(n_tuples), sigs, uint32_t(n_tuples), false, out_codes);
}

int32_t b200_fast_aggregate_verify_batch_indexed(const uint32_t* indices, const uint32_t* offsets, const uint8_t* msgs32,
                                                 const uint8_t* sigs, size_t n_tuples, int32_t* out_codes) {
    return verify_batch_indexed(nullptr, 0, indices, offsets, msgs32, sigs, n_tuples, out_codes);
}

int32_t b200_fast_aggregate_verify_batch_mixed(const uint8_t* extra_pks, size_t n_extra, const uint32_t* indices,
                                               const uint32_t* offsets, const uint8_t* msgs32, const uint8_t* sigs,
                                               size_t n_tuples, int32_t* out_codes) {
    return verify_batch_indexed(extra_pks, n_extra, indices, offsets, msgs32, sigs, n_tuples, out_codes);
}

// crypto/bls.rs:114-132 — `public_keys: &[&PublicKey]` is an array of pointers into the validator registry
int32_t b200_fast_aggregate_verify(const uint8_t* const* pks, size_t k, const uint8_t* msg, size_t msg_len,
                                   const uint8_t sig[96]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if ((!pks && k) || (!msg && msg_len) || !sig || k > 0x7fffffffu || msg_len > 0x7fffffffu) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    std::vector<uint8_t> flat(k * 48);
    for (size_t i = 0; i < k; i++) memcpy(flat.data() + 48 * i, pks[i], 48);
    const uint32_t koff[2] = {0, uint32_t(k)}, moff[2] = {0, uint32_t(msg_len)};
    int32_t code = B200_ERR_CUDA;
    rc = run_verify(e, *s, MODE_FAST_AGGREGATE, flat.data(), uint32_t(k), nullptr, 0, koff, msg, moff, 1, sig, 1, false, &code);
    return rc ? rc : code;
}

// crypto/bls.rs:150-160
int32_t b200_eth_fast_aggregate_verify(const uint8_t* const* pks, size_t k, const uint8_t* msg, size_t msg_len,
                                       const uint8_t sig[96]) {
    if (k == 0 && sig) {
        bool inf = sig[0] == 0xc0;
        for (int i = 1; i < 96 && inf; i++) inf = sig[i] == 0;
        if (inf) return B200_SUCCESS;  // G2_POINT_AT_INFINITY with no participants (byte comparison, bls.rs:343-347)
    }
    return b200_fast_aggregate_verify(pks, k, msg, msg_len, sig);
}

// crypto/bls.rs:64-77
int32_t b200_verify_signature(const uint8_t pk[48], const uint8_t* msg, size_t msg_len, const uint8_t sig[96]) {
    if (!pk) return B200_ERR_BAD_ARG;
    const uint8_t* one[1] = {pk};
    return b200_fast_aggregate_verify(one, 1, msg, msg_len, sig);
}

// crypto/bls.rs:95-112
int32_t b200_aggregate_verify(const uint8_t* pks_flat, size_t n_pks, const uint8_t* const* msgs, const size_t* msg_lens,
                              size_t n_msgs, const uint8_t sig[96]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if ((!pks_flat && n_pks) || ((!msgs || !msg_lens) && n_msgs) || !sig || n_pks > 0x3fffffffu || n_msgs > 0x3fffffffu)
        return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    const bool shape_fail = (n_pks == 0 || n_pks != n_msgs);
    std::vector<uint32_t> moff(1, 0);
    std::vector<uint8_t> flat;
    if (!shape_fail) {
        size_t total = 0;
        for (size_t i = 0; i < n_msgs; i++) {
            if (msg_lens[i] > 0xffffffffu - total) { e.last_error = "aggregate_verify: messages exceed 4 GiB in total"; return B200_ERR_BAD_ARG; }
            total += msg_lens[i];
        }
        for (size_t i = 0; i < n_msgs; i++) {
            flat.insert(flat.end(), msgs[i], msgs[i] + msg_lens[i]);
            moff.push_back(uint32_t(flat.size()));
        }
    }
    int32_t code = B200_ERR_CUDA;
    rc = run_verify(e, *s, MODE_AGGREGATE, pks_flat, uint32_t(n_pks), nullptr, 0, nullptr, flat.data(), moff.data(),
                    uint32_t(moff.size() - 1), sig, 1, shape_fail, &code);
    return rc ? rc : code;
}

// crypto/bls.rs:79-93
int32_t b200_aggregate(const uint8_t* sigs_flat, size_t n, uint8_t out[96]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (n == 0) return B200_EMPTY_AGGREGATE;
    if (!sigs_flat || !out || n > 0x3fffffffu) return B200_ERR_BAD_ARG;
    BlsState* s;
    rc = bls_state(e, &s);
    if (rc) return rc;
    B200_CUDA_TRY(s->sigs.reserve(n * 96 + 64));
    B200_CUDA_TRY(s->g2pts.reserve((n + 1) * sizeof(G2Aff)));
    B200_CUDA_TRY(s->sig_code.reserve((n + 1) * 4));
    B200_CUDA_TRY(s->out.reserve(256));
    B200_CUDA_TRY(s->stage.reserve(256));
    cudaStream_t sa = e.stream;
    B200_CUDA_TRY(cudaMemcpyAsync(s->sigs.p, sigs_flat, n * 96, cudaMemcpyHostToDevice, sa));
    launch_g2_sig_decode(static_cast<const uint8_t*>(s->sigs.p), uint32_t(n), static_cast<G2Aff*>(s->g2pts.p),
                         static_cast<int32_t*>(s->sig_code.p), sa);
    uint8_t* d_out = static_cast<uint8_t*>(s->out.p);
    launch_g2_sum_compress(static_cast<const G2Aff*>(s->g2pts.p), static_cast<const int32_t*>(s->sig_code.p), uint32_t(n),
                           d_out + 16, reinterpret_cast<int32_t*>(d_out), sa);
    e.launches += 2;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(s->stage.p, d_out, 16 + 96, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    const int32_t code = *static_cast<const int32_t*>(s->stage.p);
    if (code == B200_SUCCESS) memcpy(out, static_cast<const uint8_t*>(s->stage.p) + 16, 96);
    return code;
}

// crypto/bls.rs:135-148
}  // extern "C"

namespace b200 {
int32_t eth_aggregate_public_keys_locked(Engine& e, const uint8_t* pks_flat, size_t n, uint8_t out[48]) {
    if (n == 0) return B200_EMPTY_AGGREGATE;
    if (!pks_flat || !out || n > 0x3fffffffu) return B200_ERR_BAD_ARG;
    BlsState* s;
    int32_t rc = bls_state(e, &s);
    if (rc) return rc;
    B200_CUDA_TRY(s->keys.reserve(n * 48 + 64));
    B200_CUDA_TRY(s->key_aff.reserve((n + 1) * sizeof(G1Aff)));
    B200_CUDA_TRY(s->key_code.reserve((n + 1) * 4));
    B200_CUDA_TRY(s->g1pts.reserve(2 * sizeof(G1Aff)));
    B200_CUDA_TRY(s->pk_code.reserve(16));
    B200_CUDA_TRY(s->flags.reserve(16));
    B200_CUDA_TRY(s->small.reserve(64));
    B200_CUDA_TRY(s->out.reserve(256));
    B200_CUDA_TRY(s->stage.reserve(256));
    cudaStream_t sa = e.stream;
    uint32_t* h = static_cast<uint32_t*>(s->stage.p);
    h[0] = 0; h[1] = uint32_t(n);
    B200_CUDA_TRY(cudaMemcpyAsync(s->small.p, h, 8, cudaMemcpyHostToDevice, sa));
    B200_CUDA_TRY(cudaMemcpyAsync(s->keys.p, pks_flat, n * 48, cudaMemcpyHostToDevice, sa));
    launch_g1_validate(static_cast<const uint8_t*>(s->keys.p), uint32_t(n), static_cast<G1Aff*>(s->key_aff.p),
                       static_cast<int32_t*>(s->key_code.p), sa);
    launch_g1_aggregate(static_cast<const G1Aff*>(s->key_aff.p), static_cast<const int32_t*>(s->key_code.p), nullptr,
                        static_cast<const uint32_t*>(s->small.p), 1, static_cast<G1Aff*>(s->g1pts.p), nullptr,
                        static_cast<int32_t*>(s->pk_code.p), static_cast<uint32_t*>(s->flags.p), 0u, sa);
    uint8_t* d_out = static_cast<uint8_t*>(s->out.p);
    launch_g1_compress(static_cast<const G1Aff*>(s->g1pts.p), d_out, sa);
    e.launches += 3;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(h + 4, s->pk_code.p, 4, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaMemcpyAsync(h + 8, d_out, 48, cudaMemcpyDeviceToHost, sa));
    B200_CUDA_TRY(cudaStreamSynchronize(sa));
    const int32_t code = int32_t(h[4]);
    if (code == B200_SUCCESS) memcpy(out, h + 8, 48);
    return code;
}
}  // namespace b200

extern "C" {

int32_t b200_eth_aggregate_public_keys(const uint8_t* pks_flat, size_t n, uint8_t out[48]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    return eth_aggregate_public_keys_locked(e, pks_flat, n, out);
}

}  // extern "C"
