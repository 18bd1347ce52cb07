// deneb process_epoch / process_slots on a device-resident BeaconState (deneb/spec/mod.rs:965-1004, :3150-3240).
//
// The per-validator work (the sums behind every balance threshold, inactivity scores + rewards and penalties, registry
// marking, slashings + effective balances, the participation rotation) runs as sweeps over the resident lists; what
// is inherently sequential and small (justification, the exit-queue loop, the activation-queue top-k, sync-committee
// sampling) runs on the host from a few counters and compacted candidate lists.  Small fields are written through
// state_patch_bytes, list-length changes (eth1_data_votes reset, historical_summaries append) through state_relayout.
//
// The spec treats any uint64 overflow as an invalid transition; the kernels raise a device flag and the call returns
// B200_STATE_TRANSITION_INVALID (the reference Rust code wraps or panics instead).
#include <algorithm>
#include <cstring>
#include <vector>

#include "sha256_hd.cuh"
#include "shuffle.h"
#include "state_handle.h"

namespace b200 {
namespace {

constexpr uint64_t FAR_FUTURE = ~uint64_t(0);
constexpr uint64_t U64MAX = ~uint64_t(0);
// phase0/presets/*.rs, altair/presets/*.rs, bellatrix/presets/*.rs, configs/*.rs (identical in both presets)
constexpr uint64_t EFFECTIVE_BALANCE_INCREMENT = 1000000000ull;
constexpr uint64_t MAX_EFFECTIVE_BALANCE = 32000000000ull;
constexpr uint64_t EJECTION_BALANCE = 16000000000ull;
constexpr uint64_t BASE_REWARD_FACTOR = 64;
constexpr uint64_t HYSTERESIS_QUOTIENT = 4, HYSTERESIS_DOWNWARD_MULTIPLIER = 1, HYSTERESIS_UPWARD_MULTIPLIER = 5;
constexpr uint64_t MIN_SEED_LOOKAHEAD = 1, MAX_SEED_LOOKAHEAD = 4;
constexpr uint64_t MIN_EPOCHS_TO_INACTIVITY_PENALTY = 4;
constexpr uint64_t INACTIVITY_PENALTY_QUOTIENT_BELLATRIX = 16777216;
constexpr uint64_t PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX = 3;
constexpr uint64_t INACTIVITY_SCORE_BIAS = 4, INACTIVITY_SCORE_RECOVERY_RATE = 16;
constexpr uint64_t MIN_VALIDATOR_WITHDRAWABILITY_DELAY = 256;
constexpr uint64_t WEIGHT_DENOMINATOR = 64;
// TIMELY_SOURCE, TIMELY_TARGET, TIMELY_HEAD weights: 14, 26, 14
__host__ __device__ constexpr uint64_t flag_weight(int f) { return f == 1 ? 26 : 14; }
constexpr uint8_t DOMAIN_SYNC_COMMITTEE[4] = {7, 0, 0, 0};

struct PresetConsts {
    uint64_t slots_per_epoch, slots_per_historical_root, epochs_per_historical_vector, epochs_per_slashings_vector,
        sync_committee_size, epochs_per_sync_committee_period, epochs_per_eth1_voting_period, shuffle_round_count,
        min_per_epoch_churn_limit, max_per_epoch_activation_churn_limit, churn_limit_quotient, historical_roots_limit;
};
const PresetConsts kConsts[2] = {
    {32, 8192, 65536, 8192, 512, 256, 64, 90, 4, 8, 65536, 1ull << 24},   // mainnet
    {8, 64, 64, 64, 32, 8, 4, 10, 2, 4, 32, 1ull << 24},                 // minimal
};

// Validator record (phase0/validator.rs:10-26): byte offsets of the fields the epoch reads
constexpr uint32_t V_EB = 80, V_SLASHED = 88, V_AEE = 89, V_ACT = 97, V_EXIT = 105, V_WD = 113, V_SIZE = 121;

constexpr int kThreads = 256;

struct Rec {
    uint64_t eb, aee, act, exit, wd;
    bool slashed;
};

__host__ __device__ inline uint64_t ld64(const uint8_t* p) {
    uint64_t v = 0;
    for (int k = 7; k >= 0; k--) v = (v << 8) | p[k];
    return v;
}
__device__ inline void st64(uint8_t* p, uint64_t v) {
    for (int k = 0; k < 8; k++) p[k] = uint8_t(v >> (8 * k));
}

// The block's 256 records land in shared memory through coalesced 16-byte loads (256 x 121 B = 1936 x 16 B; the field
// buffer is 256-byte aligned, so every block's slice is 16-byte aligned).
__device__ inline Rec load_rec(const uint8_t* __restrict__ recs, uint64_t n, uint8_t* sm, uint64_t i) {
    const uint64_t first = uint64_t(blockIdx.x) * kThreads;
    const uint64_t cnt = first < n ? min(uint64_t(kThreads), n - first) : 0;
    const size_t bytes = size_t(cnt) * V_SIZE;
    const uint4* src = reinterpret_cast<const uint4*>(recs + first * V_SIZE);
    uint4* dst = reinterpret_cast<uint4*>(sm);
    const size_t nv = bytes / 16;
    for (size_t k = threadIdx.x; k < nv; k += kThreads) dst[k] = src[k];
    for (size_t k = nv * 16 + threadIdx.x; k < bytes; k += kThreads) sm[k] = recs[first * V_SIZE + k];
    __syncthreads();
    Rec r{};
    if (i < n) {
        const uint8_t* p = sm + size_t(threadIdx.x) * V_SIZE;
        r.eb = ld64(p + V_EB); r.slashed = p[V_SLASHED] != 0; r.aee = ld64(p + V_AEE);
        r.act = ld64(p + V_ACT); r.exit = ld64(p + V_EXIT); r.wd = ld64(p + V_WD);
    }
    return r;
}

__device__ inline bool is_active(const Rec& r, uint64_t epoch) { return r.act <= epoch && epoch < r.exit; }

// ---- sums: [0] active count, [1] total active balance, [2..4] previous-epoch unslashed participating balance per
// flag, [5] current-epoch target balance, [6] max exit epoch != FAR_FUTURE (atomicMax); carry[k] counts 2^64 wraps
struct Sums {
    unsigned long long v[8];
    unsigned long long carry[8];
    unsigned int flags, ej_n, act_n, pad;
    unsigned long long exit_count;
};

__device__ inline void warp_sum_atomic(uint64_t x, unsigned long long* dst, unsigned long long* carry) {
    uint64_t c = 0;
    for (int off = 16; off; off >>= 1) {
        const uint64_t y = __shfl_down_sync(0xffffffffu, x, off);
        const uint64_t cy = __shfl_down_sync(0xffffffffu, c, off);
        const uint64_t s = x + y;
        c += cy + (s < x ? 1 : 0);
        x = s;
    }
    if ((threadIdx.x & 31) == 0) {
        if (x) {
            const unsigned long long old = atomicAdd(dst, (unsigned long long)x);
            if (old + x < old) c++;
        }
        if (c) atomicAdd(carry, (unsigned long long)c);
    }
}

__global__ void __launch_bounds__(kThreads) k_epoch_sums(const uint8_t* __restrict__ recs, uint64_t n,
                                                         const uint8_t* __restrict__ prev_part,
                                                         const uint8_t* __restrict__ cur_part, uint64_t cur_epoch,
                                                         uint64_t prev_epoch, Sums* out) {
    __shared__ __align__(16) uint8_t sm[kThreads * V_SIZE];
    const uint64_t i = uint64_t(blockIdx.x) * kThreads + threadIdx.x;
    const Rec r = load_rec(recs, n, sm, i);
    uint64_t v[6] = {0, 0, 0, 0, 0, 0};
    uint64_t max_exit = 0;
    if (i < n) {
        const bool act_cur = is_active(r, cur_epoch), act_prev = is_active(r, prev_epoch);
        if (act_cur) { v[0] = 1; v[1] = r.eb; }
        const uint8_t pf = prev_part[i], cf = cur_part[i];
        for (int f = 0; f < 3; f++)
            if (act_prev && !r.slashed && ((pf >> f) & 1)) v[2 + f] = r.eb;
        if (act_cur && !r.slashed && ((cf >> 1) & 1)) v[5] = r.eb;
        if (r.exit != FAR_FUTURE) max_exit = r.exit + 1;   // +1: 0 means "none"
    }
    for (int k = 0; k < 6; k++) warp_sum_atomic(v[k], &out->v[k], &out->carry[k]);
    for (int off = 16; off; off >>= 1) max_exit = max(max_exit, __shfl_down_sync(0xffffffffu, max_exit, off));
    if ((threadIdx.x & 31) == 0 && max_exit) atomicMax(&out->v[6], (unsigned long long)max_exit);
}

__global__ void __launch_bounds__(kThreads) k_exit_count(const uint8_t* __restrict__ recs, uint64_t n, uint64_t epoch,
                                                         Sums* out) {
    const uint64_t i = uint64_t(blockIdx.x) * kThreads + threadIdx.x;
    const bool hit = i < n && ld64(recs + i * V_SIZE + V_EXIT) == epoch;
    const unsigned c = __popc(__ballot_sync(0xffffffffu, hit));
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&out->exit_count, (unsigned long long)c);
}

// ---- stages 1 + 2: inactivity scores, then the four (reward, penalty) pairs in spec order, per eligible validator
struct RewardParams {
    uint64_t prev_epoch, brpi, active_incr, part_incr[3];
    int do_inact, do_rewards, leak;
};

__device__ inline bool mul_ovf(uint64_t a, uint64_t b, uint64_t* r) {
    *r = a * b;
    return __umul64hi(a, b) != 0;
}

__global__ void __launch_bounds__(kThreads) k_epoch_rewards(const uint8_t* __restrict__ recs, uint64_t n,
                                                            uint64_t* __restrict__ bal, const uint8_t* __restrict__ prev_part,
                                                            uint64_t* __restrict__ inact, RewardParams p, Sums* out) {
    __shared__ __align__(16) uint8_t sm[kThreads * V_SIZE];
    const uint64_t i = uint64_t(blockIdx.x) * kThreads + threadIdx.x;
    const Rec r = load_rec(recs, n, sm, i);
    if (i >= n) return;
    const bool act_prev = is_active(r, p.prev_epoch);
    if (!(act_prev || (r.slashed && p.prev_epoch + 1 < r.wd))) return;   // not eligible
    const uint8_t pf = prev_part[i];
    const bool target = act_prev && !r.slashed && ((pf >> 1) & 1);
    bool ovf = false;
    uint64_t score = inact[i];
    if (p.do_inact) {
        if (target) score -= min(uint64_t(1), score);
        else { ovf |= score > U64MAX - INACTIVITY_SCORE_BIAS; score += INACTIVITY_SCORE_BIAS; }
        if (!p.leak) score -= min(INACTIVITY_SCORE_RECOVERY_RATE, score);
        inact[i] = score;
    }
    if (p.do_rewards) {
        uint64_t b = bal[i], base, t;
        ovf |= mul_ovf(r.eb / EFFECTIVE_BALANCE_INCREMENT, p.brpi, &base);
        for (int f = 0; f < 3; f++) {
            uint64_t reward = 0, penalty = 0;
            if (act_prev && !r.slashed && ((pf >> f) & 1)) {
                if (!p.leak) {
                    ovf |= mul_ovf(base, flag_weight(f), &t);
                    ovf |= mul_ovf(t, p.part_incr[f], &t);
                    reward = t / (p.active_incr * WEIGHT_DENOMINATOR);
                }
            } else if (f != 2) {
                ovf |= mul_ovf(base, flag_weight(f), &t);
                penalty = t / WEIGHT_DENOMINATOR;
            }
            ovf |= b > U64MAX - reward;
            b += reward;
            b = b > penalty ? b - penalty : 0;
        }
        if (!target) {
            ovf |= mul_ovf(r.eb, score, &t);
            const uint64_t penalty = t / (INACTIVITY_SCORE_BIAS * INACTIVITY_PENALTY_QUOTIENT_BELLATRIX);
            b = b > penalty ? b - penalty : 0;
        }
        bal[i] = b;
    }
    if (ovf) atomicOr(&out->flags, 1u);
}

// ---- stage 3 marking: activation-queue eligibility is written in place; ejection and activation candidates are
// compacted (unordered; the host sorts them)
__global__ void __launch_bounds__(kThreads) k_registry_mark(uint8_t* __restrict__ recs, uint64_t n, uint64_t cur_epoch,
                                                            uint64_t fin_epoch, uint64_t* __restrict__ ej,
                                                            uint64_t* __restrict__ act_q, Sums* out) {
    __shared__ __align__(16) uint8_t sm[kThreads * V_SIZE];
    const uint64_t i = uint64_t(blockIdx.x) * kThreads + threadIdx.x;
    const Rec r = load_rec(recs, n, sm, i);
    if (i >= n) return;
    if (r.aee == FAR_FUTURE && r.eb == MAX_EFFECTIVE_BALANCE) st64(recs + i * V_SIZE + V_AEE, cur_epoch + 1);
    if (is_active(r, cur_epoch) && r.eb <= EJECTION_BALANCE && r.exit == FAR_FUTURE) ej[atomicAdd(&out->ej_n, 1u)] = i;
    if (r.aee <= fin_epoch && r.act == FAR_FUTURE) {
        const unsigned k = atomicAdd(&out->act_n, 1u);
        act_q[2 * k] = r.aee; act_q[2 * k + 1] = i;
    }
}

// (byte offset in the validator list, u64 value) pairs
__global__ void k_write_u64(uint8_t* __restrict__ recs, const uint64_t* __restrict__ w, uint32_t n) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) st64(recs + w[2 * k], w[2 * k + 1]);
}

// ---- stages 4 + 6: slashings penalty, then hysteresis on the post-slashing balance
struct BalanceParams {
    uint64_t cur_epoch, adjusted, total;
    int do_slash, do_eb;
};

__global__ void __launch_bounds__(kThreads) k_epoch_balances(uint8_t* __restrict__ recs, uint64_t n,
                                                             uint64_t* __restrict__ bal, BalanceParams p, uint64_t half_vec,
                                                             Sums* out) {
    __shared__ __align__(16) uint8_t sm[kThreads * V_SIZE];
    const uint64_t i = uint64_t(blockIdx.x) * kThreads + threadIdx.x;
    const Rec r = load_rec(recs, n, sm, i);
    if (i >= n) return;
    bool ovf = false;
    uint64_t b = bal[i];
    if (p.do_slash && r.slashed && p.cur_epoch + half_vec == r.wd) {
        uint64_t num;
        ovf |= mul_ovf(r.eb / EFFECTIVE_BALANCE_INCREMENT, p.adjusted, &num);
        const uint64_t penalty = num / p.total * EFFECTIVE_BALANCE_INCREMENT;
        b = b > penalty ? b - penalty : 0;
        bal[i] = b;
    }
    if (p.do_eb) {
        constexpr uint64_t inc = EFFECTIVE_BALANCE_INCREMENT / HYSTERESIS_QUOTIENT;
        constexpr uint64_t down = inc * HYSTERESIS_DOWNWARD_MULTIPLIER, up = inc * HYSTERESIS_UPWARD_MULTIPLIER;
        ovf |= b > U64MAX - down || r.eb > U64MAX - up;
        if (b + down < r.eb || r.eb + up < b)
            st64(recs + i * V_SIZE + V_EB, min(b - b % EFFECTIVE_BALANCE_INCREMENT, MAX_EFFECTIVE_BALANCE));
    }
    if (ovf) atomicOr(&out->flags, 1u);
}

// sync-committee sampling inputs: effective balance of every shuffled candidate; public keys of the chosen ones
__global__ void k_gather_eb(const uint8_t* __restrict__ recs, const uint64_t* __restrict__ idx, uint64_t n, uint64_t* out) {
    const uint64_t k = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (k < n) out[k] = ld64(recs + idx[k] * V_SIZE + V_EB);
}
__global__ void k_gather_pk(const uint8_t* __restrict__ recs, const uint64_t* __restrict__ idx, uint32_t n, uint8_t* out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n * 48) out[k] = recs[idx[k / 48] * V_SIZE + k % 48];
}

// ------------------------------------------------------------------------------------------------ host side

uint64_t integer_squareroot(uint64_t n) {
    uint64_t x = n, y = (x >> 1) + (x & 1);
    while (y < x) { x = y; y = (x + n / x) / 2; }
    return x;
}

void sha256_host(const uint8_t* d, size_t n, uint8_t out[32]) {
    Sha256Ctx c;
    sha_init(c);
    sha_update(c, d, n);
    sha_final(c, out);
}

void hash_pair(const uint8_t a[32], const uint8_t b[32], uint8_t out[32]) {
    uint8_t buf[64];
    memcpy(buf, a, 32); memcpy(buf + 32, b, 32);
    sha256_host(buf, 64, out);
}

void u64_le(uint64_t v, uint8_t* p) { for (int k = 0; k < 8; k++) p[k] = uint8_t(v >> (8 * k)); }

struct Ctx {
    Engine& e;
    b200_state* h;
    const PresetConsts& C;
    uint64_t n;
    Sums* d_sums() { return static_cast<Sums*>(h->epoch_scratch.p); }
    uint8_t* scratch() { return static_cast<uint8_t*>(h->epoch_scratch.p) + 256; }
    uint8_t* list(int f) {
        uint64_t off = 0; size_t nb = 0;
        h->plan.chain_field(f, &off, &nb);
        return static_cast<uint8_t*>(h->fields.p) + off;
    }
    uint64_t rd(size_t off) const { return ld64(h->shadow + off); }
    int32_t patch(size_t off, const uint8_t* d, size_t nb) { return state_patch_bytes(e, h, off, d, nb); }
    int32_t patch_u64(size_t off, uint64_t v) { uint8_t b[8]; u64_le(v, b); return patch(off, b, 8); }
    unsigned blocks() const { return unsigned((n + kThreads - 1) / kThreads); }
};

int32_t invalid(Engine& e, const char* why) {
    e.last_error = std::string("state transition invalid: ") + why;
    return B200_STATE_TRANSITION_INVALID;
}

// get_block_root(state, epoch) from the shadow (phase0 get_block_root_at_slot: slot < state.slot <= slot + SPHR)
int32_t block_root_at_epoch(Ctx& c, uint64_t epoch, uint8_t out[32]) {
    const uint64_t slot = epoch * c.C.slots_per_epoch, state_slot = c.rd(40);
    if (!(slot < state_slot && state_slot <= slot + c.C.slots_per_historical_root)) return invalid(c.e, "block root out of range");
    memcpy(out, c.h->shadow + c.h->so.block_roots + 32 * (slot % c.C.slots_per_historical_root), 32);
    return B200_SUCCESS;
}

// stage 0 on the host: weigh_justification_and_finalization (deneb/spec/mod.rs:1469)
int32_t justification(Ctx& c, uint64_t cur, uint64_t prev, uint64_t total, uint64_t prev_target, uint64_t cur_target) {
    const size_t cp = c.h->so.checkpoints, jb = c.h->so.justification_bits;
    uint8_t ck[120];
    memcpy(ck, c.h->shadow + cp, 120);   // previous_justified, current_justified, finalized
    uint8_t old_prev[40], old_cur[40];
    memcpy(old_prev, ck, 40); memcpy(old_cur, ck + 40, 40);
    memcpy(ck, old_cur, 40);
    uint8_t bits = uint8_t((c.h->shadow[jb] << 1) & 0x0f);
    // the spec multiplies u64 balances by 3 and 2: an overflow there is an invalid transition too
    if (prev_target > U64MAX / 3 || cur_target > U64MAX / 3 || total > U64MAX / 2) return invalid(c.e, "justification weight overflow");
    if (prev_target * 3 >= total * 2) {
        u64_le(prev, ck + 40);
        int32_t rc = block_root_at_epoch(c, prev, ck + 48);
        if (rc) return rc;
        bits |= 2;
    }
    if (cur_target * 3 >= total * 2) {
        u64_le(cur, ck + 40);
        int32_t rc = block_root_at_epoch(c, cur, ck + 48);
        if (rc) return rc;
        bits |= 1;
    }
    const uint64_t op = ld64(old_prev), oc = ld64(old_cur);
    auto all = [&](int lo, int hi) { for (int k = lo; k < hi; k++) if (!((bits >> k) & 1)) return false; return true; };
    if (all(1, 4) && op + 3 == cur) memcpy(ck + 80, old_prev, 40);
    if (all(1, 3) && op + 2 == cur) memcpy(ck + 80, old_prev, 40);
    if (all(0, 3) && oc + 2 == cur) memcpy(ck + 80, old_cur, 40);
    if (all(0, 2) && oc + 1 == cur) memcpy(ck + 80, old_cur, 40);
    int32_t rc = c.patch(jb, &bits, 1);
    return rc ? rc : c.patch(cp, ck, 120);
}

// stage 3 on the host: the exit-queue loop over the ejections (index order) and the activation-queue top-k
int32_t registry_updates(Ctx& c, uint64_t cur, uint64_t active_count, uint64_t max_exit_plus1, Sums& hs) {
    Engine& e = c.e;
    uint64_t* d_ej = reinterpret_cast<uint64_t*>(c.scratch());
    uint64_t* d_act = d_ej + c.n;
    uint8_t* recs = c.list(0);
    k_registry_mark<<<c.blocks(), kThreads, 0, e.stream>>>(recs, c.n, cur, c.rd(c.h->so.checkpoints + 80), d_ej, d_act, c.d_sums());
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(&hs, c.d_sums(), sizeof(Sums), cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    std::vector<uint64_t> ej(hs.ej_n), aq(2 * size_t(hs.act_n));
    if (hs.ej_n) B200_CUDA_TRY(cudaMemcpyAsync(ej.data(), d_ej, 8 * size_t(hs.ej_n), cudaMemcpyDeviceToHost, e.stream));
    if (hs.act_n) B200_CUDA_TRY(cudaMemcpyAsync(aq.data(), d_act, 16 * size_t(hs.act_n), cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    const uint64_t churn = std::max(c.C.min_per_epoch_churn_limit, active_count / c.C.churn_limit_quotient);
    const uint64_t act_exit_epoch = cur + 1 + MAX_SEED_LOOKAHEAD;   // compute_activation_exit_epoch
    std::vector<uint64_t> w;   // (byte offset, value) pairs
    if (!ej.empty()) {
        std::sort(ej.begin(), ej.end());
        // initiate_validator_exit with the exit-queue epoch and its churn kept as running values
        uint64_t max_exit = max_exit_plus1 ? max_exit_plus1 - 1 : 0, count_at_max = 0;
        if (max_exit_plus1) {
            B200_CUDA_TRY(cudaMemsetAsync(&c.d_sums()->exit_count, 0, 8, e.stream));
            k_exit_count<<<c.blocks(), kThreads, 0, e.stream>>>(recs, c.n, max_exit, c.d_sums());
            e.launches++;
            B200_CUDA_TRY(cudaGetLastError());
            B200_CUDA_TRY(cudaMemcpyAsync(&hs.exit_count, &c.d_sums()->exit_count, 8, cudaMemcpyDeviceToHost, e.stream));
            B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
            count_at_max = hs.exit_count;
        }
        bool have_max = max_exit_plus1 != 0;
        for (uint64_t i : ej) {
            uint64_t q = act_exit_epoch, churn_q = 0;
            if (have_max && max_exit >= q) { q = max_exit; churn_q = count_at_max; }
            if (churn_q >= churn) {
                if (q == U64MAX) return invalid(e, "exit queue epoch overflow");
                q += 1; churn_q = 0;
            }
            if (q > U64MAX - MIN_VALIDATOR_WITHDRAWABILITY_DELAY) return invalid(e, "withdrawable epoch overflow");
            w.push_back(i * V_SIZE + V_EXIT); w.push_back(q);
            w.push_back(i * V_SIZE + V_WD); w.push_back(q + MIN_VALIDATOR_WITHDRAWABILITY_DELAY);
            // q is the largest exit epoch now (q >= every existing one), with churn_q + 1 exits
            max_exit = q; count_at_max = churn_q + 1; have_max = true;
        }
    }
    if (!aq.empty()) {
        std::vector<std::pair<uint64_t, uint64_t>> q(hs.act_n);
        for (size_t k = 0; k < q.size(); k++) q[k] = {aq[2 * k], aq[2 * k + 1]};
        const size_t take = size_t(std::min<uint64_t>(q.size(), std::min(c.C.max_per_epoch_activation_churn_limit, churn)));
        std::partial_sort(q.begin(), q.begin() + take, q.end());
        for (size_t k = 0; k < take; k++) { w.push_back(q[k].second * V_SIZE + V_ACT); w.push_back(act_exit_epoch); }
    }
    if (!w.empty()) {
        const uint32_t nw = uint32_t(w.size() / 2);
        B200_CUDA_TRY(c.h->scatter.reserve(w.size() * 8));
        B200_CUDA_TRY(cudaMemcpyAsync(c.h->scatter.p, w.data(), w.size() * 8, cudaMemcpyHostToDevice, e.stream));
        k_write_u64<<<(nw + 255) / 256, 256, 0, e.stream>>>(recs, static_cast<const uint64_t*>(c.h->scatter.p), nw);
        e.launches++;
        B200_CUDA_TRY(cudaGetLastError());
        B200_CUDA_TRY(cudaStreamSynchronize(e.stream));   // `w` is about to go
    }
    return B200_SUCCESS;
}

// stage 11: get_next_sync_committee (deneb/spec/mod.rs:1973-2060) — device shuffle, host sampling, device key aggregation
int32_t sync_committee_updates(Ctx& c, uint64_t cur) {
    Engine& e = c.e;
    b200_state* h = c.h;
    const size_t sc_bytes = 48 * c.C.sync_committee_size + 48;
    std::vector<uint8_t> next(h->shadow + h->so.next_sync_committee, h->shadow + h->so.next_sync_committee + sc_bytes);
    const uint64_t epoch = cur + 1;
    uint8_t seed_in[44], seed[32];
    memcpy(seed_in, DOMAIN_SYNC_COMMITTEE, 4);
    u64_le(epoch, seed_in + 4);
    const uint64_t mix = (epoch + c.C.epochs_per_historical_vector - MIN_SEED_LOOKAHEAD - 1) % c.C.epochs_per_historical_vector;
    memcpy(seed_in + 12, h->shadow + h->so.randao_mixes + 32 * mix, 32);
    sha256_host(seed_in, 44, seed);
    uint64_t *d_act, *d_shuf;
    int32_t rc = shuffle_scratch(e, c.n, &d_act, &d_shuf);
    if (rc) return rc;
    uint64_t cnt = 0;
    const uint8_t* recs = c.list(0);
    rc = active_indices_on_device(e, recs, c.n, epoch, d_act, &cnt);
    if (rc) return rc;
    if (cnt == 0) return invalid(e, "no active validator for the next sync committee");
    rc = shuffle_on_device(e, d_act, cnt, seed, uint32_t(c.C.shuffle_round_count), d_shuf);
    if (rc) return rc;
    uint64_t* d_eb = reinterpret_cast<uint64_t*>(c.scratch());
    k_gather_eb<<<unsigned((cnt + 255) / 256), 256, 0, e.stream>>>(recs, d_shuf, cnt, d_eb);
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    std::vector<uint64_t> shuf(cnt), eb(cnt);
    B200_CUDA_TRY(cudaMemcpyAsync(shuf.data(), d_shuf, 8 * cnt, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaMemcpyAsync(eb.data(), d_eb, 8 * cnt, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    std::vector<uint64_t> chosen;
    uint8_t hin[40], rnd[32];
    memcpy(hin, seed, 32);
    uint64_t rnd_block = U64MAX;
    for (uint64_t i = 0; chosen.size() < c.C.sync_committee_size; i++) {
        const uint64_t k = i % cnt;
        if (i / 32 != rnd_block) { rnd_block = i / 32; u64_le(rnd_block, hin + 32); sha256_host(hin, 40, rnd); }
        // effective_balance * 255 >= MAX_EFFECTIVE_BALANCE * random_byte (the left side cannot overflow when eb fits the
        // spec's own bound; a larger eb makes the product overflow: invalid)
        if (eb[k] > U64MAX / 255) return invalid(e, "sync committee sampling overflow");
        if (eb[k] * 255 >= MAX_EFFECTIVE_BALANCE * rnd[i % 32]) chosen.push_back(shuf[k]);
    }
    const uint32_t m = uint32_t(chosen.size());
    B200_CUDA_TRY(h->scatter.reserve(8 * m + 48 * m));
    uint64_t* d_idx = static_cast<uint64_t*>(h->scatter.p);
    uint8_t* d_pk = reinterpret_cast<uint8_t*>(d_idx + m);
    B200_CUDA_TRY(cudaMemcpyAsync(d_idx, chosen.data(), 8 * m, cudaMemcpyHostToDevice, e.stream));
    k_gather_pk<<<(48 * m + 255) / 256, 256, 0, e.stream>>>(recs, d_idx, m, d_pk);
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    std::vector<uint8_t> fresh(sc_bytes);
    B200_CUDA_TRY(cudaMemcpyAsync(fresh.data(), d_pk, 48 * m, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    rc = eth_aggregate_public_keys_locked(e, fresh.data(), m, fresh.data() + 48 * m);
    if (rc) return rc;   // a bad key: its blst code (1..7)
    rc = c.patch(h->so.current_sync_committee, next.data(), sc_bytes);
    return rc ? rc : c.patch(h->so.next_sync_committee, fresh.data(), sc_bytes);
}

int32_t process_epoch_locked(Engine& e, b200_state* h, uint32_t mask) {
    const PresetConsts& C = kConsts[h->preset];
    Ctx c{e, h, C, big_count(h, 0)};
    const uint64_t cur = c.rd(40) / C.slots_per_epoch;
    const uint64_t prev = cur == 0 ? 0 : cur - 1;
    const uint64_t next = cur + 1;
    auto on = [&](int s) { return (mask >> s) & 1; };
    B200_CUDA_TRY(h->epoch_scratch.reserve(256 + 24 * c.n));
    int32_t rc;
    // ---- the sums behind stages 0..4 (effective balances, flags and epochs do not change before stage 4 reads them)
    Sums hs{};
    uint64_t total = 0, flag_bal[3] = {0, 0, 0}, cur_target = 0, active_count = 0, max_exit_plus1 = 0;
    B200_CUDA_TRY(cudaMemsetAsync(c.d_sums(), 0, sizeof(Sums), e.stream));   // counters and the overflow flag
    if (mask & 0x1f) {
        k_epoch_sums<<<c.blocks(), kThreads, 0, e.stream>>>(c.list(0), c.n, c.list(2), c.list(3), cur, prev, c.d_sums());
        e.launches++;
        B200_CUDA_TRY(cudaGetLastError());
        B200_CUDA_TRY(cudaMemcpyAsync(&hs, c.d_sums(), sizeof(Sums), cudaMemcpyDeviceToHost, e.stream));
        B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
        for (int k = 1; k < 6; k++)
            if (hs.carry[k]) return invalid(e, "total balance overflow");
        // get_total_balance is floored at EFFECTIVE_BALANCE_INCREMENT
        auto floor_inc = [](uint64_t x) { return std::max(x, EFFECTIVE_BALANCE_INCREMENT); };
        active_count = hs.v[0];
        total = floor_inc(hs.v[1]);
        for (int f = 0; f < 3; f++) flag_bal[f] = floor_inc(hs.v[2 + f]);
        cur_target = floor_inc(hs.v[5]);
        max_exit_plus1 = hs.v[6];
    }
    // stage 0: justification_and_finalization
    if (on(0) && cur > 1) {
        rc = justification(c, cur, prev, total, flag_bal[1], cur_target);
        if (rc) return rc;
    }
    // stages 1 + 2: inactivity_updates, rewards_and_penalties (after stage 0: the leak reads the new finalized epoch)
    if ((on(1) || on(2)) && cur > 0) {
        const uint64_t fin = c.rd(h->so.checkpoints + 80);
        if (fin > prev) return invalid(e, "finality delay underflow");
        RewardParams p{};
        p.prev_epoch = prev;
        p.leak = prev - fin > MIN_EPOCHS_TO_INACTIVITY_PENALTY;
        p.brpi = EFFECTIVE_BALANCE_INCREMENT * BASE_REWARD_FACTOR / integer_squareroot(total);
        p.active_incr = total / EFFECTIVE_BALANCE_INCREMENT;
        for (int f = 0; f < 3; f++) p.part_incr[f] = flag_bal[f] / EFFECTIVE_BALANCE_INCREMENT;
        p.do_inact = on(1); p.do_rewards = on(2);
        k_epoch_rewards<<<c.blocks(), kThreads, 0, e.stream>>>(c.list(0), c.n, reinterpret_cast<uint64_t*>(c.list(1)), c.list(2),
                                                               reinterpret_cast<uint64_t*>(c.list(4)), p, c.d_sums());
        e.launches++;
        B200_CUDA_TRY(cudaGetLastError());
        h->all_dirty = true;
    }
    // stage 3: registry_updates
    if (on(3)) {
        rc = registry_updates(c, cur, active_count, max_exit_plus1, hs);
        if (rc) return rc;
        h->all_dirty = true;
    }
    // stages 4 + 6: slashings, effective_balance_updates (stage 5 touches neither balances nor the registry)
    if (on(4) || on(6)) {
        BalanceParams p{};
        p.cur_epoch = cur; p.total = total; p.do_slash = on(4); p.do_eb = on(6);
        if (on(4)) {
            unsigned __int128 sum = 0;
            for (uint64_t k = 0; k < C.epochs_per_slashings_vector; k++) sum += c.rd(h->so.slashings + 8 * k);
            sum *= PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX;
            if (sum > U64MAX) return invalid(e, "slashings sum overflow");
            p.adjusted = std::min<uint64_t>(uint64_t(sum), total);
        }
        k_epoch_balances<<<c.blocks(), kThreads, 0, e.stream>>>(c.list(0), c.n, reinterpret_cast<uint64_t*>(c.list(1)), p,
                                                                C.epochs_per_slashings_vector / 2, c.d_sums());
        e.launches++;
        B200_CUDA_TRY(cudaGetLastError());
        h->all_dirty = true;
    }
    if (mask & 0x56) {   // a kernel of stages 1, 2, 4 or 6 ran: its overflow flag
        unsigned flags = 0;
        B200_CUDA_TRY(cudaMemcpyAsync(&flags, &c.d_sums()->flags, 4, cudaMemcpyDeviceToHost, e.stream));
        B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
        if (flags) return invalid(e, "uint64 overflow in a per-validator stage");
    }
    // stage 5: eth1_data_reset — empties a list
    if (on(5) && next % C.epochs_per_eth1_voting_period == 0 && h->so.var[2] != h->so.var[1]) {
        rc = state_relayout(e, h, 1, nullptr, 0);
        if (rc) return rc;
    }
    // stage 7: slashings_reset
    if (on(7)) {
        rc = c.patch_u64(h->so.slashings + 8 * (next % C.epochs_per_slashings_vector), 0);
        if (rc) return rc;
    }
    // stage 8: randao_mixes_reset
    if (on(8)) {
        uint8_t mix[32];
        memcpy(mix, h->shadow + h->so.randao_mixes + 32 * (cur % C.epochs_per_historical_vector), 32);
        rc = c.patch(h->so.randao_mixes + 32 * (next % C.epochs_per_historical_vector), mix, 32);
        if (rc) return rc;
    }
    // stage 9: historical_summaries_update — appends to a list
    if (on(9) && next % (C.slots_per_historical_root / C.slots_per_epoch) == 0) {
        const size_t old = size_t(h->so.var[9] - h->so.var[8]);
        if (old / 64 + 1 > C.historical_roots_limit) return invalid(e, "historical_summaries full");
        SszPlan p;
        const int d = depth_for(C.slots_per_historical_root);
        const uint32_t br = p.wide_chunks(p.stage_field(h->shadow + h->so.block_roots, 32 * C.slots_per_historical_root),
                                          C.slots_per_historical_root, d);
        const uint32_t sr = p.wide_chunks(p.stage_field(h->shadow + h->so.state_roots, 32 * C.slots_per_historical_root),
                                          C.slots_per_historical_root, d);
        std::vector<uint8_t> list(old + 64);
        memcpy(list.data(), h->shadow + h->so.var[8], old);
        rc = p.run(e, e.arena, e.fields, e.planbuf, COPY_ALL, std::vector<uint32_t>{br, sr}, list.data() + old);
        if (rc) return rc;
        rc = state_relayout(e, h, 8, list.data(), list.size());
        if (rc) return rc;
    }
    // stage 10: participation_flag_updates
    if (on(10)) {
        B200_CUDA_TRY(cudaMemcpyAsync(c.list(2), c.list(3), c.n, cudaMemcpyDeviceToDevice, e.stream));
        B200_CUDA_TRY(cudaMemsetAsync(c.list(3), 0, c.n, e.stream));
        h->all_dirty = true;
    }
    // stage 11: sync_committee_updates
    if (on(11) && next % C.epochs_per_sync_committee_period == 0) {
        rc = sync_committee_updates(c, cur);
        if (rc) return rc;
    }
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    return B200_SUCCESS;
}

int32_t check_epoch_handle(Engine& e, b200_state* h) {
    if (!h || !h->uploaded || h->failed || h->sharded) return B200_ERR_BAD_ARG;
    const uint64_t n = big_count(h, 0);
    if (n == 0) { e.last_error = "epoch processing: empty validator registry"; return B200_ERR_BAD_ARG; }
    for (int f = 1; f < 5; f++)
        if (big_count(h, f) != n) { e.last_error = "epoch processing: list lengths differ from the registry"; return B200_ERR_BAD_ARG; }
    return B200_SUCCESS;
}

// a failure after the first write leaves a partial state: refuse the handle from then on
int32_t fail_if(b200_state* h, int32_t rc) {
    if (rc) h->failed = true;
    return rc;
}

struct Guard {
    std::unique_lock<std::mutex> lk;
    explicit Guard(Engine& e) : lk(e.mu) {}
};

int32_t ready(Engine& e) {
    if (!e.ready) { e.last_error = "b200_init has not been called (or failed)"; return B200_ERR_NOT_INITIALIZED; }
    cudaError_t ce = cudaSetDevice(e.device);
    if (ce != cudaSuccess) { e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    return B200_SUCCESS;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int32_t b200_state_process_epoch_deneb(b200_state* h, uint32_t stage_mask) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = ready(e);
    if (rc) return rc;
    rc = check_epoch_handle(e, h);
    if (rc) return rc;
    if (stage_mask & ~uint32_t(B200_EPOCH_ALL)) return B200_ERR_BAD_ARG;
    return fail_if(h, process_epoch_locked(e, h, stage_mask));
}

int32_t b200_state_process_slots_deneb(b200_state* h, uint64_t slot) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = ready(e);
    if (rc) return rc;
    rc = check_epoch_handle(e, h);
    if (rc) return rc;
    const PresetConsts& C = kConsts[h->preset];
    Ctx c{e, h, C, big_count(h, 0)};
    if (slot <= c.rd(40)) { e.last_error = "process_slots: TransitionToPreviousSlot"; return B200_ERR_BAD_ARG; }
    while (c.rd(40) < slot) {
        const uint64_t s = c.rd(40);
        // process_slot: cache the state root, fill in the header's state root, cache the block root
        uint8_t root[32];
        rc = state_root_locked(e, h, true, root);
        if (rc) return fail_if(h, rc);
        rc = c.patch(h->so.state_roots + 32 * (s % C.slots_per_historical_root), root, 32);
        if (rc) return fail_if(h, rc);
        constexpr size_t kHeader = 64;   // latest_block_header: slot, proposer_index, parent_root, state_root, body_root
        static const uint8_t zero[32] = {0};
        if (memcmp(h->shadow + kHeader + 48, zero, 32) == 0) {
            rc = c.patch(kHeader + 48, root, 32);
            if (rc) return fail_if(h, rc);
        }
        uint8_t leaves[8][32] = {{0}}, l1[4][32], l2[2][32], hr[32];
        memcpy(leaves[0], h->shadow + kHeader, 8);
        memcpy(leaves[1], h->shadow + kHeader + 8, 8);
        for (int k = 0; k < 3; k++) memcpy(leaves[2 + k], h->shadow + kHeader + 16 + 32 * k, 32);
        for (int k = 0; k < 4; k++) hash_pair(leaves[2 * k], leaves[2 * k + 1], l1[k]);
        for (int k = 0; k < 2; k++) hash_pair(l1[2 * k], l1[2 * k + 1], l2[k]);
        hash_pair(l2[0], l2[1], hr);
        rc = c.patch(h->so.block_roots + 32 * (s % C.slots_per_historical_root), hr, 32);
        if (rc) return fail_if(h, rc);
        if ((s + 1) % C.slots_per_epoch == 0) {
            rc = process_epoch_locked(e, h, B200_EPOCH_ALL);
            if (rc) return fail_if(h, rc);
        }
        rc = c.patch_u64(40, s + 1);
        if (rc) return fail_if(h, rc);
    }
    return B200_SUCCESS;
}

}  // extern "C"
