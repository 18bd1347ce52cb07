// extern "C" entry points — engine life cycle and the SSZ half of include/b200_consensus.h.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <vector>

#include "comm.h"
#include "engine.h"
#include "sha256.cuh"
#include "shuffle.h"
#include "ssz_plan.h"
#include "state_handle.h"

namespace b200 {

Engine& engine() {
    static Engine e;
    return e;
}

namespace {

// crypto::hash on the device: one thread, arbitrary length (parity helper; not a throughput path)
__global__ void k_sha256_bytes(const uint8_t* data, size_t len, uint32_t* out_words) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    uint32_t st[8], w[16];
    sha256_init(st);
    size_t nblocks = (len + 9 + 63) / 64;
    for (size_t b = 0; b < nblocks; b++) {
        for (int i = 0; i < 16; i++) {
            uint32_t v = 0;
            for (int k = 0; k < 4; k++) {
                size_t pos = b * 64 + size_t(i) * 4 + size_t(k);
                uint32_t byte = 0;
                if (pos < len) byte = data[pos];
                else if (pos == len) byte = 0x80;
                else if (pos >= nblocks * 64 - 8) byte = uint32_t((uint64_t(len) * 8) >> (8 * (nblocks * 64 - 1 - pos))) & 0xff;
                v = (v << 8) | byte;
            }
            w[i] = v;
        }
        sha256_compress(st, w);
    }
    for (int i = 0; i < 8; i++) out_words[i] = st[i];
}

struct Guard {
    std::unique_lock<std::mutex> lk;
    explicit Guard(Engine& e) : lk(e.mu) {}
};

int32_t check_ready(Engine& e) {
    if (!e.ready) { e.last_error = "b200_init has not been called (or failed)"; return B200_ERR_NOT_INITIALIZED; }
    cudaError_t ce = cudaSetDevice(e.device);
    if (ce != cudaSuccess) { e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    return B200_SUCCESS;
}

int32_t run_oneshot(Engine& e, SszPlan& plan, const std::vector<uint32_t>& outputs, uint8_t* out) {
    return plan.run(e, e.arena, e.fields, e.planbuf, COPY_ALL, outputs, out);
}

}  // namespace
}  // namespace b200

using namespace b200;

namespace {
// first-job input covering element i of big list f: a Validator record, or the 32-byte chunk of a packed list
inline uint32_t big_input_of(int f, uint64_t i) { return uint32_t(f == 0 ? i : (i * kBigElem[f]) / 32); }
}  // namespace

extern "C" {

int32_t b200_init(int32_t device) {
    Engine& e = engine();
    Guard g(e);
    if (e.ready) return e.device == device ? B200_SUCCESS : B200_ERR_BAD_ARG;
    int n = 0;
    cudaError_t ce = cudaGetDeviceCount(&n);
    if (ce != cudaSuccess || n == 0) {
        e.last_error = std::string("no CUDA device: ") + cudaGetErrorString(ce);
        return B200_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { e.last_error = "device index out of range"; return B200_ERR_BAD_ARG; }
    B200_CUDA_TRY(cudaSetDevice(device));
    B200_CUDA_TRY(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
    B200_CUDA_TRY(cudaStreamCreateWithFlags(&e.copy_stream, cudaStreamNonBlocking));
    B200_CUDA_TRY(cudaEventCreate(&e.ev0));
    B200_CUDA_TRY(cudaEventCreate(&e.ev1));
    for (auto& ev : e.ev_copy) B200_CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    e.device = device;
    const char* a = getenv("B200_SSZ_MINB_VALIDATORS");
    const char* b = getenv("B200_SSZ_MINB_STAGE");
    set_ssz_tuning(a ? atoi(a) : 0, b ? atoi(b) : 0);
    e.ready = true;
    return ensure_zero_nodes(e);
}

void b200_shutdown(void) {
    Engine& e = engine();
    Guard g(e);
    if (!e.ready) return;
    cudaSetDevice(e.device);
    cudaStreamSynchronize(e.stream);
    e.arena.release(); e.fields.release(); e.planbuf.release(); e.staging.release();
    if (e.d_zero) cudaFree(e.d_zero);
    e.d_zero = nullptr;
    cudaEventDestroy(e.ev0); cudaEventDestroy(e.ev1);
    for (auto& ev : e.ev_copy) cudaEventDestroy(ev);
    cudaStreamDestroy(e.stream); cudaStreamDestroy(e.copy_stream);
    e.ready = false;
}

const char* b200_last_error(void) { return engine().last_error.c_str(); }
uint64_t b200_launch_count(void) { return engine().launches; }
float b200_last_kernel_ms(void) { return engine().last_kernel_ms; }

int32_t b200_sha256(const uint8_t* data, size_t len, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!out || (!data && len)) return B200_ERR_BAD_ARG;
    B200_CUDA_TRY(e.fields.reserve(len + 64));
    B200_CUDA_TRY(e.staging.reserve(64));
    if (len) B200_CUDA_TRY(cudaMemcpyAsync(e.fields.p, data, len, cudaMemcpyHostToDevice, e.stream));
    uint32_t* d_out = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(e.fields.p) + ((len + 31) & ~size_t(31)));
    k_sha256_bytes<<<1, 32, 0, e.stream>>>(static_cast<const uint8_t*>(e.fields.p), len, d_out);
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaMemcpyAsync(e.staging.p, d_out, 32, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    const uint32_t* w = static_cast<const uint32_t*>(e.staging.p);
    for (int k = 0; k < 8; k++) {
        out[4 * k] = uint8_t(w[k] >> 24); out[4 * k + 1] = uint8_t(w[k] >> 16);
        out[4 * k + 2] = uint8_t(w[k] >> 8); out[4 * k + 3] = uint8_t(w[k]);
    }
    return B200_SUCCESS;
}

int32_t b200_merkleize(const uint8_t* chunks, size_t n_chunks, uint64_t limit, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!out || (!chunks && n_chunks)) return B200_ERR_BAD_ARG;
    if (limit == 0) limit = n_chunks ? n_chunks : 1;
    if (limit > (uint64_t(1) << 63)) return B200_ERR_BAD_ARG;
    if (n_chunks > limit) return B200_ERR_LIMIT;
    SszPlan p;
    std::vector<uint32_t> outs{p.wide_chunks(p.stage_field(chunks, 32 * n_chunks), n_chunks, depth_for(limit))};
    return run_oneshot(e, p, outs, out);
}

int32_t b200_mix_in_length(const uint8_t root[32], uint64_t length, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!root || !out) return B200_ERR_BAD_ARG;
    SszPlan p;
    std::vector<uint32_t> outs{p.mix_in_length(p.leaf(root), length)};
    return run_oneshot(e, p, outs, out);
}

int32_t b200_is_valid_merkle_branch(const uint8_t leaf[32], const uint8_t* branch, size_t depth, uint64_t index,
                                    const uint8_t root[32], int32_t* ok) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!leaf || !root || !ok || (!branch && depth) || depth > 64) return B200_ERR_BAD_ARG;
    SszPlan p;
    uint32_t v = p.leaf(leaf);
    for (size_t i = 0; i < depth; i++) {
        uint32_t sib = p.leaf(branch + 32 * i);
        v = ((index >> i) & 1) ? p.hash2(sib, v) : p.hash2(v, sib);
    }
    uint8_t got[32];
    std::vector<uint32_t> outs{v};
    rc = run_oneshot(e, p, outs, got);
    if (rc) return rc;
    *ok = memcmp(got, root, 32) == 0 ? 1 : 0;
    return B200_SUCCESS;
}

int32_t b200_htr_validators(const uint8_t* ssz, size_t n, uint64_t limit, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!out || (!ssz && n)) return B200_ERR_BAD_ARG;
    if (limit == 0) limit = n ? n : 1;
    if (limit > (uint64_t(1) << 63)) return B200_ERR_BAD_ARG;
    if (n > limit) return B200_ERR_LIMIT;
    SszPlan p;
    uint32_t r = p.wide_records(JOB_VALIDATORS, p.stage_field(ssz, 121 * n), n, depth_for(limit));
    std::vector<uint32_t> outs{p.mix_in_length(r, n)};
    return run_oneshot(e, p, outs, out);
}

int32_t b200_htr_packed(const uint8_t* data, size_t nbytes, uint64_t limit_chunks, int32_t is_list, uint64_t length,
                        uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!out || (!data && nbytes)) return B200_ERR_BAD_ARG;
    uint64_t n = (nbytes + 31) / 32;
    if (limit_chunks == 0) limit_chunks = n ? n : 1;
    if (limit_chunks > (uint64_t(1) << 63)) return B200_ERR_BAD_ARG;
    if (n > limit_chunks) return B200_ERR_LIMIT;
    SszPlan p;
    uint32_t r = p.wide_chunks(p.stage_field(data, nbytes), n, depth_for(limit_chunks));
    if (is_list) r = p.mix_in_length(r, length);
    std::vector<uint32_t> outs{r};
    return run_oneshot(e, p, outs, out);
}

int32_t b200_htr_beacon_state_deneb(const uint8_t* ssz, size_t len, int32_t preset, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !out) return B200_ERR_BAD_ARG;
    SszPlan p;
    std::vector<uint32_t> outs;
    rc = build_beacon_state_plan(p, ssz, len, preset, outs);
    if (rc) { e.last_error = "malformed deneb BeaconState SSZ"; return rc; }
    return run_oneshot(e, p, outs, out);
}

int32_t b200_state_upload_deneb(const uint8_t* ssz, size_t len, int32_t preset, b200_state** out_handle) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !out_handle) return B200_ERR_BAD_ARG;
    std::unique_ptr<b200_state> h(new b200_state());
    {
        SszPlan first;  // reads the caller's buffer
        std::vector<uint32_t> outs;
        rc = build_beacon_state_plan(first, ssz, len, preset, outs);
        if (rc) { e.last_error = "malformed deneb BeaconState SSZ"; return rc; }
        uint8_t root[32];
        rc = first.run(e, h->arena, h->fields, h->planbuf, COPY_ALL, outs, root);  // uploads + first hash
        if (rc) return rc;  // ~b200_state releases the device buffers
    }
    // keep what is needed to re-plan without the caller's buffer: the serialization minus the big lists
    if (!parse_beacon_state(ssz, len, preset, h->so)) return B200_ERR_SSZ_MALFORMED;
    h->len = len; h->preset = preset;
    h->shadow = static_cast<uint8_t*>(calloc(len ? len : 1, 1));
    if (!h->shadow) { e.last_error = "out of host memory for the state shadow"; return B200_ERR_CUDA; }
    memcpy(h->shadow, ssz, h->so.var[2]);
    memcpy(h->shadow + h->so.var[7], ssz + h->so.var[7], len - h->so.var[7]);
    h->pin();
    rc = build_beacon_state_plan(h->plan, h->shadow, len, preset, h->outputs);  // same layout: it depends on lengths only
    if (rc) return rc;
    h->uploaded = true;
    *out_handle = h.release();
    return B200_SUCCESS;
}

// pending small-field updates: re-plan from the shadow (same arena / field layout, fresh small leaves)
static int32_t replan_if_small_dirty(Engine& e, b200_state* h) {
    if (!h->small_dirty) return B200_SUCCESS;
    SszPlan np;
    std::vector<uint32_t> outs;
    int32_t rc = build_beacon_state_plan(np, h->shadow, h->len, h->preset, outs);
    if (rc) return rc;
    if (np.arena_nodes() != h->plan.arena_nodes() || np.field_bytes() != h->plan.field_bytes() || outs != h->outputs) {
        e.last_error = "state root: plan layout changed";
        return B200_ERR_BAD_ARG;
    }
    h->plan = std::move(np);
    return B200_SUCCESS;
}

}  // extern "C"

namespace b200 {
int32_t state_root_locked(Engine& e, b200_state* h, bool incremental, uint8_t out[32]) {
    int32_t rc = replan_if_small_dirty(e, h);  // updates made through b200_state_update_* are honoured here too
    if (rc) return rc;
    const CopyMode copy = (h->small_dirty || h->relaid) ? COPY_SMALL_ONLY : COPY_NONE;
    // after a re-layout every small field is re-staged (no range filter)
    const auto* ranges = h->relaid ? nullptr : &h->small_ranges;
    if (incremental && !h->all_dirty && !h->relaid) {
        std::vector<std::vector<uint32_t>> dirty(h->plan.n_chains());
        for (int f = 0; f < 9 && size_t(f) < dirty.size(); f++) {
            dirty[size_t(f)] = h->dirty[f];
            std::sort(dirty[size_t(f)].begin(), dirty[size_t(f)].end());
            dirty[size_t(f)].erase(std::unique(dirty[size_t(f)].begin(), dirty[size_t(f)].end()), dirty[size_t(f)].end());
        }
        rc = h->plan.run(e, h->arena, h->fields, h->planbuf, copy, h->outputs, out, &dirty, &h->selbuf, ranges);
    } else {
        rc = h->plan.run(e, h->arena, h->fields, h->planbuf, copy, h->outputs, out, nullptr, nullptr, ranges);
    }
    if (rc) return rc;
    for (auto& d : h->dirty) d.clear();  // a full re-hash covers every dirty path
    h->small_dirty = h->all_dirty = h->relaid = false;
    h->small_ranges.clear();
    return B200_SUCCESS;
}
}  // namespace b200

extern "C" {

int32_t b200_state_root(b200_state* h, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || !out) return B200_ERR_BAD_ARG;
    if (h->sharded)   // every rank of the communicator calls this together: stages | ncclAllGather | finisher
        return h->plan.run(e, h->arena, h->fields, h->planbuf, COPY_NONE, h->outputs, out);
    return state_root_locked(e, h, false, out);
}

void b200_state_free(b200_state* h) {
    if (!h) return;
    Engine& e = engine();
    Guard g(e);
    if (e.ready) { cudaSetDevice(e.device); cudaStreamSynchronize(e.stream); }
    delete h;
}

int32_t b200_state_update_elements(b200_state* h, int32_t field, const uint64_t* indices, const uint8_t* values, size_t n) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || field < 0 || field > 4 || (n && (!indices || !values)) || n > 0xffffffffull) return B200_ERR_BAD_ARG;
    if (!n) return B200_SUCCESS;
    const uint64_t count = big_count(h, field);
    for (size_t i = 0; i < n; i++)
        if (indices[i] >= count) { e.last_error = "state_update_elements: index beyond the list length"; return B200_ERR_BAD_ARG; }
    uint64_t field_off = 0; size_t nbytes = 0;
    if (!h->plan.chain_field(field, &field_off, &nbytes)) return B200_ERR_BAD_ARG;
    const uint32_t elem = kBigElem[field];
    // [indices | values] through pinned staging, then a scatter kernel into the resident list
    const size_t off_vals = n * 8;
    const size_t total = off_vals + n * elem;
    B200_CUDA_TRY(e.staging.reserve(total));
    B200_CUDA_TRY(h->scatter.reserve(total));
    memcpy(e.staging.p, indices, n * 8);
    memcpy(static_cast<uint8_t*>(e.staging.p) + off_vals, values, n * elem);
    B200_CUDA_TRY(cudaMemcpyAsync(h->scatter.p, e.staging.p, total, cudaMemcpyHostToDevice, e.stream));
    launch_scatter(static_cast<uint8_t*>(h->fields.p) + field_off, static_cast<const uint64_t*>(h->scatter.p),
                   static_cast<const uint8_t*>(h->scatter.p) + off_vals, uint32_t(n), elem, e.stream);
    e.launches++;
    B200_CUDA_TRY(cudaGetLastError());
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    for (size_t i = 0; i < n; i++) h->dirty[field].push_back(big_input_of(field, indices[i]));
    return B200_SUCCESS;
}

int32_t b200_state_update_bytes(b200_state* h, uint64_t ssz_offset, const uint8_t* data, size_t n) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || (n && !data) || ssz_offset > h->len || n > h->len - ssz_offset) return B200_ERR_BAD_ARG;
    if (!n) return B200_SUCCESS;
    return state_patch_bytes(e, h, ssz_offset, data, n);
}

}  // extern "C"

namespace b200 {
int32_t state_patch_bytes(Engine& e, b200_state* h, uint64_t ssz_offset, const uint8_t* data, size_t n) {
    const uint64_t lo = ssz_offset, hi = ssz_offset + n;
    // (1) the parts outside the big lists: patch the shadow; the variable-size offsets must not change
    std::vector<uint8_t> saved;
    auto patch_small = [&](uint64_t a, uint64_t b) {  // [a, b) is a small region of the serialization
        const uint64_t x = std::max(a, lo), y = std::min(b, hi);
        if (x >= y) return;
        saved.insert(saved.end(), h->shadow + x, h->shadow + y);
        memcpy(h->shadow + x, data + (x - lo), y - x);
        h->small_ranges.emplace_back(h->shadow + x, h->shadow + y);
    };
    auto restore_small = [&](uint64_t a, uint64_t b, size_t& pos) {
        const uint64_t x = std::max(a, lo), y = std::min(b, hi);
        if (x >= y) return;
        memcpy(h->shadow + x, saved.data() + pos, y - x);
        pos += y - x;
    };
    patch_small(0, h->so.var[2]);
    patch_small(h->so.var[7], h->len);
    if (!saved.empty()) {
        StateOffsets so2;
        bool ok = parse_beacon_state(h->shadow, h->len, h->preset, so2);
        for (int i = 0; ok && i < 10; i++) ok = so2.var[i] == h->so.var[i];
        if (!ok) {  // would move or resize a variable-size field: not an in-place update
            size_t pos = 0;
            restore_small(0, h->so.var[2], pos);
            restore_small(h->so.var[7], h->len, pos);
            // (the ranges stay recorded: re-copying unchanged bytes is harmless)
            e.last_error = "state_update_bytes: the update changes a variable-size field's offset or length; re-upload instead";
            return B200_ERR_BAD_ARG;
        }
        h->small_dirty = true;
    }
    // (2) the parts inside big lists and inside the four big vectors (chains 5..8): copy into the resident field, mark the
    //     covered inputs dirty
    const uint64_t vec_lo[4] = {h->so.block_roots, h->so.state_roots, h->so.randao_mixes, h->so.slashings};
    for (int f = 0; f < 9; f++) {
        if (size_t(f) >= h->plan.n_chains()) break;
        uint64_t field_off = 0; size_t nbytes = 0;
        const bool staged = h->plan.chain_field(f, &field_off, &nbytes);
        const uint64_t a = f < 5 ? h->so.var[kBigVar[f]] : vec_lo[f - 5];
        const uint64_t b = f < 5 ? h->so.var[kBigVar[f] + 1] : a + nbytes;
        const uint64_t x = std::max(a, lo), y = std::min(b, hi);
        if (x >= y) continue;
        if (!staged) return B200_ERR_BAD_ARG;
        B200_CUDA_TRY(e.staging.reserve(y - x));
        memcpy(e.staging.p, data + (x - lo), y - x);
        B200_CUDA_TRY(cudaMemcpyAsync(static_cast<uint8_t*>(h->fields.p) + field_off + (x - a), e.staging.p, y - x,
                                      cudaMemcpyHostToDevice, e.stream));
        B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
        const uint32_t unit = f == 0 ? 121u : 32u;
        for (uint64_t u = (x - a) / unit; u <= (y - 1 - a) / unit; u++) h->dirty[f].push_back(uint32_t(u));
    }
    return B200_SUCCESS;
}

// Variable-size offsets live in the fixed part: the position of each one (StateOffsets::var order, var[9] = end excluded)
static void var_offset_positions(const StateOffsets& so, size_t sc_bytes, size_t pos[9]) {
    pos[0] = so.eth1_data - 4;
    pos[1] = so.eth1_deposit_index - 4;
    pos[2] = so.eth1_deposit_index + 8;
    pos[3] = pos[2] + 4;
    pos[4] = so.justification_bits - 8;
    pos[5] = so.justification_bits - 4;
    pos[6] = so.checkpoints + 120;
    pos[7] = so.next_sync_committee + sc_bytes;
    pos[8] = so.next_withdrawal_validator_index + 8;
}

int32_t state_relayout(Engine& e, b200_state* h, int var, const uint8_t* bytes, size_t n) {
    if (var < 0 || var > 8 || (var >= 2 && var <= 6)) return B200_ERR_BAD_ARG;   // never a big list
    const StateOffsets old = h->so;
    const size_t old_n = size_t(old.var[var + 1] - old.var[var]);
    const size_t new_len = h->len - old_n + n;
    if (new_len > 0xffffffffull) return B200_ERR_BAD_ARG;
    uint8_t* ns = static_cast<uint8_t*>(calloc(new_len ? new_len : 1, 1));
    if (!ns) { e.last_error = "out of host memory for the state shadow"; return B200_ERR_CUDA; }
    // head and tail without the big lists (their ranges stay zero pages), with `var` replaced
    auto copy_shifted = [&](size_t a, size_t b) {  // old range [a, b) that lies entirely before or after `var`
        const size_t shift = a >= old.var[var + 1] ? (n - old_n) : 0;
        memcpy(ns + a + shift, h->shadow + a, b - a);
    };
    if (var < 2) {
        copy_shifted(0, old.var[var]);
        memcpy(ns + old.var[var], bytes, n);
        copy_shifted(old.var[var + 1], old.var[2]);
        copy_shifted(old.var[7], h->len);
    } else {
        copy_shifted(0, old.var[2]);
        copy_shifted(old.var[7], old.var[var]);
        memcpy(ns + old.var[var], bytes, n);
        copy_shifted(old.var[var + 1], h->len);
    }
    size_t pos[9];
    const size_t sc_bytes = old.current_sync_committee < old.next_sync_committee ? old.next_sync_committee - old.current_sync_committee : 0;
    var_offset_positions(old, sc_bytes, pos);
    for (int i = var + 1; i < 9; i++) {
        const uint32_t v = uint32_t(old.var[i] + n - old_n);
        for (int k = 0; k < 4; k++) ns[pos[i] + k] = uint8_t(v >> (8 * k));
    }
    StateOffsets so2;
    if (!parse_beacon_state(ns, new_len, h->preset, so2)) { free(ns); e.last_error = "re-layout: malformed result"; return B200_ERR_BAD_ARG; }
    SszPlan np;
    std::vector<uint32_t> outs;
    int32_t rc = build_beacon_state_plan(np, ns, new_len, h->preset, outs);
    if (rc || np.n_chains() != h->plan.n_chains()) { free(ns); return rc ? rc : B200_ERR_BAD_ARG; }
    // fresh field buffer; every chain (big lists and big vectors) moves device to device, padding included
    DevBuf nf;
    cudaError_t ce = nf.reserve(np.field_bytes() + 256);
    if (ce != cudaSuccess) { free(ns); e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    for (int c = 0; c < int(np.n_chains()); c++) {
        uint64_t fo = 0, fn = 0; size_t nb = 0, nb2 = 0;
        const bool a = h->plan.chain_field(c, &fo, &nb), b = np.chain_field(c, &fn, &nb2);
        if (a != b || nb != nb2) { nf.release(); free(ns); e.last_error = "re-layout: chain size changed"; return B200_ERR_BAD_ARG; }
        if (!a || !nb) continue;
        const size_t padded = (nb + 255) & ~size_t(255);
        ce = cudaMemcpyAsync(static_cast<uint8_t*>(nf.p) + fn, static_cast<const uint8_t*>(h->fields.p) + fo, padded,
                             cudaMemcpyDeviceToDevice, e.stream);
        if (ce != cudaSuccess) { nf.release(); free(ns); e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    }
    ce = cudaStreamSynchronize(e.stream);
    if (ce != cudaSuccess) { nf.release(); free(ns); e.last_error = cudaGetErrorString(ce); return B200_ERR_CUDA; }
    h->unpin();
    free(h->shadow);
    h->fields.release();
    h->fields = nf;
    h->shadow = ns; h->len = new_len; h->so = so2;
    h->plan = std::move(np); h->outputs = std::move(outs);
    h->pin();
    h->relaid = true;
    h->small_dirty = false;
    h->small_ranges.clear();
    return B200_SUCCESS;
}
}  // namespace b200

extern "C" {

int32_t b200_state_root_incremental(b200_state* h, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || !out) return B200_ERR_BAD_ARG;
    return state_root_locked(e, h, true, out);
}

int32_t b200_state_serialized_len(b200_state* h, size_t* out_len) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || !out_len) return B200_ERR_BAD_ARG;
    *out_len = h->len;
    return B200_SUCCESS;
}

// The shadow with the five big lists copied back from HBM
int32_t b200_state_download_deneb(b200_state* h, uint8_t* out, size_t cap) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || !out || cap < h->len) return B200_ERR_BAD_ARG;
    memcpy(out, h->shadow, h->so.var[2]);
    memcpy(out + h->so.var[7], h->shadow + h->so.var[7], h->len - h->so.var[7]);
    for (int f = 0; f < 5; f++) {
        const size_t nb = size_t(h->so.var[kBigVar[f] + 1] - h->so.var[kBigVar[f]]);
        if (!nb) continue;
        uint64_t field_off = 0; size_t staged = 0;
        if (!h->plan.chain_field(f, &field_off, &staged) || staged != nb) return B200_ERR_BAD_ARG;
        B200_CUDA_TRY(cudaMemcpyAsync(out + h->so.var[kBigVar[f]], static_cast<const uint8_t*>(h->fields.p) + field_off, nb,
                                      cudaMemcpyDeviceToHost, e.stream));
    }
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    return B200_SUCCESS;
}

int32_t b200_htr_beacon_state_deneb_shard(const uint8_t* ssz, size_t len, int32_t preset, int32_t rank, int32_t world,
                                          uint8_t* out_roots) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !out_roots) return B200_ERR_BAD_ARG;
    SszPlan p;
    std::vector<uint32_t> outs;
    rc = build_beacon_state_shard_plan(p, ssz, len, preset, rank, world, outs);
    if (rc) return rc;
    return run_oneshot(e, p, outs, out_roots);
}

int32_t b200_htr_beacon_state_deneb_combine(const uint8_t* ssz, size_t len, int32_t preset, int32_t world,
                                            const uint8_t* all_roots, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !all_roots || !out) return B200_ERR_BAD_ARG;
    SszPlan p;
    std::vector<uint32_t> outs;
    rc = build_beacon_state_combine_plan(p, ssz, len, preset, world, all_roots, outs);
    if (rc) return rc;
    return run_oneshot(e, p, outs, out);
}

// get_active_validator_indices + compute_shuffled_indices on a device-resident state: the registry never leaves HBM;
// only the shuffled index list (8 B per active validator) comes back.
int32_t b200_state_shuffled_active_indices(b200_state* h, uint64_t epoch, const uint8_t seed[32], uint32_t rounds, uint64_t* out,
                                           size_t* out_n) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!h || !h->uploaded || h->failed || h->sharded || !seed || !out_n) return B200_ERR_BAD_ARG;
    *out_n = 0;
    const uint64_t n = big_count(h, 0);
    if (n == 0) return B200_SUCCESS;
    if (!out) return B200_ERR_BAD_ARG;
    uint64_t field_off = 0; size_t nbytes = 0;
    if (!h->plan.chain_field(0, &field_off, &nbytes)) return B200_ERR_BAD_ARG;
    uint64_t *d_act, *d_out;
    rc = shuffle_scratch(e, n, &d_act, &d_out);
    if (rc) return rc;
    B200_CUDA_TRY(cudaEventRecord(e.ev0, e.stream));
    uint64_t cnt = 0;
    rc = active_indices_on_device(e, static_cast<const uint8_t*>(h->fields.p) + field_off, n, epoch, d_act, &cnt);
    if (rc) return rc;
    rc = shuffle_on_device(e, d_act, cnt, seed, rounds, d_out);
    if (rc) return rc;
    B200_CUDA_TRY(cudaEventRecord(e.ev1, e.stream));
    if (cnt) B200_CUDA_TRY(cudaMemcpyAsync(out, d_out, cnt * 8, cudaMemcpyDeviceToHost, e.stream));
    B200_CUDA_TRY(cudaStreamSynchronize(e.stream));
    B200_CUDA_TRY(cudaEventElapsedTime(&e.last_kernel_ms, e.ev0, e.ev1));
    *out_n = size_t(cnt);
    return B200_SUCCESS;
}

// A state resident across the ranks of the communicator: every rank keeps its slices of the five big lists (and all small
// fields) in HBM; b200_state_root on such a handle is kernels + one ncclAllGather, no PCIe traffic.  Root only: the
// update / incremental entry points apply to single-GPU handles.
int32_t b200_state_upload_deneb_sharded(const uint8_t* ssz, size_t len, int32_t preset, b200_state** out_handle) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !out_handle) return B200_ERR_BAD_ARG;
    const Comm& c = comm();
    if (!c.ready) { e.last_error = "b200_comm_init has not been called"; return B200_ERR_NOT_INITIALIZED; }
    std::unique_ptr<b200_state> h(new b200_state());
    rc = build_beacon_state_sharded_plan(h->plan, ssz, len, preset, c.rank, c.world, h->outputs);
    if (rc) { e.last_error = "sharded state upload: malformed SSZ or world not a power of two"; return rc; }
    uint8_t root[32];
    rc = h->plan.run(e, h->arena, h->fields, h->planbuf, COPY_ALL, h->outputs, root);   // uploads + first (collective) hash
    if (rc) return rc;
    h->len = len; h->preset = preset;
    h->sharded = true;
    h->uploaded = true;
    *out_handle = h.release();
    return B200_SUCCESS;
}

// One call, all ranks: slices + small fields -> ncclAllGather of 5 x 32 B on the engine stream -> finisher.
int32_t b200_htr_beacon_state_deneb_sharded(const uint8_t* ssz, size_t len, int32_t preset, uint8_t out[32]) {
    Engine& e = engine();
    Guard g(e);
    int32_t rc = check_ready(e);
    if (rc) return rc;
    if (!ssz || !out) return B200_ERR_BAD_ARG;
    const Comm& c = comm();
    if (!c.ready) { e.last_error = "b200_comm_init has not been called"; return B200_ERR_NOT_INITIALIZED; }
    SszPlan p;
    std::vector<uint32_t> outs;
    rc = build_beacon_state_sharded_plan(p, ssz, len, preset, c.rank, c.world, outs);
    if (rc) { e.last_error = "sharded hash_tree_root: malformed SSZ or world not a power of two"; return rc; }
    return run_oneshot(e, p, outs, out);
}

}  // extern "C"
