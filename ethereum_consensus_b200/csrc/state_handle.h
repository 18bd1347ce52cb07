// The device-resident deneb BeaconState handle (b200_state), shared by the SSZ entry points (capi_ssz.cu) and epoch
// processing (epoch.cu).  Callers of every function here hold the engine lock and have selected the device.
#pragma once
#include <cstdlib>
#include <utility>
#include <vector>

#include "engine.h"
#include "ssz_plan.h"

struct b200_state {
    b200::SszPlan plan;
    std::vector<uint32_t> outputs;
    b200::DevBuf arena, fields, planbuf, selbuf, scatter, epoch_scratch;
    bool uploaded = false;
    // ---- incremental re-hash (b200_state_update_* / b200_state_root_incremental) ----
    // Host shadow of the serialization with everything EXCEPT the five big lists filled in (their byte ranges stay
    // untouched zero pages of an anonymous mapping): small-field updates patch it and the plan is rebuilt from it.
    uint8_t* shadow = nullptr;
    size_t len = 0;
    int preset = 0;
    b200::StateOffsets so;
    // per chain (5 big lists, then block_roots / state_roots / randao_mixes / slashings): changed first-job inputs
    // (Validator records / 32-byte chunks), unsorted
    std::vector<uint32_t> dirty[9];
    // a kernel rewrote whole lists (epoch processing): the next root re-hashes everything instead of dirty paths
    bool all_dirty = false;
    // the field buffer was re-laid out (a variable-size field changed length): every small field must be re-staged
    bool relaid = false;
    // epoch processing failed part-way: the state is not a valid post-state, every call refuses the handle
    bool failed = false;
    bool small_dirty = false;
    std::vector<std::pair<const uint8_t*, const uint8_t*>> small_ranges;  // patched shadow bytes since the last root
    bool pinned_head = false, pinned_tail = false;
    bool sharded = false;   // b200_state_upload_deneb_sharded: this rank's slices only; root is a collective, no updates
    void unpin() {
        if (pinned_head) cudaHostUnregister(shadow);
        if (pinned_tail) cudaHostUnregister(shadow + so.var[7]);
        pinned_head = pinned_tail = false;
    }
    // page-lock the two populated ranges (a few MB) so that re-staging a patched small field is a real async DMA
    void pin() {
        pinned_head = cudaHostRegister(shadow, so.var[2], cudaHostRegisterDefault) == cudaSuccess;
        pinned_tail = cudaHostRegister(shadow + so.var[7], len - so.var[7], cudaHostRegisterDefault) == cudaSuccess;
        cudaGetLastError();  // registration is an optimisation: pageable copies work too
    }
    ~b200_state() {
        unpin();
        free(shadow);
        arena.release(); fields.release(); planbuf.release(); selbuf.release(); scatter.release(); epoch_scratch.release();
    }
};

namespace b200 {

constexpr int kBigVar[5] = {2, 3, 4, 5, 6};         // StateOffsets::var index of each big list
constexpr uint32_t kBigElem[5] = {121, 8, 1, 1, 8};  // element size in bytes
inline uint64_t big_count(const b200_state* h, int f) {
    return uint64_t(h->so.var[kBigVar[f] + 1] - h->so.var[kBigVar[f]]) / kBigElem[f];
}

// Overwrite bytes [off, off + n) of the resident serialization: the shadow, the device copies of the big lists and
// big vectors, and the dirty sets stay coherent.  Rejects a change of any variable-size field's offset or length.
int32_t state_patch_bytes(Engine& e, b200_state* h, uint64_t off, const uint8_t* data, size_t n);
// Replace the contents of variable-size field `var` (StateOffsets::var index; not one of the five big lists) with
// `bytes`: new shadow and plan, a fresh field buffer into which every big list and big vector is copied device to
// device, and the next root is a full one.
int32_t state_relayout(Engine& e, b200_state* h, int var, const uint8_t* bytes, size_t n);
// hash_tree_root of the resident state (full, or only the dirty paths when `incremental`)
int32_t state_root_locked(Engine& e, b200_state* h, bool incremental, uint8_t out[32]);
// eth_aggregate_public_keys over n host keys (capi_bls.cu)
int32_t eth_aggregate_public_keys_locked(Engine& e, const uint8_t* pks_flat, size_t n, uint8_t out[48]);

}  // namespace b200
