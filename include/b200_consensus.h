/*
 * b200_consensus.h — C ABI of the B200-native batch-crypto engine.
 *
 * This is the drop-in boundary for ralexstokes/ethereum_consensus' hot path (SURVEY.md §8b):
 *   - BLS:  the seven free functions re-exported at
 *           /root/reference/ethereum-consensus/src/crypto/mod.rs:4-8 (bodies in crypto/bls.rs:64-160), whose only
 *           backend today is `use blst::{min_pk as bls_impl, BLST_ERROR}` (crypto/bls.rs:4);
 *   - SSZ:  `HashTreeRoot::hash_tree_root` / `merkleize` / `is_valid_merkle_branch` from
 *           `pub use ssz_rs::prelude::*` (/root/reference/ethereum-consensus/src/ssz/mod.rs:6).
 * Plain pointers and sizes only; the caller owns every buffer; calls are synchronous and thread-safe (one
 * process-global context per device).  INTEGRATION.md shows the Rust `extern "C"` block that binds these.
 *
 * Return codes: 0..7 are blst's BLST_ERROR values (order pinned by
 * /root/reference/ethereum-consensus/src/crypto/bls.rs:48-62); >= 0x100 are engine failures (CUDA, bad
 * arguments, malformed SSZ) and are NEVER conflated with a signature verdict.  There is no CPU fallback: if
 * the device or the CUDA library is unavailable every entry point returns B200_ERR_NO_DEVICE / B200_ERR_CUDA.
 */
#ifndef B200_CONSENSUS_H
#define B200_CONSENSUS_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes -------------------------------------------------------------------------------- */
enum {
    B200_SUCCESS = 0,            /* BLST_SUCCESS */
    B200_BAD_ENCODING = 1,       /* BLST_BAD_ENCODING */
    B200_POINT_NOT_ON_CURVE = 2, /* BLST_POINT_NOT_ON_CURVE */
    B200_POINT_NOT_IN_GROUP = 3, /* BLST_POINT_NOT_IN_GROUP */
    B200_AGGR_TYPE_MISMATCH = 4, /* BLST_AGGR_TYPE_MISMATCH */
    B200_VERIFY_FAIL = 5,        /* BLST_VERIFY_FAIL  -> Error::InvalidSignature (crypto/bls.rs:127-131) */
    B200_PK_IS_INFINITY = 6,     /* BLST_PK_IS_INFINITY */
    B200_BAD_SCALAR = 7,         /* BLST_BAD_SCALAR */
    B200_EMPTY_AGGREGATE = 16,   /* Error::EmptyAggregate (crypto/bls.rs:80-82,136-138) */
    B200_KZG_BAD_ARGS = 17,      /* kzg::Error::CKzg(..) (crypto/kzg.rs:47-53): malformed KZG input, see the KZG section */
    B200_STATE_TRANSITION_INVALID = 18, /* epoch / slot processing: a uint64 overflow or a failed spec assertion */
    B200_ERR_CUDA = 0x100,
    B200_ERR_NO_DEVICE = 0x101,
    B200_ERR_BAD_ARG = 0x102,
    B200_ERR_SSZ_MALFORMED = 0x103, /* offsets / lengths inconsistent with the container schema */
    B200_ERR_NOT_INITIALIZED = 0x104,
    B200_ERR_LIMIT = 0x105,         /* more chunks than the declared limit (MerkleizationError) */
    B200_ERR_COMM = 0x106           /* NCCL missing / communicator failure (multi-GPU entry points) */
};

enum { B200_PRESET_MAINNET = 0, B200_PRESET_MINIMAL = 1 };

/* ---- life cycle ------------------------------------------------------------------------------------ */
/* Binds the calling process to CUDA device `device` (one process per GPU).  Idempotent. */
B200_API int32_t b200_init(int32_t device);
B200_API void b200_shutdown(void);
/* Human-readable text for the last engine failure (>= 0x100) on this thread's context. */
B200_API const char* b200_last_error(void);
/* Number of kernel launches issued by the library since b200_init (bench.py's gpu_launches). */
B200_API uint64_t b200_launch_count(void);
/* Device time (ms, CUDA events on the library stream) of the kernels of the last SSZ / BLS call. */
B200_API float b200_last_kernel_ms(void);

/* ---- SSZ / SHA-256 Merkle (replaces ssz_rs merkleize / hash_tree_root; sha2 one-shot) -------------- */
/* crypto::hash — /root/reference/ethereum-consensus/src/crypto/bls.rs:12-20 (computed on the device). */
B200_API int32_t b200_sha256(const uint8_t* data, size_t len, uint8_t out[32]);

/* merkleize(chunks, limit): `n_chunks` 32-byte chunks, virtually zero-padded to `limit` chunks
 * (limit == 0: next power of two of n_chunks).  ssz_rs `merkleize`. */
B200_API int32_t b200_merkleize(const uint8_t* chunks, size_t n_chunks, uint64_t limit, uint8_t out[32]);
/* mix_in_length(root, len) */
B200_API int32_t b200_mix_in_length(const uint8_t root[32], uint64_t length, uint8_t out[32]);
/* is_valid_merkle_branch(leaf, branch[depth], depth, index, root): *ok = 1/0.
 * Used at /root/reference/ethereum-consensus/src/phase0/block_processing.rs:428-437 and deneb/blob_sidecar.rs:58-63. */
B200_API int32_t b200_is_valid_merkle_branch(const uint8_t leaf[32], const uint8_t* branch, size_t depth, uint64_t index,
                                    const uint8_t root[32], int32_t* ok);

/* hash_tree_root(List<Validator, limit>) from N x 121 bytes of SSZ (phase0/validator.rs:10-26). */
B200_API int32_t b200_htr_validators(const uint8_t* ssz, size_t n, uint64_t limit, uint8_t out[32]);
/* hash_tree_root of a packed basic List (is_list=1, mixes `length`) or Vector (is_list=0):
 * `nbytes` of little-endian elements, limit in chunks. */
B200_API int32_t b200_htr_packed(const uint8_t* data, size_t nbytes, uint64_t limit_chunks, int32_t is_list, uint64_t length,
                        uint8_t out[32]);

/* hash_tree_root(deneb::BeaconState) from its SSZ serialization
 * (/root/reference/ethereum-consensus/src/deneb/beacon_state.rs:13-64; called at deneb/spec/mod.rs:3215,3288). */
B200_API int32_t b200_htr_beacon_state_deneb(const uint8_t* ssz, size_t len, int32_t preset, uint8_t out[32]);

/* Device-resident state: upload once, re-hash many times (kernel-only cost; SURVEY.md §8f-2 groundwork). */
typedef struct b200_state b200_state;
B200_API int32_t b200_state_upload_deneb(const uint8_t* ssz, size_t len, int32_t preset, b200_state** out_handle);
B200_API int32_t b200_state_root(b200_state* handle, uint8_t out[32]);
B200_API void b200_state_free(b200_state* handle);

/* Incremental re-hash of a device-resident state (SURVEY.md §8b `b200_state_update_leaves`, §8f-2): the two
 * `state.hash_tree_root()` calls per block (deneb/spec/mod.rs:3215,3288) then cost O(changed x depth), not O(N).
 *  - b200_state_update_elements: overwrite elements `indices[i]` of one of the five big lists with `values`
 *    (n x 121 / 8 / 1 bytes, SSZ encoding of Validator / u64 / participation flags).  List lengths do not change;
 *    an index may appear more than once only with identical values (elements are written in parallel).
 *  - b200_state_update_bytes: overwrite bytes [ssz_offset, ssz_offset + n) of the serialization that was uploaded
 *    (any field; must not change a variable-size field's offset or length — re-upload for that).
 *  - b200_state_root_incremental: root after the updates.  Dirty paths of the big lists only; everything small
 *    (~1 % of the hashes) is re-hashed in full.  b200_state_root stays the full O(N) re-hash. */
#define B200_FIELD_VALIDATORS 0
#define B200_FIELD_BALANCES 1
#define B200_FIELD_PREVIOUS_EPOCH_PARTICIPATION 2
#define B200_FIELD_CURRENT_EPOCH_PARTICIPATION 3
#define B200_FIELD_INACTIVITY_SCORES 4
B200_API int32_t b200_state_update_elements(b200_state* handle, int32_t field, const uint64_t* indices, const uint8_t* values, size_t n);
B200_API int32_t b200_state_update_bytes(b200_state* handle, uint64_t ssz_offset, const uint8_t* data, size_t n);
B200_API int32_t b200_state_root_incremental(b200_state* handle, uint8_t out[32]);

/* Multi-GPU sharding of hash_tree_root(BeaconState) (SURVEY.md §8e): rank r of `world` hashes its contiguous
 * power-of-two-aligned slice of the five big lists and returns one subtree root per list
 * (out_roots: 5 x 32 bytes, order validators, balances, previous/current participation, inactivity_scores);
 * after an allgather of those roots, b200_htr_beacon_state_deneb_combine finishes the tree on any rank. */
B200_API int32_t b200_htr_beacon_state_deneb_shard(const uint8_t* ssz, size_t len, int32_t preset, int32_t rank, int32_t world,
                                          uint8_t* out_roots /* 5*32 */);
B200_API int32_t b200_htr_beacon_state_deneb_combine(const uint8_t* ssz, size_t len, int32_t preset, int32_t world,
                                            const uint8_t* all_roots /* world*5*32 */, uint8_t out[32]);

/* ---- committee shuffling (SURVEY.md §8f-3): the step before the BLS hot path ---------------------------------- */
/* compute_shuffled_indices — /root/reference/ethereum-consensus/src/phase0/helpers.rs:287-360 (whole list; equal to
 * mapping every position through compute_shuffled_index, :249-283): out[i] = indices[shuffled_index(i, n, seed)].
 * `indices` == NULL means the identity list 0..n-1; `rounds` = SHUFFLE_ROUND_COUNT (90 on mainnet, 10 on minimal). */
B200_API int32_t b200_compute_shuffled_indices(const uint64_t* indices, size_t n, const uint8_t seed[32], uint32_t rounds,
                                               uint64_t* out);
/* get_active_validator_indices — phase0/helpers.rs:646-676 over n x 121 bytes of SSZ Validator records
 * (activation_epoch <= epoch < exit_epoch); `out` must hold n entries, *out_n receives the count. */
B200_API int32_t b200_get_active_validator_indices(const uint8_t* validators_ssz, size_t n, uint64_t epoch, uint64_t* out,
                                                   size_t* out_n);
/* Both steps on a device-resident state (b200_state_upload_deneb): the registry never leaves HBM, only the shuffled
 * active-index list returns.  get_beacon_committee (phase0/helpers.rs:775-806) is then the slice
 * [len*index/count, len*(index+1)/count) of `out` (compute_committee, :459-483). */
B200_API int32_t b200_state_shuffled_active_indices(b200_state* handle, uint64_t epoch, const uint8_t seed[32], uint32_t rounds,
                                                    uint64_t* out, size_t* out_n);

/* ---- epoch and slot processing on a device-resident state (deneb/spec/mod.rs:965-1004, :3150-3240) ---------------
 * b200_state_process_epoch_deneb runs the process_epoch stages whose bits are set in `stage_mask`, in this order:
 *   0 justification_and_finalization, 1 inactivity_updates, 2 rewards_and_penalties, 3 registry_updates, 4 slashings,
 *   5 eth1_data_reset, 6 effective_balance_updates, 7 slashings_reset, 8 randao_mixes_reset,
 *   9 historical_summaries_update, 10 participation_flag_updates, 11 sync_committee_updates.
 * B200_EPOCH_ALL is process_epoch; a single bit is one epoch_processing sub-function.  The state stays in HBM: the
 * next b200_state_root / b200_state_root_incremental returns the post-state root.
 * b200_state_process_slots_deneb follows process_slots up to `slot` (process_epoch at each epoch boundary);
 * slot <= state.slot returns B200_ERR_BAD_ARG (TransitionToPreviousSlot).
 * Codes: B200_STATE_TRANSITION_INVALID for a uint64 overflow (the spec's rule; the reference Rust wraps or panics) or
 * a failed spec assertion; 1..7 for an invalid public key in the next sync committee (as b200_eth_aggregate_public_keys).
 * After either, the handle is failed: every later call on it returns B200_ERR_BAD_ARG until it is freed.  Sharded
 * handles, an empty registry and lists whose lengths differ from the registry's return B200_ERR_BAD_ARG. */
#define B200_EPOCH_JUSTIFICATION_AND_FINALIZATION (1u << 0)
#define B200_EPOCH_INACTIVITY_UPDATES (1u << 1)
#define B200_EPOCH_REWARDS_AND_PENALTIES (1u << 2)
#define B200_EPOCH_REGISTRY_UPDATES (1u << 3)
#define B200_EPOCH_SLASHINGS (1u << 4)
#define B200_EPOCH_ETH1_DATA_RESET (1u << 5)
#define B200_EPOCH_EFFECTIVE_BALANCE_UPDATES (1u << 6)
#define B200_EPOCH_SLASHINGS_RESET (1u << 7)
#define B200_EPOCH_RANDAO_MIXES_RESET (1u << 8)
#define B200_EPOCH_HISTORICAL_SUMMARIES_UPDATE (1u << 9)
#define B200_EPOCH_PARTICIPATION_FLAG_UPDATES (1u << 10)
#define B200_EPOCH_SYNC_COMMITTEE_UPDATES (1u << 11)
#define B200_EPOCH_ALL 0xfffu
B200_API int32_t b200_state_process_epoch_deneb(b200_state* handle, uint32_t stage_mask);
B200_API int32_t b200_state_process_slots_deneb(b200_state* handle, uint64_t slot);
/* SSZ serialization of the current resident state (small fields from the host shadow, the five big lists copied back
 * from HBM).  `cap` must be at least b200_state_serialized_len. */
B200_API int32_t b200_state_serialized_len(b200_state* handle, size_t* out_len);
B200_API int32_t b200_state_download_deneb(b200_state* handle, uint8_t* out, size_t cap);

/* ---- multi-GPU: one process per GPU, the exchange step lives INSIDE the library (SURVEY.md §8b `b200_init(n_gpus)`,
 * §8e).  The reference is single-process (no counterpart, SURVEY.md §2a); a Rust host with one process per GPU calls:
 *   rank 0:   b200_comm_unique_id(id)  -> ships the 128 bytes to the other ranks by any means it likes (pipe, file, TCP)
 *   all ranks: b200_init(local_gpu); b200_comm_init(id, rank, world)       (collective; NCCL over NVLink / NVSwitch)
 * and then the *_sharded entry points below, which every rank must call with the same arguments.  world == 1 is
 * legal (no NCCL needed) and makes the sharded calls equivalent to the single-GPU ones. */
#define B200_COMM_ID_BYTES 128
B200_API int32_t b200_comm_unique_id(uint8_t out_id[B200_COMM_ID_BYTES]);
B200_API int32_t b200_comm_init(const uint8_t id[B200_COMM_ID_BYTES], int32_t rank, int32_t world);
B200_API int32_t b200_comm_info(int32_t* rank, int32_t* world, int32_t* nccl_version);
B200_API void b200_comm_destroy(void);
/* all-gather of `bytes_per_rank` host bytes per rank into recv[world * bytes_per_rank] (rank-major): for the host's own
 * small exchanges, e.g. verdict vectors when every rank verified a different batch (weak scaling). */
B200_API int32_t b200_comm_all_gather_bytes(const uint8_t* send, size_t bytes_per_rank, uint8_t* recv);
/* NCCL collectives issued by the library since start-up (bench.py reports it next to gpu_launches). */
B200_API uint64_t b200_collective_count(void);

/* hash_tree_root(deneb::BeaconState) computed by all ranks of the communicator in ONE call (deneb/spec/mod.rs:3215,3288):
 * every rank passes the same serialization, uploads and hashes only its power-of-two-aligned slice of the five big
 * lists (parallel H2D over every GPU's own PCIe link) together with all small fields, the 5 x 32-byte slice roots are
 * exchanged with one ncclAllGather on the engine stream, and the finisher completes the tree on every rank: no host
 * round trip between the phases.  world must be a power of two.  Every rank gets the same `out`. */
B200_API int32_t b200_htr_beacon_state_deneb_sharded(const uint8_t* ssz, size_t len, int32_t preset, uint8_t out[32]);
/* The same, resident: every rank uploads its slices (and the small fields) once; b200_state_root on the returned handle is
 * then a collective of kernels + one ncclAllGather with no PCIe traffic (all ranks call it together; b200_state_free per
 * rank).  Root only — the update / incremental / shuffling entry points take single-GPU handles. */
B200_API int32_t b200_state_upload_deneb_sharded(const uint8_t* ssz, size_t len, int32_t preset, b200_state** out_handle);

/* b200_fast_aggregate_verify_batch over all ranks (BASELINE configs[4]: an epoch's attestation batch sharded over
 * 8 GPUs): every rank passes the same T tuples, verifies the contiguous block parallel.tuple_shard(T, world, rank)
 * names (only that block's keys cross PCIe), and one ncclAllGather of the int32 verdicts leaves all T codes in
 * `out_codes` on every rank — what process_block needs to pick the first failure. */
B200_API int32_t b200_fast_aggregate_verify_batch_sharded(const uint8_t* pks_flat, const uint32_t* pk_offsets,
                                                          const uint8_t* msgs32, const uint8_t* sigs, size_t n_tuples,
                                                          int32_t* out_codes);

/* ---- BLS12-381 signatures, min-pk (replaces the blst calls of crypto/bls.rs) ------------------------- */
/* Public keys are 48-byte and signatures 96-byte ZCash-compressed points (crypto/bls.rs:23-25,227-239,287-290);
 * the ciphersuite / DST is the one at crypto/bls.rs:22.  Results: 0 = Ok(()), 5 = Err(InvalidSignature),
 * 1,2,3,6 = Err(Error::BLST(..)) from key_validate / Signature::from_bytes, first offending input in order. */

/* verify_signature — crypto/bls.rs:64-77 */
B200_API int32_t b200_verify_signature(const uint8_t pk[48], const uint8_t* msg, size_t msg_len, const uint8_t sig[96]);
/* fast_aggregate_verify — crypto/bls.rs:114-132; `pks` is the array of K pointers the reference passes
 * (`&[&PublicKey]`, gathered from state.validators at phase0/helpers.rs:123-131) */
B200_API int32_t b200_fast_aggregate_verify(const uint8_t* const* pks, size_t k, const uint8_t* msg, size_t msg_len,
                                            const uint8_t sig[96]);
/* eth_fast_aggregate_verify — crypto/bls.rs:150-160 */
B200_API int32_t b200_eth_fast_aggregate_verify(const uint8_t* const* pks, size_t k, const uint8_t* msg, size_t msg_len,
                                                const uint8_t sig[96]);
/* aggregate_verify — crypto/bls.rs:95-112; n_pks x 48 contiguous bytes, n_msgs (pointer,length) messages */
B200_API int32_t b200_aggregate_verify(const uint8_t* pks_flat, size_t n_pks, const uint8_t* const* msgs,
                                       const size_t* msg_lens, size_t n_msgs, const uint8_t sig[96]);
/* aggregate — crypto/bls.rs:79-93; n == 0 -> B200_EMPTY_AGGREGATE; out = compressed sum */
B200_API int32_t b200_aggregate(const uint8_t* sigs_flat, size_t n, uint8_t out[96]);
/* eth_aggregate_public_keys — crypto/bls.rs:135-148 */
B200_API int32_t b200_eth_aggregate_public_keys(const uint8_t* pks_flat, size_t n, uint8_t out[48]);

/* The throughput path: T independent fast_aggregate_verify tuples in one call (the batch of attestation checks
 * `process_block` issues one by one at deneb/block_processing.rs:104-108).  Tuple t uses public keys
 * pk_offsets[t] .. pk_offsets[t+1] of `pks_flat`, the 32-byte signing root msgs32[32t..] and sigs[96t..];
 * out_codes[t] is exactly what b200_fast_aggregate_verify would return for that tuple (strict mode: every key is
 * decompressed and validated in every call, as crypto/bls.rs:119-123 does). */
B200_API int32_t b200_fast_aggregate_verify_batch(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                                  const uint8_t* sigs, size_t n_tuples, int32_t* out_codes);
/* Optimistic WHOLE-BATCH check by random linear combination (north_star: "Miller loops fused across the batch, partial Gt
 * products reduced with warp shuffles"): *all_ok = 1 iff every tuple of the batch would return 0 above — decided with
 * T Miller loops and ONE final exponentiation instead of 2T and T:  prod_t e(r_t agg_t, H(msg_t)) * e(-g1, sum_t r_t sig_t) == 1
 * for 64-bit scalars r_t = SHA-256(seed || t).  Valid batches are always accepted; a batch with an invalid tuple is
 * accepted with probability <= 2^-64 over the seed (seed32 == NULL: the library draws one from the OS; tests pass a fixed
 * seed).  This is the normal-case path of process_block (every signature of a block is expected to verify); on
 * *all_ok == 0 the caller asks b200_fast_aggregate_verify_batch, which remains the only source of per-tuple codes. */
B200_API int32_t b200_fast_aggregate_verify_batch_all(const uint8_t* pks_flat, const uint32_t* pk_offsets, const uint8_t* msgs32,
                                                      const uint8_t* sigs, size_t n_tuples, const uint8_t* seed32, int32_t* all_ok);
/* Registry mode: validate the (append-only, immutable-pubkey) validator registry once, keep the affine keys in
 * HBM, then verify tuples that name their signers by validator index.  Same per-tuple codes as the strict path. */
B200_API int32_t b200_registry_load(const uint8_t* pks_flat, size_t n);
B200_API int32_t b200_registry_key_codes(int32_t* out_codes, size_t n);
B200_API int32_t b200_fast_aggregate_verify_batch_indexed(const uint32_t* indices, const uint32_t* offsets,
                                                          const uint8_t* msgs32, const uint8_t* sigs, size_t n_tuples,
                                                          int32_t* out_codes);
/* Registry mode for a whole block's signature set in ONE call: `extra_pks` are the n_extra (<= 65 536) 48-byte keys that
 * are not in the registry because they arrive in the block itself (deposits `phase0/block_processing.rs:387-392`, bls-to-
 * execution changes `capella/block_processing.rs:43-56`); they are decompressed + validated by this call exactly like
 * the strict path does, and an index i >= n_registry names extra key i - n_registry.  Codes as the strict path's. */
B200_API int32_t b200_fast_aggregate_verify_batch_mixed(const uint8_t* extra_pks, size_t n_extra, const uint32_t* indices,
                                                        const uint32_t* offsets, const uint8_t* msgs32, const uint8_t* sigs,
                                                        size_t n_tuples, int32_t* out_codes);
/* RLC whole-batch check over registry indices, and over all ranks of the communicator: every rank passes the same batch
 * and the same (non-NULL) seed, verifies its block, and ONE ncclAllGather moves the per-rank Gt partial (576 B) and G2
 * partial (288 B); every rank then finishes the same final exponentiation and returns the same boolean. */
B200_API int32_t b200_fast_aggregate_verify_batch_indexed_all(const uint32_t* indices, const uint32_t* offsets,
                                                              const uint8_t* msgs32, const uint8_t* sigs, size_t n_tuples,
                                                              const uint8_t* seed32, int32_t* all_ok);
B200_API int32_t b200_fast_aggregate_verify_batch_all_sharded(const uint8_t* pks_flat, const uint32_t* pk_offsets,
                                                              const uint8_t* msgs32, const uint8_t* sigs, size_t n_tuples,
                                                              const uint8_t seed32[32], int32_t* all_ok);
/* Device time (ms) of the dominant kernel (per-key validation) of the last BLS call. */
B200_API float b200_last_dominant_kernel_ms(void);
/* Measured integer-pipe peak on this device, 1e9 ops/s: kind 0 IMAD.WIDE.U32 (Montgomery multiply-add), 1 IMAD.U32,
 * 2 LOP3/SHF/IADD3 mix (SHA-256 round ops).  Roofline denominators for bench.py. */
B200_API int32_t b200_measure_int_peak(int32_t kind, double* gops);
/* Scheduling knobs of the BLS batch pipeline, settable at run time (the same names, upper-cased with a B200_ prefix, are
 * read from the environment when the pipeline is first used).  They change launch shapes only, never a result:
 *   "bls_chunks" (key ranges per strict batch, 1 = off), "bls_chunk_min_tuples", "bls_chunk_k1_cta" (128 | 384),
 *   "bls_chunk_alt" (0 | 1: alternate key ranges over two streams), "bls_key_split" (0 | 1: big strict batches copy most
 *   of their keys under the first waves of the per-key kernel), "bls_k1_first_cta" (128 | 384: CTA size of those first waves),
 *   "bls_small_cta" (0 = by batch size | 32 | 64 | 128: CTA size of the signature / message kernels), "vm_team16_max",
 *   "vm_cta" (32 | 64 | 128).
 * Unknown knob -> B200_ERR_BAD_ARG. */
B200_API int32_t b200_tune(const char* knob, int64_t value);
/* Replaces the scheduled Miller-loop / final-exponentiation programs of one team size (8 or 16 lanes) of the lane-parallel
 * pairing kernels with another SCHEDULE of the same formulas: `blob` is what `tools/gen_pairing_vm.py <team> ... --blob F`
 * writes after executing the schedule numerically against the direct evaluation.  Opcodes and slot indices are validated;
 * a malformed blob -> B200_ERR_BAD_ARG and the programs in use stay.  Schedule tuning only: results never depend on it. */
B200_API int32_t b200_vm_load_programs(const uint32_t* blob, size_t n_words);
/* On-device self-test of the field arithmetic over `n` pseudo-random triples; *mismatches must come back 0. */
B200_API int32_t b200_fp_selftest(uint32_t n, uint32_t seed, uint32_t* mismatches);

/* ---- KZG blob proofs, deneb (replaces the c_kzg verification calls of crypto/kzg.rs) ------------------------------- */
/* Semantics of the deneb polynomial-commitments spec (what c-kzg implements).  Field elements (blob elements, z, y) are
 * 32-byte big-endian integers that must be < r; commitments and proofs are 48-byte compressed G1 points that must
 * decompress and lie in G1 (the infinity encoding is valid: the zero polynomial).  Results: 0 = Ok(()),
 * B200_VERIFY_FAIL = Err(Error::InvalidProof), B200_KZG_BAD_ARGS = Err(Error::CKzg(..)) for any malformed input;
 * engine failures stay >= 0x100.  A blob is 4 096 field elements = 131 072 bytes. */
#define B200_KZG_BYTES_PER_BLOB 131072
/* batch entry points take at most this many blobs per call (16 GiB of blobs would not fit the device anyway:
 * each blob is 128 KiB of host-to-device copy) -> B200_ERR_BAD_ARG above it */
#define B200_KZG_MAX_BLOBS 16384
typedef struct b200_kzg_settings b200_kzg_settings;
/* KzgSettings::load_trusted_setup — crypto/kzg.rs:39-45.  n_g1 must be 4 096 (g1_lagrange, natural order) and n_g2 >= 2
 * (g2_monomial); every point must decode and lie in its subgroup, else B200_KZG_BAD_ARGS.  Resident on the device:
 * [tau]G2 = g2_monomial[1] and the bit-reversed roots of unity (verification), and the prover's fixed-base table built
 * from g1_lagrange in bit-reversed order (52 x 16 multiples of each point, 327 MB; built on the device at load time). */
B200_API int32_t b200_kzg_settings_load(const uint8_t* g1_lagrange, size_t n_g1, const uint8_t* g2_monomial, size_t n_g2,
                                        b200_kzg_settings** out);
B200_API void b200_kzg_settings_free(b200_kzg_settings* settings);
/* verify_kzg_proof — crypto/kzg.rs:101-122 */
B200_API int32_t b200_verify_kzg_proof(const b200_kzg_settings* settings, const uint8_t commitment[48], const uint8_t z[32],
                                       const uint8_t y[32], const uint8_t proof[48]);
/* verify_blob_kzg_proof — crypto/kzg.rs:124-137 */
B200_API int32_t b200_verify_blob_kzg_proof(const b200_kzg_settings* settings, const uint8_t* blob, const uint8_t commitment[48],
                                            const uint8_t proof[48]);
/* verify_blob_kzg_proof_batch — crypto/kzg.rs:139-174: one code for n blobs (n x 131 072, n x 48, n x 48 bytes).  n = 0
 * returns 0; any malformed input returns B200_KZG_BAD_ARGS; otherwise 0 iff every blob's proof verifies.  The spec decides
 * this with a random linear combination, which differs only with probability <= n / r; here every blob is checked. */
B200_API int32_t b200_verify_blob_kzg_proof_batch(const b200_kzg_settings* settings, const uint8_t* blobs, const uint8_t* commitments,
                                                  const uint8_t* proofs, size_t n);
/* The throughput path (no counterpart in the reference): n independent blob checks in one call; out_codes[i] is exactly
 * what b200_verify_blob_kzg_proof returns for blob i (which is this call with n = 1). */
B200_API int32_t b200_verify_blob_kzg_proofs(const b200_kzg_settings* settings, const uint8_t* blobs, const uint8_t* commitments,
                                             const uint8_t* proofs, size_t n, int32_t* out_codes);
/* The prover.  Outputs are 48-byte compressed G1 points (the point at infinity is 0xc0 || 0^47) and, for
 * compute_kzg_proof, y = p(z) as 32 big-endian bytes.  B200_KZG_BAD_ARGS: a blob element >= r, z >= r, or a commitment that
 * does not decode or is not in G1 (infinity is valid); a failed call's outputs are zero.
 * blob_to_kzg_commitment — crypto/kzg.rs:60-69 */
B200_API int32_t b200_blob_to_kzg_commitment(const b200_kzg_settings* settings, const uint8_t* blob, uint8_t out_commitment[48]);
/* compute_kzg_proof — crypto/kzg.rs:71-86: the proof of p(z) and y = p(z) (z on the domain takes the spec's in-domain branch) */
B200_API int32_t b200_compute_kzg_proof(const b200_kzg_settings* settings, const uint8_t* blob, const uint8_t z[32],
                                        uint8_t out_proof[48], uint8_t out_y[32]);
/* compute_blob_kzg_proof — crypto/kzg.rs:88-99: the proof at z = compute_challenge(blob, commitment).  As in the spec, the
 * commitment is not checked against the blob. */
B200_API int32_t b200_compute_blob_kzg_proof(const b200_kzg_settings* settings, const uint8_t* blob, const uint8_t commitment[48],
                                             uint8_t out_proof[48]);
/* Throughput paths: n blobs in one call, one code per blob (what the single-blob call, which is this call with n = 1,
 * returns); a failed blob's 48 output bytes are zero.  n = 0 returns 0 and writes nothing; n > B200_KZG_MAX_BLOBS returns
 * B200_ERR_BAD_ARG.  Device scratch is bounded by the chunk of 1 024 blobs processed at a time (about 265 MiB). */
B200_API int32_t b200_blob_to_kzg_commitments(const b200_kzg_settings* settings, const uint8_t* blobs, size_t n,
                                              uint8_t* out_commitments, int32_t* out_codes);
B200_API int32_t b200_compute_blob_kzg_proofs(const b200_kzg_settings* settings, const uint8_t* blobs, const uint8_t* commitments,
                                              size_t n, uint8_t* out_proofs, int32_t* out_codes);

#ifdef __cplusplus
}
#endif
#endif /* B200_CONSENSUS_H */
