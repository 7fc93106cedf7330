// kernels.cuh -- host-side launchers shared between the .cu files and the C ABI (api.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

#include "../../include/dandd_b200.h"

namespace dd {

// Every kernel launch of the library is counted (dd_kernel_launches(): bench.py reports the number of
// launches inside its timed region as measured, not as a formula).
extern unsigned long long g_kernel_launches;
#define DD_COUNT_LAUNCH() ((void)__atomic_fetch_add(&dd::g_kernel_launches, 1ull, __ATOMIC_RELAXED))

// ---- K1 (pack.cu)
size_t pack_workspace_bytes(size_t chunk_bytes);
cudaError_t pack_reset(uint32_t *d_codes, size_t codes_bytes, uint32_t *d_invalid, size_t invalid_bytes,
                       dd_pack_state *d_state, cudaStream_t stream);
cudaError_t pack_fasta(const uint8_t *d_text, size_t n, uint32_t *d_codes, uint32_t *d_invalid, size_t cap_symbols,
                       dd_pack_state *d_state, void *d_ws, cudaStream_t stream);
cudaError_t pack_polyt_sentinel(const uint32_t *d_codes, uint32_t *d_invalid, const dd_pack_state *d_state,
                                uint64_t sym_begin, uint64_t sym_end, size_t max_symbols, cudaStream_t stream);
extern int g_polyt_sentinel;  // dd_set_option("polyt_sentinel"): the *_host entry points apply the pass

// ---- K2 (sketch.cu).  Workspace = [SketchWsHeader | scratch | u16 accumulators [nk][2^p] | rank-1 sink bitmaps
// [nk][2^p/32] u32 | mid-k presence bitmaps]; register = max(accumulator, sink bit)
extern int g_k_per_pass;
extern int g_midk;
extern int g_sink;
struct SketchWsHeader {
    uint8_t floor[32];  // floor[k-1] <= min(register of k): updates with rank <= floor are no-ops
    uint32_t use_floor;
    uint32_t pad[7];
};
size_t sketch_workspace_bytes(int nk, int p);
cudaError_t sketch_begin(void *d_ws, int nk, int p, cudaStream_t stream);
// Either d_state != nullptr (range read on the device: [prev_nsym, nsym), grid sized from
// max_new_symbols; a non-empty [sym_begin, sym_end) then selects a sub-range RELATIVE to prev_nsym)
// or an explicit host-known range.
cudaError_t sketch_update(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                          uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint32_t kmask, int p,
                          int canon, void *d_ws, cudaStream_t stream);
cudaError_t sketch_refresh_floor(void *d_ws, uint32_t kmask, int p, cudaStream_t stream);
// sketch_update cut at the floor schedule's boundaries, with the refreshes in between (sketch.cu).
// d_state != nullptr: [sym_begin, sym_end) is ignored, the range is the last pack call's.
cudaError_t sketch_update_sched(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                                uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint64_t seen_before,
                                uint32_t kmask, int p, int canon, void *d_ws, cudaStream_t stream);
cudaError_t sketch_end(void *d_ws, int nk, int p, uint8_t *d_regs, uint32_t *d_hist, double *d_cards,
                       cudaStream_t stream);

// ---- K3 / K4 / K6 (card.cu)
cudaError_t card_hist(const uint8_t *d_regs, int nsk, int p, uint32_t *d_hist, cudaStream_t stream);
cudaError_t mle_from_hist(const uint32_t *d_hist, int nsk, int p, double *d_cards, cudaStream_t stream);
cudaError_t union_max(const uint8_t *const *d_in, int n_in, size_t len, uint8_t *d_out, cudaStream_t stream);
cudaError_t prefix_union_hist(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                              int nk, int p, int final_only, uint32_t *d_hist, uint8_t *d_unions,
                              cudaStream_t stream);

// planes.cu: the same contract as prefix_union_hist (without materialised unions) on bit-sliced sketches
bool planes_supported(int p);
size_t planes_bytes(int64_t n_sketches, int p);
size_t prefix_union_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk, int p);
cudaError_t to_planes(const uint8_t *d_regs, int64_t n_sketches, int p, uint32_t *d_planes, cudaStream_t stream);
cudaError_t prefix_union_hist_from_planes(const uint32_t *d_planes, const int32_t *d_order, int n_ord, int n_steps,
                                          int n_genomes, int nk, int p, int final_only, uint32_t *d_hist, void *d_scratch,
                                          cudaStream_t stream);
cudaError_t prefix_union_hist_planes(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                                     int nk, int p, int final_only, uint32_t *d_hist, void *d_ws, cudaStream_t stream);
extern int g_prefix_planes;  // tuning knob: 1 = use the bit-plane kernel where it applies (default)
cudaError_t union_sets_hist(const uint8_t *const *d_members, int n_sets, int n_steps, int p, int final_only,
                            uint32_t *d_hist, uint8_t *d_unions, cudaStream_t stream);

// ---- K10 (leaveout.cu): union and leave-one-group-out histograms, regs [n][nk][2^p] -> hist [nk][1 + G][64] (added to).
// Workspace = [nk][64] u32 union part | [n] int2 members sorted by group.  h_group: host copy, ids in [0, G).
size_t leave_out_workspace_bytes(int n_genomes, int nk);
cudaError_t leave_out_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *h_group, int n_groups,
                           uint64_t reg_begin, uint64_t reg_end, uint32_t *d_hist, void *d_ws, cudaStream_t stream);

// ---- K11 (greedy.cu): hist(max(U, g)) for every listed candidate g, regs [n][nk][2^p], U [nk][2^p] ->
// hist [C][nk][64] and live [C][nk] (written).  Workspace = the candidate list.  h_cand / h_seg_off: host copies,
// checked by the caller.
size_t greedy_workspace_bytes(int n_cand);
cudaError_t greedy_dense_hist(const uint8_t *d_regs, int nk, int p, const uint8_t *d_union, const uint32_t *d_uhist,
                              const int32_t *h_cand, int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws,
                              cudaStream_t stream);
cudaError_t greedy_compact(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union,
                           const int32_t *h_cand, int n_cand, const int64_t *h_seg_off, int64_t *d_seg_off,
                           uint32_t *d_seg_len, uint32_t *d_entries, void *d_ws, cudaStream_t stream);
cudaError_t greedy_sparse_hist(uint32_t *d_entries, int64_t n_entries, const int64_t *d_seg_off, uint32_t *d_seg_len,
                               int nk, int p, const uint8_t *d_union, const uint32_t *d_uhist, const int32_t *h_cand,
                               int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws, cudaStream_t stream);

// ---- K5 (exact.cu).  Workspace = [ExactWsHeader | bitmap or key table]
struct ExactWsHeader {
    unsigned long long count;     // distinct keys inserted (hash-set mode; bitmap mode counts on demand)
    unsigned long long overflow;  // table full
    unsigned long long saw_ones;  // the all-ones key (== the empty marker) was inserted
    unsigned long long cur_stream;  // k > 64: index (in the stream table) of the stream being inserted
    unsigned long long n_streams;   // k > 64: streams registered so far
    unsigned long long n_nodes;     // K7: co-occurrence nodes pushed so far
    unsigned long long cover_cursor;  // K12 emit: (keys << 32) | nodes reserved so far
    unsigned long long cover_bad;     // K12 emit: a reservation did not fit the caller's buffers, or a genome >= n
};
size_t exact_workspace_bytes(int k, uint64_t capacity);
cudaError_t exact_begin(void *d_ws, int k, uint64_t capacity, cudaStream_t stream);
cudaError_t exact_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                         int k, int canon, void *d_ws, uint64_t capacity, uint32_t shard_rank, uint32_t shard_world,
                         cudaStream_t stream);
cudaError_t exact_count(void *d_ws, int k, uint64_t capacity, uint64_t *d_count, cudaStream_t stream);

// ---- K7 (exact.cu): pair intersections.  Sparse: [ExactWsHeader | key table | streams | (last, head) | nodes]
constexpr uint32_t kNil = 0xFFFFFFFFu;
struct PairNode {
    uint32_t genome, next;
};
size_t pairs_lh_offset(int k, uint64_t capacity, unsigned max_streams);     // the (last, head) u32 pairs, capacity + 1
size_t pairs_node_offset(int k, uint64_t capacity, unsigned max_streams);   // the PairNode array
size_t exact_pairs_workspace_bytes(int k, uint64_t capacity, uint64_t max_nodes, unsigned max_streams);
cudaError_t exact_pairs_begin(void *d_ws, int k, uint64_t capacity, unsigned max_streams, cudaStream_t stream);
cudaError_t exact_pairs_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                               int canon, uint32_t genome, void *d_ws, uint64_t capacity, uint64_t max_nodes,
                               unsigned max_streams, uint32_t shard_rank, uint32_t shard_world, cudaStream_t stream);
cudaError_t exact_pairs_accumulate(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                   uint64_t *d_inter, int sm_count, cudaStream_t stream);
// ---- K8 (exact.cu): first-rank histograms over the K7 lists, ranks [n_rows][n_genomes] u16 -> hist [n_rows][n_genomes]
cudaError_t exact_first_rank_hist(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                  const uint16_t *d_ranks, uint64_t n_rows, uint64_t *d_hist, int sm_count, cudaStream_t stream);
// ---- K9 (exact.cu): sharing spectrum over the K7 lists -> hist [n_genomes] (keys held by c = i + 1 genomes),
// priv [n_genomes] or null (keys held by genome g alone)
cudaError_t exact_occupancy_hist(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                 uint64_t *d_hist, uint64_t *d_priv, int sm_count, cudaStream_t stream);
// ---- K13 (exact.cu): genomes 0..R-1 references, R..R+Q-1 queries on the K7 lists -> inter [Q][R], shared [Q]
// (keys of q a reference holds), *d_union (keys some reference holds); added to
cudaError_t exact_query_counts(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint32_t n_refs,
                               uint32_t n_queries, uint64_t *d_inter, uint64_t *d_shared, uint64_t *d_union, int sm_count,
                               cudaStream_t stream);
// the node counter of a K7 sparse workspace (ExactWsHeader::n_nodes) -> *d_out, a copy on the stream
cudaError_t exact_pairs_node_count(const void *d_ws, uint64_t *d_out, cudaStream_t stream);
// Dense: K5 bitmap workspaces, ws_stride bytes apart, for genomes row0.. and col0..
cudaError_t exact_pair_popc(const void *d_rows, int64_t row0, int nr, const void *d_cols, int64_t col0, int nc,
                            size_t ws_stride, int k, int64_t n_genomes, uint64_t *d_inter, int sm_count, cudaStream_t stream);

// ---- K12 (cover.cu): the exact greedy cover index over the K7 lists.  count: d_counts[2] = (distinct keys, nodes),
// all-ones on a full table or node array.  emit: offsets [n_keys + 1] u32, holders [n_nodes] u16, key_of_node
// [n_nodes] u32; d_status[2] = (keys, nodes) written, or all-ones.  step: one launch over the parts (device
// descriptors in d_parts) adds, for every key of the picked genome's node range not covered yet, 1 to lost[h] of
// every holder h.
struct CoverPart {
    const uint32_t *offsets;
    const uint16_t *holders;
    const uint32_t *key_of_node;
    uint8_t *covered;
    unsigned long long *lost;   // [n_genomes], added to
    uint64_t node_begin, node_end;
    uint64_t pad;
};
cudaError_t exact_cover_count(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t *d_counts,
                              int sm_count, cudaStream_t stream);
cudaError_t exact_cover_emit(void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint32_t n_genomes, uint64_t n_keys,
                             uint64_t n_nodes, uint32_t *d_offsets, uint16_t *d_holders, uint32_t *d_key_of_node,
                             uint64_t *d_status, int sm_count, cudaStream_t stream);
cudaError_t exact_cover_step(const CoverPart *h_parts, int n_parts, uint32_t n_genomes, void *d_ws, int sm_count,
                             cudaStream_t stream);

}  // namespace dd
