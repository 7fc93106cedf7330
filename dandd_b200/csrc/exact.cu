// exact.cu -- K5: --exact mode, the number of distinct (canonical) k-mers, KMC semantics.
//
// Replaces `kmc -ci1 -cs2 -kK [-b] -fm` + `kmc_tools info` (reference lib/sketch_classes.py:389-399,
// 434-449) and `kmc_tools complex` unions (:451-465).  KMC builds an on-disk sorted database; all
// DandD ever reads back is its size, so the GPU keeps a *set* in HBM instead:
//   k <= 16 : a presence bitmap of 4^k bits (<= 512 MiB), filled with test-then-atomicOr, counted
//             with popc -- exact by construction;
//   k  > 16 : an open-addressing table of 64-bit keys (linear probing, atomicCAS); the key is the
//             k-mer value itself, so there are no false merges -- exact as long as the table is
//             not full, which is reported, never ignored;
//   k  > 32 : (to 64) the same with 128-bit keys and `atom.cas.b128`;
//   k  > 64 : (to 256, KMC's own limit) no atomic is wide enough for the key, so a 16-byte entry holds a
//             64-bit fingerprint of the canonical k-mer plus a REFERENCE to one occurrence (stream,
//             position); entries are still claimed with one `atom.cas.b128`, and a fingerprint match
//             is settled by comparing the k-mer at the referenced position word for word -- exact,
//             fingerprints only save comparisons.
// Inserting several genomes into one set gives the union count; reading the count after each
// insertion gives the progressive exact unions in one sweep (the reference re-merges databases
// n(n+1)/2 times).
#include <cuda_runtime.h>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr int kExactThreads = 256;
constexpr unsigned long long kEmptyKey = 0xFFFFFFFFFFFFFFFFull;

static size_t exact_table_bytes(int k, uint64_t capacity) {
    if (k <= DD_EXACT_BITMAP_MAXK) {
        const size_t bits = (size_t)1 << (2 * k);
        return bits < 128 ? 16 : bits / 8;
    }
    return (size_t)capacity * (k > 32 ? 2 : 1) * sizeof(unsigned long long);
}
constexpr unsigned kMaxStreams = 512;   // k > 64: streams whose k-mers one set may reference
static size_t exact_stream_table_bytes(int k) { return k > 64 ? kMaxStreams * sizeof(const uint32_t *) : 0; }
size_t exact_workspace_bytes(int k, uint64_t capacity) { return 256 + exact_table_bytes(k, capacity) + exact_stream_table_bytes(k); }
static ExactWsHeader *ex_hdr(void *ws) { return static_cast<ExactWsHeader *>(ws); }
static void *ex_tab(void *ws) { return static_cast<uint8_t *>(ws) + 256; }

// fmix64 (MurmurHash3 finaliser) -- only spreads keys over slots, never decides equality
__device__ __forceinline__ uint64_t slot_hash(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return x;
}

// Key-range sharding over ranks (SURVEY.md 8e): a k-mer belongs to rank (hash >> 40) % world -- the
// high hash bits, so the low bits that pick the slot stay uniform inside every shard.  Each rank
// scans everything but stores only its own keys; the per-rank distinct counts add up exactly.
__device__ __forceinline__ bool mine(uint64_t h, uint32_t shard_rank, uint32_t shard_world) {
    return shard_world <= 1u || (uint32_t)(h >> 40) % shard_world == shard_rank;
}

// What an insert kernel does once it has found or claimed the slot of a k-mer.  The probe loops are
// shared; K5 counts the keys it claimed, K7 (pair intersections) records which genome holds the key.
struct CountFresh {  // K5: distinct keys
    unsigned long long fresh = 0;
    __device__ __forceinline__ void key(uint64_t, bool claimed) { fresh += claimed; }
    __device__ __forceinline__ void ones(ExactWsHeader *hdr) { if (atomicExch(&hdr->saw_ones, 1ull) == 0ull) ++fresh; }
    __device__ __forceinline__ void finish(ExactWsHeader *hdr) {   // one global add per warp
        fresh = __reduce_add_sync(0xffffffffu, (unsigned)fresh);
        if ((threadIdx.x & 31) == 0 && fresh) atomicAdd(&hdr->count, fresh);
    }
};

// K7: slot s keeps (last genome pushed, head of its node list) in lh[s]; the all-ones key, which cannot
// live in the table, uses the extra slot lh[capacity].  Genomes are inserted one after another, so the
// first thread of genome g to reach a slot is the one whose exchange returns something other than g.
struct PushGenome {
    uint2 *lh;
    PairNode *nodes;
    uint64_t max_nodes, capacity;
    uint32_t genome;
    ExactWsHeader *hdr;
    __device__ __forceinline__ void push(uint64_t slot) {
        if (atomicExch(&lh[slot].x, genome) == genome) return;
        const unsigned long long n = atomicAdd(&hdr->n_nodes, 1ull);
        if (n >= max_nodes) { hdr->overflow = 1; return; }
        nodes[n].genome = genome;
        nodes[n].next = atomicExch(&lh[slot].y, (uint32_t)n);
    }
    __device__ __forceinline__ void key(uint64_t slot, bool) { push(slot); }
    __device__ __forceinline__ void ones(ExactWsHeader *) { push(capacity); }
    __device__ __forceinline__ void finish(ExactWsHeader *) {}
};

template <bool kBitmap, class Action>
__global__ void __launch_bounds__(kExactThreads)
exact_insert_kernel(const uint32_t *__restrict__ codes, const uint32_t *__restrict__ invalid, uint64_t sym_begin,
                    uint64_t sym_end, int k, int canon, ExactWsHeader *hdr, void *table, uint64_t capacity,
                    uint32_t shard_rank, uint32_t shard_world, Action act) {
    const uint64_t w = (sym_begin >> 4) + (uint64_t)blockIdx.x * kExactThreads + threadIdx.x;
    const uint64_t s0 = w << 4;
    if (s0 < sym_end) {
        const uint32_t w0 = __ldg(codes + w);
        const uint32_t w1 = w >= 1 ? __ldg(codes + w - 1) : 0u;
        const uint32_t w2 = w >= 2 ? __ldg(codes + w - 2) : 0u;
        const uint64_t iw = w >> 1;
        const uint32_t i0 = __ldg(invalid + iw);
        const uint32_t i1 = iw >= 1 ? __ldg(invalid + iw - 1) : 0xffffffffu;
        const uint32_t r0 = revcomp_word(w0), r1 = revcomp_word(w1), r2 = revcomp_word(w2);
        const int j_lo = sym_begin > s0 ? (int)(sym_begin - s0) : 0;
        const int j_hi = sym_end - s0 < 16 ? (int)(sym_end - s0) : 16;
        const uint32_t sm_base = (uint32_t)(s0 & 31);
        for (int j = j_lo; j < j_hi; ++j) {
            if (valid_run(invalid_window(i0, i1, sm_base + (uint32_t)j)) < k) continue;
            const Window win = window_at(w0, w1, w2, r0, r1, r2, j);
            const uint64_t v = kmer_value_rt(win, k, canon != 0);
            if (!mine(slot_hash(v), shard_rank, shard_world)) continue;  // another rank's key range
            if (kBitmap) {
                uint32_t *bm = static_cast<uint32_t *>(table);
                const uint32_t bit = 1u << (v & 31);
                uint32_t *word = bm + (v >> 5);
                if (!(__ldcg(word) & bit)) atomicOr(word, bit);
            } else {
                if (v == kEmptyKey) {  // cannot be stored: it is the empty marker
                    act.ones(hdr);
                    continue;
                }
                unsigned long long *tab = static_cast<unsigned long long *>(table);
                const uint64_t mask = capacity - 1;
                uint64_t slot = slot_hash(v) & mask;
                uint64_t probes = 0;
                for (;;) {
                    unsigned long long cur = __ldcg(tab + slot);
                    if (cur == kEmptyKey) cur = atomicCAS(tab + slot, kEmptyKey, (unsigned long long)v);
                    if (cur == kEmptyKey) { act.key(slot, true); break; }
                    if (cur == v) { act.key(slot, false); break; }
                    slot = (slot + 1) & mask;
                    if (++probes > mask) { hdr->overflow = 1; break; }
                }
            }
        }
    }
    if (!kBitmap) act.finish(hdr);
}

// ---- k = 33..64: 128-bit keys ---------------------------------------------------------------------
__device__ __forceinline__ ulonglong2 cas128(ulonglong2 *addr, ulonglong2 cmp, ulonglong2 val) {
    ulonglong2 old;
    asm volatile(
        "{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
        "atom.global.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
        : "=l"(old.x), "=l"(old.y)
        : "l"(cmp.x), "l"(cmp.y), "l"(val.x), "l"(val.y), "l"(addr)
        : "memory");
    return old;
}

template <class Action>
__global__ void __launch_bounds__(kExactThreads)
exact_insert_wide_kernel(const uint32_t *__restrict__ codes, const uint32_t *__restrict__ invalid, uint64_t sym_begin,
                         uint64_t sym_end, int k, int canon, ExactWsHeader *hdr, ulonglong2 *tab, uint64_t capacity,
                         uint32_t shard_rank, uint32_t shard_world, Action act) {
    const uint64_t w = (sym_begin >> 4) + (uint64_t)blockIdx.x * kExactThreads + threadIdx.x;
    const uint64_t s0 = w << 4;
    if (s0 < sym_end) {
        uint32_t c[5], I[5];
        const uint64_t iw = w >> 1;
#pragma unroll
        for (int t = 0; t < 5; ++t) {
            c[t] = w >= (uint64_t)t ? __ldg(codes + w - t) : 0u;
            I[t] = iw >= (uint64_t)t ? __ldg(invalid + iw - t) : 0xffffffffu;  // before the stream: breaks
        }
        const int j_lo = sym_begin > s0 ? (int)(sym_begin - s0) : 0;
        const int j_hi = sym_end - s0 < 16 ? (int)(sym_end - s0) : 16;
        const uint32_t sm_base = (uint32_t)(s0 & 31);
        const ulonglong2 empty = make_ulonglong2(kEmptyKey, kEmptyKey);
        const uint64_t mask = capacity - 1;
        for (int j = j_lo; j < j_hi; ++j) {
            if (valid_run_long(I, sm_base + (uint32_t)j) < k) continue;
            const U128 v = kmer128_at(c, j, k, canon != 0);
            if (v.lo == kEmptyKey && v.hi == kEmptyKey) {  // cannot be stored: it is the empty marker (rank 0's)
                if (shard_rank == 0u) act.ones(hdr);
                continue;
            }
            const uint64_t hv = slot_hash(v.lo ^ slot_hash(v.hi));
            if (!mine(hv, shard_rank, shard_world)) continue;
            const ulonglong2 key = make_ulonglong2(v.lo, v.hi);
            uint64_t slot = hv & mask;
            uint64_t probes = 0;
            for (;;) {
                // a matching read settles it; anything else is decided by the CAS result alone
                const ulonglong2 seen = __ldcg(tab + slot);
                if (seen.x == key.x && seen.y == key.y) { act.key(slot, false); break; }
                const ulonglong2 old = cas128(tab + slot, empty, key);
                if (old.x == kEmptyKey && old.y == kEmptyKey) { act.key(slot, true); break; }
                if (old.x == key.x && old.y == key.y) { act.key(slot, false); break; }
                slot = (slot + 1) & mask;
                if (++probes > mask) { hdr->overflow = 1; break; }
            }
        }
    }
    act.finish(hdr);
}

// ---- k = 65..256: (fingerprint, reference) entries ------------------------------------------------
constexpr int kRefPosBits = 48;

// one thread: find or append `codes` in the set's stream table; publish its index for the insert kernel
__global__ void exact_register_stream_kernel(ExactWsHeader *hdr, const uint32_t **streams, const uint32_t *codes,
                                             unsigned max_streams) {
    unsigned long long n = hdr->n_streams, i = 0;
    while (i < n && streams[i] != codes) ++i;
    if (i == n) {
        if (n >= max_streams) {
            hdr->overflow = 1;
            i = 0;
        } else {
            streams[n] = codes;
            hdr->n_streams = n + 1;
        }
    }
    hdr->cur_stream = i;
}

template <class Action>
__global__ void __launch_bounds__(kExactThreads)
exact_insert_long_kernel(const uint32_t *__restrict__ codes, const uint32_t *__restrict__ invalid, uint64_t sym_begin,
                         uint64_t sym_end, int k, int canon, ExactWsHeader *hdr, ulonglong2 *tab, uint64_t capacity,
                         const uint32_t *const *streams, uint32_t shard_rank, uint32_t shard_world, Action act) {
    const uint64_t w = (sym_begin >> 4) + (uint64_t)blockIdx.x * kExactThreads + threadIdx.x;
    const uint64_t s0 = w << 4;
    if (s0 < sym_end) {
        const int j_lo = sym_begin > s0 ? (int)(sym_begin - s0) : 0;
        const int j_hi = sym_end - s0 < 16 ? (int)(sym_end - s0) : 16;
        const ulonglong2 empty = make_ulonglong2(kEmptyKey, kEmptyKey);
        const uint64_t mask = capacity - 1;
        const unsigned long long me = hdr->cur_stream << kRefPosBits;
        int run = 0;
        for (int j = j_lo; j < j_hi; ++j) {
            const uint64_t s = s0 + j;
            // valid symbols ending at s (saturating at k): the first position of the word walks the break
            // bits backwards, the others extend its count
            if (j == j_lo) {
                run = valid_run_upto(invalid, s, k);
            } else {
                const bool bad = (invalid[s >> 5] >> (31u - (uint32_t)(s & 31))) & 1u;
                run = bad ? 0 : (run < k ? run + 1 : k);
            }
            if (run < k) continue;
            uint64_t key[kLongWords];
            const int W = kmer_long_at(codes, s, k, canon != 0, key);
            uint64_t h = 0;
            for (int t = 0; t < W; ++t) h = slot_hash(h ^ key[t]);
            if (!mine(h, shard_rank, shard_world)) continue;
            const ulonglong2 entry = make_ulonglong2(h, me | s);
            uint64_t slot = h & mask;
            uint64_t probes = 0;
            for (;;) {
                ulonglong2 seen = __ldcg(tab + slot);
                if (seen.x == kEmptyKey && seen.y == kEmptyKey) {
                    seen = cas128(tab + slot, empty, entry);
                    if (seen.x == kEmptyKey && seen.y == kEmptyKey) { act.key(slot, true); break; }
                }
                if (seen.x == h) {   // same fingerprint: the k-mer at the referenced occurrence decides
                    uint64_t other[kLongWords];
                    kmer_long_at(streams[seen.y >> kRefPosBits], seen.y & ((1ull << kRefPosBits) - 1ull), k, canon != 0, other);
                    bool same = true;
                    for (int t = 0; t < W; ++t) same = same && other[t] == key[t];
                    if (same) { act.key(slot, false); break; }
                }
                slot = (slot + 1) & mask;
                if (++probes > mask) { hdr->overflow = 1; break; }
            }
        }
    }
    act.finish(hdr);
}

__global__ void __launch_bounds__(256) bitmap_count_kernel(const uint32_t *__restrict__ bm, size_t nwords,
                                                           unsigned long long *out) {
    unsigned long long c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords; i += (size_t)gridDim.x * blockDim.x)
        c += __popc(__ldg(bm + i));
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}
// Hash-set mode: publish the running count; a full table can never yield a silent wrong answer --
// the count is replaced by the all-ones marker, which the host turns into DD_ERR_WORKSPACE.
__global__ void exact_publish_kernel(const ExactWsHeader *hdr, unsigned long long *out) {
    *out = hdr->overflow ? kEmptyKey : hdr->count;
}

cudaError_t exact_begin(void *d_ws, int k, uint64_t capacity, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(d_ws, 0, 256, stream);
    if (e != cudaSuccess) return e;
    const int fill = k <= DD_EXACT_BITMAP_MAXK ? 0x00 : 0xff;
    if ((e = cudaMemsetAsync(ex_tab(d_ws), fill, exact_table_bytes(k, capacity), stream)) != cudaSuccess) return e;
    if (k > 64)
        return cudaMemsetAsync(static_cast<uint8_t *>(ex_tab(d_ws)) + exact_table_bytes(k, capacity), 0, exact_stream_table_bytes(k), stream);
    return cudaSuccess;
}

// The probe loops of the three key layouts, for either action.  kBitmap: k <= DD_EXACT_BITMAP_MAXK sets of K5.
template <class Action>
static cudaError_t insert_with(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                               int k, int canon, ExactWsHeader *hdr, void *table, uint64_t capacity, const uint32_t **streams,
                               unsigned max_streams, bool bitmap, uint32_t shard_rank, uint32_t shard_world, Action act,
                               cudaStream_t stream) {
    if (sym_end <= sym_begin) return cudaSuccess;
    const size_t nwords = (size_t)((sym_end - sym_begin + 15) / 16 + 2);  // +2: the range need not start on a word boundary
    const unsigned grid = (unsigned)((nwords + kExactThreads - 1) / kExactThreads);
    if (k > 64) {
        if (sym_end >> kRefPosBits) return cudaErrorInvalidValue;
        DD_COUNT_LAUNCH(), exact_register_stream_kernel<<<1, 1, 0, stream>>>(hdr, streams, d_codes, max_streams);
        DD_COUNT_LAUNCH(), exact_insert_long_kernel<<<grid, kExactThreads, 0, stream>>>(d_codes, d_invalid, sym_begin, sym_end, k, canon,
                                                                    hdr, static_cast<ulonglong2 *>(table),
                                                                    capacity, streams, shard_rank, shard_world, act);
    } else if (k > 32)
        DD_COUNT_LAUNCH(), exact_insert_wide_kernel<<<grid, kExactThreads, 0, stream>>>(d_codes, d_invalid, sym_begin, sym_end, k, canon,
                                                                    hdr, static_cast<ulonglong2 *>(table),
                                                                    capacity, shard_rank, shard_world, act);
    else if (bitmap)
        DD_COUNT_LAUNCH(), exact_insert_kernel<true><<<grid, kExactThreads, 0, stream>>>(d_codes, d_invalid, sym_begin, sym_end, k, canon,
                                                                     hdr, table, capacity, shard_rank, shard_world, act);
    else
        DD_COUNT_LAUNCH(), exact_insert_kernel<false><<<grid, kExactThreads, 0, stream>>>(d_codes, d_invalid, sym_begin, sym_end, k,
                                                                      canon, hdr, table, capacity, shard_rank,
                                                                      shard_world, act);
    return cudaGetLastError();
}

cudaError_t exact_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                         int k, int canon, void *d_ws, uint64_t capacity, uint32_t shard_rank, uint32_t shard_world,
                         cudaStream_t stream) {
    const uint32_t **streams = reinterpret_cast<const uint32_t **>(static_cast<uint8_t *>(ex_tab(d_ws)) + exact_table_bytes(k, capacity));
    return insert_with(d_codes, d_invalid, sym_begin, sym_end, k, canon, ex_hdr(d_ws), ex_tab(d_ws), capacity, streams,
                       kMaxStreams, k <= DD_EXACT_BITMAP_MAXK, shard_rank, shard_world, CountFresh{}, stream);
}

cudaError_t exact_count(void *d_ws, int k, uint64_t capacity, uint64_t *d_count, cudaStream_t stream) {
    (void)capacity;
    if (k <= DD_EXACT_BITMAP_MAXK) {
        cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(uint64_t), stream);
        if (e != cudaSuccess) return e;
        const size_t nwords = exact_table_bytes(k, 0) / 4;
        size_t blocks = (nwords + 256 * 8 - 1) / (256 * 8);
        if (blocks < 1) blocks = 1;
        if (blocks > 148 * 8) blocks = 148 * 8;
        DD_COUNT_LAUNCH(), bitmap_count_kernel<<<(unsigned)blocks, 256, 0, stream>>>(static_cast<const uint32_t *>(ex_tab(d_ws)), nwords,
                                                                 reinterpret_cast<unsigned long long *>(d_count));
    } else {
        DD_COUNT_LAUNCH(), exact_publish_kernel<<<1, 1, 0, stream>>>(ex_hdr(d_ws), reinterpret_cast<unsigned long long *>(d_count));
    }
    return cudaGetLastError();
}

// ---- K7: |A n B| for every pair of genomes ------------------------------------------------------
// Sparse path.  Workspace = [header | K5 key table (hash layout at every k) | k > 64: stream table |
// (last, head) u32 pairs for capacity + 1 slots | node array].  Each genome's insert pushes one node
// {genome, next} per key it holds onto that key's list; the accumulate kernel then adds 1 to pair (a, b)
// for every two genomes on one list -- sum over keys of occ(occ-1)/2 increments.
static size_t pairs_key_bytes(int k, uint64_t capacity) { return (size_t)capacity * (k > 32 ? 2 : 1) * sizeof(unsigned long long); }
static size_t pairs_stream_bytes(int k, unsigned max_streams) { return k > 64 ? (size_t)max_streams * sizeof(const uint32_t *) : 0; }
size_t pairs_lh_offset(int k, uint64_t capacity, unsigned max_streams) {
    return 256 + pairs_key_bytes(k, capacity) + pairs_stream_bytes(k, max_streams);
}
size_t pairs_node_offset(int k, uint64_t capacity, unsigned max_streams) {
    return pairs_lh_offset(k, capacity, max_streams) + (size_t)(capacity + 1) * sizeof(uint2);
}
size_t exact_pairs_workspace_bytes(int k, uint64_t capacity, uint64_t max_nodes, unsigned max_streams) {
    return pairs_node_offset(k, capacity, max_streams) + (size_t)max_nodes * sizeof(PairNode);
}

cudaError_t exact_pairs_begin(void *d_ws, int k, uint64_t capacity, unsigned max_streams, cudaStream_t stream) {
    uint8_t *ws = static_cast<uint8_t *>(d_ws);
    cudaError_t e = cudaMemsetAsync(ws, 0, 256, stream);
    if (e != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(ws + 256, 0xff, pairs_key_bytes(k, capacity), stream)) != cudaSuccess) return e;
    if (k > 64 && (e = cudaMemsetAsync(ws + 256 + pairs_key_bytes(k, capacity), 0, pairs_stream_bytes(k, max_streams), stream)) != cudaSuccess)
        return e;
    return cudaMemsetAsync(ws + pairs_lh_offset(k, capacity, max_streams), 0xff, (size_t)(capacity + 1) * sizeof(uint2), stream);
}

cudaError_t exact_pairs_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                               int canon, uint32_t genome, void *d_ws, uint64_t capacity, uint64_t max_nodes,
                               unsigned max_streams, uint32_t shard_rank, uint32_t shard_world, cudaStream_t stream) {
    uint8_t *ws = static_cast<uint8_t *>(d_ws);
    PushGenome act;
    act.lh = reinterpret_cast<uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams));
    act.nodes = reinterpret_cast<PairNode *>(ws + pairs_node_offset(k, capacity, max_streams));
    act.max_nodes = max_nodes;
    act.capacity = capacity;
    act.genome = genome;
    act.hdr = ex_hdr(d_ws);
    const uint32_t **streams = reinterpret_cast<const uint32_t **>(ws + 256 + pairs_key_bytes(k, capacity));
    return insert_with(d_codes, d_invalid, sym_begin, sym_end, k, canon, ex_hdr(d_ws), ws + 256, capacity, streams,
                       max_streams, /*bitmap=*/false, shard_rank, shard_world, act, stream);
}

// PushGenome pushes one node per (genome, slot) and a key owns exactly one slot in all three layouts, so the
// counter's growth over one genome's insert is that genome's distinct keys in the pass (the family job's singles).
cudaError_t exact_pairs_node_count(const void *d_ws, uint64_t *d_out, cudaStream_t stream) {
    const ExactWsHeader *hdr = static_cast<const ExactWsHeader *>(d_ws);
    return cudaMemcpyAsync(d_out, &hdr->n_nodes, sizeof(uint64_t), cudaMemcpyDeviceToDevice, stream);
}

__device__ __forceinline__ uint64_t pair_row(uint64_t a, uint64_t b, uint64_t n) {  // a < b
    return a * (2 * n - a - 1) / 2 + (b - a - 1);
}

// Each warp takes 32 slots at a time (grid-stride) and walks the list of every occupied one in turn.  A
// list is read 32 nodes at a time, every lane loading the
// same node (one broadcast transaction); lane j keeps the j-th genome of the chunk.  Pairs inside a
// chunk come from shuffles; a chunk is then paired with every later chunk of the list.  kSmem: the
// pair counters of the whole job fit in shared memory, and each CTA adds its counters to the output
// once at the end.
template <bool kSmem>
__global__ void __launch_bounds__(256)
exact_pairs_accumulate_kernel(const ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh,
                              const PairNode *__restrict__ nodes, uint64_t n_slots, uint64_t n_genomes,
                              unsigned long long *out, uint64_t n_pairs) {
    extern __shared__ uint32_t sm_count[];
    if (hdr->overflow) {   // a full table or node array: the marker, never a count
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += (uint64_t)gridDim.x * blockDim.x)
            out[i] = kEmptyKey;
        return;
    }
    if (kSmem) {
        for (uint64_t i = threadIdx.x; i < n_pairs; i += blockDim.x) sm_count[i] = 0;
        __syncthreads();
    }
    const unsigned lane = threadIdx.x & 31;
    auto add = [&](uint32_t a, uint32_t b) {
        if (a >= n_genomes || b >= n_genomes) return;   // outside the caller's genome range: never written out of bounds
        const uint64_t r = a < b ? pair_row(a, b, n_genomes) : pair_row(b, a, n_genomes);
        if (kSmem) atomicAdd(&sm_count[r], 1u);
        else atomicAdd(&out[r], 1ull);
    };
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t base = ((uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < n_slots; base += warps * 32) {
        // 32 slots per coalesced load; the warp then walks the lists of the occupied ones one by one
        const uint32_t head = base + lane < n_slots ? __ldg(&lh[base + lane].y) : kNil;
        for (unsigned occ = __ballot_sync(0xffffffffu, head != kNil); occ; occ &= occ - 1) {
            uint32_t a_at = __shfl_sync(0xffffffffu, head, __ffs(occ) - 1);
            while (a_at != kNil) {
                uint32_t ga = 0, cur = a_at;
                int na = 0;
                for (; na < 32 && cur != kNil; ++na) {
                    const PairNode nd = nodes[cur];
                    if (lane == (unsigned)na) ga = nd.genome;
                    cur = nd.next;
                }
                a_at = cur;
                for (int d = 1; d < na; ++d) {
                    const uint32_t gb = __shfl_down_sync(0xffffffffu, ga, d);
                    if ((int)lane + d < na) add(ga, gb);
                }
                for (uint32_t b_at = a_at; b_at != kNil;) {
                    uint32_t gb = 0;
                    int nb = 0;
                    for (; nb < 32 && b_at != kNil; ++nb) {
                        const PairNode nd = nodes[b_at];
                        if (lane == (unsigned)nb) gb = nd.genome;
                        b_at = nd.next;
                    }
                    for (int i = 0; i < na; ++i) {
                        const uint32_t g = __shfl_sync(0xffffffffu, ga, i);
                        if ((int)lane < nb) add(g, gb);
                    }
                }
            }
        }
    }
    if (kSmem) {
        __syncthreads();
        for (uint64_t i = threadIdx.x; i < n_pairs; i += blockDim.x)
            if (sm_count[i]) atomicAdd(&out[i], (unsigned long long)sm_count[i]);
    }
}

constexpr size_t kPairSmemBytes = 96 * 1024;

cudaError_t exact_pairs_accumulate(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                   uint64_t *d_inter, int sm_count, cudaStream_t stream) {
    const uint8_t *ws = static_cast<const uint8_t *>(d_ws);
    const uint64_t n_pairs = n_genomes * (n_genomes - 1) / 2;
    if (n_pairs == 0) return cudaSuccess;
    const ExactWsHeader *hdr = static_cast<const ExactWsHeader *>(d_ws);
    const uint2 *lh = reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams));
    const PairNode *nodes = reinterpret_cast<const PairNode *>(ws + pairs_node_offset(k, capacity, max_streams));
    unsigned long long *out = reinterpret_cast<unsigned long long *>(d_inter);
    const uint64_t n_slots = capacity + 1;
    const size_t smem = (size_t)n_pairs * sizeof(uint32_t);
    if (smem <= kPairSmemBytes) {
        cudaError_t e = cudaFuncSetAttribute(exact_pairs_accumulate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)kPairSmemBytes);
        if (e != cudaSuccess) return e;
        // few CTAs: every CTA pays one pass over the counters at the start and one at the end
        const unsigned grid = (unsigned)(sm_count * 2);
        DD_COUNT_LAUNCH(), exact_pairs_accumulate_kernel<true><<<grid, 256, smem, stream>>>(hdr, lh, nodes, n_slots, n_genomes, out, n_pairs);
    } else {
        const uint64_t want = (n_slots + 255) / 256;   // one 32-slot group per warp
        const unsigned grid = (unsigned)(want < (uint64_t)sm_count * 16 ? (want ? want : 1) : (uint64_t)sm_count * 16);
        DD_COUNT_LAUNCH(), exact_pairs_accumulate_kernel<false><<<grid, 256, 0, stream>>>(hdr, lh, nodes, n_slots, n_genomes, out, n_pairs);
    }
    return cudaGetLastError();
}

// ---- K8: first-rank histograms over the K7 lists ---------------------------------------------------
// Row r of the rank table gives every genome a rank (ties allowed, 0xFFFF = not in the row's family);
// hist[r][m] counts the keys whose minimum rank over the genomes on their list is m.  A progressive
// ordering is a row of positions (prefix i holds the keys of bins < i), a set a row of zeros (its union
// is bin 0).  The work per slot is occ x ceil(R / 32): linear in the list, so no bitmap path is needed.
//
// Row blocks are the outer loop: lane j owns row rb*32 + j for a whole pass over the slots, so bin 0 --
// where almost every key of a progressive row or a set lands -- is a register counter, flushed once per
// lane and row block.  kSmemHist: the other bins count in shared memory (u32, row stride odd so that 32
// rows hitting one bin hit 32 banks); kSmemRanks: the table sits transposed in shared memory, [genome][row],
// so the 32 lanes of a row block read 32 adjacent entries.
constexpr uint16_t kNoRank = 0xFFFF;

template <bool kSmemHist, bool kSmemRanks>
__global__ void __launch_bounds__(256)
exact_first_rank_kernel(const ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh, const PairNode *__restrict__ nodes,
                        uint64_t n_slots, uint32_t n_genomes, const uint16_t *__restrict__ ranks, uint32_t n_rows,
                        uint32_t hist_stride, uint32_t rank_stride, unsigned long long *out) {
    extern __shared__ uint32_t smem[];
    const uint64_t n_cells = (uint64_t)n_rows * n_genomes;
    if (hdr->overflow) {   // a full table or node array: the marker, never a count
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cells; i += (uint64_t)gridDim.x * blockDim.x)
            out[i] = kEmptyKey;
        return;
    }
    uint32_t *sm_hist = smem;
    uint16_t *sm_rank = reinterpret_cast<uint16_t *>(smem + (kSmemHist ? (size_t)n_rows * hist_stride : 0));
    if (kSmemHist)
        for (uint64_t i = threadIdx.x; i < (uint64_t)n_rows * hist_stride; i += blockDim.x) sm_hist[i] = 0;
    if (kSmemRanks)
        for (uint64_t i = threadIdx.x; i < (uint64_t)n_genomes * rank_stride; i += blockDim.x) {
            const uint32_t g = (uint32_t)(i / rank_stride), r = (uint32_t)(i % rank_stride);
            sm_rank[i] = r < n_rows ? __ldg(ranks + (size_t)r * n_genomes + g) : kNoRank;
        }
    if (kSmemHist || kSmemRanks) __syncthreads();

    const unsigned lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    const uint64_t warp0 = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (uint32_t rb = 0; rb * 32 < n_rows; ++rb) {
        const uint32_t row = rb * 32 + lane;
        unsigned long long zero = 0;   // this lane's bin-0 count
        for (uint64_t base = warp0 * 32; base < n_slots; base += warps * 32) {
            const uint32_t head = base + lane < n_slots ? __ldg(&lh[base + lane].y) : kNil;
            for (unsigned occ = __ballot_sync(0xffffffffu, head != kNil); occ; occ &= occ - 1) {
                uint32_t at = __shfl_sync(0xffffffffu, head, __ffs(occ) - 1);
                uint32_t best = kNoRank;
                while (at != kNil) {   // the list, 32 nodes at a time: lane i keeps the i-th genome of the chunk
                    uint32_t gl = 0;
                    int na = 0;
                    for (; na < 32 && at != kNil; ++na) {
                        const PairNode nd = nodes[at];
                        if (lane == (unsigned)na) gl = nd.genome;
                        at = nd.next;
                    }
                    for (int i = 0; i < na; ++i) {
                        const uint32_t g = __shfl_sync(0xffffffffu, gl, i);
                        if (g >= n_genomes) continue;   // outside the caller's genome range: never read out of bounds
                        uint32_t rk;
                        if (kSmemRanks) rk = sm_rank[(size_t)g * rank_stride + row];
                        else rk = row < n_rows ? __ldg(ranks + (size_t)row * n_genomes + g) : kNoRank;
                        best = rk < best ? rk : best;
                    }
                }
                if (best == 0) ++zero;
                else if (best < n_genomes) {   // (kNoRank: no genome of the row holds the key; a rank >= n is not counted)
                    if (kSmemHist) atomicAdd(&sm_hist[(size_t)row * hist_stride + best], 1u);
                    else atomicAdd(&out[(size_t)row * n_genomes + best], 1ull);
                }
            }
        }
        if (row < n_rows && zero) atomicAdd(&out[(size_t)row * n_genomes], zero);
    }
    if (kSmemHist) {
        __syncthreads();
        for (uint64_t i = threadIdx.x; i < n_cells; i += blockDim.x) {
            const uint64_t r = i / n_genomes, m = i % n_genomes;
            const uint32_t v = sm_hist[r * hist_stride + m];
            if (v) atomicAdd(&out[i], (unsigned long long)v);
        }
    }
}

constexpr size_t kRankSmemBytes = 128 * 1024;   // counters + transposed rank table, per CTA

cudaError_t exact_first_rank_hist(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                  const uint16_t *d_ranks, uint64_t n_rows, uint64_t *d_hist, int sm_count, cudaStream_t stream) {
    if (n_genomes == 0 || n_rows == 0) return cudaSuccess;
    const uint8_t *ws = static_cast<const uint8_t *>(d_ws);
    const ExactWsHeader *hdr = static_cast<const ExactWsHeader *>(d_ws);
    const uint2 *lh = reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams));
    const PairNode *nodes = reinterpret_cast<const PairNode *>(ws + pairs_node_offset(k, capacity, max_streams));
    unsigned long long *out = reinterpret_cast<unsigned long long *>(d_hist);
    const uint64_t n_slots = capacity + 1;
    const uint32_t hist_stride = (uint32_t)(n_genomes | 1);                  // odd: one bank per row
    const uint32_t rank_stride = (uint32_t)((n_rows + 31) / 32 * 32);        // whole row blocks, padded with kNoRank
    const size_t hist_bytes = (size_t)n_rows * hist_stride * sizeof(uint32_t);
    const size_t rank_bytes = (size_t)n_genomes * rank_stride * sizeof(uint16_t);
    const bool smem_hist = hist_bytes <= kPairSmemBytes;
    const bool smem_rank = (smem_hist ? hist_bytes : 0) + rank_bytes <= kRankSmemBytes;
    const size_t smem = (smem_hist ? hist_bytes : 0) + (smem_rank ? rank_bytes : 0);
    unsigned grid;
    if (smem_hist) {
        grid = (unsigned)(sm_count * 2);   // every CTA pays one pass over its counters at the start and one at the end
    } else {
        const uint64_t want = (n_slots + 255) / 256;   // one 32-slot group per warp
        grid = (unsigned)(want < (uint64_t)sm_count * 16 ? (want ? want : 1) : (uint64_t)sm_count * 16);
    }
    auto launch = [&](auto kernel) -> cudaError_t {
        if (smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        DD_COUNT_LAUNCH(), kernel<<<grid, 256, smem, stream>>>(hdr, lh, nodes, n_slots, (uint32_t)n_genomes, d_ranks,
                                                              (uint32_t)n_rows, hist_stride, rank_stride, out);
        return cudaGetLastError();
    };
    if (smem_hist && smem_rank) return launch(exact_first_rank_kernel<true, true>);
    if (smem_hist) return launch(exact_first_rank_kernel<true, false>);
    if (smem_rank) return launch(exact_first_rank_kernel<false, true>);
    return launch(exact_first_rank_kernel<false, false>);
}

// ---- K9: the sharing spectrum over the K7 lists ------------------------------------------------------
// A key's list holds one node per genome that holds it, so its length is the key's sharing count c:
// hist[c - 1] counts the keys held by exactly c genomes, priv[g] (optional) the keys held by genome g alone.
// Only the length and, for a list of one, its genome are needed -- so unlike K7 and K8, where a warp walks
// one list at a time with broadcast loads, every lane walks the list of its own slot: 32 independent pointer
// chases per warp.  kSmem: both counter arrays fit in shared memory (u32), flushed once per CTA.
template <bool kSmem>
__global__ void __launch_bounds__(256)
exact_occupancy_kernel(const ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh, const PairNode *__restrict__ nodes,
                       uint64_t n_slots, uint64_t n_genomes, unsigned long long *hist, unsigned long long *priv) {
    extern __shared__ uint32_t sm_occ[];
    if (hdr->overflow) {   // a full table or node array: the marker, never a count
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_genomes; i += (uint64_t)gridDim.x * blockDim.x) {
            hist[i] = kEmptyKey;
            if (priv) priv[i] = kEmptyKey;
        }
        return;
    }
    uint32_t *sm_hist = sm_occ, *sm_priv = sm_occ + n_genomes;
    if (kSmem) {
        for (uint64_t i = threadIdx.x; i < (priv ? 2 : 1) * n_genomes; i += blockDim.x) sm_occ[i] = 0;
        __syncthreads();
    }
    const uint64_t threads = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n_slots; s += threads) {   // 32 slots per warp load
        uint32_t at = __ldg(&lh[s].y);
        uint64_t c = 0;
        uint32_t only = 0;
        while (at != kNil) {
            const PairNode nd = nodes[at];
            if (nd.genome < n_genomes) {   // outside the caller's genome range: never counted, never an address
                only = nd.genome;
                ++c;
            }
            at = nd.next;
        }
        if (c == 0 || c > n_genomes) continue;   // (c > n: a genome pushed twice, against the insert contract)
        if (kSmem) {
            atomicAdd(&sm_hist[c - 1], 1u);
            if (priv && c == 1) atomicAdd(&sm_priv[only], 1u);
        } else {
            atomicAdd(&hist[c - 1], 1ull);
            if (priv && c == 1) atomicAdd(&priv[only], 1ull);
        }
    }
    if (kSmem) {
        __syncthreads();
        for (uint64_t i = threadIdx.x; i < n_genomes; i += blockDim.x) {
            if (sm_hist[i]) atomicAdd(&hist[i], (unsigned long long)sm_hist[i]);
            if (priv && sm_priv[i]) atomicAdd(&priv[i], (unsigned long long)sm_priv[i]);
        }
    }
}

cudaError_t exact_occupancy_hist(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t n_genomes,
                                 uint64_t *d_hist, uint64_t *d_priv, int sm_count, cudaStream_t stream) {
    if (n_genomes == 0) return cudaSuccess;
    const uint8_t *ws = static_cast<const uint8_t *>(d_ws);
    const ExactWsHeader *hdr = static_cast<const ExactWsHeader *>(d_ws);
    const uint2 *lh = reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams));
    const PairNode *nodes = reinterpret_cast<const PairNode *>(ws + pairs_node_offset(k, capacity, max_streams));
    unsigned long long *hist = reinterpret_cast<unsigned long long *>(d_hist);
    unsigned long long *priv = reinterpret_cast<unsigned long long *>(d_priv);
    const uint64_t n_slots = capacity + 1;
    const size_t smem = (size_t)(d_priv ? 2 : 1) * n_genomes * sizeof(uint32_t);
    const uint64_t want = (n_slots + 255) / 256;   // one slot per thread
    if (smem <= kPairSmemBytes) {
        // a latency-bound walk wants full occupancy; every CTA pays one pass over its counters at each end
        const uint64_t per_sm = smem <= 8 * 1024 ? 8 : 2;
        const unsigned grid = (unsigned)(want < (uint64_t)sm_count * per_sm ? want : (uint64_t)sm_count * per_sm);
        if (smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(exact_occupancy_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                       (int)kPairSmemBytes);
            if (e != cudaSuccess) return e;
        }
        DD_COUNT_LAUNCH(), exact_occupancy_kernel<true><<<grid, 256, smem, stream>>>(hdr, lh, nodes, n_slots, n_genomes, hist, priv);
    } else {
        const unsigned grid = (unsigned)(want < (uint64_t)sm_count * 16 ? want : (uint64_t)sm_count * 16);
        DD_COUNT_LAUNCH(), exact_occupancy_kernel<false><<<grid, 256, 0, stream>>>(hdr, lh, nodes, n_slots, n_genomes, hist, priv);
    }
    return cudaGetLastError();
}

// ---- K13: query genomes against a reference collection over the K7 lists -------------------------------
// Genomes 0 .. R-1 are the references, R .. R+Q-1 the queries.  Per key: union_R += 1 if a reference holds it,
// shared[q] += 1 for every query on such a list, inter[q][r] += 1 for every (query, reference) pair on it --
// occ + q_on * r_on work per key where K7 pays occ(occ-1)/2.
// The walk depends on the list order: PushGenome links every node at the list head, and genomes are inserted
// one after another in id order, so every list is in DECREASING genome order -- its query nodes come before its
// reference nodes.  A list whose head is a reference holds no query (one node load), and the references that
// pair with a chunk of queries are those after the chunk's queries: one walk of the rest of the list per chunk.
// Queries go in chunks of <= 32, one per lane, broadcast by shuffle while every lane owns one reference node,
// so the lanes of a warp hit one counter row at distinct columns.  kSmem: the Q*R + Q counters fit in shared
// memory (u32) and each CTA flushes them once; union_R is a per-lane register count, flushed once.
template <bool kSmem>
__global__ void __launch_bounds__(256)
exact_query_kernel(const ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh, const PairNode *__restrict__ nodes,
                   uint64_t n_slots, uint32_t n_refs, uint32_t n_queries, unsigned long long *inter,
                   unsigned long long *shared, unsigned long long *union_r) {
    extern __shared__ uint32_t sm_q[];
    const uint64_t n_inter = (uint64_t)n_queries * n_refs;
    if (hdr->overflow) {   // a full table or node array: the marker, never a count
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_inter + n_queries + 1;
             i += (uint64_t)gridDim.x * blockDim.x) {
            if (i < n_inter) inter[i] = kEmptyKey;
            else if (i < n_inter + n_queries) shared[i - n_inter] = kEmptyKey;
            else *union_r = kEmptyKey;
        }
        return;
    }
    if (kSmem) {
        for (uint64_t i = threadIdx.x; i < n_inter + n_queries; i += blockDim.x) sm_q[i] = 0;
        __syncthreads();
    }
    const uint32_t n_all = n_refs + n_queries;
    const unsigned lane = threadIdx.x & 31;
    unsigned long long keys_r = 0;   // lane 0's union_R count
    auto add_pair = [&](uint32_t q, uint32_t r) {   // q: a query index, r: a reference genome
        const uint64_t c = (uint64_t)q * n_refs + r;
        if (kSmem) atomicAdd(&sm_q[c], 1u);
        else atomicAdd(&inter[c], 1ull);
    };
    // up to 32 nodes from `at`, lane j keeps the j-th genome (kNil past the chunk); returns the node after it
    auto load = [&](uint32_t at, uint32_t &g) {
        g = kNil;
        for (unsigned i = 0; i < 32 && at != kNil; ++i) {
            const PairNode nd = nodes[at];
            if (lane == i) g = nd.genome;
            at = nd.next;
        }
        return at;
    };
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t base = ((uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < n_slots; base += warps * 32) {
        // 32 slots per coalesced load; the warp then walks the lists of the occupied ones one by one
        const uint32_t head = base + lane < n_slots ? __ldg(&lh[base + lane].y) : kNil;
        for (unsigned occ = __ballot_sync(0xffffffffu, head != kNil); occ; occ &= occ - 1) {
            uint32_t at = __shfl_sync(0xffffffffu, head, __ffs(occ) - 1);
            if (nodes[at].genome < n_refs) {   // a reference at the head: no query on this list
                keys_r += lane == 0;
                continue;
            }
            bool has_ref = false;
            while (at != kNil) {
                uint32_t gq;
                const uint32_t after = load(at, gq);
                const bool is_q = gq >= n_refs && gq < n_all, is_r = gq < n_refs;
                const unsigned qm = __ballot_sync(0xffffffffu, is_q), rm = __ballot_sync(0xffffffffu, is_r);
                if (qm) {
                    // the references of this chunk (after its queries), then every later chunk
                    bool own_r = is_r;
                    uint32_t gr = gq, b_at = after;
                    for (;;) {
                        has_ref |= __any_sync(0xffffffffu, own_r);
                        for (unsigned m = qm; m; m &= m - 1) {
                            const uint32_t q = __shfl_sync(0xffffffffu, gq, __ffs(m) - 1) - n_refs;
                            if (own_r) add_pair(q, gr);
                        }
                        if (b_at == kNil) break;
                        b_at = load(b_at, gr);
                        own_r = gr < n_refs;
                    }
                    if (has_ref && is_q) {
                        if (kSmem) atomicAdd(&sm_q[n_inter + (gq - n_refs)], 1u);
                        else atomicAdd(&shared[gq - n_refs], 1ull);
                    }
                }
                if (rm) {   // references began in this chunk: no query follows (decreasing order)
                    has_ref = true;
                    break;
                }
                at = after;
            }
            keys_r += lane == 0 && has_ref;
        }
    }
    if (keys_r) atomicAdd(union_r, keys_r);
    if (kSmem) {
        __syncthreads();
        for (uint64_t i = threadIdx.x; i < n_inter + n_queries; i += blockDim.x) {
            const uint32_t v = sm_q[i];
            if (!v) continue;
            if (i < n_inter) atomicAdd(&inter[i], (unsigned long long)v);
            else atomicAdd(&shared[i - n_inter], (unsigned long long)v);
        }
    }
}

cudaError_t exact_query_counts(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint32_t n_refs,
                               uint32_t n_queries, uint64_t *d_inter, uint64_t *d_shared, uint64_t *d_union, int sm_count,
                               cudaStream_t stream) {
    const uint8_t *ws = static_cast<const uint8_t *>(d_ws);
    const ExactWsHeader *hdr = static_cast<const ExactWsHeader *>(d_ws);
    const uint2 *lh = reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams));
    const PairNode *nodes = reinterpret_cast<const PairNode *>(ws + pairs_node_offset(k, capacity, max_streams));
    auto *inter = reinterpret_cast<unsigned long long *>(d_inter);
    auto *shared = reinterpret_cast<unsigned long long *>(d_shared);
    auto *union_r = reinterpret_cast<unsigned long long *>(d_union);
    const uint64_t n_slots = capacity + 1;
    const size_t smem = ((size_t)n_queries * n_refs + n_queries) * sizeof(uint32_t);
    if (smem <= kPairSmemBytes) {
        if (smem > 48 * 1024) {
            const cudaError_t e = cudaFuncSetAttribute(exact_query_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                       (int)kPairSmemBytes);
            if (e != cudaSuccess) return e;
        }
        // few CTAs: every CTA pays one pass over the counters at the start and one at the end
        const unsigned grid = (unsigned)(sm_count * 2);
        DD_COUNT_LAUNCH(), exact_query_kernel<true><<<grid, 256, smem, stream>>>(hdr, lh, nodes, n_slots, n_refs, n_queries,
                                                                                 inter, shared, union_r);
    } else {
        const uint64_t want = (n_slots + 255) / 256;   // one 32-slot group per warp
        const unsigned grid = (unsigned)(want < (uint64_t)sm_count * 16 ? (want ? want : 1) : (uint64_t)sm_count * 16);
        DD_COUNT_LAUNCH(), exact_query_kernel<false><<<grid, 256, 0, stream>>>(hdr, lh, nodes, n_slots, n_refs, n_queries,
                                                                               inter, shared, union_r);
    }
    return cudaGetLastError();
}

// Dense path: popc(A & B) over K5 presence bitmaps.  A CTA owns a tile of 8 row genomes x 8 column
// genomes and a slice of the bitmap words: each word range of the 16 bitmaps is read once per tile
// (from L2 when other tiles have just read it) and feeds 64 pair counters.
constexpr int kPopcTile = 8;
__global__ void __launch_bounds__(256)
exact_pair_popc_kernel(const uint8_t *__restrict__ rows, int64_t row0, int nr, const uint8_t *__restrict__ cols, int64_t col0,
                       int nc, size_t ws_stride, size_t nwords, int64_t n_genomes, int col_tiles, int64_t tile0,
                       unsigned long long *out) {
    const int64_t t = tile0 + blockIdx.y;
    const int tr = (int)(t / col_tiles), tc = (int)(t % col_tiles);
    const int r_lo = tr * kPopcTile, c_lo = tc * kPopcTile;
    const int c_hi = min(nc, c_lo + kPopcTile);
    if (row0 + r_lo >= col0 + c_hi - 1) return;   // no pair a < b in this tile
    const uint32_t *ra[kPopcTile], *cb[kPopcTile];
#pragma unroll
    for (int i = 0; i < kPopcTile; ++i) {
        const int r = min(r_lo + i, nr - 1), c = min(c_lo + i, nc - 1);   // clamped rows/columns are never counted
        ra[i] = reinterpret_cast<const uint32_t *>(rows + (size_t)r * ws_stride + 256);
        cb[i] = reinterpret_cast<const uint32_t *>(cols + (size_t)c * ws_stride + 256);
    }
    uint32_t acc[kPopcTile][kPopcTile];
#pragma unroll
    for (int i = 0; i < kPopcTile; ++i)
#pragma unroll
        for (int j = 0; j < kPopcTile; ++j) acc[i][j] = 0;
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += (size_t)gridDim.x * blockDim.x) {
        uint32_t a[kPopcTile], b[kPopcTile];
#pragma unroll
        for (int i = 0; i < kPopcTile; ++i) {
            a[i] = __ldg(ra[i] + w);
            b[i] = __ldg(cb[i] + w);
        }
#pragma unroll
        for (int i = 0; i < kPopcTile; ++i)
#pragma unroll
            for (int j = 0; j < kPopcTile; ++j) acc[i][j] += __popc(a[i] & b[j]);
    }
    __shared__ unsigned long long tile[kPopcTile * kPopcTile];
    if (threadIdx.x < kPopcTile * kPopcTile) tile[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kPopcTile; ++i)
#pragma unroll
        for (int j = 0; j < kPopcTile; ++j) {
            const uint32_t v = __reduce_add_sync(0xffffffffu, acc[i][j]);
            if ((threadIdx.x & 31) == 0 && v) atomicAdd(&tile[i * kPopcTile + j], (unsigned long long)v);
        }
    __syncthreads();
    if (threadIdx.x < kPopcTile * kPopcTile) {
        const int i = threadIdx.x / kPopcTile, j = threadIdx.x % kPopcTile;
        const int64_t a = row0 + r_lo + i, b = col0 + c_lo + j;
        if (r_lo + i < nr && c_lo + j < nc && a < b && tile[threadIdx.x])
            atomicAdd(&out[pair_row((uint64_t)a, (uint64_t)b, (uint64_t)n_genomes)], tile[threadIdx.x]);
    }
}

cudaError_t exact_pair_popc(const void *d_rows, int64_t row0, int nr, const void *d_cols, int64_t col0, int nc,
                            size_t ws_stride, int k, int64_t n_genomes, uint64_t *d_inter, int sm_count, cudaStream_t stream) {
    if (nr <= 0 || nc <= 0) return cudaSuccess;
    const size_t nwords = exact_table_bytes(k, 0) / 4;
    const int row_tiles = (nr + kPopcTile - 1) / kPopcTile, col_tiles = (nc + kPopcTile - 1) / kPopcTile;
    const uint64_t tiles = (uint64_t)row_tiles * col_tiles;
    // enough word slices to give every SM a few CTAs, none shorter than 4 words per thread
    uint64_t slices = ((uint64_t)sm_count * 8 + tiles - 1) / tiles;
    const uint64_t most = (nwords + 256 * 4 - 1) / (256 * 4);
    if (slices > most) slices = most;
    if (slices < 1) slices = 1;
    for (uint64_t t0 = 0; t0 < tiles; t0 += 65535) {   // grid.y holds at most 65535 tiles per launch
        const uint64_t nt = tiles - t0 < 65535 ? tiles - t0 : 65535;
        const dim3 grid((unsigned)slices, (unsigned)nt);
        DD_COUNT_LAUNCH(), exact_pair_popc_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint8_t *>(d_rows), row0, nr,
                                                                         static_cast<const uint8_t *>(d_cols), col0, nc, ws_stride,
                                                                         nwords, n_genomes, col_tiles, (int64_t)t0,
                                                                         reinterpret_cast<unsigned long long *>(d_inter));
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace dd
