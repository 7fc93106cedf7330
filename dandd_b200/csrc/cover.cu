// cover.cu -- K12: the exact greedy cover index, built once per (k, key-range pass) from the K7 lists.
//
// For a greedy ordering by exact union counts (helpers/greedy.py --tool kmc): with A_g genome g's distinct keys and U
// the union of the genomes chosen so far, |U u A_g| = |U| + |A_g| - lost[g], lost[g] = |A_g n U|.  When g* joins U,
// every key of A_g* that U did not cover yet becomes covered, and every genome h holding it gains lost[h] += 1.  A key
// is covered once, so a whole ordering costs sum |A_g| holder visits per k, whatever the number of steps.
//
// The index of one part (k, pass) needs no k-mer:
//   offsets      [keys + 1] u32   key-major CSR over
//   holders      [nodes]    u16   the genomes holding each key (one entry per K7 node)
//   key_of_node  [nodes]    u32   the key id of every K7 node.  PushGenome pushes exactly one node per (genome, key),
//                                 and genomes are inserted one after another on one stream, so genome g's nodes are
//                                 the contiguous range between the node-counter readings before and after its
//                                 insert: that range, mapped through key_of_node, is g's key list.
//   covered      [keys]     u8    (the caller's; zeroed at the start of an ordering)
#include <cuda_runtime.h>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr unsigned long long kAllOnes = 0xFFFFFFFFFFFFFFFFull;
constexpr size_t kCoverSmemBytes = 48 * 1024;   // u32 lost counters of n <= 12288 genomes per CTA

// Distinct keys = occupied slots (a list head), including the all-ones key's extra slot `capacity`.
__global__ void __launch_bounds__(256)
exact_cover_count_kernel(const ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh, uint64_t n_slots,
                         unsigned long long *out) {
    if (hdr->overflow) {   // a full table or node array: the marker, never a count
        if (blockIdx.x == 0 && threadIdx.x == 0) out[0] = out[1] = kAllOnes;
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[1] = hdr->n_nodes;
    unsigned c = 0;
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n_slots; s += (uint64_t)gridDim.x * blockDim.x)
        c += __ldg(&lh[s].y) != kNil;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, (unsigned long long)c);
}

// Every lane owns one slot and walks its list twice: once for its length, once to write.  A warp reserves its key ids
// and holder spans together with one 64-bit atomic on (keys << 32 | nodes), so the offsets of consecutive key ids are
// consecutive spans and offsets[] is non-decreasing.  (Nodes number below 2^32 - 1, so the low half never carries.)
__global__ void __launch_bounds__(256)
exact_cover_emit_kernel(ExactWsHeader *__restrict__ hdr, const uint2 *__restrict__ lh, const PairNode *__restrict__ nodes,
                        uint64_t n_slots, uint32_t n_genomes, uint64_t n_keys, uint64_t n_nodes, uint32_t *offsets,
                        uint16_t *holders, uint32_t *key_of_node) {
    if (hdr->overflow) return;   // reported by the finishing kernel
    const unsigned lane = threadIdx.x & 31;
    const uint64_t warps = (uint64_t)gridDim.x * (blockDim.x >> 5);
    for (uint64_t base = ((uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; base < n_slots; base += warps * 32) {
        const uint32_t head = base + lane < n_slots ? __ldg(&lh[base + lane].y) : kNil;
        uint32_t c = 0;
        bool bad = false;
        for (uint32_t at = head; at != kNil;) {
            if (at >= n_nodes) { bad = true; break; }
            const PairNode nd = nodes[at];
            bad |= nd.genome >= n_genomes;
            ++c;
            at = nd.next;
        }
        const unsigned occ = __ballot_sync(0xffffffffu, c != 0);
        uint32_t incl = c;   // inclusive prefix of the list lengths over the warp
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d) incl += v;
        }
        unsigned long long at0 = 0;
        if (lane == 31 && occ) at0 = atomicAdd(&hdr->cover_cursor, ((unsigned long long)__popc(occ) << 32) | incl);
        at0 = __shfl_sync(0xffffffffu, at0, 31);
        if (c == 0) continue;
        const uint64_t key = (at0 >> 32) + __popc(occ & ((1u << lane) - 1u));
        const uint64_t off = (at0 & 0xFFFFFFFFull) + incl - c;
        if (bad || key >= n_keys || off + c > n_nodes) {   // never an index: the finishing kernel reports it
            hdr->cover_bad = 1;
            continue;
        }
        offsets[key] = (uint32_t)off;
        uint32_t i = 0;
        for (uint32_t at = head; at != kNil; ++i) {
            const PairNode nd = nodes[at];
            holders[off + i] = (uint16_t)nd.genome;
            key_of_node[at] = (uint32_t)key;
            at = nd.next;
        }
    }
}

__global__ void exact_cover_finish_kernel(const ExactWsHeader *hdr, uint64_t n_keys, uint64_t n_nodes, uint32_t *offsets,
                                          unsigned long long *status) {
    const unsigned long long keys = hdr->cover_cursor >> 32, nodes = hdr->cover_cursor & 0xFFFFFFFFull;
    if (hdr->overflow || hdr->cover_bad || keys != n_keys || nodes != n_nodes) {
        status[0] = status[1] = kAllOnes;
        return;
    }
    offsets[n_keys] = (uint32_t)n_nodes;
    status[0] = keys;
    status[1] = nodes;
}

// One step over every part (blockIdx.y): the picked genome's nodes, 32 per warp round.  Each lane looks up its node's
// key; the keys not covered yet are covered, and for each of them in turn the warp walks its holder span 32 entries at
// a time, adding 1 to lost[h].  kSmem: u32 counters of the part in shared memory, flushed with 64-bit atomics.
template <bool kSmem>
__global__ void __launch_bounds__(256)
exact_cover_step_kernel(const CoverPart *__restrict__ parts, uint32_t n_genomes) {
    extern __shared__ uint32_t sm_lost[];
    const CoverPart P = parts[blockIdx.y];
    const uint64_t todo = P.node_end - P.node_begin;
    if ((uint64_t)blockIdx.x * blockDim.x >= todo) return;   // CTA-uniform, before any barrier
    if (kSmem) {
        for (uint32_t i = threadIdx.x; i < n_genomes; i += blockDim.x) sm_lost[i] = 0;
        __syncthreads();
    }
    const unsigned lane = threadIdx.x & 31;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < todo;
         base += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t key = 0;
        bool fresh = false;
        if (base + lane < todo) {
            key = __ldg(P.key_of_node + P.node_begin + base + lane);
            // A key appears once in a genome's node range (one node per (genome, key)), so no other thread of this step
            // touches covered[key]: a plain load and store, no atomic.
            fresh = !P.covered[key];
            if (fresh) P.covered[key] = 1;
        }
        for (unsigned m = __ballot_sync(0xffffffffu, fresh); m; m &= m - 1) {
            const uint32_t kk = __shfl_sync(0xffffffffu, key, __ffs(m) - 1);
            const uint32_t b = __ldg(P.offsets + kk), e = __ldg(P.offsets + kk + 1);
            for (uint32_t j = b + lane; j < e; j += 32) {
                const uint32_t h = __ldg(P.holders + j);
                if (h >= n_genomes) continue;   // the emit never writes one; never an address either
                if (kSmem) atomicAdd(&sm_lost[h], 1u);
                else atomicAdd(P.lost + h, 1ull);
            }
        }
    }
    if (kSmem) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_genomes; i += blockDim.x)
            if (sm_lost[i]) atomicAdd(P.lost + i, (unsigned long long)sm_lost[i]);
    }
}

static unsigned slot_grid(uint64_t n_slots, int sm_count) {
    const uint64_t want = (n_slots + 255) / 256;   // one slot per thread
    const uint64_t most = (uint64_t)sm_count * 16;
    return (unsigned)(want < 1 ? 1 : want < most ? want : most);
}

cudaError_t exact_cover_count(const void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint64_t *d_counts,
                              int sm_count, cudaStream_t stream) {
    const uint8_t *ws = static_cast<const uint8_t *>(d_ws);
    const cudaError_t e = cudaMemsetAsync(d_counts, 0, sizeof(uint64_t), stream);
    if (e != cudaSuccess) return e;
    const uint64_t n_slots = capacity + 1;
    DD_COUNT_LAUNCH(), exact_cover_count_kernel<<<slot_grid(n_slots, sm_count), 256, 0, stream>>>(
        static_cast<const ExactWsHeader *>(d_ws), reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams)),
        n_slots, reinterpret_cast<unsigned long long *>(d_counts));
    return cudaGetLastError();
}

cudaError_t exact_cover_emit(void *d_ws, int k, uint64_t capacity, unsigned max_streams, uint32_t n_genomes, uint64_t n_keys,
                             uint64_t n_nodes, uint32_t *d_offsets, uint16_t *d_holders, uint32_t *d_key_of_node,
                             uint64_t *d_status, int sm_count, cudaStream_t stream) {
    uint8_t *ws = static_cast<uint8_t *>(d_ws);
    ExactWsHeader *hdr = static_cast<ExactWsHeader *>(d_ws);
    cudaError_t e = cudaMemsetAsync(&hdr->cover_cursor, 0, 2 * sizeof(unsigned long long), stream);   // cursor, bad
    if (e != cudaSuccess) return e;
    const uint64_t n_slots = capacity + 1;
    DD_COUNT_LAUNCH(), exact_cover_emit_kernel<<<slot_grid(n_slots, sm_count), 256, 0, stream>>>(
        hdr, reinterpret_cast<const uint2 *>(ws + pairs_lh_offset(k, capacity, max_streams)),
        reinterpret_cast<const PairNode *>(ws + pairs_node_offset(k, capacity, max_streams)), n_slots, n_genomes, n_keys,
        n_nodes, d_offsets, d_holders, d_key_of_node);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    DD_COUNT_LAUNCH(), exact_cover_finish_kernel<<<1, 1, 0, stream>>>(hdr, n_keys, n_nodes, d_offsets,
                                                                       reinterpret_cast<unsigned long long *>(d_status));
    return cudaGetLastError();
}

cudaError_t exact_cover_step(const CoverPart *h_parts, int n_parts, uint32_t n_genomes, void *d_ws, int sm_count,
                             cudaStream_t stream) {
    uint64_t most = 0;
    for (int i = 0; i < n_parts; ++i) most = h_parts[i].node_end - h_parts[i].node_begin > most ? h_parts[i].node_end - h_parts[i].node_begin : most;
    if (most == 0) return cudaSuccess;
    // pageable source: the call returns once the bytes are staged, so the caller may reuse h_parts at once
    cudaError_t e = cudaMemcpyAsync(d_ws, h_parts, (size_t)n_parts * sizeof(CoverPart), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;
    const CoverPart *d_parts = static_cast<const CoverPart *>(d_ws);
    // a few CTAs per SM over all parts: with shared counters every CTA pays one pass over n counters at each end
    const uint64_t want = (most + 255) / 256;
    uint64_t cap = ((uint64_t)sm_count * 8 + n_parts - 1) / n_parts;
    if (cap < 1) cap = 1;
    const dim3 grid((unsigned)(want < cap ? want : cap), (unsigned)n_parts);
    const size_t smem = (size_t)n_genomes * sizeof(uint32_t);
    if (smem <= kCoverSmemBytes)
        DD_COUNT_LAUNCH(), exact_cover_step_kernel<true><<<grid, 256, smem, stream>>>(d_parts, n_genomes);
    else
        DD_COUNT_LAUNCH(), exact_cover_step_kernel<false><<<grid, 256, 0, stream>>>(d_parts, n_genomes);
    return cudaGetLastError();
}

}  // namespace dd
