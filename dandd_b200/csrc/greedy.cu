// greedy.cu -- K11: one step of a greedy ordering, the histogram of max(U, g) for every remaining candidate g and k.
//
//   progressive -r <greedy ordering>, one SubSpider union per candidate per step   reference lib/huffman_dandd.py:618-663
//     -> greedy_dense_kernel, greedy_compact (greedy_dense_kernel<true>), greedy_sparse_kernel
//
// U is the running union [nk][2^p].  hist(max(U, g)) is hist(U) moved by one -1 / +1 pair per register where g > U
// (a "live" register), so a step only has to find the live registers.  U only grows: the live set of a candidate only
// shrinks, to about 1/(t+1) of the registers at step t for independent genomes.
//
//   dense    reads every register of every listed candidate.  Lane = candidate, warp = a slab of registers of one k:
//            the 32 lanes of a warp count into 32 different shared-memory rows of odd stride, so the -1 / +1 pairs
//            never collide on a bank (lanes over the registers of one candidate would pile onto the one or two bins
//            where most HLL ranks sit).  U's bytes are the same for the whole warp (broadcast loads).
//   compact  the same scan, writing every live register as one u32 entry `j << 6 | value` (p <= 26, values < 64)
//            into per-(genome, k) segments whose capacities the caller took from the dense step's live counts.
//   sparse   one CTA per (candidate, k) segment: drop the entries with value <= U[k][j], compact the rest in place
//            (ballot + CTA prefix), and count their pairs in thread-private byte counters.  The kept entries are the
//            next step's live set.
// All three write hist[C][nk][64] (u32) and live[C][nk]; greedy_finish_kernel adds hist(U) to every row.
#include <cuda_runtime.h>

#include <vector>

#include "common.cuh"
#include "hist.cuh"
#include "kernels.cuh"
#include "swar.cuh"

namespace dd {

constexpr int kGrThreads = 256;
constexpr int kGrWarps = kGrThreads / 32;
constexpr int kGrRow = DD_HIST_BINS + 1;      // odd row stride; slot 64 counts the live registers
constexpr int kGrVec = 4;                     // 16-byte loads in flight per lane: 64 registers
constexpr int kGrWarpRegs = 2048;             // registers of one k a warp covers per CTA
constexpr int kGrCtaRegs = kGrWarps * kGrWarpRegs;
constexpr int kSpRounds = 255;                // byte counters: at most one increment per thread and round

__device__ __forceinline__ uint32_t word_at(const uint4 &w, int i) { return i == 0 ? w.x : i == 1 ? w.y : i == 2 ? w.z : w.w; }

// grid (batches * slabs, nk); batch = 32 candidates (one per lane), slab = kGrCtaRegs registers.
//   kEmit false: -1 / +1 pairs into hist[c][k][*] (wrapping u32, added to) and live counts into live[c * nk + k].
//   kEmit true:  every live register of candidate g at k becomes an entry of segment g * nk + k: position from an
//                atomic cursor seg_len[s], written only below the segment's capacity seg_off[s + 1] - seg_off[s].
template <bool kEmit>
__global__ void __launch_bounds__(kGrThreads)
greedy_dense_kernel(const uint8_t *__restrict__ regs, int nk, int p, const uint8_t *__restrict__ uni,
                    const int32_t *__restrict__ cand, int n_cand, unsigned slabs, uint32_t *__restrict__ hist,
                    uint32_t *__restrict__ live, const int64_t *__restrict__ seg_off, uint32_t *__restrict__ seg_len,
                    uint32_t *__restrict__ entries) {
    __shared__ int s_cnt[32 * kGrRow];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = blockIdx.y;
    const unsigned batch = blockIdx.x / slabs, slab = blockIdx.x % slabs;
    const int c = (int)batch * 32 + lane;
    const bool has = c < n_cand;
    const size_t m = (size_t)1 << p;
    const int g = has ? __ldg(&cand[c]) : 0;
    const uint8_t *grow = regs + ((size_t)g * nk + k) * m;
    const uint8_t *urow = uni + (size_t)k * m;
    const size_t j0 = (size_t)slab * kGrCtaRegs + (size_t)warp * kGrWarpRegs;
    const size_t j1 = min(j0 + (size_t)kGrWarpRegs, m);
    int *row = s_cnt + lane * kGrRow;
    if (!kEmit) {
        for (int i = threadIdx.x; i < 32 * kGrRow; i += kGrThreads) s_cnt[i] = 0;
        __syncthreads();
    }
    const size_t s = (size_t)g * nk + k;
    int64_t base = 0, cap = 0;
    if (kEmit && has) {
        base = seg_off[s];
        cap = seg_off[s + 1] - base;
    }
    uint32_t n_live = 0;
    if (has) {
        for (size_t j = j0; j < j1; j += 16 * kGrVec) {
            uint4 x[kGrVec], u[kGrVec];
#pragma unroll
            for (int b = 0; b < kGrVec; ++b) {
                x[b] = u[b] = make_uint4(0, 0, 0, 0);
                if (j + 16 * b < j1) {
                    x[b] = __ldcs(reinterpret_cast<const uint4 *>(grow + j + 16 * b));
                    u[b] = __ldg(reinterpret_cast<const uint4 *>(urow + j + 16 * b));
                }
            }
            uint32_t pos = 0;
            if (kEmit) {   // reserve this lane's entries of the 64 registers at once
                uint32_t cnt = 0;
#pragma unroll
                for (int b = 0; b < kGrVec; ++b)
#pragma unroll
                    for (int w = 0; w < 4; ++w) cnt += __popc(gt_top(word_at(x[b], w), word_at(u[b], w)));
                if (cnt) pos = atomicAdd(&seg_len[s], cnt);
            }
#pragma unroll
            for (int b = 0; b < kGrVec; ++b) {
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const uint32_t gw = word_at(x[b], w), uw = word_at(u[b], w);
                    uint32_t gt = gt_top(gw, uw);
                    if (!kEmit) n_live += __popc(gt);
                    while (gt) {
                        const int sh = __ffs(gt) - 8;   // bit 7 of the live byte
                        gt &= gt - 1;
                        const uint32_t gv = (gw >> sh) & 0xffu;
                        if (kEmit) {
                            const uint32_t jj = (uint32_t)(j + 16 * b + 4 * w + (sh >> 3));
                            if ((int64_t)pos < cap) entries[base + pos] = jj << 6 | (gv & 63u);
                            ++pos;
                        } else {
                            atomicSub(&row[ph_bin((uw >> sh) & 0xffu)], 1);
                            atomicAdd(&row[ph_bin(gv)], 1);
                        }
                    }
                }
            }
        }
    }
    if (kEmit) return;
    if (n_live) atomicAdd(&row[DD_HIST_BINS], (int)n_live);
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * kGrRow; i += kGrThreads) {
        const int cc = i / kGrRow, b = i - cc * kGrRow;
        const int d = s_cnt[i];
        const int ci = (int)batch * 32 + cc;
        if (!d || ci >= n_cand) continue;
        if (b < DD_HIST_BINS) atomicAdd(&hist[((size_t)ci * nk + k) * DD_HIST_BINS + b], (uint32_t)d);
        else atomicAdd(&live[(size_t)ci * nk + k], (uint32_t)d);
    }
}

// grid (C, nk): the segment of candidate cand[blockIdx.x] at k = blockIdx.y.  Entries with value <= U[k][j] are
// dropped, the rest are moved down in place (a write never passes the reads of its round, which all precede it)
// and their pairs counted; seg_len and live get the kept count.  A segment is clipped to its capacity and to the
// entry buffer, so no offsets can make it read or write outside them.
__global__ void __launch_bounds__(kGrThreads)
greedy_sparse_kernel(uint32_t *__restrict__ entries, int64_t n_entries, const int64_t *__restrict__ seg_off,
                     uint32_t *__restrict__ seg_len, int nk, int p, const uint8_t *__restrict__ uni,
                     const int32_t *__restrict__ cand, uint32_t *__restrict__ hist, uint32_t *__restrict__ live) {
    __shared__ __align__(16) uint8_t s_add[kPhBytes];
    __shared__ __align__(16) uint8_t s_sub[kPhBytes];
    __shared__ uint32_t s_warp[2][kGrWarps];
    const int c = blockIdx.x, k = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t s = (size_t)__ldg(&cand[c]) * nk + k;
    const int64_t off = seg_off[s];
    int64_t cap = seg_off[s + 1] - off;
    if (off < 0 || off > n_entries) cap = 0;
    cap = min(cap, n_entries - off);
    const uint32_t len = (uint32_t)max((int64_t)0, min((int64_t)seg_len[s], cap));
    uint32_t *seg = entries + (cap > 0 ? off : 0);
    const uint32_t mask = (uint32_t)(((size_t)1 << p) - 1);   // p = 26 fills all 26 index bits
    const uint8_t *urow = uni + (size_t)k * ((size_t)1 << p);
    uint32_t *out = hist + ((size_t)c * nk + k) * DD_HIST_BINS;
    const uint32_t slot = ph_slot();
    uint32_t kept = 0;   // CTA-uniform
    int parity = 0;
    for (uint32_t r0 = 0; r0 < len; r0 += (uint32_t)kGrThreads * kSpRounds) {
        ph_zero(s_add);
        ph_zero(s_sub);
        __syncthreads();
        const uint32_t r1 = min(len, r0 + (uint32_t)kGrThreads * kSpRounds);
        for (uint32_t i0 = r0; i0 < r1; i0 += kGrThreads) {
            const uint32_t i = i0 + threadIdx.x;
            uint32_t e = 0;
            bool keep = false;
            if (i < r1) {
                e = seg[i];
                const uint32_t v = e & 63u, uv = __ldg(&urow[(e >> 6) & mask]);
                keep = v > uv;
                if (keep) {
                    s_add[ph_bin(v) * kPhThreads + slot]++;
                    s_sub[ph_bin(uv) * kPhThreads + slot]++;
                }
            }
            const uint32_t ballot = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) s_warp[parity][warp] = __popc(ballot);
            __syncthreads();   // every read of this round precedes every write below
            uint32_t before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < kGrWarps; ++w) {
                const uint32_t x = s_warp[parity][w];
                before += w < warp ? x : 0;
                total += x;
            }
            if (keep) seg[kept + before + __popc(ballot & ((1u << lane) - 1u))] = e;
            kept += total;
            parity ^= 1;
        }
        __syncthreads();
        for (int b = warp; b < DD_HIST_BINS; b += kGrWarps) {
            const int d = (int)ph_total(s_add, b) - (int)ph_total(s_sub, b);
            if (lane == 0 && d) atomicAdd(&out[b], (uint32_t)d);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (cap > 0) seg_len[s] = kept;
        live[(size_t)c * nk + k] = kept;
    }
}

// hist[c][k][*] += uhist[k][*]: every row starts from the histogram of U.
__global__ void __launch_bounds__(256)
greedy_finish_kernel(const uint32_t *__restrict__ uhist, int nk, size_t cells, uint32_t *__restrict__ hist) {
    const size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= cells) return;
    hist[i] += uhist[(i / DD_HIST_BINS) % (size_t)nk * DD_HIST_BINS + (i & (DD_HIST_BINS - 1))];
}

size_t greedy_workspace_bytes(int n_cand) { return ((size_t)n_cand * sizeof(int32_t) + 15) & ~(size_t)15; }

static cudaError_t upload_cand(const int32_t *h_cand, int n_cand, void *d_ws, cudaStream_t stream) {
    // pageable source: the call returns once the bytes are staged, so the caller may reuse h_cand at once
    return cudaMemcpyAsync(d_ws, h_cand, (size_t)n_cand * sizeof(int32_t), cudaMemcpyHostToDevice, stream);
}

static cudaError_t finish(const uint32_t *d_uhist, int n_cand, int nk, uint32_t *d_hist, cudaStream_t stream) {
    const size_t cells = (size_t)n_cand * nk * DD_HIST_BINS;
    DD_COUNT_LAUNCH(), greedy_finish_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, stream>>>(d_uhist, nk, cells, d_hist);
    return cudaGetLastError();
}

static unsigned dense_slabs(int p) { return (unsigned)((((size_t)1 << p) + kGrCtaRegs - 1) / kGrCtaRegs); }

cudaError_t greedy_dense_hist(const uint8_t *d_regs, int nk, int p, const uint8_t *d_union, const uint32_t *d_uhist,
                              const int32_t *h_cand, int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws,
                              cudaStream_t stream) {
    const int32_t *d_cand = static_cast<const int32_t *>(d_ws);
    cudaError_t e = upload_cand(h_cand, n_cand, d_ws, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_hist, 0, (size_t)n_cand * nk * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_live, 0, (size_t)n_cand * nk * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    const unsigned slabs = dense_slabs(p), batches = (unsigned)((n_cand + 31) / 32);
    DD_COUNT_LAUNCH(), greedy_dense_kernel<false><<<dim3(batches * slabs, (unsigned)nk), kGrThreads, 0, stream>>>(
        d_regs, nk, p, d_union, d_cand, n_cand, slabs, d_hist, d_live, nullptr, nullptr, nullptr);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return finish(d_uhist, n_cand, nk, d_hist, stream);
}

cudaError_t greedy_compact(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union,
                           const int32_t *h_cand, int n_cand, const int64_t *h_seg_off, int64_t *d_seg_off,
                           uint32_t *d_seg_len, uint32_t *d_entries, void *d_ws, cudaStream_t stream) {
    const int32_t *d_cand = static_cast<const int32_t *>(d_ws);
    const size_t n_seg = (size_t)n_genomes * nk;
    cudaError_t e = upload_cand(h_cand, n_cand, d_ws, stream);
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(d_seg_off, h_seg_off, (n_seg + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_seg_len, 0, n_seg * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    const unsigned slabs = dense_slabs(p), batches = (unsigned)((n_cand + 31) / 32);
    DD_COUNT_LAUNCH(), greedy_dense_kernel<true><<<dim3(batches * slabs, (unsigned)nk), kGrThreads, 0, stream>>>(
        d_regs, nk, p, d_union, d_cand, n_cand, slabs, nullptr, nullptr, d_seg_off, d_seg_len, d_entries);
    return cudaGetLastError();
}

cudaError_t greedy_sparse_hist(uint32_t *d_entries, int64_t n_entries, const int64_t *d_seg_off, uint32_t *d_seg_len,
                               int nk, int p, const uint8_t *d_union, const uint32_t *d_uhist, const int32_t *h_cand,
                               int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws, cudaStream_t stream) {
    const int32_t *d_cand = static_cast<const int32_t *>(d_ws);
    cudaError_t e = upload_cand(h_cand, n_cand, d_ws, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_hist, 0, (size_t)n_cand * nk * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    DD_COUNT_LAUNCH(), greedy_sparse_kernel<<<dim3((unsigned)n_cand, (unsigned)nk), kGrThreads, 0, stream>>>(
        d_entries, n_entries, d_seg_off, d_seg_len, nk, p, d_union, d_cand, d_hist, d_live);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    return finish(d_uhist, n_cand, nk, d_hist, stream);
}

}  // namespace dd
