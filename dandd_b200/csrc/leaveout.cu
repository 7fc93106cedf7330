// leaveout.cu -- K10: the register histograms of every leave-one-group-out union, one read of the registers.
//
//   DeltaTree.find_delta_delta(subset)   reference lib/huffman_dandd.py:559-566   -> leave_out_kernel
//
// Leave group G out of a collection, and register j of the union of the rest is the union's max1(j), unless every
// genome that holds max1(j) is in G; then it is max2(j), the largest value among the genomes outside that leading
// group.  One pass over regs[n][nk][2^p] keeps (max1, max2, lead) per register and gives the union's histogram plus
// one -1 / +1 pair per register with a single leading group: the histogram of "all but group g" is the union's
// histogram moved by the pairs of the registers g leads.
//
// The genomes are visited sorted by group, so "lead == current group" is a byte mask that starts at zero with every
// group; the lead's group id is written out only where the mask is set when a group ends.  Per 16 registers and
// genome that is one 16-byte load and about 18 integer instructions per 4 registers, whatever the lead is.
#include <cuda_runtime.h>

#include <vector>

#include "common.cuh"
#include "hist.cuh"
#include "kernels.cuh"
#include "swar.cuh"

namespace dd {

constexpr int kLoThreads = kPhThreads;   // 16 registers per thread: a CTA covers 4096 registers of one k
constexpr int kLoBatch = 4;              // genome loads in flight per thread
constexpr int kLoSmemCorrBytes = 48 << 10;

// One genome of the current group c over 4 registers.  mine: lead == c, multi: lead is MULTI (top-bit flags).
//   v >  max1: not mine -> max2 = max1, lead = c; max1 = v
//   v == max1: not mine -> lead = MULTI
//   v <  max1: not mine -> max2 = max(max2, v)
// max(max2, min(v, max1)) covers the first and third case; in the second it sets max2 = max1, which is never read
// while the lead is MULTI and is overwritten when a single group takes the lead again.
__device__ __forceinline__ void lo_step(uint32_t v, uint32_t &m1, uint32_t &m2, uint32_t &mine, uint32_t &multi) {
    const uint32_t gt = gt_top(v, m1), eq = eq_top(v, m1);
    const uint32_t gt_mask = spread(gt);
    const uint32_t lo = pick(gt_mask, m1, v);
    m1 = pick(gt_mask, v, m1);
    m2 = pick(spread(gt_top(lo, m2) & ~mine), lo, m2);
    multi = (multi | (eq & ~mine)) & ~gt;
    mine |= gt;
}

// grid (ceil(nvec / 256), nk).  members[n] = {genome, group}, sorted by group.  The union histogram of this CTA's
// registers goes to union_ws[k]; the corrections go straight to hist[k][1 + g] (u32, wrapping: the union part that
// leave_out_finish_kernel adds brings every cell back to a count).  kSmem: corrections counted per CTA in shared
// memory [G][64] (signed), else one global atomic each.
template <bool kSmem>
__global__ void __launch_bounds__(kLoThreads, 4)
leave_out_kernel(const uint8_t *__restrict__ regs, int n, int nk, int p, const int2 *__restrict__ members, int n_groups,
                 uint64_t reg_begin, uint64_t nvec, uint32_t *__restrict__ union_ws, uint32_t *__restrict__ hist) {
    extern __shared__ __align__(16) uint8_t s_mem[];
    const int k = blockIdx.y;
    const size_t m = (size_t)1 << p;
    const uint64_t v = (uint64_t)blockIdx.x * kLoThreads + threadIdx.x;
    const bool live = v < nvec;
    const uint8_t *base = regs + (size_t)k * m + reg_begin + v * 16;
    const size_t gstride = (size_t)nk * m;

    uint4 m1 = make_uint4(0, 0, 0, 0), m2 = m1, mine = m1, multi = make_uint4(kTop, kTop, kTop, kTop);
    uint32_t lead[8];            // u16 group id of register b in the half (b & 1) of lead[b >> 1]
#pragma unroll
    for (int b = 0; b < 8; ++b) lead[b] = 0;
    int cur = __ldg(&members[0].y);
    auto close_group = [&]() {   // the bytes the current group leads now record it
        if (mine.x | mine.y | mine.z | mine.w) {
#pragma unroll
            for (int b = 0; b < 16; ++b)
                if (byte_at(mine, b)) lead[b >> 1] = __byte_perm(lead[b >> 1], (uint32_t)cur, (b & 1) ? 0x5410 : 0x3254);
            mine = make_uint4(0, 0, 0, 0);
        }
    };
    for (int i0 = 0; i0 < n; i0 += kLoBatch) {
        uint4 x[kLoBatch];
        int c[kLoBatch];
#pragma unroll
        for (int b = 0; b < kLoBatch; ++b) {
            c[b] = cur;
            x[b] = make_uint4(0, 0, 0, 0);
            if (i0 + b < n) {
                const int2 e = __ldg(&members[i0 + b]);
                c[b] = e.y;
                if (live) x[b] = __ldcs(reinterpret_cast<const uint4 *>(base + (size_t)e.x * gstride));
            }
        }
#pragma unroll
        for (int b = 0; b < kLoBatch; ++b) {
            if (i0 + b >= n) break;
            if (c[b] != cur) {   // CTA-uniform
                close_group();
                cur = c[b];
            }
            lo_step(x[b].x, m1.x, m2.x, mine.x, multi.x);
            lo_step(x[b].y, m1.y, m2.y, mine.y, multi.y);
            lo_step(x[b].z, m1.z, m2.z, mine.z, multi.z);
            lo_step(x[b].w, m1.w, m2.w, mine.w, multi.w);
        }
    }
    close_group();

    // the union: thread-private byte counters, 16 values per thread
    const uint32_t slot = ph_slot();
    ph_zero(s_mem);
    __syncthreads();
    if (live) {
        ph_add_word(s_mem, slot, m1.x);
        ph_add_word(s_mem, slot, m1.y);
        ph_add_word(s_mem, slot, m1.z);
        ph_add_word(s_mem, slot, m1.w);
    }
    __syncthreads();
    ph_flush(s_mem, union_ws + (size_t)k * DD_HIST_BINS);
    __syncthreads();

    // the corrections: row 1 + lead loses max1 and gains max2 (max2 < max1 under a single lead)
    uint32_t *rows = hist + ((size_t)k * (n_groups + 1) + 1) * DD_HIST_BINS;
    int *s_corr = reinterpret_cast<int *>(s_mem);
    const int cells = n_groups * DD_HIST_BINS;
    if (kSmem) {
        for (int i = threadIdx.x; i < cells; i += kLoThreads) s_corr[i] = 0;
        __syncthreads();
    }
    if (live) {
#pragma unroll
        for (int b = 0; b < 16; ++b) {
            if (byte_at(multi, b)) continue;
            const size_t row = (size_t)((lead[b >> 1] >> (16 * (b & 1))) & 0xffffu) * DD_HIST_BINS;
            const uint32_t hi = ph_bin(byte_at(m1, b)), lo = ph_bin(byte_at(m2, b));
            if (kSmem) {
                atomicSub(&s_corr[row + hi], 1);
                atomicAdd(&s_corr[row + lo], 1);
            } else {
                atomicAdd(&rows[row + hi], 0xffffffffu);
                atomicAdd(&rows[row + lo], 1u);
            }
        }
    }
    if (kSmem) {
        __syncthreads();
        for (int i = threadIdx.x; i < cells; i += kLoThreads)
            if (const int d = s_corr[i]) atomicAdd(&rows[i], (uint32_t)d);
    }
}

// hist[k][r][*] += union_ws[k][*] for r = 0 .. G: the union row, and the part every leave-out row shares.
__global__ void __launch_bounds__(256)
leave_out_finish_kernel(const uint32_t *__restrict__ union_ws, int n_rows, uint32_t *__restrict__ hist) {
    const int k = blockIdx.y;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n_rows * DD_HIST_BINS) return;
    hist[(size_t)k * n_rows * DD_HIST_BINS + i] += union_ws[(size_t)k * DD_HIST_BINS + (i & (DD_HIST_BINS - 1))];
}

size_t leave_out_workspace_bytes(int n_genomes, int nk) {
    return (size_t)nk * DD_HIST_BINS * sizeof(uint32_t) + (size_t)n_genomes * sizeof(int2);
}

cudaError_t leave_out_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *h_group, int n_groups,
                           uint64_t reg_begin, uint64_t reg_end, uint32_t *d_hist, void *d_ws, cudaStream_t stream) {
    // genomes sorted by group (counting sort; the ids were checked against [0, n_groups) by the caller)
    std::vector<int> first(n_groups + 1, 0);
    for (int g = 0; g < n_genomes; ++g) first[h_group[g] + 1]++;
    for (int c = 0; c < n_groups; ++c) first[c + 1] += first[c];
    std::vector<int2> members(n_genomes);
    for (int g = 0; g < n_genomes; ++g) members[first[h_group[g]]++] = make_int2(g, h_group[g]);

    uint32_t *union_ws = static_cast<uint32_t *>(d_ws);
    int2 *d_members = reinterpret_cast<int2 *>(static_cast<uint8_t *>(d_ws) + (size_t)nk * DD_HIST_BINS * sizeof(uint32_t));
    cudaError_t e = cudaMemsetAsync(union_ws, 0, (size_t)nk * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    // pageable source: the call returns once the bytes are staged, so `members` may go out of scope
    e = cudaMemcpyAsync(d_members, members.data(), members.size() * sizeof(int2), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) return e;

    const uint64_t nvec = (reg_end - reg_begin) / 16;
    if (nvec == 0) return cudaSuccess;
    const dim3 grid((unsigned)((nvec + kLoThreads - 1) / kLoThreads), (unsigned)nk);
    const size_t corr = (size_t)n_groups * DD_HIST_BINS * sizeof(int);
    if (corr <= (size_t)kLoSmemCorrBytes) {   // <= 48 KiB: no opt-in attribute, four CTAs per SM
        const size_t smem = corr > (size_t)kPhBytes ? corr : (size_t)kPhBytes;
        DD_COUNT_LAUNCH(), leave_out_kernel<true><<<grid, kLoThreads, smem, stream>>>(
            d_regs, n_genomes, nk, p, d_members, n_groups, reg_begin, nvec, union_ws, d_hist);
    } else {
        DD_COUNT_LAUNCH(), leave_out_kernel<false><<<grid, kLoThreads, kPhBytes, stream>>>(
            d_regs, n_genomes, nk, p, d_members, n_groups, reg_begin, nvec, union_ws, d_hist);
    }
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int n_rows = n_groups + 1;
    DD_COUNT_LAUNCH(), leave_out_finish_kernel<<<dim3((unsigned)((n_rows * DD_HIST_BINS + 255) / 256), (unsigned)nk), 256, 0,
                                                 stream>>>(union_ws, n_rows, d_hist);
    return cudaGetLastError();
}

}  // namespace dd
