// lattice.cu -- K3 for small jobs: every prefix union of up to 12 sketches from one pass over the registers.
//
// The planes kernel (planes.cu) redoes the same work for every (ordering, step): one more member max-ed
// into the running union, then a 64-value histogram of all 2^p registers.  Here the union of ANY subset S
// of the job's n <= 12 sketches is read from one table per k instead:
//   * for register r and value v >= 1 let M_v(r) = {g : x_g(r) >= v}, an n-bit mask; max_{g in S} x_g(r) >= v
//     exactly when M_v(r) meets S;
//   * F_v[M] = #{r : M_v(r) = M} (F_v[0] is not kept) and its subset sum Z_v[T] = sum_{0 != M subset T} F_v[M] give
//     cnt>=_S(v) = Z_v[full] - Z_v[full \ S], and hist_S[v] = cnt>=_S(v) - cnt>=_S(v + 1), hist_S[0] = 2^p - cnt>=_S(1).
// Only integers are counted, so every histogram is bit-identical to the planes kernel's.
//
// A register whose distinct non-zero values are u_1 > ... > u_d (u_{d+1} = 0) has d levels; level i has mask
// M^(i) = {g : x_g >= u_i} and covers v in (u_{i+1}, u_i], which in difference form over v is two updates:
// D[u_{i+1} + 1][M^(i)] += 1 and D[u_i + 1][M^(i)] -= 1 (the second dropped at u_i = 63).  A prefix sum over v
// turns D into F.  The cost is one read of the registers and ~2d table updates per register, whatever the
// number of orderings and steps.  On the 12 x 5 Mbp bench genomes d averages 2.7 (k = 21) to 3.2 (k = 32);
// the full set, the full set less one genome and single genomes make 58-67 % of the level masks, and those
// updates go to a per-CTA shared-memory table -- the rest, 1.8 (k = 21) to 2.6 (k = 32) per register, are L2
// reductions into D.
#include <cuda_runtime.h>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr int kLatMaxGenomes = 12;
constexpr int kLatThreads = 256;
constexpr int kLatValues = DD_HIST_BINS;   // register values 0..63

// shared-memory part of D for the masks most registers produce: the full set, the full set less genome g,
// genome g alone
struct LatticeSmem {
    uint32_t full[kLatValues];
    uint32_t miss[kLatValues][kLatMaxGenomes];
    uint32_t one[kLatValues][kLatMaxGenomes];
};

__device__ __forceinline__ void lattice_update(LatticeSmem &s, uint32_t *__restrict__ dk, int n, uint32_t full, int v,
                                               uint32_t mask, uint32_t delta) {
    if (mask == full) {
        atomicAdd(&s.full[v], delta);
        return;
    }
    const int c = __popc(mask);
    if (c == n - 1) atomicAdd(&s.miss[v][__ffs((int)(~mask & full)) - 1], delta);
    else if (c == 1) atomicAdd(&s.one[v][__ffs((int)mask) - 1], delta);
    else atomicAdd(&dk[((size_t)v << n) + mask], delta);
}

// grid (CTAs per k, nk).  A thread reads 16 consecutive registers of every sketch as one uint4 each and
// walks the levels of each register from the top: the genomes at or above the current level form its mask,
// the largest value below it is the next level.
__global__ void __launch_bounds__(kLatThreads)
lattice_levels_kernel(const uint8_t *__restrict__ regs, int n, int nk, int p, uint32_t *__restrict__ diff) {
    __shared__ LatticeSmem s;
    for (int i = threadIdx.x; i < (int)(sizeof(LatticeSmem) / 4); i += kLatThreads) reinterpret_cast<uint32_t *>(&s)[i] = 0u;
    __syncthreads();
    const int k = blockIdx.y;
    const size_t m = (size_t)1 << p, nvec = m / 16;
    const uint32_t full = (1u << n) - 1u;
    uint32_t *dk = diff + ((size_t)k * kLatValues << n);
    uint32_t base1 = 0;   // registers whose lowest level is the full set: D[1][full] += 1, too hot for a shared atomic
    for (size_t vec = (size_t)blockIdx.x * kLatThreads + threadIdx.x; vec < nvec; vec += (size_t)gridDim.x * kLatThreads) {
        uint4 x[kLatMaxGenomes];
#pragma unroll
        for (int g = 0; g < kLatMaxGenomes; ++g)
            x[g] = g < n ? __ldg(reinterpret_cast<const uint4 *>(regs + ((size_t)g * nk + k) * m) + vec) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t w[kLatMaxGenomes];
            uint32_t top = 0u;
#pragma unroll
            for (int g = 0; g < kLatMaxGenomes; ++g) {
                const uint32_t word = c == 0 ? x[g].x : c == 1 ? x[g].y : c == 2 ? x[g].z : x[g].w;
                w[g] = __vminu4(word, 0x3f3f3f3fu);
                top = __vmaxu4(top, w[g]);
            }
            if (top == 0u) continue;   // four registers that are 0 in every sketch
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                int hi = (int)((top >> (8 * b)) & 0xffu);
                while (hi > 0) {
                    uint32_t mask = 0u;
                    int lo = 0;
#pragma unroll
                    for (int g = 0; g < kLatMaxGenomes; ++g) {
                        const int v = (int)((w[g] >> (8 * b)) & 0xffu);   // 0 for g >= n
                        if (v >= hi) mask |= 1u << g;
                        else lo = max(lo, v);
                    }
                    if (lo == 0 && mask == full) ++base1;
                    else lattice_update(s, dk, n, full, lo + 1, mask, 1u);
                    if (hi < kLatValues - 1) lattice_update(s, dk, n, full, hi + 1, mask, 0xffffffffu);
                    hi = lo;
                }
            }
        }
    }
    base1 = __reduce_add_sync(0xffffffffu, base1);
    if ((threadIdx.x & 31) == 0 && base1) atomicAdd(&s.full[1], base1);
    __syncthreads();
    for (int i = threadIdx.x; i < kLatValues * (1 + 2 * kLatMaxGenomes); i += kLatThreads) {
        const int v = i / (1 + 2 * kLatMaxGenomes), j = i % (1 + 2 * kLatMaxGenomes);
        if (j > 2 * n) continue;
        const uint32_t c = j == 0 ? s.full[v] : j <= n ? s.miss[v][j - 1] : s.one[v][j - 1 - n];
        const uint32_t mask = j == 0 ? full : j <= n ? full & ~(1u << (j - 1)) : 1u << (j - 1 - n);
        if (c) atomicAdd(&dk[((size_t)v << n) + mask], c);
    }
}

// D -> F: running sum over v, one thread per (k, mask)
__global__ void __launch_bounds__(256) lattice_prefix_kernel(uint32_t *__restrict__ diff, int n) {
    const uint32_t mask = blockIdx.x * 256u + threadIdx.x;
    if (mask >= (1u << n)) return;
    uint32_t *col = diff + ((size_t)blockIdx.y * kLatValues << n) + mask;
    uint32_t run = 0u;
    for (int v = 1; v < kLatValues; ++v) {
        run += col[(size_t)v << n];
        col[(size_t)v << n] = run;
    }
}

// the set of every requested (ordering, step): members of order[o][0..step] that are genomes of the job
__global__ void lattice_sets_kernel(const int32_t *__restrict__ order, int n_ord, int n_steps, int n_genomes,
                                    uint32_t *__restrict__ sets) {
    const int o = blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_ord) return;
    uint32_t s = 0u;
    for (int st = 0; st < n_steps; ++st) {
        const int g = order[(size_t)o * n_steps + st];
        if (g >= 0 && g < n_genomes) s |= 1u << g;
        sets[(size_t)o * n_steps + st] = s;
    }
}

// grid (63, nk), CTA (v, k): F_v -> Z_v in shared memory (n passes), then cnt>=_S(v) into bin v of every
// requested row; lattice_finish_kernel turns the counts into the histogram
__global__ void __launch_bounds__(256)
lattice_zeta_kernel(const uint32_t *__restrict__ diff, const uint32_t *__restrict__ sets, int n_ord, int n_steps, int n,
                    int nk, int final_only, uint32_t *__restrict__ hist) {
    extern __shared__ uint32_t z[];
    const int v = blockIdx.x + 1, k = blockIdx.y;
    const uint32_t size = 1u << n, full = size - 1u;
    const uint32_t *row = diff + (((size_t)k * kLatValues + v) << n);
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) z[i] = i ? row[i] : 0u;
    __syncthreads();
    for (int b = 0; b < n; ++b) {
        const uint32_t bit = 1u << b;
        for (uint32_t i = threadIdx.x; i < size / 2; i += blockDim.x) {
            const uint32_t t = ((i >> b) << (b + 1)) | bit | (i & (bit - 1u));   // i-th mask with bit b set
            z[t] += z[t ^ bit];
        }
        __syncthreads();
    }
    const uint32_t total = z[full];
    const int out_steps = final_only ? 1 : n_steps;
    const size_t rows = (size_t)n_ord * out_steps;
    for (size_t r = threadIdx.x; r < rows; r += blockDim.x) {
        const size_t o = r / out_steps;
        const int st = final_only ? n_steps - 1 : (int)(r % out_steps);
        const uint32_t s = sets[o * n_steps + st];
        hist[(r * nk + k) * DD_HIST_BINS + v] = total - z[full & ~s];
    }
}

// one warp per row: bins 1..63 hold cnt>=(v); hist[v] = cnt>=(v) - cnt>=(v + 1) with cnt>=(0) = 2^p, cnt>=(64) = 0
__global__ void __launch_bounds__(256) lattice_finish_kernel(uint32_t *__restrict__ hist, size_t rows, int p) {
    const size_t r = ((size_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (r >= rows) return;   // whole warps leave together
    const int lane = threadIdx.x & 31;
    uint32_t *h = hist + r * DD_HIST_BINS;
    const uint32_t lo = lane ? h[lane] : 1u << p, hi = h[lane + 32];
    const uint32_t lo_next = __shfl_down_sync(0xffffffffu, lo, 1), hi_next = __shfl_down_sync(0xffffffffu, hi, 1);
    const uint32_t hi0 = __shfl_sync(0xffffffffu, hi, 0);
    h[lane] = lo - (lane == 31 ? hi0 : lo_next);
    h[lane + 32] = hi - (lane == 31 ? 0u : hi_next);
}

// ---- host side ----------------------------------------------------------------------------------
int g_prefix_lattice = 1;

bool lattice_supported(int n_genomes, int p) { return n_genomes >= 1 && n_genomes <= kLatMaxGenomes && p >= 12; }

static size_t lattice_table_bytes(int n_genomes, int nk) {
    return (((size_t)nk * kLatValues * sizeof(uint32_t) << n_genomes) + 255) / 256 * 256;
}
size_t prefix_lattice_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk) {
    return lattice_table_bytes(n_genomes, nk) + ((size_t)n_ord * n_steps * sizeof(uint32_t) + 255) / 256 * 256;
}

cudaError_t prefix_union_hist_lattice(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                                      int nk, int p, int final_only, uint32_t *d_hist, void *d_ws, cudaStream_t stream) {
    const size_t rows = (size_t)n_ord * (final_only ? 1 : n_steps) * nk;
    if (rows == 0) return cudaSuccess;
    uint32_t *diff = reinterpret_cast<uint32_t *>(d_ws);
    uint32_t *sets = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(d_ws) + lattice_table_bytes(n_genomes, nk));
    const size_t cols = (size_t)1 << n_genomes;
    cudaError_t e = cudaMemsetAsync(diff, 0, (size_t)nk * kLatValues * cols * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    // ~8 CTAs per SM over all k: each flushes its shared table once
    const size_t nvec = ((size_t)1 << p) / 16;
    size_t per_k = ((size_t)148 * 8 + nk - 1) / nk, most = (nvec + kLatThreads - 1) / kLatThreads;
    if (per_k > most) per_k = most;
    DD_COUNT_LAUNCH(), lattice_levels_kernel<<<dim3((unsigned)per_k, (unsigned)nk), kLatThreads, 0, stream>>>(d_regs, n_genomes,
                                                                                                             nk, p, diff);
    DD_COUNT_LAUNCH(), lattice_prefix_kernel<<<dim3((unsigned)((cols + 255) / 256), (unsigned)nk), 256, 0, stream>>>(diff,
                                                                                                                   n_genomes);
    DD_COUNT_LAUNCH(), lattice_sets_kernel<<<(n_ord + 255) / 256, 256, 0, stream>>>(d_order, n_ord, n_steps, n_genomes, sets);
    DD_COUNT_LAUNCH(), lattice_zeta_kernel<<<dim3(kLatValues - 1, (unsigned)nk), 256, cols * sizeof(uint32_t), stream>>>(
        diff, sets, n_ord, n_steps, n_genomes, nk, final_only, d_hist);
    DD_COUNT_LAUNCH(), lattice_finish_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, stream>>>(d_hist, rows, p);
    return cudaGetLastError();
}

}  // namespace dd
