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
// number of orderings and steps.  On the 12 x 5 Mbp bench genomes d averages 2.7 (k = 21) to 3.2 (k = 32).
//
// Level pass: one CTA per SM, each owning a contiguous register range of one k and a dense shared-memory table
// D[1..V][every mask] (V = as many values as fit in shared memory: 14 at n = 12, 63 for n <= 9).  At exit the
// table is stored whole to the CTA's own slab; lattice_prefix_kernel sums the slabs of each k while it runs the
// sum over v.  Updates at v > V (a register >= V in some sketch, rare) are L2 reductions into the rows v > V of
// the F table, the only part of the workspace that is zeroed per call.  The full set is the lowest level of
// every register that is non-zero in all n sketches, so its cells D[1][full] and D[min + 1][full] at small
// minima take most registers: they are counted in thread-private registers and added to the table once per warp.
#include <cuda_runtime.h>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr int kLatMaxGenomes = 12;
constexpr int kLatThreads = 896;
constexpr int kLatValues = DD_HIST_BINS;   // register values 0..63
constexpr int kLatPrivateMins = 4;         // full-set levels at minimum 1..4 are counted per thread, not in shared memory

// words of one CTA's table and slab, rounded up to whole uint4s
__host__ __device__ __forceinline__ size_t lattice_slab_words(int values, int n) { return (((size_t)values << n) + 3) & ~(size_t)3; }

struct LatticeTable {
    uint32_t *tab;      // shared: D[v][mask] at ((v - 1) << n) | mask, v = 1..V
    uint32_t *spill;    // global, this k: D[v][mask] at (v << n) | mask for v > V
    int n, values;
    uint32_t full;
    uint32_t base1;                    // D[1][full] += 1 of every register non-zero in all sketches
    uint32_t mins[kLatPrivateMins];    // D[m + 1][full] -= 1 of those whose minimum m is 1..4

    __device__ __forceinline__ void add(int v, uint32_t mask, uint32_t delta) {
        if (v <= values) atomicAdd(&tab[((v - 1) << n) | mask], delta);
        else atomicAdd(&spill[((size_t)v << n) | mask], delta);
    }
    // the level [lo + 1, hi] of mask
    __device__ __forceinline__ void level(int hi, int lo, uint32_t mask) {
        if (mask == full) {   // the lowest level: lo = 0 and hi is the minimum over the sketches
            ++base1;
#pragma unroll
            for (int m = 0; m < kLatPrivateMins; ++m) mins[m] += hi == m + 1;
            if (hi > kLatPrivateMins && hi < kLatValues - 1) add(hi + 1, full, 0xffffffffu);
            return;
        }
        add(lo + 1, mask, 1u);
        if (hi < kLatValues - 1) add(hi + 1, mask, 0xffffffffu);
    }
};

// w[g]: 4 consecutive registers of genome g (0 for g >= n).  Each register's levels are walked from the top: the
// genomes at or above the current level form its mask, the largest value below it is the next level.
template <int NW>
__device__ __forceinline__ void lattice_registers(LatticeTable &tb, uint32_t (&w)[4 * NW]) {
    uint32_t any = 0u;
#pragma unroll
    for (int g = 0; g < 4 * NW; ++g) any |= w[g];
    if (any == 0u) return;   // four registers that are 0 in every sketch
    if (any & 0xc0c0c0c0u) {
#pragma unroll
        for (int g = 0; g < 4 * NW; ++g) w[g] = __vminu4(w[g], 0x3f3f3f3fu);
    }
    uint32_t top = 0u;
#pragma unroll
    for (int g = 0; g < 4 * NW; ++g) top = __vmaxu4(top, w[g]);
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        int hi = (int)((top >> (8 * b)) & 0xffu);
        while (hi > 0) {
            uint32_t mask = 0u;
            int lo = 0;
#pragma unroll
            for (int g = 0; g < 4 * NW; ++g) {
                const int v = (int)((w[g] >> (8 * b)) & 0xffu);   // 0 for g >= n
                if (v >= hi) mask |= 1u << g;
                else lo = max(lo, v);
            }
            tb.level(hi, lo, mask);
            hi = lo;
        }
    }
}

// grid (per_k * nk): CTA c of k walks words [c, c + 1) * nwords / per_k of k's registers, 4 registers of every
// sketch per thread and step (the next step's words are loaded before the current ones are walked), then
// stores its table D[1..V] to slab blockIdx.x.
template <int NW>
__global__ void __launch_bounds__(kLatThreads, 1)
lattice_levels_kernel(const uint8_t *__restrict__ regs, int n, int nk, int p, int per_k, int values, uint32_t *__restrict__ slabs,
                      uint32_t *__restrict__ table) {
    extern __shared__ uint4 lattice_smem[];
    const size_t cols = (size_t)1 << n, words4 = lattice_slab_words(values, n) / 4;
    for (size_t i = threadIdx.x; i < words4; i += kLatThreads) lattice_smem[i] = make_uint4(0u, 0u, 0u, 0u);
    const int k = blockIdx.x / per_k, c = blockIdx.x % per_k;
    LatticeTable tb;
    tb.tab = reinterpret_cast<uint32_t *>(lattice_smem);
    tb.spill = table + (size_t)k * kLatValues * cols;
    tb.n = n;
    tb.values = values;
    tb.full = (uint32_t)cols - 1u;
    tb.base1 = 0u;
#pragma unroll
    for (int m = 0; m < kLatPrivateMins; ++m) tb.mins[m] = 0u;
    __syncthreads();

    const size_t m = (size_t)1 << p, nwords = m / 4;
    const size_t end = nwords * (c + 1) / per_k;
    const uint32_t *src = reinterpret_cast<const uint32_t *>(regs + (size_t)k * m);   // genome g at src + g * stride
    const size_t stride = (size_t)nk * nwords;
    uint32_t w[4 * NW];
    size_t i = nwords * c / per_k + threadIdx.x;
#pragma unroll
    for (int g = 0; g < 4 * NW; ++g) w[g] = i < end && g < n ? __ldg(src + g * stride + i) : 0u;
    for (; i < end; i += kLatThreads) {
        uint32_t nx[4 * NW];
#pragma unroll
        for (int g = 0; g < 4 * NW; ++g) nx[g] = i + kLatThreads < end && g < n ? __ldg(src + g * stride + i + kLatThreads) : 0u;
        lattice_registers<NW>(tb, w);
#pragma unroll
        for (int g = 0; g < 4 * NW; ++g) w[g] = nx[g];
    }

    const uint32_t base1 = __reduce_add_sync(0xffffffffu, tb.base1);
    uint32_t mins[kLatPrivateMins];
#pragma unroll
    for (int mi = 0; mi < kLatPrivateMins; ++mi) mins[mi] = __reduce_add_sync(0xffffffffu, tb.mins[mi]);
    if ((threadIdx.x & 31) == 0) {
        if (base1) atomicAdd(&tb.tab[tb.full], base1);
#pragma unroll
        for (int mi = 0; mi < kLatPrivateMins; ++mi)   // minimum mi + 1: D[mi + 2][full], row mi + 1
            if (mins[mi]) atomicAdd(&tb.tab[((size_t)(mi + 1) << n) | tb.full], 0u - mins[mi]);
    }
    __syncthreads();
    uint4 *slab = reinterpret_cast<uint4 *>(slabs + blockIdx.x * lattice_slab_words(values, n));
    for (size_t j = threadIdx.x; j < words4; j += kLatThreads) slab[j] = lattice_smem[j];
}

// D -> F, one thread per (k, mask): the slabs of k's CTAs hold D[1..V], the table's own rows hold D[V + 1..63]
__global__ void __launch_bounds__(256) lattice_prefix_kernel(const uint32_t *__restrict__ slabs, uint32_t *__restrict__ table, int n,
                                                             int per_k, int values) {
    const uint32_t mask = blockIdx.x * 256u + threadIdx.x;
    if (mask >= (1u << n)) return;
    const int k = blockIdx.y;
    const size_t cols = (size_t)1 << n;
    uint32_t *col = table + (size_t)k * kLatValues * cols + mask;
    const size_t slab_words = lattice_slab_words(values, n);
    const uint32_t *d = slabs + (size_t)k * per_k * slab_words + mask;
    uint32_t run = 0u;
    for (int v = 1; v <= values; ++v) {
        for (int c = 0; c < per_k; ++c) run += d[c * slab_words + (size_t)(v - 1) * cols];
        col[(size_t)v * cols] = run;
    }
    for (int v = values + 1; v < kLatValues; ++v) {
        run += col[(size_t)v * cols];
        col[(size_t)v * cols] = run;
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

// The level pass's shape on the current device, shared by the workspace size and the launch: V = the values
// a CTA's shared table holds, per_k = CTAs (and slabs) per k -- one CTA per SM over all k, no more than k's
// registers keep busy.
struct LatticeGeometry {
    int values, per_k;
};
static LatticeGeometry lattice_geometry(int n_genomes, int nk, int p) {
    int dev = 0, sms = 0, smem = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || sms <= 0 || smem <= 0) {
        cudaGetLastError();
        sms = 148;            // B200
        smem = 227 * 1024;
    }
    LatticeGeometry geo;
    geo.values = (int)((size_t)smem / (sizeof(uint32_t) << n_genomes));
    if (geo.values > kLatValues - 1) geo.values = kLatValues - 1;
    const size_t busy = (((size_t)1 << p) / 4 + kLatThreads - 1) / kLatThreads;
    size_t per_k = (size_t)sms / (size_t)nk;
    if (per_k > busy) per_k = busy;
    geo.per_k = per_k > 0 ? (int)per_k : 1;
    return geo;
}

static size_t round256(size_t b) { return (b + 255) / 256 * 256; }
static size_t lattice_table_bytes(int n_genomes, int nk) { return round256((size_t)nk * kLatValues * sizeof(uint32_t) << n_genomes); }
static size_t lattice_slab_bytes(const LatticeGeometry &geo, int n_genomes, int nk) {
    return round256((size_t)nk * geo.per_k * lattice_slab_words(geo.values, n_genomes) * sizeof(uint32_t));
}
size_t prefix_lattice_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk, int p) {
    const LatticeGeometry geo = lattice_geometry(n_genomes, nk, p);
    return lattice_table_bytes(n_genomes, nk) + lattice_slab_bytes(geo, n_genomes, nk) + round256((size_t)n_ord * n_steps * sizeof(uint32_t));
}

cudaError_t prefix_union_hist_lattice(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                                      int nk, int p, int final_only, uint32_t *d_hist, void *d_ws, cudaStream_t stream) {
    const size_t rows = (size_t)n_ord * (final_only ? 1 : n_steps) * nk;
    if (rows == 0) return cudaSuccess;
    const LatticeGeometry geo = lattice_geometry(n_genomes, nk, p);
    uint32_t *table = reinterpret_cast<uint32_t *>(d_ws);
    uint32_t *slabs = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(d_ws) + lattice_table_bytes(n_genomes, nk));
    uint32_t *sets = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(slabs) + lattice_slab_bytes(geo, n_genomes, nk));
    const size_t cols = (size_t)1 << n_genomes, row_bytes = cols * sizeof(uint32_t);
    cudaError_t e;
    if (geo.values < kLatValues - 1) {   // the spill rows v > V of every k
        e = cudaMemset2DAsync(table + (size_t)(geo.values + 1) * cols, kLatValues * row_bytes, 0,
                              (size_t)(kLatValues - 1 - geo.values) * row_bytes, (size_t)nk, stream);
        if (e != cudaSuccess) return e;
    }
    const size_t smem = lattice_slab_words(geo.values, n_genomes) * sizeof(uint32_t);
    const int nw = (n_genomes + 3) / 4;
    auto fn = nw == 1 ? lattice_levels_kernel<1> : nw == 2 ? lattice_levels_kernel<2> : lattice_levels_kernel<3>;
    if ((e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    DD_COUNT_LAUNCH(), fn<<<(unsigned)(geo.per_k * nk), kLatThreads, smem, stream>>>(d_regs, n_genomes, nk, p, geo.per_k, geo.values,
                                                                                     slabs, table);
    DD_COUNT_LAUNCH(), lattice_prefix_kernel<<<dim3((unsigned)((cols + 255) / 256), (unsigned)nk), 256, 0, stream>>>(
        slabs, table, n_genomes, geo.per_k, geo.values);
    DD_COUNT_LAUNCH(), lattice_sets_kernel<<<(n_ord + 255) / 256, 256, 0, stream>>>(d_order, n_ord, n_steps, n_genomes, sets);
    DD_COUNT_LAUNCH(), lattice_zeta_kernel<<<dim3(kLatValues - 1, (unsigned)nk), 256, cols * sizeof(uint32_t), stream>>>(
        table, sets, n_ord, n_steps, n_genomes, nk, final_only, d_hist);
    DD_COUNT_LAUNCH(), lattice_finish_kernel<<<(unsigned)((rows * 32 + 255) / 256), 256, 0, stream>>>(d_hist, rows, p);
    return cudaGetLastError();
}

}  // namespace dd
