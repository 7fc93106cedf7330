// spectrum.cu -- K14: the register sharing spectrum, one read of the registers.
//
//   helpers/spectrum.py --tool dashing: the growth curve averaged over all n! orderings from HLL sketches
//
// For register r and value v >= 1 let c_v(r) = #{g : x_g(r) >= v}.  The union of a subset S has max_{g in S} x_g(r) >= v
// exactly when S meets that set of c_v(r) genomes, and prefix m of a uniformly random ordering is a uniformly random
// m-subset, so the mean register histogram of the m-prefix union over all orderings follows from
//     T[k][v][c] = #{r : c_v(r) = c}      (v = 1..63, c = 1..n)
// with the weights of the exact spectrum (helpers/spectrum.py hit_weights).  Row v sums to the union's cnt>=(v), bit for
// bit: values are clamped at 63 as hist_kernel clamps them (ph_bin).
//
// A thread owns 4 registers of one k (one u32 word per genome) and streams the n genomes, 32 loads in flight, into
// thread-private u16 value counters in shared memory ([register][value][thread], every lane of a warp on its own bank,
// no atomics).  Then it walks each register's counters from its own max down to its own min: the level of distinct
// value u_i covers v in (u_{i+1}, u_i] with c_i genomes at or above u_i, which in difference form over v is
// D[u_{i+1} + 1][c_i] += 1 and D[u_i + 1][c_i] -= 1 (the second dropped at u_i = 63) -- lattice.cu's level walk with a
// count in place of the mask.  The lowest level of almost every register (c = n from v = 1) is counted in a lane
// register and warp-reduced.  D goes to a per-CTA shared table: the whole [64][n] when it takes <= 32 KiB, else the
// c = n and c = 1 columns, and the other cells are L2 reductions into the [nk][64][n] workspace.  A running sum over v,
// one thread per (k, c), adds T into the caller's table, so calls over disjoint register ranges add up.
#include <cuda_runtime.h>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr int kSpThreads = 128;
constexpr int kSpRegs = 4;        // registers per thread: one u32 word of every genome
constexpr int kSpBatch = 32;      // genome loads in flight per thread
constexpr int kSpValues = DD_HIST_BINS;
constexpr size_t kSpCounterBytes = (size_t)kSpRegs * kSpValues * kSpThreads * sizeof(uint16_t);   // 64 KiB
constexpr size_t kSpSmemTableBytes = 32 << 10;

// u16 slot of this thread in a counter row of 128: lane l of warp w owns half (w >> 1) of word l + 32 (w & 1), so the
// 32 lanes of a warp touch 32 consecutive words
__device__ __forceinline__ uint32_t sp_slot() {
    return (((threadIdx.x & 31u) + (((threadIdx.x >> 5) & 1u) << 5)) << 1) | (threadIdx.x >> 6);
}

// grid (CTAs per k, nk).  kWhole: the whole per-CTA table [64][n] in shared memory, else [64][2] (c = n, c = 1).
template <bool kWhole>
__global__ void __launch_bounds__(kSpThreads)
register_spectrum_kernel(const uint8_t *__restrict__ regs, int n, int nk, int p, uint64_t reg_begin, uint64_t nword,
                         uint32_t *__restrict__ diff) {
    extern __shared__ __align__(16) uint8_t s_mem[];
    uint16_t *cnt = reinterpret_cast<uint16_t *>(s_mem);
    uint32_t *tab = reinterpret_cast<uint32_t *>(s_mem + kSpCounterBytes);
    const int cols = kWhole ? n : 2;
    for (int i = threadIdx.x; i < (int)(kSpCounterBytes / 16); i += kSpThreads) reinterpret_cast<uint4 *>(s_mem)[i] = make_uint4(0, 0, 0, 0);
    for (int i = threadIdx.x; i < kSpValues * cols; i += kSpThreads) tab[i] = 0u;
    __syncthreads();

    const int k = blockIdx.y;
    const size_t m = (size_t)1 << p, gstride = (size_t)nk * m / 4;   // in words
    const uint32_t *base = reinterpret_cast<const uint32_t *>(regs + (size_t)k * m + reg_begin);
    uint32_t *dk = diff + (size_t)k * kSpValues * n;
    const uint32_t slot = sp_slot();
    uint32_t base1 = 0;   // registers whose lowest level is c = n from v = 1: T[1][n] += 1, too hot for a shared atomic
    auto update = [&](int v, int c, uint32_t delta) {
        if (kWhole) atomicAdd(&tab[v * n + c - 1], delta);
        else if (c == n) atomicAdd(&tab[2 * v], delta);
        else if (c == 1) atomicAdd(&tab[2 * v + 1], delta);
        else atomicAdd(&dk[(size_t)v * n + c - 1], delta);
    };

    for (uint64_t w = (uint64_t)blockIdx.x * kSpThreads + threadIdx.x; w < nword; w += (uint64_t)gridDim.x * kSpThreads) {
        const uint32_t *src = base + w;
        uint32_t lo = 0x3f3f3f3fu, hi = 0u;
        for (int g0 = 0; g0 < n; g0 += kSpBatch) {
            uint32_t x[kSpBatch];
#pragma unroll
            for (int b = 0; b < kSpBatch; ++b) x[b] = g0 + b < n ? __ldcs(src + (size_t)(g0 + b) * gstride) : 0u;
#pragma unroll
            for (int b = 0; b < kSpBatch; ++b) {
                if (g0 + b >= n) break;
                const uint32_t v = __vminu4(x[b], 0x3f3f3f3fu);
                lo = __vminu4(lo, v);
                hi = __vmaxu4(hi, v);
                // four different rows: load all four counters, then store, so the increments do not wait on each other
                uint16_t *a0 = cnt + (0 * kSpValues + (v & 0xffu)) * kSpThreads + slot;
                uint16_t *a1 = cnt + (1 * kSpValues + ((v >> 8) & 0xffu)) * kSpThreads + slot;
                uint16_t *a2 = cnt + (2 * kSpValues + ((v >> 16) & 0xffu)) * kSpThreads + slot;
                uint16_t *a3 = cnt + (3 * kSpValues + (v >> 24)) * kSpThreads + slot;
                const uint16_t c0 = *a0, c1 = *a1, c2 = *a2, c3 = *a3;
                *a0 = c0 + 1;
                *a1 = c1 + 1;
                *a2 = c2 + 1;
                *a3 = c3 + 1;
            }
        }
#pragma unroll
        for (int j = 0; j < kSpRegs; ++j) {
            const int vlo = (int)((lo >> (8 * j)) & 0xffu), vhi = (int)((hi >> (8 * j)) & 0xffu);
            uint16_t *col = cnt + j * kSpValues * kSpThreads + slot;
            int above = 0, up = 0;   // genomes at or above the current level, and its value (0: no level yet)
            for (int v = vhi; v >= vlo; --v) {
                const int h = col[v * kSpThreads];
                if (!h) continue;
                col[v * kSpThreads] = 0;   // the counters are clean again for the next word
                if (up) {                  // level (up, above) covers (v, up]
                    update(v + 1, above, 1u);
                    if (up < kSpValues - 1) update(up + 1, above, 0xffffffffu);
                }
                above += h;
                up = v;
            }
            if (vlo > 0) {                 // the lowest level: every genome, (0, vlo]
                ++base1;
                if (vlo < kSpValues - 1) update(vlo + 1, n, 0xffffffffu);
            }
        }
    }
    base1 = __reduce_add_sync(0xffffffffu, base1);
    if ((threadIdx.x & 31) == 0 && base1) atomicAdd(kWhole ? &tab[n + n - 1] : &tab[2], base1);
    __syncthreads();
    for (int i = threadIdx.x; i < kSpValues * cols; i += kSpThreads) {
        const uint32_t c = tab[i];
        if (!c) continue;
        const int v = i / cols, j = i % cols;
        atomicAdd(&dk[(size_t)v * n + (kWhole ? j : j == 0 ? n - 1 : 0)], c);
    }
}

// D -> T: running sum over v, one thread per (k, c), added into the caller's table
__global__ void __launch_bounds__(256)
register_spectrum_finish_kernel(const uint32_t *__restrict__ diff, int n, uint32_t *__restrict__ spec) {
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c >= n) return;
    const size_t off = (size_t)blockIdx.y * kSpValues * n + c;
    uint32_t run = 0u;
    for (int v = 1; v < kSpValues; ++v) {
        run += diff[off + (size_t)v * n];
        spec[off + (size_t)v * n] += run;
    }
}

size_t register_spectrum_workspace_bytes(int n_genomes, int nk) {
    return (size_t)nk * kSpValues * n_genomes * sizeof(uint32_t);
}

cudaError_t register_spectrum(const uint8_t *d_regs, int n_genomes, int nk, int p, uint64_t reg_begin, uint64_t reg_end,
                              uint32_t *d_spec, void *d_ws, cudaStream_t stream) {
    const uint64_t nword = (reg_end - reg_begin) / 4;
    if (nword == 0) return cudaSuccess;
    uint32_t *diff = static_cast<uint32_t *>(d_ws);
    cudaError_t e = cudaMemsetAsync(diff, 0, register_spectrum_workspace_bytes(n_genomes, nk), stream);
    if (e != cudaSuccess) return e;
    const bool whole = (size_t)kSpValues * n_genomes * sizeof(uint32_t) <= kSpSmemTableBytes;
    const size_t smem = kSpCounterBytes + (whole ? (size_t)kSpValues * n_genomes : (size_t)kSpValues * 2) * sizeof(uint32_t);
    const void *fn = whole ? reinterpret_cast<const void *>(register_spectrum_kernel<true>)
                           : reinterpret_cast<const void *>(register_spectrum_kernel<false>);
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int dev = 0, sms = 0, per_sm = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return e;
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return e;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kSpThreads, smem)) != cudaSuccess) return e;
    // one wave of resident CTAs over all k (rounded down: a second, partial wave would double the time); each CTA
    // flushes its shared table once
    size_t per_k = (size_t)sms * (per_sm > 0 ? per_sm : 1) / nk, most = (nword + kSpThreads - 1) / kSpThreads;
    if (per_k < 1) per_k = 1;
    if (per_k > most) per_k = most;
    const dim3 grid((unsigned)per_k, (unsigned)nk);
    if (whole)
        DD_COUNT_LAUNCH(), register_spectrum_kernel<true><<<grid, kSpThreads, smem, stream>>>(d_regs, n_genomes, nk, p, reg_begin,
                                                                                             nword, diff);
    else
        DD_COUNT_LAUNCH(), register_spectrum_kernel<false><<<grid, kSpThreads, smem, stream>>>(d_regs, n_genomes, nk, p,
                                                                                              reg_begin, nword, diff);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    DD_COUNT_LAUNCH(), register_spectrum_finish_kernel<<<dim3((unsigned)((n_genomes + 255) / 256), (unsigned)nk), 256, 0,
                                                         stream>>>(diff, n_genomes, d_spec);
    return cudaGetLastError();
}

}  // namespace dd
