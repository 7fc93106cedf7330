// card.cu -- K3 (unions / progressive prefix unions), K4 (register histogram + Ertl MLE) and the
// K6 all-pairs shape.  All three are HBM/L2-streaming kernels over u8 register arrays.
//
//   dashing union -z -o OUT in...      reference lib/sketch_classes.py:368-373   -> union_max_kernel
//   dashing card --presketched p...    reference lib/sketch_classes.py:306-321   -> hist_kernel + mle_kernel
//   progressive unions                 reference lib/huffman_dandd.py:624-663    -> prefix_union_kernel
//   pairwise two-leaf spiders          reference lib/huffman_dandd.py:666-695    -> prefix_union_kernel (2 steps)
//
// Histograms use thread-private counters in shared memory laid out [bin][thread]: a warp's 32
// increments land in 32 different banks, so they cost two conflict-free shared accesses each
// instead of a serialised shared-memory atomic (register values concentrate in a handful of bins,
// the worst case for atomics).
#include <cuda_runtime.h>

#include "common.cuh"
#include "hist.cuh"
#include "kernels.cuh"

namespace dd {

// -------------------------------------------------------------------------------------------------
// K4a: histogram of u8 registers.  grid (slices, nsk); a thread counts at most 240 registers
// between flushes.
// -------------------------------------------------------------------------------------------------
constexpr int kHistVecPerFlush = 15;  // 15 x 16 registers = 240 <= 255

__global__ void __launch_bounds__(kPhThreads)
hist_kernel(const uint8_t *__restrict__ regs, int p, uint32_t *__restrict__ hist) {
    __shared__ __align__(16) uint8_t s_hist[kPhBytes];
    const uint32_t slot = ph_slot();
    const size_t m = (size_t)1 << p;
    const int sk = blockIdx.y;
    uint32_t *g_hist = hist + (size_t)sk * DD_HIST_BINS;
    const uint4 *src = reinterpret_cast<const uint4 *>(regs + (size_t)sk * m);
    const size_t nvec = m / 16;
    const size_t per = (nvec + gridDim.x - 1) / gridDim.x;
    const size_t v0 = (size_t)blockIdx.x * per, v1 = min(nvec, v0 + per);
    for (size_t base = v0; base < v1; base += (size_t)kPhThreads * kHistVecPerFlush) {
        ph_zero(s_hist);
        __syncthreads();
#pragma unroll 5
        for (int i = 0; i < kHistVecPerFlush; ++i) {
            const size_t v = base + (size_t)i * kPhThreads + threadIdx.x;
            if (v < v1) {
                const uint4 x = __ldg(src + v);
                ph_add_word(s_hist, slot, x.x);
                ph_add_word(s_hist, slot, x.y);
                ph_add_word(s_hist, slot, x.z);
                ph_add_word(s_hist, slot, x.w);
            }
        }
        __syncthreads();
        ph_flush(s_hist, g_hist);
        __syncthreads();
    }
}

// -------------------------------------------------------------------------------------------------
// K4b: Ertl MLE, one WARP per sketch.  dd::ertl_mle (common.cuh) walks the ranks one after another
// with a doubling identity -- ~45 dependent f64 divisions per secant step, ~10 us for a lone thread.
// Here lane L owns ranks L and L+32: it evaluates h(t) = 1 - t/(e^t - 1) at t = x 2^-j directly
// (Taylor series below 2^-3, expm1 above) and the weighted sum is a butterfly reduction, so a
// secant step is one expm1 deep.  Same equation, same starting point, same stopping rule; the
// results differ from the sequential form by rounding only (<= 1e-14 relative, tests/ pin 1e-9).
// -------------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}
__device__ __forceinline__ double mle_h(double t) {
    if (t < 0.125) {
        const double y = 0.5 * t, y2 = y * y;
        return y - y2 * (1.0 / 3.0 - y2 * (1.0 / 45.0 - y2 * (1.0 / 472.5 - y2 * (1.0 / 4725.0 - y2 * (1.0 / 46777.5)))));
    }
    return 1.0 - t / expm1(t);
}
// T = uint32_t: integer histograms; T = double: fractional ones (mean histograms, K14).  The arithmetic is the same
// for both: every count is read as a double.
template <typename T>
__device__ double ertl_mle_warp(T c_lo, T c_hi, int p, int lane) {
    const unsigned full = 0xffffffffu;
    const int q = 64 - p;
    const double m = ldexp(1.0, p);
    auto count_at = [&](int j) { return __shfl_sync(full, j < 32 ? c_lo : c_hi, j & 31); };
    const double c0 = (double)count_at(0), ctop_reg = (double)count_at(q + 1);
    if (ctop_reg == m) return INFINITY;  // every register saturated
    unsigned long long nz = (unsigned long long)__ballot_sync(full, c_lo != T(0)) |
                            ((unsigned long long)__ballot_sync(full, c_hi != T(0)) << 32);
    if (q + 2 < 64) nz &= (1ull << (q + 2)) - 1ull;
    if (nz == 0ull) return nan("");      // not a histogram of 2^p registers
    const int lo = __ffsll((long long)nz) - 1, hi = 63 - __clzll((long long)nz);
    const int jlo = lo < 1 ? 1 : lo, jhi = hi > q ? q : hi;
    const double occupied = m - c0;
    if (occupied == 0.0 || jhi < jlo) return 0.0;  // empty sketch
    const double c_jhi = (double)count_at(jhi);
    const double ctop = ctop_reg + c_jhi;
    // my two ranks and their weights in z (plain counts) and in g (the top rank carries ctop)
    const int j1 = lane, j2 = lane + 32;
    const bool in1 = j1 >= jlo && j1 <= jhi, in2 = j2 >= jlo && j2 <= jhi;
    const double n1 = in1 ? (double)c_lo : 0.0, n2 = in2 ? (double)c_hi : 0.0;
    const double w1 = in1 ? (j1 == jhi ? ctop : n1) : 0.0, w2 = in2 ? (j2 == jhi ? ctop : n2) : 0.0;
    const double z = warp_sum_f64(ldexp(n1, -j1) + ldexp(n2, -j2));
    const double a = z + c0;
    const double b = z + ldexp(ctop_reg, -q);
    double x = (b <= 1.5 * a) ? occupied / (0.5 * b + a) : occupied / b * log1p(b / a);
    double step = x, g_prev = 0.0;
    const double tol = 1e-2 / sqrt(m);
    while (step > x * tol) {  // warp-uniform: every lane holds the same x and step
        double part = 0.0;
        if (in1) part += w1 * mle_h(ldexp(x, -j1));
        if (in2) part += w2 * mle_h(ldexp(x, -j2));
        const double g = warp_sum_f64(part) + x * a;
        if (g_prev < g && g <= occupied) step *= (g - occupied) / (g_prev - g);
        else step = 0.0;
        x += step;
        g_prev = g;
    }
    return x * m;
}

constexpr int kMleWarps = 4;
template <typename T>
__global__ void __launch_bounds__(32 * kMleWarps)
mle_kernel(const T *__restrict__ hist, int nsk, int p, double *__restrict__ cards) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * kMleWarps + (threadIdx.x >> 5);
    if (i >= nsk) return;  // whole warps leave together
    const T *row = hist + (size_t)i * DD_HIST_BINS;
    const double card = ertl_mle_warp(row[lane], row[lane + 32], p, lane);
    if (lane == 0) cards[i] = card;
}

// -------------------------------------------------------------------------------------------------
// K3a: n-ary union, element-wise max over a device array of pointers
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
union_max_kernel(const uint8_t *const *__restrict__ in, int n_in, size_t len, uint8_t *__restrict__ out) {
    const size_t nvec = len / 16;
    for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (size_t)gridDim.x * blockDim.x) {
        uint4 acc = make_uint4(0, 0, 0, 0);
        for (int j = 0; j < n_in; ++j) {
            const uint4 x = __ldg(reinterpret_cast<const uint4 *>(in[j]) + v);
            acc.x = __vmaxu4(acc.x, x.x);
            acc.y = __vmaxu4(acc.y, x.y);
            acc.z = __vmaxu4(acc.z, x.z);
            acc.w = __vmaxu4(acc.w, x.w);
        }
        reinterpret_cast<uint4 *>(out)[v] = acc;
    }
    // tail (len not a multiple of 16)
    for (size_t i = nvec * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < len;
         i += (size_t)gridDim.x * blockDim.x) {
        uint8_t a = 0;
        for (int j = 0; j < n_in; ++j) a = max(a, in[j][i]);
        out[i] = a;
    }
}

// -------------------------------------------------------------------------------------------------
// K3b: progressive prefix unions with fused histograms.
// Each thread keeps the running max of 128 registers (8 x uint4) in registers while the members of
// a set stream past; after every step the CTA histograms its 32 KiB slice of the running union with
// thread-private byte counters and adds the bin totals to the global row of that (set, step).
// (An incremental variant that only moved the counters of changed registers was measured 1.6x
// SLOWER: under SIMT a byte position is processed as soon as one lane of the warp changed, so
// nothing is skipped and every change costs two read-modify-writes -- profiles/r01_notes.md.)
// -------------------------------------------------------------------------------------------------
constexpr int kPfxThreads = kPhThreads;
constexpr int kPfxVec = 8;                                 // uint4 per thread (128 registers <= 255)
constexpr int kPfxSliceBytes = kPfxThreads * kPfxVec * 16; // 32 KiB

// kPtrTable = false: members are genome indices into regs[n_genomes][nk][2^p], grid (n_ord, slices, nk)
// kPtrTable = true : members are device pointers to 2^p-byte sketches,      grid (n_sets, slices, 1)
// The ordering / set index is the FASTEST grid dimension on purpose: the CTAs that are resident
// together then work on the same register slice of the same genomes under different orderings, so
// all but the first read of a slice hit in L2 (ncu, before: L2 hit rate 2 %, 8.3 GB from DRAM per
// launch for 30 orderings of 12 genomes; the data itself is only 276 MiB).
template <bool kPtrTable>
__global__ void __launch_bounds__(kPfxThreads)
prefix_union_kernel(const uint8_t *__restrict__ regs, const int32_t *__restrict__ order,
                    const uint8_t *const *__restrict__ members, int n_steps, int n_genomes, int nk, int p,
                    int final_only, uint32_t *__restrict__ hist, uint8_t *__restrict__ unions) {
    __shared__ __align__(16) uint8_t s_hist[kPhBytes];
    const uint32_t slot = ph_slot();
    const size_t m = (size_t)1 << p;
    const int o = kPtrTable ? 0 : (int)blockIdx.x;
    const int k = kPtrTable ? (int)blockIdx.x : (int)blockIdx.z;   // pointer mode: k is the set index
    const size_t slice0 = (size_t)blockIdx.y * kPfxSliceBytes;
    uint4 run[kPfxVec];
#pragma unroll
    for (int q = 0; q < kPfxVec; ++q) run[q] = make_uint4(0, 0, 0, 0);

    for (int step = 0; step < n_steps; ++step) {
        const uint8_t *src = nullptr;
        if (kPtrTable) {
            src = members[(size_t)k * n_steps + step];
        } else {
            const int g = order[(size_t)o * n_steps + step];
            if (g >= 0 && g < n_genomes) src = regs + ((size_t)g * nk + k) * m;
        }
        if (src) {
            src += slice0;
#pragma unroll
            for (int q = 0; q < kPfxVec; ++q) {
                const size_t off = ((size_t)q * kPfxThreads + threadIdx.x) * 16;
                if (slice0 + off < m) {
                    const uint4 x = __ldg(reinterpret_cast<const uint4 *>(src + off));
                    run[q].x = __vmaxu4(run[q].x, x.x);
                    run[q].y = __vmaxu4(run[q].y, x.y);
                    run[q].z = __vmaxu4(run[q].z, x.z);
                    run[q].w = __vmaxu4(run[q].w, x.w);
                }
            }
        }
        if (final_only && step != n_steps - 1) continue;
        const size_t row = kPtrTable ? (final_only ? (size_t)k : (size_t)k * n_steps + step)
                                     : (final_only ? (size_t)o * nk + k : ((size_t)o * n_steps + step) * nk + k);
        ph_zero(s_hist);
        __syncthreads();
#pragma unroll
        for (int q = 0; q < kPfxVec; ++q) {
            const size_t off = ((size_t)q * kPfxThreads + threadIdx.x) * 16;
            if (slice0 + off < m) {
                ph_add_word(s_hist, slot, run[q].x);
                ph_add_word(s_hist, slot, run[q].y);
                ph_add_word(s_hist, slot, run[q].z);
                ph_add_word(s_hist, slot, run[q].w);
                if (unions) *reinterpret_cast<uint4 *>(unions + row * m + slice0 + off) = run[q];
            }
        }
        __syncthreads();
        ph_flush(s_hist, hist + row * DD_HIST_BINS);
        __syncthreads();
    }
}

// -------------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------------
int g_prefix_planes = 1;

cudaError_t card_hist(const uint8_t *d_regs, int nsk, int p, uint32_t *d_hist, cudaStream_t stream) {
    cudaError_t e = cudaMemsetAsync(d_hist, 0, (size_t)nsk * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    if (nsk == 0) return cudaSuccess;
    const size_t m = (size_t)1 << p;
    // one flush round (256 threads x 240 registers = 60 KiB) per CTA where the sketch is big enough
    int slices = (int)((m + (size_t)kPhThreads * kHistVecPerFlush * 16 - 1) / ((size_t)kPhThreads * kHistVecPerFlush * 16));
    if (slices < 1) slices = 1;
    for (int s0 = 0; s0 < nsk; s0 += 65535) {  // gridDim.y limit
        const int cnt = nsk - s0 < 65535 ? nsk - s0 : 65535;
        DD_COUNT_LAUNCH(), hist_kernel<<<dim3(slices, cnt), kPhThreads, 0, stream>>>(d_regs + (size_t)s0 * m, p,
                                                                    d_hist + (size_t)s0 * DD_HIST_BINS);
    }
    return cudaGetLastError();
}

cudaError_t mle_from_hist(const uint32_t *d_hist, int nsk, int p, double *d_cards, cudaStream_t stream) {
    if (nsk == 0) return cudaSuccess;
    DD_COUNT_LAUNCH(), mle_kernel<<<(nsk + kMleWarps - 1) / kMleWarps, 32 * kMleWarps, 0, stream>>>(d_hist, nsk, p, d_cards);
    return cudaGetLastError();
}

cudaError_t mle_from_hist_f64(const double *d_hist, int nsk, int p, double *d_cards, cudaStream_t stream) {
    if (nsk == 0) return cudaSuccess;
    DD_COUNT_LAUNCH(), mle_kernel<<<(nsk + kMleWarps - 1) / kMleWarps, 32 * kMleWarps, 0, stream>>>(d_hist, nsk, p, d_cards);
    return cudaGetLastError();
}

cudaError_t union_max(const uint8_t *const *d_in, int n_in, size_t len, uint8_t *d_out, cudaStream_t stream) {
    if (len == 0) return cudaSuccess;
    size_t blocks = (len / 16 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 16) blocks = 148 * 16;
    DD_COUNT_LAUNCH(), union_max_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_in, n_in, len, d_out);
    return cudaGetLastError();
}

cudaError_t prefix_union_hist(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                              int nk, int p, int final_only, uint32_t *d_hist, uint8_t *d_unions,
                              cudaStream_t stream) {
    const int out_steps = final_only ? 1 : n_steps;
    const size_t rows = (size_t)n_ord * out_steps * nk;
    cudaError_t e = cudaMemsetAsync(d_hist, 0, rows * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    if (rows == 0) return cudaSuccess;
    const size_t m = (size_t)1 << p;
    const unsigned slices = (unsigned)((m + kPfxSliceBytes - 1) / kPfxSliceBytes);
    DD_COUNT_LAUNCH(), prefix_union_kernel<false><<<dim3((unsigned)n_ord, slices, (unsigned)nk), kPfxThreads, 0, stream>>>(
        d_regs, d_order, nullptr, n_steps, n_genomes, nk, p, final_only, d_hist, d_unions);
    return cudaGetLastError();
}

// Pointer-table form: set s is the list members[s][0..n_steps) of device sketches (NULL = skip).
// With nk := n_sets and one "ordering" the row arithmetic of the kernel gives row = s (final_only)
// or s * n_steps + step.
cudaError_t union_sets_hist(const uint8_t *const *d_members, int n_sets, int n_steps, int p, int final_only,
                            uint32_t *d_hist, uint8_t *d_unions, cudaStream_t stream) {
    const int out_steps = final_only ? 1 : n_steps;
    const size_t rows = (size_t)n_sets * out_steps;
    cudaError_t e = cudaMemsetAsync(d_hist, 0, rows * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    if (rows == 0) return cudaSuccess;
    const size_t m = (size_t)1 << p;
    const unsigned slices = (unsigned)((m + kPfxSliceBytes - 1) / kPfxSliceBytes);
    DD_COUNT_LAUNCH(), prefix_union_kernel<true><<<dim3((unsigned)n_sets, slices, 1), kPfxThreads, 0, stream>>>(
        nullptr, nullptr, d_members, n_steps, 0, n_sets, p, final_only, d_hist, d_unions);
    return cudaGetLastError();
}

}  // namespace dd
