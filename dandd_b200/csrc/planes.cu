// planes.cu -- K3 on bit-sliced sketches: progressive prefix unions with fused histograms.
//
// The byte kernel (card.cu) spends ~7 instructions per register per step, almost all of it in the
// thread-private histogram (extract byte, address, LDS, add, STS).  Here a sketch is first
// transposed once per call into 6 bit-planes: plane b, word g holds bit b of registers 32g..32g+31
// (ranks are <= 64-p+1 < 64).  On planes
//   * the running max of two sketches is a bit-serial compare-and-select, 2 LOP3 per plane
//     (12 per 32 registers), and
//   * "how many registers equal v" is AND-ing the six planes (or their complements) and a POPC:
//     1.5 LOP3 + POPC + IADD per value per 32 registers.
// Values are counted in four buckets of 16 (top two planes); a bucket nobody in the warp populates
// is skipped, a thinly populated one is walked register by register, a dense one runs the unrolled
// 16-value loop -- so the cost follows the actual value range of the data and every register is
// counted exactly once.  ~3.3 instructions per register per step instead of ~7.
//
// Same contract as prefix_union_hist (index mode, no materialised unions); replaces the reference's
// n(n+1)/2 `dashing union` + `dashing card` processes per ordering (lib/huffman_dandd.py:624-663).
#include <cuda_runtime.h>

#include <utility>

#include "common.cuh"
#include "kernels.cuh"

namespace dd {

constexpr int kPlThreads = 64;   // measured (bench prefix unions): 64 -> 1.51 ms, 128 -> 1.54, 256 -> 1.60, 512 -> 1.74
constexpr int kPlanes = 6;

// ---- u8 registers -> bit planes -------------------------------------------------------------------
// One thread per group of 32 registers: two 128-bit loads, then a SWAR transpose -- for each of the
// six bits, the four bytes of a word give a nibble with one mask, one multiply and one shift
// (same gather as dd::gather_bit7), eight nibbles make the plane word.  Stores are one word per
// plane per thread, contiguous across the warp.
__device__ __forceinline__ uint32_t bit_nibble(uint32_t w, int b) {   // bit b of bytes 0..3 -> bits 0..3
    return ((((w >> b) & 0x01010101u) * 0x00204081u) >> 21) & 0xFu;
}
__global__ void __launch_bounds__(256)
to_planes_kernel(const uint8_t *__restrict__ regs, uint32_t *__restrict__ planes, int p, size_t total_groups) {
    const size_t ngroups = (size_t)1 << (p - 5);
    for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < total_groups; g += (size_t)gridDim.x * blockDim.x) {
        const uint4 lo = __ldg(reinterpret_cast<const uint4 *>(regs) + 2 * g);
        const uint4 hi = __ldg(reinterpret_cast<const uint4 *>(regs) + 2 * g + 1);
        const uint32_t w[8] = {__vminu4(lo.x, 0x3f3f3f3fu), __vminu4(lo.y, 0x3f3f3f3fu), __vminu4(lo.z, 0x3f3f3f3fu),
                               __vminu4(lo.w, 0x3f3f3f3fu), __vminu4(hi.x, 0x3f3f3f3fu), __vminu4(hi.y, 0x3f3f3f3fu),
                               __vminu4(hi.z, 0x3f3f3f3fu), __vminu4(hi.w, 0x3f3f3f3fu)};
        const size_t sketch = g >> (p - 5), group = g & (ngroups - 1);
        uint32_t *dst = planes + sketch * kPlanes * ngroups + group;
#pragma unroll
        for (int b = 0; b < kPlanes; ++b) {
            uint32_t word = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) word |= bit_nibble(w[j], b) << (4 * j);
            dst[(size_t)b * ngroups] = word;
        }
    }
}

// running max of bit-sliced values: R = max(R, X).  "R < X" is the borrow of R - X, carried from the
// least significant plane up: where the bits differ the higher plane decides, where they agree the
// verdict so far stands -- a three-input function, one LOP3 per plane; then one select per plane.
__device__ __forceinline__ void plane_max(uint32_t (&R)[kPlanes], const uint32_t (&X)[kPlanes]) {
    uint32_t lt = 0u;
#pragma unroll
    for (int b = 0; b < kPlanes; ++b) lt = (~R[b] & X[b]) | (~(R[b] ^ X[b]) & lt);
#pragma unroll
    for (int b = 0; b < kPlanes; ++b) R[b] = (X[b] & lt) | (R[b] & ~lt);
}

// Counting a dense bucket (16 values sharing the two top planes).  The four combinations of planes 0
// and 1 inside the bucket are formed once per 32-register chunk (one LOP3 each); a value's registers are
// then one more LOP3 away (that combination AND planes 2, 3 in the right polarity) -- 1.25 LOP3 per
// (value, chunk) instead of 4.
struct BucketLow2 {
    uint32_t m[4][4];   // [chunk][value & 3]
};
__device__ __forceinline__ BucketLow2 bucket_low2(const uint32_t (&P)[4][kPlanes], const uint32_t (&mem)[4]) {
    BucketLow2 b;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        b.m[c][0] = mem[c] & ~P[c][0] & ~P[c][1];
        b.m[c][1] = mem[c] & P[c][0] & ~P[c][1];
        b.m[c][2] = mem[c] & ~P[c][0] & P[c][1];
        b.m[c][3] = mem[c] & P[c][0] & P[c][1];
    }
    return b;
}
template <int J>
__device__ __forceinline__ uint32_t count_value(const uint32_t (&P)[4][kPlanes], const BucketLow2 &b) {
    uint32_t n = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c)
        n += __popc(b.m[c][J & 3] & ((J & 4) ? P[c][2] : ~P[c][2]) & ((J & 8) ? P[c][3] : ~P[c][3]));
    return n;
}

// Two values per warp reduction (a lane holds at most 128 registers, so a warp sum fits 16 bits);
// lane J keeps the warp's count of value J, and the sixteen lanes issue one shared-memory add
// together at the end -- no branch, vote or atomic per value.
template <int J>
__device__ __forceinline__ uint32_t count_pair(const uint32_t (&P)[4][kPlanes], const BucketLow2 &b) {
    return __reduce_add_sync(0xffffffffu, count_value<J>(P, b) | (count_value<J + 1>(P, b) << 16));
}

template <int... Js>
__device__ __forceinline__ void count_bucket_dense(std::integer_sequence<int, Js...>, const uint32_t (&P)[4][kPlanes],
                                                   const uint32_t (&mem)[4], uint32_t *s_cnt, int lane) {
    const BucketLow2 low = bucket_low2(P, mem);
    uint32_t mine = 0;
    (([&] {
         const uint32_t both = count_pair<2 * Js>(P, low);
         if (lane == 2 * Js) mine = both & 0xFFFFu;
         if (lane == 2 * Js + 1) mine = both >> 16;
     }()),
     ...);
    if (lane < 16 && mine) atomicAdd(&s_cnt[lane], mine);
}

__device__ __forceinline__ void count_bucket_sparse(const uint32_t (&P)[4][kPlanes], const uint32_t (&mem)[4],
                                                    uint32_t *s_cnt_all) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint32_t left = mem[c];
        while (left) {
            const int i = __ffs((int)left) - 1;
            left &= left - 1;
            uint32_t v = 0;
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) v |= ((P[c][b] >> i) & 1u) << b;
            atomicAdd(&s_cnt_all[v], 1u);
        }
    }
}

// ---- identical prefixes --------------------------------------------------------------------------
// Two orderings whose first s+1 entries are the same SET have the same union at step s (always true
// for the last step of permutations of one set, frequent at the first and last few steps of random
// ones): only the lowest-numbered ordering of each such class (among the first kDedupWindow orderings)
// counts, the others get a copy of its histogram row.  Sets are 64-bit masks, so this applies to n_genomes <= 64; beyond that every
// ordering is its own representative.
constexpr int kDedupWindow = 256;   // representatives are looked for among the first 256 orderings

__global__ void __launch_bounds__(1024)
prefix_dedup_kernel(const int32_t *__restrict__ order, int n_ord, int n_steps, int n_genomes,
                    unsigned long long *__restrict__ masks, int32_t *__restrict__ rep) {
    const int total = n_ord * n_steps;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int o = i / n_steps, st = i % n_steps;
        unsigned long long m = 0ull;
        for (int j = 0; j <= st; ++j) {
            const int g = order[(size_t)o * n_steps + j];
            if (g >= 0 && g < n_genomes && n_genomes <= 64) m |= 1ull << g;
        }
        masks[i] = m;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int o = i / n_steps, st = i % n_steps;
        int r = o;
        if (n_genomes <= 64) {
            const unsigned long long m = masks[i];
            const int qmax = o < kDedupWindow ? o : kDedupWindow;   // bounded search: linear in n_ord
            for (int q = 0; q < qmax; ++q)
                if (masks[(size_t)q * n_steps + st] == m) {
                    r = q;
                    break;
                }
        }
        rep[i] = r;
    }
}

// hist rows of non-representative (ordering, step) pairs <- the representative's rows
__global__ void prefix_copy_rows_kernel(const int32_t *__restrict__ rep, int n_ord, int n_steps, int nk, int final_only,
                                        uint32_t *__restrict__ hist) {
    const int out_steps = final_only ? 1 : n_steps;
    const size_t rows = (size_t)n_ord * out_steps * nk;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * DD_HIST_BINS; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / DD_HIST_BINS, bin = i % DD_HIST_BINS;
        const int k = (int)(row % nk);
        const int os = (int)(row / nk);  // o * out_steps + step'
        const int o = os / out_steps, st = final_only ? n_steps - 1 : os % out_steps;
        const int r = rep[(size_t)o * n_steps + st];
        if (r != o) {
            const size_t src = final_only ? (size_t)r * nk + k : ((size_t)r * n_steps + st) * nk + k;
            hist[i] = hist[src * DD_HIST_BINS + bin];
        }
    }
}

// grid (n_ord, slices, nk); a thread owns 4 groups (128 registers), a CTA 128 x kPlThreads registers.
// kCopyFirst: the first member is copied instead of max-ed with the all-zero start (pairs: half of
// their max work; for long orderings the extra branch costs more than the one saved step).
template <bool kCopyFirst>
__global__ void __launch_bounds__(kPlThreads, 1024 / kPlThreads)
prefix_union_planes_kernel(const uint32_t *__restrict__ planes, const int32_t *__restrict__ order, int n_steps,
                           int n_genomes, int nk, int p, int final_only, const int32_t *__restrict__ rep,
                           uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_cnt[DD_HIST_BINS];
    const size_t ngroups = (size_t)1 << (p - 5);
    const size_t nvec = ngroups >> 2;  // uint4 per plane
    const int o = blockIdx.x, k = blockIdx.z;
    const size_t vec = (size_t)blockIdx.y * kPlThreads + threadIdx.x;
    const bool owner = vec < nvec;
    const int lane = threadIdx.x & 31;
    uint32_t R[4][kPlanes];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int b = 0; b < kPlanes; ++b) R[c][b] = 0u;

    for (int step = 0; step < n_steps; ++step) {
        const int g = order[(size_t)o * n_steps + step];
        if (g >= 0 && g < n_genomes && owner) {
            const uint4 *src = reinterpret_cast<const uint4 *>(planes + ((size_t)g * nk + k) * kPlanes * ngroups);
            uint4 x[kPlanes];
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) x[b] = __ldg(src + (size_t)b * nvec + vec);
            if (kCopyFirst && step == 0) {  // max(0, X) = X
#pragma unroll
                for (int b = 0; b < kPlanes; ++b) {
                    R[0][b] = x[b].x;
                    R[1][b] = x[b].y;
                    R[2][b] = x[b].z;
                    R[3][b] = x[b].w;
                }
            } else {
                uint32_t X[kPlanes];
#pragma unroll
                for (int b = 0; b < kPlanes; ++b) X[b] = x[b].x;
                plane_max(R[0], X);
#pragma unroll
                for (int b = 0; b < kPlanes; ++b) X[b] = x[b].y;
                plane_max(R[1], X);
#pragma unroll
                for (int b = 0; b < kPlanes; ++b) X[b] = x[b].z;
                plane_max(R[2], X);
#pragma unroll
                for (int b = 0; b < kPlanes; ++b) X[b] = x[b].w;
                plane_max(R[3], X);
            }
        }
        if (final_only && step != n_steps - 1) continue;
        if (rep && rep[(size_t)o * n_steps + step] != o) continue;  // same set as an earlier ordering: row copied afterwards
        const size_t row = final_only ? (size_t)o * nk + k : ((size_t)o * n_steps + step) * nk + k;

        if (threadIdx.x < DD_HIST_BINS) s_cnt[threadIdx.x] = 0u;
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // bucket q: values 16q .. 16q+15
            uint32_t mem[4];
            uint32_t any = 0u, n = 0u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                mem[c] = owner ? (((q & 1) ? R[c][4] : ~R[c][4]) & ((q & 2) ? R[c][5] : ~R[c][5])) : 0u;
                any |= mem[c];
            }
            if (!__any_sync(0xffffffffu, any != 0u)) continue;  // nobody in the warp has such values
#pragma unroll
            for (int c = 0; c < 4; ++c) n += __popc(mem[c]);
            if (__any_sync(0xffffffffu, n > 12u)) count_bucket_dense(std::make_integer_sequence<int, 8>{}, R, mem, s_cnt + 16 * q, lane);
            else count_bucket_sparse(R, mem, s_cnt);
        }
        __syncthreads();
        if (threadIdx.x < DD_HIST_BINS) {
            const uint32_t c = s_cnt[threadIdx.x];
            if (c) atomicAdd(&hist[row * DD_HIST_BINS + threadIdx.x], c);
        }
        __syncthreads();
    }
}

// ---- pairs (K6) -----------------------------------------------------------------------------------
// The prefix kernel above gives every 8192-register slice of every (set, k) its own CTA and flushes a
// histogram per CTA.  For an all-pairs job -- half a million pairs x 23 k x 32 slices -- that is 4e8
// tiny CTAs whose fixed cost (start-up, two loads' latency, three barriers, a dozen global atomics)
// dwarfs the ~14k instructions of useful work.  Here ONE CTA owns a whole (pair, k): it walks all the
// slices, keeps the per-value counts of dense buckets in registers (lane J of a warp holds value J's
// running count), and writes the 64-bin row once.  grid = (pairs, Y, nk); Y > 1 only when there are too
// few pairs to fill the chip, in which case the rows are accumulated with atomics.
template <int... Js>
__device__ __forceinline__ uint32_t count_bucket_dense_reg(std::integer_sequence<int, Js...>, const uint32_t (&P)[4][kPlanes],
                                                           const uint32_t (&mem)[4], int lane) {
    const BucketLow2 low = bucket_low2(P, mem);
    uint32_t mine = 0;
    (([&] {
         const uint32_t both = count_pair<2 * Js>(P, low);
         if (lane == 2 * Js) mine = both & 0xFFFFu;
         if (lane == 2 * Js + 1) mine = both >> 16;
     }()),
     ...);
    return mine;
}

__global__ void __launch_bounds__(kPlThreads, 1024 / kPlThreads)
pair_union_planes_kernel(const uint32_t *__restrict__ planes, const int32_t *__restrict__ pairs, int n_genomes, int nk, int p,
                         uint32_t *__restrict__ hist) {
    __shared__ uint32_t s_cnt[DD_HIST_BINS];
    const size_t ngroups = (size_t)1 << (p - 5);
    const size_t nvec = ngroups >> 2;  // uint4 per plane
    const int pr = blockIdx.x, k = blockIdx.z;
    const int lane = threadIdx.x & 31;
    const int ga = pairs[2 * (size_t)pr], gb = pairs[2 * (size_t)pr + 1];
    const bool have_a = ga >= 0 && ga < n_genomes, have_b = gb >= 0 && gb < n_genomes;
    const uint4 *pa = reinterpret_cast<const uint4 *>(planes + ((size_t)(have_a ? ga : 0) * nk + k) * kPlanes * ngroups);
    const uint4 *pb = reinterpret_cast<const uint4 *>(planes + ((size_t)(have_b ? gb : 0) * nk + k) * kPlanes * ngroups);
    if (threadIdx.x < DD_HIST_BINS) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    uint32_t acc[4] = {0u, 0u, 0u, 0u};   // lane J < 16: registers equal to 16 q + J seen by this warp so far
    // every warp runs the same number of iterations (the warp-wide reductions need all lanes)
    const size_t stride = (size_t)gridDim.y * kPlThreads;
    for (size_t base = (size_t)blockIdx.y * kPlThreads; base < nvec; base += stride) {
        const size_t vec = base + threadIdx.x;
        const bool owner = vec < nvec;
        uint32_t R[4][kPlanes];
        uint4 xa[kPlanes], xb[kPlanes];
#pragma unroll
        for (int b = 0; b < kPlanes; ++b) {
            xa[b] = owner && have_a ? __ldg(pa + (size_t)b * nvec + vec) : make_uint4(0, 0, 0, 0);
            xb[b] = owner && have_b ? __ldg(pb + (size_t)b * nvec + vec) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int b = 0; b < kPlanes; ++b) {
            R[0][b] = xa[b].x;
            R[1][b] = xa[b].y;
            R[2][b] = xa[b].z;
            R[3][b] = xa[b].w;
        }
        {
            uint32_t X[kPlanes];
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) X[b] = xb[b].x;
            plane_max(R[0], X);
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) X[b] = xb[b].y;
            plane_max(R[1], X);
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) X[b] = xb[b].z;
            plane_max(R[2], X);
#pragma unroll
            for (int b = 0; b < kPlanes; ++b) X[b] = xb[b].w;
            plane_max(R[3], X);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // bucket q: values 16q .. 16q+15
            uint32_t mem[4];
            uint32_t any = 0u, n = 0u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                mem[c] = owner ? (((q & 1) ? R[c][4] : ~R[c][4]) & ((q & 2) ? R[c][5] : ~R[c][5])) : 0u;
                any |= mem[c];
            }
            if (!__any_sync(0xffffffffu, any != 0u)) continue;  // nobody in the warp has such values
#pragma unroll
            for (int c = 0; c < 4; ++c) n += __popc(mem[c]);
            if (__any_sync(0xffffffffu, n > 12u)) acc[q] += count_bucket_dense_reg(std::make_integer_sequence<int, 8>{}, R, mem, lane);
            else count_bucket_sparse(R, mem, s_cnt);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (lane < 16 && acc[q]) atomicAdd(&s_cnt[16 * q + lane], acc[q]);
    __syncthreads();
    if (threadIdx.x < DD_HIST_BINS) {
        const uint32_t c = s_cnt[threadIdx.x];
        uint32_t *cell = &hist[((size_t)pr * nk + k) * DD_HIST_BINS + threadIdx.x];
        if (gridDim.y == 1) *cell = c;           // the row is this CTA's alone
        else if (c) atomicAdd(cell, c);
    }
}

// ---- host side ----------------------------------------------------------------------------------
bool planes_supported(int p) { return p >= 12; }   // whole uint4s of groups per plane, >= 1 CTA of work
size_t planes_bytes(int64_t n_sketches, int p) { return (size_t)n_sketches * kPlanes * (((size_t)1 << p) / 8); }

static size_t dedup_bytes(int n_ord, int n_steps) {
    return (size_t)n_ord * n_steps * (sizeof(unsigned long long) + sizeof(int32_t));
}
// scratch of the register-input entry: [planes | identical-prefix masks | representatives], or the subset
// table of lattice.cu, whichever is larger where that path applies
size_t prefix_union_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk, int p) {
    const size_t pl = (planes_bytes((int64_t)n_genomes * nk, p) + 255) / 256 * 256;
    const size_t planes_path = pl + (dedup_bytes(n_ord, n_steps) + 255) / 256 * 256;
    const size_t lattice_path = lattice_supported(n_genomes, p) ? prefix_lattice_workspace_bytes(n_ord, n_steps, n_genomes, nk, p) : 0;
    return (planes_path > lattice_path ? planes_path : lattice_path) + 256;
}

cudaError_t to_planes(const uint8_t *d_regs, int64_t n_sketches, int p, uint32_t *d_planes, cudaStream_t stream) {
    const size_t total_groups = ((size_t)n_sketches << p) >> 5;
    if (total_groups == 0) return cudaSuccess;
    size_t blocks = (total_groups + 255) / 256;
    if (blocks > (size_t)148 * 64) blocks = (size_t)148 * 64;
    DD_COUNT_LAUNCH(), to_planes_kernel<<<(unsigned)blocks, 256, 0, stream>>>(d_regs, d_planes, p, total_groups);
    return cudaGetLastError();
}

// d_scratch: dedup_bytes(n_ord, n_steps) bytes, or nullptr (no identical-prefix search)
cudaError_t prefix_union_hist_from_planes(const uint32_t *d_planes, const int32_t *d_order, int n_ord, int n_steps,
                                          int n_genomes, int nk, int p, int final_only, uint32_t *d_hist, void *d_scratch,
                                          cudaStream_t stream) {
    const int out_steps = final_only ? 1 : n_steps;
    const size_t rows = (size_t)n_ord * out_steps * nk;
    if (rows == 0) return cudaSuccess;
    const size_t m = (size_t)1 << p;
    if (final_only && n_steps == 2) {   // pairs: one CTA per (pair, k) -- or a few, when the job is too small to fill the chip
        const size_t nvec_p = (m >> 5) >> 2;
        const size_t max_y = (nvec_p + kPlThreads - 1) / kPlThreads;
        size_t y = 1;
        while (y < max_y && (size_t)n_ord * nk * y < (size_t)148 * 64) y <<= 1;
        cudaError_t e0 = y > 1 ? cudaMemsetAsync(d_hist, 0, rows * DD_HIST_BINS * sizeof(uint32_t), stream) : cudaSuccess;
        if (e0 != cudaSuccess) return e0;
        DD_COUNT_LAUNCH(), pair_union_planes_kernel<<<dim3((unsigned)n_ord, (unsigned)y, (unsigned)nk), kPlThreads, 0, stream>>>(
            d_planes, d_order, n_genomes, nk, p, d_hist);
        return cudaGetLastError();
    }
    cudaError_t e = cudaMemsetAsync(d_hist, 0, rows * DD_HIST_BINS * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    const size_t pairs = (size_t)n_ord * n_steps;
    unsigned long long *masks = reinterpret_cast<unsigned long long *>(d_scratch);
    int32_t *rep = d_scratch ? reinterpret_cast<int32_t *>(masks + pairs) : nullptr;
    // one CTA compares every (ordering, step) with the first kDedupWindow orderings: the big classes
    // (last steps, first steps) are always found there; pointless for a batch of distinct pairs
    const bool dedup = d_scratch && n_genomes <= 64 && n_ord > 1 && !(final_only && n_steps == 2) &&
                       (double)n_ord * (n_ord < kDedupWindow ? n_ord : kDedupWindow) * n_steps <= 5e7;
    if (dedup) DD_COUNT_LAUNCH(), prefix_dedup_kernel<<<1, 1024, 0, stream>>>(d_order, n_ord, n_steps, n_genomes, masks, rep);
    else rep = nullptr;
    const size_t nvec = (m >> 5) >> 2;
    const unsigned slices = (unsigned)((nvec + kPlThreads - 1) / kPlThreads);
    // the ordering / pair index is the fastest grid dimension (co-resident CTAs share slices in L2);
    // gridDim.x has room for 2^31-1 of them
    const dim3 grid((unsigned)n_ord, slices, (unsigned)nk);
    DD_COUNT_LAUNCH(), prefix_union_planes_kernel<false><<<grid, kPlThreads, 0, stream>>>(d_planes, d_order, n_steps, n_genomes, nk, p, final_only,
                                                                      rep, d_hist);
    if (dedup) {
        const size_t cells = rows * DD_HIST_BINS;
        const unsigned cb = (unsigned)((cells + 255) / 256 < 1184 ? (cells + 255) / 256 : 1184);
        DD_COUNT_LAUNCH(), prefix_copy_rows_kernel<<<cb, 256, 0, stream>>>(rep, n_ord, n_steps, nk, final_only, d_hist);
    }
    return cudaGetLastError();
}

// register input: transpose into the caller's workspace, then the planes path
cudaError_t prefix_union_hist_planes(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                                     int nk, int p, int final_only, uint32_t *d_hist, void *d_ws, cudaStream_t stream) {
    uint32_t *planes = reinterpret_cast<uint32_t *>(d_ws);
    const size_t pl = (planes_bytes((int64_t)n_genomes * nk, p) + 255) / 256 * 256;
    cudaError_t e = to_planes(d_regs, (int64_t)n_genomes * nk, p, planes, stream);
    if (e != cudaSuccess) return e;
    return prefix_union_hist_from_planes(planes, d_order, n_ord, n_steps, n_genomes, nk, p, final_only, d_hist,
                                         static_cast<uint8_t *>(d_ws) + pl, stream);
}

}  // namespace dd
