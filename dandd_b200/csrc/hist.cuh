// hist.cuh -- thread-private shared-memory byte histograms shared by card.cu and sketch.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/dandd_b200.h"

namespace dd {

// -------------------------------------------------------------------------------------------------
// Thread-private byte counters in shared memory for CTAs of 256 threads: row `bin` is 256 bytes,
// thread t owns byte slot(t).  slot() gives every lane of a warp its own 32-bit word (= its own
// bank); the four bytes of a word belong to four different warps, so a warp's 32 increments are
// conflict-free and, being plain byte stores, never race.  A thread may count at most 255.
// -------------------------------------------------------------------------------------------------
constexpr int kPhThreads = 256;
constexpr int kPhBytes = DD_HIST_BINS * kPhThreads;  // 16 KiB

__device__ __forceinline__ uint32_t ph_slot() {
    return ((threadIdx.x & 31u) << 2) | ((threadIdx.x >> 5) & 3u) | ((threadIdx.x >> 7) << 7);
}
__device__ __forceinline__ void ph_zero(uint8_t *s_hist) {
    for (int i = threadIdx.x; i < kPhBytes / 16; i += kPhThreads) reinterpret_cast<uint4 *>(s_hist)[i] = make_uint4(0, 0, 0, 0);
}
__device__ __forceinline__ uint32_t ph_bin(uint32_t byte) { return min(byte, (uint32_t)(DD_HIST_BINS - 1)); }
__device__ __forceinline__ void ph_add_word(uint8_t *s_hist, uint32_t slot, uint32_t w) {
#pragma unroll
    for (int b = 0; b < 4; ++b) s_hist[ph_bin((w >> (8 * b)) & 0xffu) * kPhThreads + slot]++;
}
// Bin b summed over the 256 threads, in every lane of the calling warp: a lane adds the 8 byte counters of one
// 64-bit word with SWAR adds.
__device__ __forceinline__ uint32_t ph_total(const uint8_t *s_hist, int b) {
    const uint2 x = reinterpret_cast<const uint2 *>(s_hist + b * kPhThreads)[threadIdx.x & 31];
    uint32_t s = (x.x & 0x00ff00ffu) + ((x.x >> 8) & 0x00ff00ffu) + (x.y & 0x00ff00ffu) + ((x.y >> 8) & 0x00ff00ffu);
    s = (s & 0xffffu) + (s >> 16);
    return __reduce_add_sync(0xffffffffu, s);
}
// Sum every bin over the 256 threads and add the totals to a global histogram row.  Each warp
// takes 8 bins.
__device__ __forceinline__ void ph_flush(const uint8_t *s_hist, uint32_t *g_hist) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll 2
    for (int b = warp; b < DD_HIST_BINS; b += kPhThreads / 32) {
        const uint32_t s = ph_total(s_hist, b);
        if (lane == 0 && s) atomicAdd(&g_hist[b], s);
    }
}

}  // namespace dd
