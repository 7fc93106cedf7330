// swar.cuh -- byte-wise register comparisons on 4 HLL registers per 32-bit word, shared by K10 (leaveout.cu) and
// K11 (greedy.cu).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace dd {

__device__ __forceinline__ uint32_t byte_at(const uint4 &w, int b) {
    const uint32_t x = b < 4 ? w.x : b < 8 ? w.y : b < 12 ? w.z : w.w;
    return (x >> (8 * (b & 3))) & 0xffu;
}

// SWAR on 4 registers per 32-bit word.  Registers hold ranks <= 64 - p + 1 < 128, so with the top bit of every
// byte forced on, a byte difference never borrows from its neighbour: the top bit of each result byte is the
// comparison, and flags stay in that bit (0x80) until a full byte mask is needed.
constexpr uint32_t kTop = 0x80808080u, kOne = 0x01010101u;
__device__ __forceinline__ uint32_t gt_top(uint32_t a, uint32_t b) { return ((a | kTop) - b - kOne) & kTop; }   // a > b
__device__ __forceinline__ uint32_t eq_top(uint32_t a, uint32_t b) { return ~((a ^ b) + 0x7f7f7f7fu) & kTop; }  // a == b
__device__ __forceinline__ uint32_t spread(uint32_t top) {   // 0x80 -> 0xff per byte (PRMT sign replication)
    uint32_t r;
    asm("prmt.b32 %0, %1, 0, 0xba98;" : "=r"(r) : "r"(top));
    return r;
}
__device__ __forceinline__ uint32_t pick(uint32_t mask, uint32_t a, uint32_t b) { return (a & mask) | (b & ~mask); }

}  // namespace dd
