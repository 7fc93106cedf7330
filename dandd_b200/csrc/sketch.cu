// sketch.cu -- K2: fused all-k canonical k-mer HyperLogLog sketch.
//
// Replaces `parallel -j 95% ' dashing sketch -k{} -S p ... ' ::: k...` (reference
// lib/huffman_dandd.py:217 over lib/sketch_classes.py:351-366): ONE pass over the packed symbol
// stream updates the registers of every requested k with Dashing's own hash (Wang) and register
// rule, so the registers are bit-identical to nk separate `dashing sketch` runs.
//
// Mapping: one thread per 16-symbol code word.  The 64-bit forward window and its reverse
// complement for any symbol of the word are two funnel shifts over three consecutive words (the
// reverse-complement words are computed once per thread), so there is no rolling state and no
// dependence between symbols or between k values; validity of a k-mer is "at least k symbols
// since the last break", one funnel shift + ctz on the break-bit words.  The k loop is unrolled
// at compile time (masks and shifts are immediates; k <= 16 keeps the k-mer in one register); the
// symbol loop is not, which keeps the body (~1.1k instructions for 31 k) inside the instruction
// cache.
//
// There is no byte-wide atomic max, and one u32 per register (nk x 4 MiB per genome at p=20) does
// not stay L2-resident: ncu showed 51 % of the RED sectors missing and 2.4 GB of DRAM write-back
// per 5 Mbp genome (profiles/r01).  Registers are therefore accumulated two to a 32-bit word with
// REDG.E.MAX.F16x2 (`red.global.max.noftz.v2.f16`): a rank r <= 45 is stored as the f16 *subnormal*
// whose bit pattern is r, positive f16 values order like their bit patterns, .noftz keeps
// subnormals, and the other half of the operand is +0.0, the identity of max over ranks -- so each
// half is an independent, exact integer max.  dd_sketch_end narrows the u16 halves to u8.
// Bound: INT32 issue and the L2 reduction rate -- not HBM (see DESIGN.md).
//
// Small k.  For k <= 9 there are at most 4^k distinct k-mers, so every update of such a k lands on
// a handful of addresses and same-address L2 reductions serialise (measured at 1 Gbp: k=2 alone
// 190 ms, k=3 87 ms, against 5.5 ms for k >= 8).  The kernel is therefore persistent (a few CTAs per
// SM, grid-stride over 4096-symbol tiles) and each CTA keeps a presence bitmap of the canonical
// k-mers it has already sent, for every k <= 9 (43.7 KB of shared memory): a k-mer whose bit is
// set is dropped before hashing -- exact, because the same k-mer always produces the same
// (register, rank) -- so a CTA issues at most 4^k reductions per small k over its whole life.
#include <cuda_runtime.h>

#include <utility>

#include "common.cuh"
#include "hist.cuh"
#include "kernels.cuh"

namespace dd {

// CTA shapes, measured on B200 (profiles/r02_k2_variants.md).  Sweeps without a small k (no presence
// bitmaps, short genomes dominate: config 2) run best as 256-thread CTAs, one tile each; sweeps with
// small k are persistent and share one 43.7 KB bitmap set among the 32 warps of a 1024-thread CTA
// (two CTAs per SM instead of five 256-thread ones: 64 resident warps instead of 40).
#ifndef DD_SKETCH_THREADS_PLAIN
#define DD_SKETCH_THREADS_PLAIN 256
#endif
#ifndef DD_SKETCH_THREADS_SMALLK
#define DD_SKETCH_THREADS_SMALLK 1024
#endif
constexpr int kThreadsPlain = DD_SKETCH_THREADS_PLAIN, kThreadsSmallK = DD_SKETCH_THREADS_SMALLK;
constexpr int min_ctas_for(int threads) { return threads >= 1024 ? 2 : threads >= 512 ? 3 : 5; }
#ifndef DD_XORSHIFT_ON_FMA
#define DD_XORSHIFT_ON_FMA 0  // measured: no gain (3.1 Gbp 210 vs 203 ms); IMAD.WIDE is not cheaper than SHF here
#endif

struct SketchArgs {
    const uint32_t *codes;
    const uint32_t *invalid;
    const dd_pack_state *state;  // if non-null the symbol range is [state->prev_nsym, state->nsym)
    uint64_t sym_begin, sym_end;
    uint32_t kmask;               // every k of the sketch (defines the accumulator slots)
    uint32_t kmask_run;           // the k values this launch updates (subset of kmask)
    int p;
    uint32_t *acc;                // [nk][2^p / 2] words, two u16 registers per word
    uint32_t *midk;               // presence bitmaps for k = 10..14 (kMidK variants only)
    int midk_hi;                  // largest k whose bitmap this launch consults (12..14)
    const SketchWsHeader *hdr;
    uint32_t ntiles;              // upper bound on the (CTA size)-word tiles of the symbol range
};

// Presence bitmaps for k = 1..kBitmapMaxK: 4^k bits each (at least one word).
constexpr int kBitmapMaxK = 9;
__host__ __device__ constexpr uint32_t bitmap_words(int k) { return (1u << (2 * k)) >= 32u ? (1u << (2 * k)) / 32u : 1u; }
__host__ __device__ constexpr uint32_t bitmap_offset(int k) {  // words before the bitmap of k
    uint32_t o = 0;
    for (int j = 1; j < k; ++j) o += bitmap_words(j);
    return o;
}
constexpr uint32_t kBitmapWords = bitmap_offset(kBitmapMaxK + 1);  // 10924 words = 43.7 KB
constexpr uint32_t kSmallKMask = (1u << kBitmapMaxK) - 1u;

// Mid k (10..12) on LONG genomes.  4^k is still far below the number of k-mers of a multi-Gbp genome
// (k = 12: 8.4 M canonical k-mers against 3.1 G windows), so almost every window repeats one already
// hashed -- but the bitmaps (128 KiB + 512 KiB + 2 MiB) no longer fit in shared memory.  They live in
// the workspace, shared by all CTAs through L2: one 4-byte load per (symbol, k) replaces the hash,
// compare and branch of a repeat.  Sound by construction: a bit is only ever set by the thread that goes
// on to issue that k-mer's update, and the same k-mer always yields the same (register, rank).  Only
// launches deep inside a long stream use it (the host decides); short genomes keep the plain path,
// where the extra L2 loads would compete with the reductions that bound it.
constexpr int kMidKLo = 10, kMidKHi = 14;   // k = 13 (8 MiB) and 14 (32 MiB) join once the stream is >= 4^k symbols long
__host__ __device__ constexpr uint32_t midk_offset(int k) {   // words before the bitmap of k
    uint32_t o = 0;
    for (int j = kMidKLo; j < k; ++j) o += (1u << (2 * j)) / 32u;
    return o;
}
constexpr uint32_t kMidKWords = midk_offset(kMidKHi + 1);     // 42.6 MiB in all; k <= 12 alone: 2.6 MiB

// 64-bit x times 32-bit constant: IMAD.WIDE.U32 + IMAD, both on the FMA pipe (PTX spelled out so
// that ptxas does not split the high-word multiply-add).
__device__ __forceinline__ uint64_t mul64x32(uint64_t x, uint32_t c) {
    uint32_t xl, xh, rl, rh;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(xl), "=r"(xh) : "l"(x));
    uint64_t r;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(r) : "r"(xl), "r"(c));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(rl), "=r"(rh) : "l"(r));
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(rh) : "r"(xh), "r"(c), "r"(rh));
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(rl), "r"(rh));
    return r;
}
// ... plus a 64-bit addend folded into the wide multiply.
__device__ __forceinline__ uint64_t mad64x32(uint64_t x, uint32_t c, uint64_t add) {
    uint32_t xl, xh, rl, rh;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(xl), "=r"(xh) : "l"(x));
    uint64_t r;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(xl), "r"(c), "l"(add));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(rl), "=r"(rh) : "l"(r));
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(rh) : "r"(xh), "r"(c), "r"(rh));
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(rl), "r"(rh));
    return r;
}

// h ^= h >> S with the two 32-bit right shifts done as widening multiplies by 2^(32-S) on the
// FMA pipe (the high word of x * 2^(32-S) is x >> S, the low word is x << (32-S)), leaving only the
// two XOR/OR LOP3s on the ALU pipe, which is the binding pipe of this kernel (ncu: ALU 67 %, FMA 11 %).
template <int S>
__device__ __forceinline__ uint64_t xorshr_fma(uint64_t h) {
    uint32_t hl, hh, tl, th, ul, uh;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(hl), "=r"(hh) : "l"(h));
    uint64_t t, u;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(t) : "r"(hh), "r"(1u << (32 - S)));
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(u) : "r"(hl), "r"(1u << (32 - S)));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(tl), "=r"(th) : "l"(t));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(ul), "=r"(uh) : "l"(u));
    const uint32_t nl = hl ^ (uh | tl), nh = hh ^ th;
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(nl), "r"(nh));
    return r;
}

// h ^= h >> S with only the HIGH word's shift moved to the FMA pipe (mul.hi by 2^(32-S) == >> S):
// one ALU instruction less per xor-shift, one IMAD.HI more.
#ifndef DD_K2_MULHI
#define DD_K2_MULHI 0
#endif
#ifndef DD_K2_VOTE_TAIL
#define DD_K2_VOTE_TAIL 0
#endif
template <int S>
__device__ __forceinline__ uint64_t xorshr(uint64_t h) {
#if DD_K2_MULHI
    uint32_t hl, hh, sh;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(hl), "=r"(hh) : "l"(h));
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(sh) : "r"(hh), "r"(1u << (32 - S)));
    const uint32_t nl = hl ^ __funnelshift_r(hl, hh, S), nh = hh ^ sh;
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(nl), "r"(nh));
    return r;
#else
    return h ^ (h >> S);
#endif
}

// dd::wang64 (common.cuh) with the multiplications pinned to the FMA pipe
__device__ __forceinline__ uint64_t wang64_fma(uint64_t v, uint64_t minus_one) {
    uint64_t h = mad64x32(v, 0x1FFFFFu, minus_one);
#if DD_XORSHIFT_ON_FMA
    h = xorshr_fma<24>(h);
    h = mul64x32(h, 265u);
    h = xorshr_fma<14>(h);
    h = mul64x32(h, 21u);
    h = xorshr_fma<28>(h);
#else
    h = xorshr<24>(h);
    h = mul64x32(h, 265u);
    h = xorshr<14>(h);
    h = mul64x32(h, 21u);
    h = xorshr<28>(h);
#endif
    return mul64x32(h, 0x80000001u);
}

// Rank of a hash whose 32 bits below the register index are t (lo = its low word): clz(t) + 1 unless
// they are all zero.
__device__ __forceinline__ uint32_t rank_of(uint32_t t, uint32_t lo, int p) {
    return t ? (uint32_t)__clz((int)t) + 1u : 33u + (uint32_t)__clz((int)((lo << p) | (1u << (p - 1))));
}

// acc[slot_off + register / 2] = max(.., rank) on the register's u16 half (register = hi >> (32 - p))
__device__ __forceinline__ void red_max_register(uint32_t *acc, uint32_t slot_off, uint32_t hi, uint32_t rank, int p) {
    // register idx = hi >> (32-p) lives in word idx>>1, half idx&1
    const uint32_t val = rank << ((hi >> (28 - p)) & 16u);
    uint32_t *word = acc + (slot_off + (hi >> (33 - p)));
    asm volatile("{ .reg .b16 l, h; mov.b32 {l, h}, %1; red.global.max.noftz.v2.f16 [%0], {l, h}; }" ::"l"(word), "r"(val) : "memory");
}

// The packed words behind the 16 symbols of code word w: every window ending in it is two funnel
// shifts over w0..w2 (r0..r2 = their reverse complements), its validity a ctz over i0:i1.  Only
// symbols j_lo <= j < j_hi lie in the range being sketched; a word out of range has none.
struct WordSpan {
    uint32_t w0, w1, w2, r0, r1, r2, i0, i1;
    uint32_t sm_base;
    int j_lo, j_hi;
    bool all_valid;
};
// the five loads behind code word w, apart from what is computed from them (so that they can be issued a tile early)
struct RawWord {
    uint32_t w0, w1, w2, i0, i1;
};
__device__ __forceinline__ RawWord load_raw(const uint32_t *codes, const uint32_t *invalid, uint64_t w, bool in_range) {
    RawWord r;
    r.w0 = in_range ? __ldg(codes + w) : 0u;
    r.w1 = in_range && w >= 1 ? __ldg(codes + w - 1) : 0u;
    r.w2 = in_range && w >= 2 ? __ldg(codes + w - 2) : 0u;
    const uint64_t iw = w >> 1;
    r.i0 = in_range ? __ldg(invalid + iw) : 0xffffffffu;
    r.i1 = in_range && iw >= 1 ? __ldg(invalid + iw - 1) : 0xffffffffu;  // before the stream: breaks
    return r;
}
__device__ __forceinline__ WordSpan span_of(const RawWord &r, uint64_t w, bool in_range, uint64_t sym_begin, uint64_t sym_end) {
    WordSpan s;
    const uint64_t s0 = w << 4;
    s.w0 = r.w0;
    s.w1 = r.w1;
    s.w2 = r.w2;
    s.i0 = r.i0;
    s.i1 = r.i1;
    s.r0 = revcomp_word(s.w0);
    s.r1 = revcomp_word(s.w1);
    s.r2 = revcomp_word(s.w2);
    s.all_valid = (s.i0 | s.i1) == 0u;
    s.j_lo = sym_begin > s0 ? (int)(sym_begin - s0) : 0;
    s.j_hi = !in_range ? 0 : (sym_end - s0 < 16 ? (int)(sym_end - s0) : 16);
    s.sm_base = (uint32_t)(s0 & 31);
    return s;
}
__device__ __forceinline__ WordSpan load_word(const uint32_t *codes, const uint32_t *invalid, uint64_t w, bool in_range,
                                              uint64_t sym_begin, uint64_t sym_end) {
    return span_of(load_raw(codes, invalid, w, in_range), w, in_range, sym_begin, sym_end);
}
__device__ __forceinline__ Window span_window(const WordSpan &s, int j) { return window_at(s.w0, s.w1, s.w2, s.r0, s.r1, s.r2, j); }
// valid symbols ending at symbol j of the word (0 outside the range)
__device__ __forceinline__ int span_run(const WordSpan &s, int j) {
    int run = s.all_valid ? 32 : valid_run(invalid_window(s.i0, s.i1, s.sm_base + (uint32_t)j));
    if (j < s.j_lo || j >= s.j_hi) run = 0;
    return run;
}

// Canonical (or forward) k-mer ending at the current symbol.  For K <= 16 the whole k-mer lives in
// one 32-bit register: mask, shift and min are single instructions.
template <int K, bool kCanon>
__device__ __forceinline__ uint64_t kmer_of(const Window &win) {
    if constexpr (K <= 16) {
        const uint32_t f = (uint32_t)win.fwd & (K == 16 ? 0xffffffffu : ((1u << (2 * (K & 15))) - 1u));
        if (!kCanon) return f;
        const uint32_t r = (uint32_t)(win.rc >> 32) >> (32 - 2 * K);
        return min(f, r);
    } else {
        return kmer_value<K>(win, kCanon);
    }
}

// Per-k constants of one launch, in shared memory (a load with an immediate address per use; kept
// in registers they cost 64 of them): thresh[k-1] = largest value of the top 32 remainder bits whose
// rank still exceeds the floor of k (rank > floor <=> clz(t) >= floor <=> t <= 0xffffffff >> floor),
// floor[k-1] itself for the exact re-check that only matters when floor > 32.
struct KConsts {
    uint32_t thresh[32];
    uint32_t floor[32];
};

// One (symbol, k) update.  `live` says whether this lane has a valid k-mer of this length; the
// warp stays converged (dead lanes are only predicated off the shared-memory and global updates),
// so the small-k early exit is a plain full-warp vote.
// kStaticMask != 0: the set of k values is known at compile time (no per-k mask tests, table slot a
// constant); 0: generic, driven by kmask / kmask_run.
// Cost after the hash (SASS, profiles/r02_k2_sass.md): the common case -- rank <= floor on a long
// genome -- is one funnel shift, one compare and one branch; rank, register index and address are
// only computed by the lanes that actually update.
template <int K, bool kCanon, uint32_t kStaticMask, bool kMidK>
__device__ __forceinline__ void update_one_k(const Window &win, int run, uint32_t kmask, uint32_t kmask_run, int p,
                                             uint32_t *acc, uint32_t &off_k, const KConsts &kc, uint32_t *s_seen,
                                             uint32_t *midk, int midk_hi, uint64_t minus_one) {
    constexpr uint32_t bit = 1u << (K - 1);
    if (kStaticMask) {
        if (!(kStaticMask & bit)) return;    // compile time
    } else {
        if (!(kmask & bit)) return;          // warp-uniform
        if (!(kmask_run & bit)) {
            off_k += 1u << (p - 1);
            return;
        }
    }
    const uint64_t v = kmer_of<K, kCanon>(win);
    bool live = run >= K;
    if (K <= kBitmapMaxK) {
        // already sent by this CTA?  (a racing duplicate only repeats an idempotent update)
        uint32_t *word = s_seen + bitmap_offset(K) + ((uint32_t)v >> 5);
        const uint32_t seen_bit = 1u << ((uint32_t)v & 31u);
        live = live && !(*word & seen_bit);
        if (live) atomicOr(word, seen_bit);
        if (!__any_sync(0xffffffffu, live)) {
            if (!kStaticMask) off_k += 1u << (p - 1);
            return;
        }
    }
    if (kMidK && K >= kMidKLo && K <= kMidKHi && (K <= 12 || K <= midk_hi)) {   // (warp-uniform)
        // already sent by ANY CTA of this sketch?  (L2-resident bitmap; a stale "not yet" only repeats an idempotent update)
        uint32_t *word = midk + midk_offset(K) + ((uint32_t)v >> 5);
        const uint32_t seen_bit = 1u << ((uint32_t)v & 31u);
        live = live && !(__ldcg(word) & seen_bit);
        if (live) atomicOr(word, seen_bit);
        if (!__any_sync(0xffffffffu, live)) {
            if (!kStaticMask) off_k += 1u << (p - 1);
            return;
        }
    }
    const uint64_t h = wang64_fma(v, minus_one);
    const uint32_t hi = (uint32_t)(h >> 32), lo = (uint32_t)h;
    // t = the 32 bits below the register index; rank = clz(t) + 1 unless they are all zero
    const uint32_t t = __funnelshift_l(lo, hi, (uint32_t)p);
    const bool pass = live && t <= kc.thresh[K - 1];
#if DD_K2_VOTE_TAIL
    if (__any_sync(0xffffffffu, pass))   // warp-uniform branch (no reconvergence barrier); the tail is predicated
#endif
    if (pass) {
        const uint32_t rank = rank_of(t, lo, p);
        if (rank > kc.floor[K - 1]) {
            const uint32_t slot_off = kStaticMask ? (uint32_t)__popc(kStaticMask & (bit - 1u)) << (p - 1) : off_k;
            red_max_register(acc, slot_off, hi, rank, p);
        }
    }
    if (!kStaticMask) off_k += 1u << (p - 1);
}

template <bool kCanon, uint32_t kStaticMask, bool kMidK, int... Ks>
__device__ __forceinline__ void update_all_k(std::integer_sequence<int, Ks...>, const Window &win, int run,
                                             uint32_t kmask, uint32_t kmask_run, int p, uint32_t *acc,
                                             const KConsts &kc, uint32_t *s_seen, uint32_t *midk, int midk_hi,
                                             uint64_t minus_one) {
    uint32_t off_k = 0;
    (update_one_k<Ks + 1, kCanon, kStaticMask, kMidK>(win, run, kmask, kmask_run, p, acc, off_k, kc, s_seen, midk, midk_hi, minus_one), ...);
}

// per-k floors (indexed by k-1) and the remainder thresholds derived from them; the caller syncs
__device__ __forceinline__ void load_kconsts(const SketchWsHeader *hdr, KConsts &kc) {
    if (threadIdx.x < 32) {
        const uint32_t f = hdr->floor[threadIdx.x];
        kc.floor[threadIdx.x] = f;
        kc.thresh[threadIdx.x] = f >= 32u ? 0u : 0xffffffffu >> f;
    }
}

// [sym_begin, sym_end) of a launch: explicit, or read from the pack state on the device
__device__ __forceinline__ void launch_range(const SketchArgs &a, uint64_t &sym_begin, uint64_t &sym_end) {
    sym_begin = a.sym_begin;
    sym_end = a.sym_end;
    if (a.state) {   // the range of the last pack call; a.sym_begin / a.sym_end select a sub-range of it, relative to its start
        const uint64_t first = a.state->prev_nsym, last = a.state->nsym;
        sym_begin = first + a.sym_begin < last ? first + a.sym_begin : last;
        sym_end = a.sym_end < last - first ? first + a.sym_end : last;
    }
}

template <bool kCanon, uint32_t kStaticMask, int kThreads, bool kMidK = false>
__global__ void __launch_bounds__(kThreads, min_ctas_for(kThreads)) sketch_allk_kernel(SketchArgs a) {
    extern __shared__ uint32_t s_seen[];  // presence bitmaps, only allocated when a k <= 9 is requested
    const bool small_k = ((kStaticMask ? kStaticMask : a.kmask_run) & kSmallKMask) != 0u;
    if (small_k) {
        for (uint32_t i = threadIdx.x; i < kBitmapWords; i += kThreads) s_seen[i] = 0u;
        __syncthreads();
    }
    __shared__ KConsts kc;
    load_kconsts(a.hdr, kc);
    __syncthreads();
    const uint64_t minus_one = ~0ull;   // (ptxas splits the addend off the IMAD.WIDE whether or not it can see its value)
    // k = 13 / 14 bitmaps: only those the header says were zeroed since dd_sketch_begin
    const int midk_hi = kMidK ? min(a.midk_hi, max(12, (int)a.hdr->pad[0])) : 0;
    uint64_t sym_begin, sym_end;
    launch_range(a, sym_begin, sym_end);

#pragma unroll 1
    for (uint32_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
        const uint64_t w = (sym_begin >> 4) + (uint64_t)tile * kThreads + threadIdx.x;
        if ((uint64_t)((sym_begin >> 4) + (uint64_t)tile * kThreads) << 4 >= sym_end) break;  // CTA-uniform
        // lanes past the end stay in the loop, predicated off
        const WordSpan ws = load_word(a.codes, a.invalid, w, (w << 4) < sym_end, sym_begin, sym_end);

#pragma unroll 1
        for (int j = 0; j < 16; ++j) {
            const Window win = span_window(ws, j);
            const int run = span_run(ws, j);
            if (!__any_sync(0xffffffffu, run != 0)) continue;  // warp-uniform
            update_all_k<kCanon, kStaticMask, kMidK>(std::make_integer_sequence<int, 32>{}, win, run, a.kmask, a.kmask_run, a.p,
                                                     a.acc, kc, s_seen, a.midk, midk_hi, minus_one);
        }
    }
}

// ---- rank-1 sink: one k per CTA, rank-1 updates absorbed in a shared-memory bitmap ---------------
// Half of all updates have rank 1, and a rank-1 update can only raise a register from 0 to 1: all it
// records is "some k-mer hit register r", one bit.  Before the floor schedule's first cut (floor 0)
// every such update is a scattered L2 reduction -- the resource that bounds K2 on short genomes.  Here
// a CTA owns one k over a contiguous slice of the stream and ORs its rank-1 updates into a 2^p-bit
// bitmap in shared memory (128 KiB at p = 20); rank >= 2 goes to L2 as in the plain kernel.  At the end
// the CTA stores its bitmap whole to its own slab of the workspace (no merge reductions), and a CTA of a
// later launch into the same workspace starts from its slab.  The register is max(acc, OR of k's slabs)
// -- finalize_kernel and floor_min_kernel read it so -- which keeps the result exact whichever kernel
// sketched which piece.  k <= 9 stays with the presence-bitmap kernel.
//
// The sink only runs at floor 0 (sketch_update_sched), so it has no threshold or floor test.  A warp whose 32 words are all in range and hold no break runs its 16 symbols unrolled, with no
// per-symbol validity test; the next tile's words are loaded before the current tile is hashed.
constexpr int kSinkThreads = 1024, kSinkMinK = kBitmapMaxK + 1, kSinkMaxP = 20;
// u32 words of one slab (the 2^p-bit bitmap, whole uint4s)
__host__ __device__ constexpr uint32_t sink_slab_words(int p) { return ((1u << (p - 5)) + 3u) & ~3u; }

// one (symbol, k) update at floor 0; acc_k = k's accumulator row, s_bits the bitmap's shared-window address.  The rank
// is computed without a branch (clz(0) = 32, so the t == 0 case only adds the low word's clz).  The shared-memory OR
// and the REDG each sit behind a short BSSY/BRA/BSYNC: ptxas wraps every predicated ATOMS or REDG so, even one
// written as a PTX predicate.  Both are spelled out in PTX on a 32-bit register index, 3 SASS instructions per update
// fewer than atomicOr and red_max_register on a 64-bit slot offset.
template <int K, bool kCanon>
__device__ __forceinline__ void sink_update(const Window &win, bool live, uint32_t s_bits, uint32_t *acc_k, int p) {
    const uint64_t h = wang64_fma(kmer_of<K, kCanon>(win), ~0ull);
    const uint32_t hi = (uint32_t)(h >> 32), lo = (uint32_t)h;
    const uint32_t t = __funnelshift_l(lo, hi, (uint32_t)p);
    const uint32_t r = hi >> (32 - p);
    const uint32_t low = (uint32_t)__clz((int)((lo << p) | (1u << (p - 1))));
    const uint32_t rank = (uint32_t)__clz((int)t) + 1u + (t == 0u ? low : 0u);
    const bool one = (int32_t)t < 0;   // rank 1
    if (live && one) asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(s_bits + ((r >> 3) & ~3u)), "r"(1u << (r & 31u)) : "memory");
    if (live && !one) {
        const uint32_t val = rank << ((hi >> (28 - p)) & 16u);   // register r's u16 half of word r / 2
        asm volatile("{ .reg .b16 l, h; .reg .b64 a; mad.wide.u32 a, %1, 4, %0; mov.b32 {l, h}, %2; red.global.max.noftz.v2.f16 [a], {l, h}; }"
                     ::"l"(acc_k), "r"(hi >> (33 - p)), "r"(val)
                     : "memory");
    }
}

template <int K, bool kCanon>
__device__ __forceinline__ void sink_slice(const SketchArgs &a, uint32_t s_bits, uint32_t *acc_k, uint64_t sym_begin,
                                           uint64_t sym_end, uint64_t w_lo, uint64_t w_hi) {
    const int p = a.p;
    RawWord next = load_raw(a.codes, a.invalid, w_lo + threadIdx.x, w_lo + threadIdx.x < w_hi);
#pragma unroll 1
    for (uint64_t base = w_lo; base < w_hi; base += kSinkThreads) {
        const uint64_t w = base + threadIdx.x;
        const RawWord cur = next;
        next = load_raw(a.codes, a.invalid, w + kSinkThreads, w + kSinkThreads < w_hi);
        const WordSpan ws = span_of(cur, w, w < w_hi, sym_begin, sym_end);
        const bool full = w < w_hi && ws.all_valid && ws.j_lo == 0 && ws.j_hi == 16;   // every symbol ends a valid 32-mer
        if (__all_sync(0xffffffffu, full)) {
#pragma unroll
            for (int j = 0; j < 16; ++j) sink_update<K, kCanon>(span_window(ws, j), true, s_bits, acc_k, p);
        } else {
#pragma unroll 1
            for (int j = 0; j < 16; ++j) {
                const bool live = span_run(ws, j) >= K;
                if (!__any_sync(0xffffffffu, live)) continue;  // warp-uniform
                sink_update<K, kCanon>(span_window(ws, j), live, s_bits, acc_k, p);
            }
        }
    }
}

// CTA-uniform dispatch to the compile-time K of this CTA (immediate masks in kmer_of)
template <bool kCanon, int... Ks>
__device__ __forceinline__ void sink_dispatch(std::integer_sequence<int, Ks...>, int k, const SketchArgs &a, uint32_t s_bits,
                                              uint32_t *acc_k, uint64_t sym_begin, uint64_t sym_end, uint64_t w_lo, uint64_t w_hi) {
    ((k == Ks + kSinkMinK ? sink_slice<Ks + kSinkMinK, kCanon>(a, s_bits, acc_k, sym_begin, sym_end, w_lo, w_hi) : void()), ...);
}

// grid = (k values of a.kmask_run, all >= kSinkMinK) x slices, CTA b owning slab b; dynamic shared memory = one slab.
// written[b] != 0: slab b holds the bits of an earlier launch into this workspace.
template <bool kCanon>
__global__ void __launch_bounds__(kSinkThreads, 1) sketch_sink_kernel(SketchArgs a, uint32_t *slabs, uint32_t *written,
                                                                        uint32_t slices, SketchWsHeader *hdr) {
    extern __shared__ uint4 s_bits4[];
    uint32_t *s_bits = reinterpret_cast<uint32_t *>(s_bits4);
    const int p = a.p;
    const uint32_t n4 = sink_slab_words(p) / 4;
    uint4 *slab = reinterpret_cast<uint4 *>(slabs + (size_t)blockIdx.x * sink_slab_words(p));
    const bool carry = written[blockIdx.x] != 0u;
    for (uint32_t i = threadIdx.x; i < n4; i += kSinkThreads) s_bits4[i] = carry ? __ldcs(slab + i) : make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();

    // this CTA's k: the (blockIdx.x / slices)-th set bit of kmask_run; its table slot counts over kmask
    uint32_t m = a.kmask_run;
    for (uint32_t u = blockIdx.x / slices; u > 0; --u) m &= m - 1u;
    const int k = __ffs((int)m);
    const uint32_t slot = (uint32_t)__popc(a.kmask & ((1u << (k - 1)) - 1u));
    // this CTA's slice: whole code words, so every symbol of the range belongs to exactly one slice
    uint64_t sym_begin, sym_end;
    launch_range(a, sym_begin, sym_end);
    const uint64_t wb = sym_begin >> 4, we = sym_end > sym_begin ? (sym_end + 15) >> 4 : wb;
    const uint64_t per = (we - wb + slices - 1) / slices, slice = blockIdx.x % slices;
    const uint64_t w_lo = min(wb + slice * per, we), w_hi = min(w_lo + per, we);
    sink_dispatch<kCanon>(std::make_integer_sequence<int, 33 - kSinkMinK>{}, k, a, (uint32_t)__cvta_generic_to_shared(s_bits),
                          a.acc + ((size_t)slot << (p - 1)), sym_begin, sym_end, w_lo, w_hi);
    __syncthreads();
    // evict-first stores: the slabs are read once, by finalize, and must not push the accumulators out of L2
    for (uint32_t i = threadIdx.x; i < n4; i += kSinkThreads) __stcs(slab + i, s_bits4[i]);
    if (threadIdx.x == 0) {
        written[blockIdx.x] = 1u;
        hdr->sink_slices = slices;                              // the same values from every CTA and launch
        hdr->sink_first = (uint32_t)__popc(a.kmask & kSmallKMask);   // table slot of the first sink k
    }
}

// marks the presence bitmap of k (13 or 14) as zeroed since dd_sketch_begin (which clears the header)
__global__ void midk_ready_kernel(SketchWsHeader *hdr, uint32_t k) {
    if (hdr->pad[0] < k) hdr->pad[0] = k;
}

// ---- per-slot min(register): the "floor" filter ---------------------------------------------------
// Rank-1 sink bits as register values: bit i of x -> byte i (0 or 1), i < 4; -> u16 half i, i < 2.
__device__ __forceinline__ uint32_t bits_to_bytes(uint32_t x) { return (x * 0x00204081u) & 0x01010101u; }
__device__ __forceinline__ uint32_t bits_to_halves(uint32_t x) { return (x & 1u) | ((x & 2u) << 15); }

// The first sink slab of table slot `table`, or null unless a sink launch has run into this workspace and the slot is
// one of its k.
__device__ __forceinline__ uint32_t *sink_slabs_of(uint32_t *slabs, const SketchWsHeader *hdr, uint32_t table, int p) {
    const uint32_t slices = hdr->sink_slices, first = hdr->sink_first;
    return slices != 0u && table >= first ? slabs + (size_t)(table - first) * slices * sink_slab_words(p) : nullptr;
}

// ORs every sink k's slabs into its first one, so that floor_min_kernel and finalize_kernel read one bitmap per k
// (byte i holding the bits of registers 8i..8i+7).  Done in a pass of its own: finalize's threads, each with 30
// octets in turn, would wait for every slab load one after the other.  grid (uint4s of a slab / 256, nk)
__global__ void __launch_bounds__(256) sink_merge_kernel(uint32_t *slabs, const SketchWsHeader *hdr, int p) {
    uint4 *s = reinterpret_cast<uint4 *>(sink_slabs_of(slabs, hdr, blockIdx.y, p));
    const uint32_t slices = hdr->sink_slices, n4 = sink_slab_words(p) / 4, i = blockIdx.x * 256u + threadIdx.x;
    if (!s || slices < 2u || i >= n4) return;
    uint4 v = s[i];
#pragma unroll 4
    for (uint32_t c = 1; c < slices; ++c) {
        const uint4 x = __ldcs(s + (size_t)c * n4 + i);
        v = make_uint4(v.x | x.x, v.y | x.y, v.z | x.z, v.w | x.w);
    }
    s[i] = v;
}
static cudaError_t sink_merge(uint32_t *slabs, const SketchWsHeader *hdr, int nk, int p, cudaStream_t stream) {
    if (p > kSinkMaxP) return cudaSuccess;   // no sink, no slabs
    DD_COUNT_LAUNCH(), sink_merge_kernel<<<dim3((sink_slab_words(p) / 4 + 255) / 256, nk), 256, 0, stream>>>(slabs, hdr, p);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) floor_min_kernel(const uint32_t *__restrict__ acc, uint32_t *__restrict__ slabs, int p,
                                                        const SketchWsHeader *hdr, uint32_t *scratch /*[nk]*/) {
    // grid (slices, nk); scratch pre-set to 0xff.  acc rows are 2^p u16 registers = 2^(p-1) words;
    // register = max(acc, sink bit).
    const size_t nwords = (size_t)1 << (p - 1);
    const uint32_t *t = acc + (size_t)blockIdx.y * nwords;
    const uint8_t *bits = reinterpret_cast<const uint8_t *>(sink_slabs_of(slabs, hdr, blockIdx.y, p));   // merged
    uint32_t mn = 0xffffu;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nwords / 4; i += (size_t)gridDim.x * blockDim.x) {
        uint4 v = reinterpret_cast<const uint4 *>(t)[i];
        const uint32_t b = bits ? bits[i] : 0u;
        v.x = __vmaxu2(v.x, bits_to_halves(b));
        v.y = __vmaxu2(v.y, bits_to_halves(b >> 2));
        v.z = __vmaxu2(v.z, bits_to_halves(b >> 4));
        v.w = __vmaxu2(v.w, bits_to_halves(b >> 6));
        const uint32_t w = __vminu2(__vminu2(v.x, v.y), __vminu2(v.z, v.w));
        mn = min(mn, min(w & 0xffffu, w >> 16));
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    if ((threadIdx.x & 31) == 0) atomicMin(&scratch[blockIdx.y], mn);
}
// scratch[slot] -> floor[k-1] for the slot-th set bit of kmask
__global__ void floor_publish_kernel(SketchWsHeader *hdr, const uint32_t *scratch, uint32_t kmask) {
    const int i = threadIdx.x;  // k - 1
    if (i < 32) {
        const bool on = (kmask >> i) & 1u;
        const int slot = __popc(kmask & ((1u << i) - 1u));
        hdr->floor[i] = on ? (uint8_t)scratch[slot] : 0;
    }
    if (i == 0) hdr->use_floor = 1;
}

// ---- finalisation: u16 accumulators -> u8 registers (+ histogram) -------------------------------
constexpr int kFinOctPerThread = 30;                                   // 30 x 8 = 240 registers <= 255 per flush
constexpr int kFinChunk = kPhThreads * kFinOctPerThread * 8;           // registers per CTA

__global__ void __launch_bounds__(kPhThreads)
finalize_kernel(const uint32_t *__restrict__ acc, uint32_t *__restrict__ slabs, const SketchWsHeader *hdr, int p,
                uint8_t *__restrict__ regs, uint32_t *__restrict__ hist) {
    __shared__ __align__(16) uint8_t s_hist[kPhBytes];
    const uint32_t slot = ph_slot();
    const size_t m = (size_t)1 << p;
    const int table = blockIdx.y;
    // 8 u16 accumulators (one uint4) and one byte of rank-1 sink bits -> 8 u8 registers (one uint2)
    const uint4 *src = reinterpret_cast<const uint4 *>(acc + (size_t)table * (m / 2));
    const uint8_t *bits = reinterpret_cast<const uint8_t *>(sink_slabs_of(slabs, hdr, (uint32_t)table, p));   // merged
    uint2 *dst = reinterpret_cast<uint2 *>(regs + (size_t)table * m);
    if (hist) ph_zero(s_hist);
    __syncthreads();
    const size_t noct = m / 8;
    const size_t q0 = (size_t)blockIdx.x * (kFinChunk / 8);
#pragma unroll 5
    for (int i = 0; i < kFinOctPerThread; ++i) {
        const size_t q = q0 + (size_t)i * kPhThreads + threadIdx.x;
        if (q < noct) {
            const uint4 v = __ldcs(src + q);
            // bytes 0 and 2 of each word are the low bytes of its two u16 registers (ranks < 256)
            const uint32_t b = bits ? __ldcs(bits + q) : 0u;
            const uint2 out = make_uint2(__vmaxu4(__byte_perm(v.x, v.y, 0x6420), bits_to_bytes(b & 15u)),
                                         __vmaxu4(__byte_perm(v.z, v.w, 0x6420), bits_to_bytes(b >> 4)));
            dst[q] = out;
            if (hist) {
                ph_add_word(s_hist, slot, out.x);
                ph_add_word(s_hist, slot, out.y);
            }
        }
    }
    if (!hist) return;
    __syncthreads();
    ph_flush(s_hist, hist + (size_t)table * DD_HIST_BINS);
}

// ---- host side ----------------------------------------------------------------------------------
int g_k_per_pass = 0;  // tuning knob, see dd_set_option("sketch_k_per_pass", n)

// The k sets that get their own instantiation (no per-k mask tests, constant table slots): the sweeps
// DandD actually runs -- config 2 (10..32), `--ksweep` default (2..32), the store's all-k prefetch
// (1..32).  Anything else takes the generic kernel.
constexpr uint32_t kMask10to32 = 0xFFFFFE00u, kMask2to32 = 0xFFFFFFFEu, kMask1to32 = 0xFFFFFFFFu;

using SketchKernel = void (*)(SketchArgs);
struct SketchVariant {
    SketchKernel fn;
    int threads;
    int id;   // index into the occupancy cache
};
static SketchVariant pick_kernel(bool canon, uint32_t kmask, uint32_t kmask_run, bool midk) {
    if (midk && kmask == kmask_run && (kmask == kMask2to32 || kmask == kMask1to32)) {
        const int id = 10 + (kmask == kMask1to32 ? 2 : 0) + (canon ? 1 : 0);
        switch (id) {
            case 10: return {sketch_allk_kernel<false, kMask2to32, kThreadsSmallK, true>, kThreadsSmallK, id};
            case 11: return {sketch_allk_kernel<true, kMask2to32, kThreadsSmallK, true>, kThreadsSmallK, id};
            case 12: return {sketch_allk_kernel<false, kMask1to32, kThreadsSmallK, true>, kThreadsSmallK, id};
            default: return {sketch_allk_kernel<true, kMask1to32, kThreadsSmallK, true>, kThreadsSmallK, id};
        }
    }
    int v = 0;
    if (kmask == kmask_run) v = kmask == kMask10to32 ? 1 : kmask == kMask2to32 ? 2 : kmask == kMask1to32 ? 3 : 0;
    const bool small_k = (kmask_run & kSmallKMask) != 0u;
    if (v == 0 && small_k) v = 4;   // generic mask with a small k: the wide persistent CTA
    const int id = 2 * v + (canon ? 1 : 0);
    switch (id) {
        case 0: return {sketch_allk_kernel<false, 0u, kThreadsPlain>, kThreadsPlain, id};
        case 1: return {sketch_allk_kernel<true, 0u, kThreadsPlain>, kThreadsPlain, id};
        case 2: return {sketch_allk_kernel<false, kMask10to32, kThreadsPlain>, kThreadsPlain, id};
        case 3: return {sketch_allk_kernel<true, kMask10to32, kThreadsPlain>, kThreadsPlain, id};
        case 4: return {sketch_allk_kernel<false, kMask2to32, kThreadsSmallK>, kThreadsSmallK, id};
        case 5: return {sketch_allk_kernel<true, kMask2to32, kThreadsSmallK>, kThreadsSmallK, id};
        case 6: return {sketch_allk_kernel<false, kMask1to32, kThreadsSmallK>, kThreadsSmallK, id};
        case 7: return {sketch_allk_kernel<true, kMask1to32, kThreadsSmallK>, kThreadsSmallK, id};
        case 8: return {sketch_allk_kernel<false, 0u, kThreadsSmallK>, kThreadsSmallK, id};
        default: return {sketch_allk_kernel<true, 0u, kThreadsSmallK>, kThreadsSmallK, id};
    }
}

// SM count x resident CTAs per SM for the persistent (small-k) launch, cached per (device, variant).
static unsigned persistent_grid(const SketchVariant &v, size_t smem) {
    constexpr int kMaxDev = 64;
    static unsigned cached[kMaxDev][14] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    unsigned local = 0;
    unsigned &g = (dev >= 0 && dev < kMaxDev) ? cached[dev][v.id] : local;
    if (g == 0) {
        int sms = 148, per_sm = 1;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (smem > 48 * 1024) cudaFuncSetAttribute(v.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, v.fn, v.threads, smem);
        g = (unsigned)(sms * (per_sm > 0 ? per_sm : 1));
    }
    return g;
}

int g_midk = 1;   // dd_set_option("sketch_midk", 0/1): tuning knob, never changes results
int g_sink = 1;   // dd_set_option("sketch_sink", 0/1): A/B switch for the rank-1 sink, never changes results

// resident sink CTAs on this device (its SM count x CTAs per SM at one slab of shared memory), cached
static unsigned sink_resident(bool canon, int p) {
    constexpr int kMaxDev = 64;
    static unsigned cached[kMaxDev][2][kSinkMaxP + 1] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) cudaGetLastError();
    unsigned local = 0;
    unsigned &g = (dev >= 0 && dev < kMaxDev) ? cached[dev][canon ? 1 : 0][p] : local;
    if (g == 0) {
        const auto fn = canon ? sketch_sink_kernel<true> : sketch_sink_kernel<false>;
        int sms = 148, per_sm = 1;   // (no device: a B200's count, for the workspace size alone)
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sink_slab_words(kSinkMaxP) * 4)) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kSinkThreads, sink_slab_words(p) * 4) != cudaSuccess) {
            cudaGetLastError();
            return 148;
        }
        g = (unsigned)(sms * (per_sm > 0 ? per_sm : 1));
    }
    return g;
}
// CTAs (and slabs) per k of a sink launch over nk_sink k values: the resident CTAs shared among them
static unsigned sink_slices(bool canon, int p, unsigned nk_sink) {
    const unsigned resident = sink_resident(canon, p);
    return resident / nk_sink > 0 ? resident / nk_sink : 1u;
}
// slabs of a workspace: nk_sink x sink_slices(nk_sink) <= max(resident, nk) for any launch into it
static size_t sink_slab_count(int nk, int p) {
    if (p > kSinkMaxP) return 0;
    const size_t resident = max(sink_resident(true, p), sink_resident(false, p));
    return max(resident, (size_t)nk);
}

static size_t round256(size_t b) { return (b + 255) / 256 * 256; }
static size_t acc_bytes(int nk, int p) { return round256((size_t)nk * sizeof(uint16_t) * ((size_t)1 << p)); }
static size_t written_bytes(int nk, int p) { return round256(sink_slab_count(nk, p) * sizeof(uint32_t)); }
static constexpr size_t kMidKBytes = (size_t)kMidKWords * sizeof(uint32_t);
// [header | scratch | accumulators | slab-written flags | mid-k bitmaps | rank-1 sink slabs [k][slice][2^p / 32] u32]
size_t sketch_workspace_bytes(int nk, int p) {
    return sizeof(SketchWsHeader) + 256 + acc_bytes(nk, p) + written_bytes(nk, p) + kMidKBytes +
           sink_slab_count(nk, p) * sink_slab_words(p) * sizeof(uint32_t);
}
static SketchWsHeader *ws_hdr(void *ws) { return static_cast<SketchWsHeader *>(ws); }
static uint32_t *ws_scratch(void *ws) { return reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(ws) + sizeof(SketchWsHeader)); }
static uint32_t *ws_acc(void *ws) { return reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(ws) + sizeof(SketchWsHeader) + 256); }
static uint32_t *ws_written(void *ws, int nk, int p) {
    return reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(ws) + sizeof(SketchWsHeader) + 256 + acc_bytes(nk, p));
}
static uint32_t *ws_midk(void *ws, int nk, int p) {
    return reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(ws_written(ws, nk, p)) + written_bytes(nk, p));
}
static uint32_t *ws_slabs(void *ws, int nk, int p) {
    return reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(ws_midk(ws, nk, p)) + kMidKBytes);
}

cudaError_t sketch_begin(void *d_ws, int nk, int p, cudaStream_t stream) {
    // header, scratch, accumulators, slab-written flags and the k <= 12 bitmaps; the 8 + 32 MiB of k = 13 / 14
    // are zeroed by the launch that first consults them (only streams longer than 4^13 symbols ever do), and a
    // slab is only read once its flag says a sink CTA has written it
    return cudaMemsetAsync(d_ws, 0,
                           sizeof(SketchWsHeader) + 256 + acc_bytes(nk, p) + written_bytes(nk, p) + (size_t)midk_offset(13) * sizeof(uint32_t),
                           stream);
}

static cudaError_t sketch_update_impl(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                                      uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint32_t kmask, int p,
                                      int canon, void *d_ws, int midk_hi, bool sink, cudaStream_t stream);

cudaError_t sketch_update(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                          uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint32_t kmask, int p,
                          int canon, void *d_ws, cudaStream_t stream) {
    return sketch_update_impl(d_codes, d_invalid, d_state, sym_begin, sym_end, max_new_symbols, kmask, p, canon, d_ws, 0, false,
                              stream);
}

// sink = the caller allows the rank-1 sink for this range (it ends before the first floor cut); it is used
// for the k >= 10 of the mask when p fits the shared-memory bitmap and every CTA gets >= 2^p / 4 symbols
static cudaError_t sketch_update_impl(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                                      uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint32_t kmask, int p,
                                      int canon, void *d_ws, int midk_hi, bool sink, cudaStream_t stream) {
    const bool midk = midk_hi >= 12;
    SketchArgs a;
    a.codes = d_codes;
    a.invalid = d_invalid;
    a.state = d_state;
    a.sym_begin = sym_begin;
    a.sym_end = sym_end;
    a.kmask = kmask;
    a.kmask_run = kmask;
    a.p = p;
    a.acc = ws_acc(d_ws);
    a.midk = ws_midk(d_ws, __builtin_popcount(kmask), p);
    a.midk_hi = midk_hi;
    a.hdr = ws_hdr(d_ws);
    if (d_state && sym_end <= sym_begin) {   // state-relative range not given: the whole last pack call
        a.sym_begin = 0;
        a.sym_end = ~0ull;
    }
    size_t nsym = d_state ? max_new_symbols : (size_t)(sym_end - sym_begin);
    if (d_state && a.sym_end != ~0ull) {      // grid sized for the sub-range only
        const uint64_t hi = a.sym_end < (uint64_t)max_new_symbols ? a.sym_end : (uint64_t)max_new_symbols;
        nsym = hi > a.sym_begin ? (size_t)(hi - a.sym_begin) : 0;
    }
    if (nsym == 0) return cudaSuccess;
    // +2 words: the range may start and end in the middle of a word
    const size_t nwords = (nsym + 15) / 16 + 2;

    // Optionally split the k set over several launches so that the accumulators touched by one
    // launch (2^(p+1) bytes per k) stay L2-resident; 0 = all k in one launch.
    const int per_pass = g_k_per_pass > 0 ? g_k_per_pass : 32;
    uint32_t todo = kmask;
    const uint32_t sink_mask = kmask & ~kSmallKMask;
    if (sink && sink_mask && p <= kSinkMaxP) {
        const unsigned nk_sink = (unsigned)__builtin_popcount(sink_mask);
        const unsigned slices = sink_slices(canon != 0, p, nk_sink);
        if (nsym >= (size_t)slices * (((size_t)1 << p) / 4)) {
            const int nk = __builtin_popcount(kmask);
            a.kmask_run = sink_mask;
            const auto fn = canon ? sketch_sink_kernel<true> : sketch_sink_kernel<false>;
            DD_COUNT_LAUNCH(), fn<<<nk_sink * slices, kSinkThreads, sink_slab_words(p) * sizeof(uint32_t), stream>>>(
                a, ws_slabs(d_ws, nk, p), ws_written(d_ws, nk, p), slices, ws_hdr(d_ws));
            todo &= kSmallKMask;
        }
    }
    while (todo) {
        uint32_t run = 0;
        for (int c = 0; c < per_pass && todo; ++c) {
            const uint32_t low = todo & (0u - todo);
            run |= low;
            todo ^= low;
        }
        a.kmask_run = run;
        // Small k present: persistent CTAs (they must live long for their bitmaps to pay off) with
        // the bitmaps in dynamic shared memory; otherwise one CTA per tile and no shared memory.
        const bool small_k = (run & kSmallKMask) != 0u;
        const size_t smem = small_k ? kBitmapWords * sizeof(uint32_t) : 0;
        const SketchVariant v = pick_kernel(canon != 0, kmask, run, midk);
        const size_t ntiles = (nwords + v.threads - 1) / v.threads;
        if (ntiles > 0xffffffffull) return cudaErrorInvalidValue;
        a.ntiles = (uint32_t)ntiles;
        unsigned grid = (unsigned)ntiles;
        if (small_k) {
            const unsigned resident = persistent_grid(v, smem);
            if (grid > resident) grid = resident;
        }
        DD_COUNT_LAUNCH(), v.fn<<<grid, v.threads, smem, stream>>>(a);
    }
    return cudaGetLastError();
}

// Update + floor schedule.  The per-k floor (min register) rises by one each time the number of
// k-mers seen doubles, first reaching 1 at about 14 x 2^p k-mers (every register occupied), and an
// update whose rank does not exceed it is dropped before the reduction.  So the range is cut at
// 16 x 2^p x 2^i symbols (i = 0, 1, ...) counted from the start of the sketch and the floor is
// refreshed at each cut: a handful of 10 us refreshes turn most of a long genome's reductions into
// one compare.  `seen_before` = symbols sketched into this workspace by earlier calls (host-side
// count; an estimate only shifts the cuts, never the result).
cudaError_t sketch_update_sched(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                                uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint64_t seen_before,
                                uint32_t kmask, int p, int canon, void *d_ws, cudaStream_t stream) {
    const uint64_t total = d_state ? (uint64_t)max_new_symbols : sym_end - sym_begin;
    const uint64_t origin = d_state ? 0 : sym_begin;   // state mode: ranges are relative to the pack call's first symbol
    uint64_t pos = 0;                       // symbols of this call already issued
    uint64_t cut = (uint64_t)16 << p;       // next cut, counted from the start of the sketch
    while (cut <= seen_before) cut <<= 1;
    cudaError_t e;
    while (pos < total) {
        const uint64_t to_cut = cut - (seen_before + pos);
        const bool refresh = to_cut <= total - pos;
        const uint64_t upto = refresh ? pos + to_cut : total;
        // a k's presence bitmap pays off once the stream is >= 4^k symbols long: k <= 12 from 2^24 symbols on,
        // k = 13 from 2^26, k = 14 from 2^28 (their bitmaps are zeroed when they are first consulted)
        const uint64_t at = seen_before + pos, at_end = seen_before + upto;
        const bool wide = kmask == kMask2to32 || kmask == kMask1to32;
        const int midk_hi = !g_midk || !wide || at < ((uint64_t)1 << 24) ? 0 : at < ((uint64_t)1 << 26) ? 12 : at < ((uint64_t)1 << 28) ? 13 : 14;
        // the piece during which the stream crosses 4^13 (4^14) symbols zeroes that bitmap for the pieces after it;
        // the kernel only trusts a bitmap the header says has been zeroed since dd_sketch_begin
        if (g_midk && wide)
            for (int k = 13; k <= kMidKHi; ++k) {
                const uint64_t T = (uint64_t)1 << (2 * k);
                if (at < T && T <= at_end) {
                    uint32_t *mk = ws_midk(d_ws, __builtin_popcount(kmask), p);
                    if ((e = cudaMemsetAsync(mk + midk_offset(k), 0, (size_t)(midk_offset(k + 1) - midk_offset(k)) * sizeof(uint32_t),
                                             stream)) != cudaSuccess)
                        return e;
                    DD_COUNT_LAUNCH(), midk_ready_kernel<<<1, 1, 0, stream>>>(ws_hdr(d_ws), (uint32_t)k);
                }
            }
        // before the first cut the floor is 0 and half of all updates have rank 1: absorb them in the sink;
        // past it the floor drops them for free and the plain kernels are the right ones.  The sink kernel has no
        // floor test, which stays exact even under a floor raised by hand: a floor is a minimum register, so an
        // update of rank <= floor cannot raise any register.
        const bool sink = g_sink && at_end <= ((uint64_t)16 << p);
        if ((e = sketch_update_impl(d_codes, d_invalid, d_state, origin + pos, origin + upto, max_new_symbols, kmask, p, canon, d_ws,
                                    midk_hi, sink, stream)) != cudaSuccess)
            return e;
        pos = upto;
        if (refresh) {
            if ((e = sketch_refresh_floor(d_ws, kmask, p, stream)) != cudaSuccess) return e;
            cut <<= 1;
        }
    }
    return cudaSuccess;
}

cudaError_t sketch_refresh_floor(void *d_ws, uint32_t kmask, int p, cudaStream_t stream) {
    const int nk = __builtin_popcount(kmask);
    cudaError_t e = cudaMemsetAsync(ws_scratch(d_ws), 0xff, 32 * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    if ((e = sink_merge(ws_slabs(d_ws, nk, p), ws_hdr(d_ws), nk, p, stream)) != cudaSuccess) return e;
    DD_COUNT_LAUNCH(), floor_min_kernel<<<dim3(16, nk), 256, 0, stream>>>(ws_acc(d_ws), ws_slabs(d_ws, nk, p), p, ws_hdr(d_ws),
                                                                          ws_scratch(d_ws));
    DD_COUNT_LAUNCH(), floor_publish_kernel<<<1, 32, 0, stream>>>(ws_hdr(d_ws), ws_scratch(d_ws), kmask);
    return cudaGetLastError();
}

cudaError_t sketch_end(void *d_ws, int nk, int p, uint8_t *d_regs, uint32_t *d_hist, double *d_cards,
                       cudaStream_t stream) {
    cudaError_t e;
    if (d_hist && (e = cudaMemsetAsync(d_hist, 0, (size_t)nk * DD_HIST_BINS * sizeof(uint32_t), stream)) != cudaSuccess)
        return e;
    if ((e = sink_merge(ws_slabs(d_ws, nk, p), ws_hdr(d_ws), nk, p, stream)) != cudaSuccess) return e;
    const unsigned slices = (unsigned)((((size_t)1 << p) + kFinChunk - 1) / kFinChunk);
    DD_COUNT_LAUNCH(), finalize_kernel<<<dim3(slices, nk), kPhThreads, 0, stream>>>(ws_acc(d_ws), ws_slabs(d_ws, nk, p), ws_hdr(d_ws), p, d_regs,
                                                                                        d_hist);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (d_hist && d_cards) return mle_from_hist(d_hist, nk, p, d_cards, stream);
    return cudaSuccess;
}

}  // namespace dd
