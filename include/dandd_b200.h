/*
 * dandd_b200.h -- C ABI of the B200-native DandD sketch-and-count hot path.
 *
 * The reference (jessicabonnie/dandd) has NO FFI: its seam to the arithmetic is a set of shell
 * command strings built by SketchObj subclasses and run through subprocess.  Each entry point
 * below replaces one of those command lines; the citation gives the reference site (paths are
 * relative to the reference repository root).  INTEGRATION.md shows the ctypes stubs a reference
 * maintainer would add at those sites.
 *
 * Conventions
 *   - Every function returns DD_OK (0) or a negative DD_ERR_* code; dd_last_error() returns a
 *     thread-local message for the last failure.  There is no CPU fallback: on a machine without
 *     an sm_100 device dd_init() fails and nothing else may be called.
 *   - The caller owns every buffer.  Pointers named d_* are DEVICE pointers (e.g. torch tensors'
 *     data_ptr()), pointers named h_* are HOST pointers.  The library allocates nothing that
 *     outlives a call; scratch space is passed in as (d_ws, ws_bytes) sized by the matching
 *     *_workspace_bytes() query.
 *   - All device work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = default
 *     stream) and is asynchronous unless the name ends in _host.
 *   - k values travel as a bit mask: bit (k-1) set <=> k-mer length k is requested, 1 <= k <= 32
 *     (`maxk<=32 for estimation`, README.md:82; lib/huffman_dandd.py:109-110).  "slot" j of a
 *     [nk][...] output is the j-th set bit of the mask in increasing k.
 *   - A sketch is 2^p one-byte HyperLogLog registers (p = --registers, default 20,
 *     lib/dandd_cmd.py:187), bit-identical to what `dashing sketch -S p` builds (SURVEY.md A.5).
 */
#ifndef DANDD_B200_H
#define DANDD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DD_ABI_VERSION 2

#define DD_OK 0
#define DD_ERR_ARG (-1)       /* bad argument (null pointer, k/p out of range, ...) */
#define DD_ERR_CUDA (-2)      /* a CUDA runtime call or kernel launch failed        */
#define DD_ERR_WORKSPACE (-3) /* workspace smaller than *_workspace_bytes() says    */
#define DD_ERR_DEVICE (-4)    /* no usable sm_100 device                            */
#define DD_ERR_FORMAT (-5)    /* input text needs dd_fastq_to_fasta_host first      */

#define DD_HIST_BINS 64 /* register-value histogram: bin j = #registers == j (j <= 64-p+1 < 64) */

typedef void *dd_stream;

#if defined(__GNUC__)
#define DD_API __attribute__((visibility("default")))
#else
#define DD_API
#endif

DD_API const char *dd_last_error(void);
DD_API int dd_abi_version(void);
/* Number of CUDA kernels this library has launched in this process so far (all threads, all streams;
 * memsets and copies are not kernels).  Lets a benchmark report its launches as a measurement. */
DD_API unsigned long long dd_kernel_launches(void);
/* Select `device` for the calling thread and verify it is compute capability 10.x. */
DD_API int dd_init(int device);
/* Tuning knobs (never change results).  "sketch_k_per_pass" = n: K2 updates at most n k values per
 * kernel launch (0 = all in one), trading re-reads of the packed stream for L2 residency of the
 * accumulators.  "prefix_planes" = 0/1: dd_prefix_union_card uses the bit-sliced kernel (default 1)
 * or the byte kernel.  "prefix_lattice" = 0/1: dd_prefix_union_card answers index-mode jobs of at most 12
 * genomes from a per-k subset table built in one pass over the registers (default 1; for A/B measurement:
 * 0 sends them to the bit-sliced kernel).  "sketch_midk" = 0/1: dd_sketch_update_sched lets pieces deep inside a long stream
 * consult L2-resident presence bitmaps for k = 10..12 before hashing (default 1).  "sketch_sink" = 0/1:
 * dd_sketch_update_sched sketches the k >= 10 of pieces before the first floor cut (p <= 20) with one k per
 * CTA, absorbing rank-1 updates in a shared-memory bitmap instead of L2 reductions (default 1; for A/B
 * measurement).  "polyt_sentinel" = 0/1: the dd_*_host entry points apply dd_pack_polyt_sentinel
 * (this one DOES change results: it selects the SURVEY.md A.6 encoder behaviour; default 0). */
DD_API int dd_set_option(const char *name, long value);
DD_API int dd_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *l2_bytes, size_t *total_mem);

/* ===========================================================================================
 * K1  FASTA text -> packed symbol stream.
 * Replaces the FASTA parsing half of `dashing sketch ... <fasta>` (lib/sketch_classes.py:351-366)
 * and of `kmc ... -fm <fasta>` (lib/sketch_classes.py:434-449).
 *
 * Stream layout (device memory, caller-owned, zero-filled by dd_pack_reset):
 *   codes   : uint32 words, 16 symbols per word, symbol s in word s/16 at bits [31-2(s%16) : 30-2(s%16)]
 *             (first symbol most significant), A/a=0 C/c=1 G/g=2 T/t=3;
 *   invalid : uint32 words, 32 symbols per word, symbol s in word s/32 at bit 31-(s%32); a set bit
 *             means "k-mer windows restart here" (any byte other than ACGTacgt, and one synthetic
 *             symbol per '>' header line so that k-mers never span records);
 *   state   : dd_pack_state, carried from chunk to chunk so a FASTA can be streamed.
 * Text rules (SURVEY.md A.1, klib kseq_read() as used by Dashing and by KMC's -fm mode): a line
 * whose first byte is '>' or '@' is a record header; '\n' and '\r' are not sequence; text before
 * the first '>' / '@' of a file must be skipped by the caller (dd_*_host do it).  A line whose
 * first byte is '+' opens a FASTQ quality section, whose extent depends on the record's sequence
 * length: the packer does not interpret it, it sets DD_PACK_FLAG_FASTQ in dd_pack_state.reserved and
 * the caller must pass such text through dd_fastq_to_fasta_host first (dd_sketch_fasta_host does).
 * =========================================================================================== */
#define DD_PACK_FLAG_OVERFLOW 1u /* more symbols than cap_symbols: the excess was dropped            */
#define DD_PACK_FLAG_FASTQ 2u    /* a line begins with '+': FASTQ, results are NOT what kseq yields  */
typedef struct dd_pack_state {
    uint64_t nsym;      /* symbols in the stream so far                                   */
    uint64_t prev_nsym; /* value of nsym before the most recent dd_pack_fasta call        */
    uint32_t in_header; /* 1 if the text consumed so far ends inside a header line        */
    uint32_t last_byte; /* last text byte consumed ('\n' initially: start of a line)      */
    uint64_t reserved;  /* DD_PACK_FLAG_* bits (sticky)                                   */
} dd_pack_state;

/* HOST helper, no GPU work: rewrite FASTA/FASTQ text the way kseq_read() walks it into plain
 * FASTA that dd_pack_fasta packs to the same symbols -- record markers found anywhere while no
 * record is open, '+' lines and quality lines (as many bytes as the record has sequence bytes, at
 * least one line) dropped, a record with a quality/sequence length mismatch and everything after
 * it dropped (kseq_read returns an error there and the reader loop ends).  h_out must hold
 * n_bytes + 16 bytes and may not overlap h_in; returns the number of bytes written. */
DD_API size_t dd_fastq_to_fasta_host(const uint8_t *h_in, size_t n_bytes, uint8_t *h_out);
/* Offset of the first record marker ('>' or '@') in host text, n_bytes if there is none. */
DD_API size_t dd_fasta_first_record_host(const uint8_t *h_text, size_t n_bytes);

DD_API size_t dd_pack_codes_bytes(size_t max_text_bytes);
DD_API size_t dd_pack_invalid_bytes(size_t max_text_bytes);
DD_API size_t dd_pack_workspace_bytes(size_t chunk_bytes);
DD_API int dd_pack_reset(uint32_t *d_codes, size_t codes_bytes, uint32_t *d_invalid, size_t invalid_bytes,
                  dd_pack_state *d_state, dd_stream stream);
/* Append the symbols of text chunk [d_text, d_text+n_bytes) to the stream.  d_text should be
 * 16-byte aligned for full speed.  cap_symbols = capacity of codes/invalid in symbols. */
DD_API int dd_pack_fasta(const uint8_t *d_text, size_t n_bytes, uint32_t *d_codes, uint32_t *d_invalid,
                  size_t cap_symbols, dd_pack_state *d_state, void *d_ws, size_t ws_bytes, dd_stream stream);

/* Optional emulation of the encoder quirk recalled in SURVEY.md A.6 (UNVERIFIED, off by default):
 * bonsai's unwindowed encoder tests its 64-bit accumulator against all-ones to detect an invalid
 * base, and 32 consecutive 'T' make a legitimate accumulator all-ones too.  With this pass every
 * 32nd 'T' of a run of T/t becomes a break symbol, for symbols [sym_begin, sym_end) -- or
 * [d_state->prev_nsym, d_state->nsym) when d_state != NULL (max_symbols bounds the grid) -- so
 * call it after each dd_pack_fasta, before dd_sketch_update.  dd_set_option("polyt_sentinel", 1)
 * makes the dd_*_host entry points do so. */
DD_API int dd_pack_polyt_sentinel(const uint32_t *d_codes, uint32_t *d_invalid, const dd_pack_state *d_state, uint64_t sym_begin,
                           uint64_t sym_end, size_t max_symbols, dd_stream stream);

/* ===========================================================================================
 * K2  fused all-k canonical-k-mer HyperLogLog sketch.
 * Replaces the whole fan-out
 *     parallel -j 95% ' dashing sketch [--no-canon] -k{} -S p --prefix DIR fasta ' ::: k1 k2 ...
 * (lib/huffman_dandd.py:217 building lib/sketch_classes.py:351-366): one pass over the packed
 * stream updates the registers of every requested k.
 *   begin  : zero the accumulators held in the workspace;
 *   update : sketch stream symbols [state.prev_nsym, state.nsym) (k-mers ENDING in that range, so
 *            chunked packing + update is exact), or an explicit [sym_begin, sym_end) range;
 *   end    : write the final u8 registers [nk][2^p], and optionally the register histograms and
 *            Ertl-MLE cardinalities (what `dashing card` would print for each of the nk sketches).
 * canon = 1 hashes min(kmer, reverse complement) (default), 0 = --no-canon
 * (lib/sketch_classes.py:20-29).
 * =========================================================================================== */
DD_API size_t dd_sketch_workspace_bytes(int nk, int p);
DD_API int dd_sketch_begin(void *d_ws, size_t ws_bytes, int nk, int p, dd_stream stream);
DD_API int dd_sketch_update(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                     size_t max_new_symbols, uint32_t kmask, int p, int canon, void *d_ws, size_t ws_bytes,
                     dd_stream stream);
DD_API int dd_sketch_update_range(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                           uint32_t kmask, int p, int canon, void *d_ws, size_t ws_bytes, dd_stream stream);
/* dd_sketch_update plus the floor schedule: the per-k lower bound min(register) rises by one every
 * time the number of k-mers seen doubles (first at about 14 x 2^p), and an update that cannot exceed
 * it is dropped before the reduction.  This entry cuts the range at 16 x 2^p x 2^i symbols counted
 * from the start of the sketch and refreshes the bound at each cut.  seen_before = symbols sketched
 * into this workspace by earlier calls (a host-side count; an estimate only moves the cuts).  With
 * d_state != NULL the range is the last dd_pack_fasta call's and [sym_begin, sym_end) is ignored. */
DD_API int dd_sketch_update_sched(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                           uint64_t sym_begin, uint64_t sym_end, size_t max_new_symbols, uint64_t seen_before,
                           uint32_t kmask, int p, int canon, void *d_ws, size_t ws_bytes, dd_stream stream);
/* Recompute the per-k lower bound min(register) used to skip no-op updates (long genomes). */
DD_API int dd_sketch_refresh_floor(void *d_ws, size_t ws_bytes, uint32_t kmask, int p, dd_stream stream);
DD_API int dd_sketch_end(void *d_ws, size_t ws_bytes, int nk, int p, uint8_t *d_regs, uint32_t *d_hist /*[nk][64] or NULL*/,
                  double *d_cards /*[nk] or NULL*/, dd_stream stream);

/* ===========================================================================================
 * K4  cardinality: register histogram + Ertl maximum-likelihood estimate.
 * Replaces `dashing card --presketched <paths...>` (lib/sketch_classes.py:306-321); d_cards[i] is
 * the number the reference would store in cardkey[path_i].  d_hist ([nsk][64] uint32) receives the
 * histograms and doubles as scratch; it must be provided.
 * =========================================================================================== */
DD_API int dd_card_ertl_mle(const uint8_t *d_regs, int nsk, int p, double *d_cards, uint32_t *d_hist, dd_stream stream);
/* Estimator alone, from histograms (host-callable building block; also used by K3/K6). */
DD_API int dd_mle_from_hist(const uint32_t *d_hist, int nsk, int p, double *d_cards, dd_stream stream);
/* The same estimator on fractional counts, d_hist [nsk][64] f64 (mean histograms: K14).  On integer counts it gives
 * the floats dd_mle_from_hist gives. */
DD_API int dd_mle_from_hist_f64(const double *d_hist, int nsk, int p, double *d_cards, dd_stream stream);

/* ===========================================================================================
 * K3  unions.
 * dd_union_max replaces `dashing union -z -o OUT in1 .. inN` (lib/sketch_classes.py:368-373):
 * d_in is a DEVICE array of n_in device pointers, each to `len` bytes; d_out = element-wise max.
 *
 * dd_prefix_union_card replaces the progressive-union loop (lib/huffman_dandd.py:624-663): for
 * every ordering o and step i it forms the union of genomes order[o][0..i] and its cardinality
 * for each of the nk sketches per genome -- as a running max, n reads instead of the reference's
 * n(n+1)/2.  Entries of d_order < 0 are skipped (ragged orderings).
 *   d_regs   [n_genomes][nk][2^p] u8         d_order [n_ord][n_steps] int32
 *   d_cards  [n_ord][n_steps][nk] f64        d_hist  [n_ord][n_steps][nk][64] u32 (scratch+output)
 *   d_unions NULL, or [n_ord][n_steps][nk][2^p] u8 to materialise every prefix union
 *   final_only != 0: only the union of each whole ordering is estimated/materialised -- the n-ary
 *   union of a tree node (lib/huffman_dandd.py:412-438); the step dimension of the outputs then
 *   has extent 1: d_cards [n_ord][nk], d_hist [n_ord][nk][64], d_unions [n_ord][nk][2^p].
 * =========================================================================================== */
/* dd_union_sets_card: the same running-max + histogram + MLE over arbitrary sketches given by
 * address.  d_members is a DEVICE array [n_sets][n_steps] of device pointers to 2^p-byte sketches
 * (NULL entries are skipped).  Set s, step i covers members[s][0..i].  This is the form the
 * drop-in sketch objects use: one launch evaluates the union of a tree node for every k
 * (n_sets = nk, final_only = 1), or every prefix of every ordering for every k.
 *   d_cards [n_sets][n_steps or 1] f64   d_hist [n_sets][n_steps or 1][64] u32
 *   d_unions NULL or [n_sets][n_steps or 1][2^p] u8 */
DD_API int dd_union_sets_card(const uint8_t *const *d_members, int n_sets, int n_steps, int p, int final_only,
                              double *d_cards, uint32_t *d_hist, uint8_t *d_unions, dd_stream stream);
DD_API int dd_union_max(const uint8_t *const *d_in, int n_in, size_t len, uint8_t *d_out, dd_stream stream);
/* Scratch: (d_ws, ws_bytes) sized by dd_prefix_union_workspace_bytes() lets the call use the bit-plane
 * kernel (it holds the transposed sketches and the identical-prefix table) or, for n_genomes <= 12 and
 * p >= 12 except pairs (final_only with two steps), the subset table ([nk][64][2^n_genomes] u32): every
 * prefix union of every ordering is then read from one pass over the registers.  With d_ws == NULL, or
 * when d_unions != NULL, the byte kernel runs, which needs no scratch. */
DD_API size_t dd_prefix_union_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk, int p);
DD_API int dd_prefix_union_card(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                         int nk, int p, int final_only, double *d_cards, uint32_t *d_hist, uint8_t *d_unions,
                         void *d_ws, size_t ws_bytes, dd_stream stream);

/* Bit planes: a sketch of 2^p one-byte registers transposed into 6 planes of 2^p bits (plane b, word
 * g = bit b of registers 32g..32g+31; ranks are <= 64-p+1 < 64), 0.75 bytes per register.  A caller
 * that unions the same sketches many times (all pairs, many orderings) transposes them ONCE with
 * dd_to_planes and passes the planes to the *_planes entry points; p >= 12.
 *   d_planes [n_sketches][6][2^p / 32] u32,  dd_planes_bytes(n_sketches, p) bytes
 * dd_prefix_union_card_planes: d_planes laid out [n_genomes][nk]; scratch only for the
 * identical-prefix table, dd_prefix_union_workspace_bytes(n_ord, n_steps, 0, 0, p) bytes (NULL = none). */
DD_API size_t dd_planes_bytes(int64_t n_sketches, int p);
DD_API int dd_to_planes(const uint8_t *d_regs, int64_t n_sketches, int p, uint32_t *d_planes, dd_stream stream);
DD_API int dd_prefix_union_card_planes(const uint32_t *d_planes, const int32_t *d_order, int n_ord, int n_steps,
                                int n_genomes, int nk, int p, int final_only, double *d_cards, uint32_t *d_hist,
                                void *d_ws, size_t ws_bytes, dd_stream stream);

/* ===========================================================================================
 * K6  all-pairs union cardinalities (the shape of lib/huffman_dandd.py:666-695 and
 * helpers/allpairs.py:360-370): for each listed pair (a,b) and each of the nk sketches,
 * card(max(regs[a], regs[b])).
 *   d_pairs [n_pairs][2] int32      d_cards [n_pairs][nk] f64     d_hist [n_pairs][nk][64] u32
 * dd_pairwise_union_card transposes d_regs into (d_ws, ws_bytes) -- dd_prefix_union_workspace_bytes(0, 0,
 * n_genomes, nk, p) bytes -- on every call (NULL: byte kernel); dd_pairwise_union_card_planes takes
 * sketches already transposed by dd_to_planes, so tiles of a large pair matrix share one transpose.
 * =========================================================================================== */
DD_API int dd_pairwise_union_card(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *d_pairs,
                           int64_t n_pairs, double *d_cards, uint32_t *d_hist, void *d_ws, size_t ws_bytes,
                           dd_stream stream);
DD_API int dd_pairwise_union_card_planes(const uint32_t *d_planes, int n_genomes, int nk, int p, const int32_t *d_pairs,
                                  int64_t n_pairs, double *d_cards, uint32_t *d_hist, dd_stream stream);

/* ===========================================================================================
 * K10  leave-one-group-out unions (what lib/huffman_dandd.py:559-566 find_delta_delta asks per subset:
 * a fresh SubSpider over the remaining genomes, climbed union by union).  One read of the registers gives
 * the histograms of the union of all genomes and of the union of every genome outside each group.
 *   d_regs  [n_genomes][nk][2^p] u8 (the layout of dd_pairwise_union_card), 16-byte aligned
 *   d_group [n_genomes] int32, group of each genome in [0, n_groups), any order;
 *           1 <= n_groups <= min(n_genomes, 65535).
 *           It is read back to the host and checked before any launch (the call synchronises the stream).
 *   [reg_begin, reg_end) register range of every k, multiples of 16, reg_end <= 2^p
 *   d_hist  [nk][1 + n_groups][64] u32, ADDED to (the caller zeroes it): row 0 is the union of all genomes,
 *           row 1 + g the union of every genome not in group g.  Calls over disjoint register ranges, on one
 *           device or on several, add up to the histograms of the whole range.
 *   d_ws    dd_leave_out_workspace_bytes(n_genomes, nk) bytes of scratch
 * nk * (1 + n_groups) * 64 < 2^31.  Cardinalities: dd_mle_from_hist over the nk * (1 + n_groups) rows.
 * =========================================================================================== */
DD_API size_t dd_leave_out_workspace_bytes(int n_genomes, int nk);
DD_API int dd_leave_out_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *d_group, int n_groups,
                             uint64_t reg_begin, uint64_t reg_end, uint32_t *d_hist, void *d_ws, size_t ws_bytes,
                             dd_stream stream);

/* ===========================================================================================
 * K14  register sharing spectrum (what `progressive -n N` samples from the orderings lib/huffman_dandd.py:618-663 climbs
 * one union at a time, averaged over all n! orderings).  For register r and value v let c_v(r) = #{g : x_g(r) >= v};
 * the union of a subset S has max >= v at r exactly when S meets those c_v(r) genomes, so the mean register histogram
 * of the m-prefix union over all orderings follows from T[k][v][c] = #{r : c_v(r) = c} in closed form.  One read of
 * the registers.
 *   d_regs  [n_genomes][nk][2^p] u8 (the layout of dd_pairwise_union_card), 16-byte aligned; 1 <= n_genomes <= 65535
 *   [reg_begin, reg_end) register range of every k, multiples of 16, reg_end <= 2^p
 *   d_spec  [nk][64][n_genomes] u32, ADDED to (the caller zeroes it): entry (k, v, c - 1) = T[k][v][c] over the range;
 *           row v = 0 stays 0.  Values are clamped at 63 as dd_card_ertl_mle's histogram clamps them, so row v sums to
 *           the union's registers >= v.  Calls over disjoint register ranges, on one device or on several, add up.
 *   d_ws    dd_register_spectrum_workspace_bytes(n_genomes, nk) bytes of scratch, 4-byte aligned
 * nk * 64 * n_genomes < 2^31.  Every argument is checked before any launch.  Cardinalities: the mean histograms
 * (helpers/spectrum.py hit_weights) through dd_mle_from_hist_f64.
 * =========================================================================================== */
DD_API size_t dd_register_spectrum_workspace_bytes(int n_genomes, int nk);
DD_API int dd_register_spectrum(const uint8_t *d_regs, int n_genomes, int nk, int p, uint64_t reg_begin, uint64_t reg_end,
                                uint32_t *d_spec, void *d_ws, size_t ws_bytes, dd_stream stream);

/* ===========================================================================================
 * K11  one step of a greedy ordering (a chosen ordering for `progressive -r`, lib/huffman_dandd.py:618-663
 * orderings_list, where the reference would climb one SubSpider union per candidate per step).  U is the running
 * union; for every listed candidate g and every k these give the histogram of max(U, g), as hist(U) plus one
 * -1 / +1 pair per "live" register where g > U, and the number of live registers.
 *   d_regs      [n_genomes][nk][2^p] u8 (the layout of dd_pairwise_union_card), 16-byte aligned
 *   d_union     [nk][2^p] u8, 16-byte aligned; register values < 64
 *   d_union_hist [nk][64] u32, the histogram of d_union (dd_card_ertl_mle's d_hist)
 *   h_cand      [n_cand] int32 HOST array of distinct genome indices in [0, n_genomes); n_cand >= 1
 *   d_hist      [n_cand][nk][64] u32, written: row (c, k) is the histogram of max(U, regs[h_cand[c]][k])
 *   d_live      [n_cand][nk] u32, written: registers where regs[h_cand[c]][k] > U[k]
 *   d_ws        dd_greedy_workspace_bytes(n_cand) bytes of scratch, 16-byte aligned
 * n_cand * nk * 64 < 2^31.  Cardinalities: dd_mle_from_hist over the n_cand * nk rows.
 *
 * dd_greedy_dense_hist reads every register of every candidate.  dd_greedy_compact writes the live registers of
 * every candidate as entries `j << 6 | value` (u32) into segment g * nk + k of d_entries:
 *   h_seg_off   [n_genomes * nk + 1] int64 HOST offsets, starting at 0, non-decreasing, last <= n_entries;
 *               the capacity of segment s is h_seg_off[s + 1] - h_seg_off[s] (live counts of an earlier U bound it)
 *   d_seg_off   [n_genomes * nk + 1] int64, written: a device copy of h_seg_off
 *   d_seg_len   [n_genomes * nk] u32, written: the live count of each listed segment, 0 elsewhere
 * dd_greedy_sparse_hist then does a step from the segments alone: it drops the entries with value <= U[k][j],
 * compacts the rest in place, sets d_seg_len to the kept count (also d_live) and counts their pairs.  A segment is
 * clipped to its capacity and to the entry buffer.  Both sparse and dense give the same d_hist and d_live.
 * =========================================================================================== */
DD_API size_t dd_greedy_workspace_bytes(int n_cand);
DD_API int dd_greedy_dense_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union,
                                const uint32_t *d_union_hist, const int32_t *h_cand, int n_cand, uint32_t *d_hist,
                                uint32_t *d_live, void *d_ws, size_t ws_bytes, dd_stream stream);
DD_API int dd_greedy_compact(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union,
                             const int32_t *h_cand, int n_cand, const int64_t *h_seg_off, int64_t *d_seg_off,
                             uint32_t *d_seg_len, uint32_t *d_entries, int64_t n_entries, void *d_ws, size_t ws_bytes,
                             dd_stream stream);
DD_API int dd_greedy_sparse_hist(uint32_t *d_entries, int64_t n_entries, const int64_t *d_seg_off, uint32_t *d_seg_len,
                                 int n_genomes, int nk, int p, const uint8_t *d_union, const uint32_t *d_union_hist,
                                 const int32_t *h_cand, int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws,
                                 size_t ws_bytes, dd_stream stream);

/* ===========================================================================================
 * K5  --exact: number of distinct (canonical) k-mers, KMC semantics (SURVEY.md Appendix B).
 * Replaces `kmc -ci1 -cs2 -kK [-b] -fm ...` + `kmc_tools info` (lib/sketch_classes.py:389-399,
 * 434-449) and, by inserting several streams into one set, `kmc_tools complex` unions (:451-465).
 * The set lives in the workspace: a 4^k-bit presence bitmap when k <= DD_EXACT_BITMAP_MAXK, else
 * an open-addressing table with `capacity` slots (power of two, must exceed the number of distinct
 * k-mers; dd_exact_count reports overflow as DD_ERR_WORKSPACE): 64-bit keys to k = 32, 128-bit keys to
 * k = 64, and for 64 < k <= 256 -- KMC's own limit; the README's "to sweep higher ks you must use KMC
 * via --exact" (README.md:82), helpers/allpairs.py:295 sweeps to 99 -- 16-byte (fingerprint, reference
 * to one occurrence) entries whose matches are verified against the packed stream, so the count stays
 * exact.  In that mode every stream inserted into a set must stay alive and unmodified until the last
 * dd_exact_insert into that set has completed (at most 512 distinct streams per set).
 * 1 <= k <= DD_EXACT_MAXK.
 * =========================================================================================== */
#define DD_EXACT_BITMAP_MAXK 16
#define DD_EXACT_MAXK 256
DD_API size_t dd_exact_workspace_bytes(int k, uint64_t capacity);
DD_API int dd_exact_begin(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, dd_stream stream);
DD_API int dd_exact_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                    int canon, void *d_ws, size_t ws_bytes, uint64_t capacity, dd_stream stream);
/* Multi-GPU exact mode (SURVEY.md 8e: "per-range local distinct + all-reduce SUM"): the same insert
 * restricted to the k-mers of key range `shard_rank` of `shard_world` (a hash of the k-mer decides).
 * Every rank scans the same streams with its own rank; the per-rank dd_exact_count values add up to
 * the count a single dd_exact_insert pass would give, with 1/shard_world of the table per rank. */
DD_API int dd_exact_insert_shard(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                          int k, int canon, void *d_ws, size_t ws_bytes, uint64_t capacity, uint32_t shard_rank,
                          uint32_t shard_world, dd_stream stream);
/* Distinct k-mers inserted since dd_exact_begin -> *d_count (device u64); cumulative, so calling
 * it after each genome gives the progressive exact unions. */
DD_API int dd_exact_count(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t *d_count, dd_stream stream);

/* ===========================================================================================
 * K7  --exact all pairs: |A n B| for every unordered pair of n_genomes genomes at one k, added into
 * d_inter [n_genomes(n_genomes-1)/2] u64, rows in the order (0,1), (0,2) .. (n-2,n-1); the caller forms
 * |A u B| = |A| + |B| - |A n B|.  Replaces the pair unions of `kmc_tools complex` that an exact all-pairs
 * run asks for, one pair and one k at a time (helpers/allpairs.py:38-44,360-370; the SubSpider of each
 * pair in lib/huffman_dandd.py:666-695), with one job that reads every genome once.
 *
 * Sparse path (any k <= DD_EXACT_MAXK): the K5 open-addressing key table (64-bit keys to k = 32, 128-bit
 * to k = 64, verified references above; at every k, no bitmap), plus a (last genome, list head) pair per
 * slot and `max_nodes` list nodes.  dd_exact_pairs_insert pushes `genome` once onto the list of every key
 * of [sym_begin, sym_end) it holds: all ranges of one genome must be inserted before the next genome's
 * (a genome may come in several ranges or streams); `genome` must be below the n_genomes later passed to
 * dd_exact_pairs_accumulate (other indices are not counted).  dd_exact_pairs_accumulate then adds 1 to
 * every pair on a list.  `capacity` (power of two >= 1024) must exceed the distinct keys of the job, `max_nodes`
 * (< 2^32 - 1) the sum over genomes of their distinct keys; `max_streams` (k > 64 only, at most 65536) bounds
 * the distinct streams inserted.  A full table or node array makes dd_exact_pairs_accumulate write all-ones
 * into every row of d_inter: a count is never silently wrong.  _shard restricts the job to key range
 * shard_rank of shard_world exactly as dd_exact_insert_shard does: the shards' results add up.
 *
 * Dense path: dd_exact_pair_popc adds popc(A & B) over K5 presence bitmaps (k <= DD_EXACT_BITMAP_MAXK,
 * filled with dd_exact_begin / dd_exact_insert[_shard]).  d_row_ws points at nr K5 workspaces, ws_stride
 * bytes apart, holding genomes row0 .. row0+nr-1; d_col_ws likewise for col0 .. col0+nc-1 (it may be
 * d_row_ws).  Every pair a < b with a a row and b a column genome is counted; blocks of genomes that do
 * not fit in memory together are covered by calling it for every (row block, column block).
 * =========================================================================================== */
DD_API size_t dd_exact_pairs_workspace_bytes(int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams);
DD_API int dd_exact_pairs_begin(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                uint32_t max_streams, dd_stream stream);
DD_API int dd_exact_pairs_insert_shard(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                                       int k, int canon, uint32_t genome, void *d_ws, size_t ws_bytes, uint64_t capacity,
                                       uint64_t max_nodes, uint32_t max_streams, uint32_t shard_rank, uint32_t shard_world,
                                       dd_stream stream);
DD_API int dd_exact_pairs_accumulate(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                     uint32_t max_streams, int64_t n_genomes, uint64_t *d_inter, dd_stream stream);
DD_API int dd_exact_pair_popc(const void *d_row_ws, int64_t row0, int nr, const void *d_col_ws, int64_t col0, int nc,
                              size_t ws_stride, int k, int64_t n_genomes, uint64_t *d_inter, dd_stream stream);

/* ===========================================================================================
 * K8  --exact unions of many genome sets at one k, from the K7 sparse workspace after every genome has
 * been inserted with dd_exact_pairs_insert_shard (same workspace, same arguments).  d_ranks [n_rows]
 * [n_genomes] u16: row r gives every genome a rank (ties allowed; 0xFFFF = not in the row's family; any
 * other value must be below n_genomes, larger ones are not counted).  Adds into d_hist [n_rows][n_genomes]
 * u64 (the caller zeroes it): hist[r][m] = number of distinct keys whose minimum rank over the genomes
 * holding them, under row r, is m; a key no genome of the row holds is not counted.  So
 *   - a progressive ordering (row = the position of every genome in it): the union of its first i genomes
 *     holds sum(hist[r][0 .. i-1]) k-mers -- the prefix unions of `kmc_tools complex` in
 *     lib/huffman_dandd.py:624-663;
 *   - a set S (row = 0 for its members, 0xFFFF elsewhere): |union of S| = hist[r][0] -- a tree node.
 * n_genomes <= 65535.  A full table or node array writes all-ones into every cell of d_hist.
 * =========================================================================================== */
DD_API int dd_exact_first_rank_hist(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                    uint32_t max_streams, int64_t n_genomes, const uint16_t *d_ranks, int64_t n_rows,
                                    uint64_t *d_hist, dd_stream stream);
/* The K7 sparse workspace's node counter, copied on the stream into the caller's device word d_out (u64; no
 * kernel, no synchronisation).  dd_exact_pairs_insert_shard pushes exactly one node per (genome, key of the
 * range) it holds, so the counter read after a genome's insert minus the one read before it is the number of
 * distinct keys of that genome in the workspace's key range: the single counts |A_g| of a family job come
 * from the lists themselves.  The counter keeps counting past max_nodes; such a job is reported full by
 * dd_exact_pairs_accumulate / dd_exact_first_rank_hist. */
DD_API int dd_exact_pairs_node_count(const void *d_ws, size_t ws_bytes, uint64_t *d_out, dd_stream stream);

/* ===========================================================================================
 * K9  --exact sharing spectrum at one k, from the K7 sparse workspace after every genome has been inserted
 * with dd_exact_pairs_insert_shard (same workspace, same arguments).  A key's list holds one node per genome
 * holding it, so its length is the key's sharing count c.  Adds into d_hist [n_genomes] u64 (the caller
 * zeroes it): d_hist[c - 1] = number of distinct keys held by exactly c of the genomes 0 .. n_genomes-1; and,
 * if d_priv is not NULL, into d_priv [n_genomes] u64: d_priv[g] = number of keys genome g alone holds.  Nodes
 * of a genome index >= n_genomes are not counted.  1 <= n_genomes < 2^32.  With the singles |A_g| (the node
 * counter, dd_exact_pairs_node_count) this gives the core / shell / cloud split of a collection and, in
 * closed form, the mean union and intersection of the first m genomes over all n! orderings.  A full table
 * or node array writes all-ones into every cell of d_hist (and of d_priv).
 * =========================================================================================== */
DD_API int dd_exact_occupancy_hist(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                   uint32_t max_streams, int64_t n_genomes, uint64_t *d_hist, uint64_t *d_priv,
                                   dd_stream stream);

/* ===========================================================================================
 * K13  --exact query genomes against a reference collection at one k, from the K7 sparse workspace after the
 * n_refs references have been inserted with dd_exact_pairs_insert_shard as genomes 0 .. n_refs-1 and then the
 * n_queries queries as genomes n_refs .. n_refs+n_queries-1, in that order (same workspace, same arguments).
 * With A_g genome g's distinct keys and U_R the union of the references, adds into caller-zeroed u64 arrays:
 *   d_inter  [n_queries][n_refs]  inter[q][r] = |A_q n A_r|   (query q is genome n_refs + q)
 *   d_shared [n_queries]          shared[q]   = |A_q n U_R|
 *   d_union  [1]                  |U_R|
 * With the singles |A_g| (the node counter, dd_exact_pairs_node_count): |U_R u A_q| = |U_R| + |A_q| - shared[q]
 * and |A_q u A_r| = |A_q| + |A_r| - inter[q][r].  It stands in for the reference's `kmc_tools complex` union +
 * `kmc_tools info` per query (the collection plus the query) and per (query, reference) pair.  The kernel relies
 * on the insert order: every list holds its genomes in decreasing order, queries first.  Nodes of a genome
 * index >= n_refs + n_queries are not counted.  n_refs >= 1, n_queries >= 1, n_refs + n_queries < 2^32 (at most
 * 65536 above k = 64), n_queries * n_refs <= DD_QUERY_MAX_CELLS.  A full table or node array writes all-ones into
 * every cell of d_inter, d_shared and d_union: never a partial count.
 * =========================================================================================== */
#define DD_QUERY_MAX_CELLS (1ll << 32)
DD_API int dd_exact_query_counts(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                 uint32_t max_streams, int64_t n_refs, int64_t n_queries, uint64_t *d_inter,
                                 uint64_t *d_shared, uint64_t *d_union, dd_stream stream);

/* ===========================================================================================
 * K12  the exact greedy cover index (a chosen ordering for `progressive -r`, lib/huffman_dandd.py:618-663
 * orderings_list, by exact counts: the greedy order where the reference would count one `kmc_tools complex` union
 * per remaining candidate per step).  With A_g genome g's distinct keys and U the union of the genomes chosen so
 * far, |U u A_g| = |U| + |A_g| - lost[g], lost[g] = |A_g n U|; when g* joins U, every key of A_g* not covered yet
 * becomes covered and adds 1 to lost[h] of every genome h holding it.
 * The index of one part (one k, one key-range pass) is built from the K7 sparse workspace after every genome has
 * been inserted with dd_exact_pairs_insert_shard as genome g (same workspace, same arguments):
 *   dd_exact_cover_count  writes d_counts [2] u64: the distinct keys of the workspace and its list nodes (one per
 *                         (genome, key)), so the caller allocates the index exactly; all-ones for a full table or
 *                         node array.
 *   dd_exact_cover_emit   writes the index: d_offsets [n_keys + 1] u32, a key-major CSR over d_holders [n_nodes]
 *                         u16 (the genomes holding each key), and d_key_of_node [n_nodes] u32 (the key id of every
 *                         list node).  Genome g's nodes are the range between the node counter read before and
 *                         after its insert (dd_exact_pairs_node_count): that range is g's key list.  d_status [2]
 *                         u64 is written: (n_keys, n_nodes), or all-ones if the table or node array was full, the
 *                         lists did not match the counts given, or a list holds a genome >= n_genomes -- never a
 *                         partial index.  1 <= n_genomes <= 65535; n_keys < 2^32; n_nodes < 2^32 - 1.
 *   dd_exact_cover_step   one launch over the n_parts parts (for example every (k, pass) of an ordering): for the
 *                         picked genome's nodes [h_node_start[genome], h_node_start[genome + 1]) of each part it
 *                         marks the keys not covered yet covered and adds 1 to d_lost[h] (u64, [n_genomes]) of every
 *                         holder h of each of them.  h_parts is a HOST array, checked before any launch: pointers
 *                         and alignment, 0 <= genome < n_genomes <= 65535, n_keys < 2^32, and node starts that do
 *                         not decrease over the pick and fit n_nodes.  d_ws: n_parts * DD_COVER_PART_BYTES bytes,
 *                         16-byte aligned (the descriptors are staged there).  d_covered [n_keys] u8 starts zeroed.
 * =========================================================================================== */
typedef struct dd_cover_part {
    const uint32_t *d_offsets;      /* [n_keys + 1] */
    const uint16_t *d_holders;      /* [n_nodes] */
    const uint32_t *d_key_of_node;  /* [n_nodes] */
    uint8_t *d_covered;             /* [n_keys] */
    uint64_t *d_lost;               /* [n_genomes], added to */
    uint64_t n_keys, n_nodes;
    const uint64_t *h_node_start;   /* HOST [n_genomes + 1]: the node counter before each genome's insert, then after the last */
} dd_cover_part;
#define DD_COVER_PART_BYTES 64
DD_API int dd_exact_cover_count(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                                uint32_t max_streams, uint64_t *d_counts, dd_stream stream);
DD_API int dd_exact_cover_emit(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                               uint32_t max_streams, int64_t n_genomes, uint64_t n_keys, uint64_t n_nodes,
                               uint32_t *d_offsets, uint16_t *d_holders, uint32_t *d_key_of_node, uint64_t *d_status,
                               dd_stream stream);
DD_API int dd_exact_cover_step(const dd_cover_part *h_parts, int n_parts, int64_t n_genomes, int64_t genome,
                               void *d_ws, size_t ws_bytes, dd_stream stream);

/* ===========================================================================================
 * Host-buffer convenience path (what bench.py's e2e number times): one FASTA held in host memory
 * -> H2D copy -> K1 -> K2 -> K4 -> D2H of cardinalities (and registers if h_regs != NULL);
 * synchronises the stream before returning.  Equivalent to the reference running
 * `dashing sketch` + `dashing card` for every k of the mask on that file.  FASTQ text (a line
 * beginning with '+') is detected by the packer, rewritten with dd_fastq_to_fasta_host and sketched
 * again, so the result is what kseq-based readers produce for it.
 * =========================================================================================== */
DD_API size_t dd_sketch_fasta_host_workspace_bytes(size_t n_bytes, int nk, int p);
DD_API int dd_sketch_fasta_host(const uint8_t *h_text, size_t n_bytes, uint32_t kmask, int p, int canon,
                         uint8_t *h_regs /*[nk][2^p] or NULL*/, double *h_cards /*[nk]*/, uint8_t *d_regs_or_null,
                         void *d_ws, size_t ws_bytes, dd_stream stream);

/* Same, but returns as soon as the work is enqueued: h_text must stay valid, and h_cards / h_regs
 * must not be read, until `stream` has been synchronised by the caller (pinned host memory makes
 * the copies truly asynchronous).  Lets a caller keep several FASTAs in flight on different streams
 * (one workspace per stream) so that H2D copies overlap the kernels of the previous file.  Nothing
 * in the call waits for the device, whatever the file size.  FASTQ text cannot be handled without
 * a host round trip: h_cards[] is then filled with NaN, and the caller falls back to
 * dd_sketch_fasta_host for that file. */
DD_API int dd_sketch_fasta_host_async(const uint8_t *h_text, size_t n_bytes, uint32_t kmask, int p, int canon,
                                      uint8_t *h_regs, double *h_cards, uint8_t *d_regs_or_null, void *d_ws,
                                      size_t ws_bytes, dd_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* DANDD_B200_H */
