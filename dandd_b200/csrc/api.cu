// api.cu -- the C ABI declared in include/dandd_b200.h: argument checking, error reporting and
// the host-buffer convenience path.  No arithmetic lives here.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "kernels.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    return fail(DD_ERR_CUDA, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}
#define DD_CUDA(call, what)                              \
    do {                                                 \
        cudaError_t e__ = (call);                        \
        if (e__ != cudaSuccess) return cuda_fail(e__, what); \
    } while (0)

cudaStream_t S(dd_stream s) { return static_cast<cudaStream_t>(s); }
size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
bool bad_p(int p) { return p < 5 || p > 26; }
int popc(uint32_t x) { return __builtin_popcount(x); }

}  // namespace

namespace dd {
unsigned long long g_kernel_launches = 0;
}

extern "C" {

unsigned long long dd_kernel_launches(void) { return __atomic_load_n(&dd::g_kernel_launches, __ATOMIC_RELAXED); }
const char *dd_last_error(void) { return g_err; }
int dd_abi_version(void) { return DD_ABI_VERSION; }

int dd_init(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(DD_ERR_DEVICE, "no CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(DD_ERR_ARG, "device %d out of range (0..%d)", device, n - 1);
    cudaDeviceProp prop;
    DD_CUDA(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
    if (prop.major != 10)
        return fail(DD_ERR_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device, prop.major,
                    prop.minor);
    DD_CUDA(cudaSetDevice(device), "cudaSetDevice");
    return DD_OK;
}

int dd_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *l2_bytes, size_t *total_mem) {
    cudaDeviceProp prop;
    DD_CUDA(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (l2_bytes) *l2_bytes = (size_t)prop.l2CacheSize;
    if (total_mem) *total_mem = prop.totalGlobalMem;
    return DD_OK;
}

int dd_set_option(const char *name, long value) {
    if (!name) return fail(DD_ERR_ARG, "dd_set_option: null name");
    if (!strcmp(name, "sketch_k_per_pass")) {
        if (value < 0 || value > 32) return fail(DD_ERR_ARG, "dd_set_option: sketch_k_per_pass must be 0..32");
        dd::g_k_per_pass = (int)value;
        return DD_OK;
    }
    if (!strcmp(name, "sketch_midk")) {
        dd::g_midk = value != 0;
        return DD_OK;
    }
    if (!strcmp(name, "sketch_sink")) {
        dd::g_sink = value != 0;
        return DD_OK;
    }
    if (!strcmp(name, "prefix_planes")) {
        dd::g_prefix_planes = value != 0;
        return DD_OK;
    }
    if (!strcmp(name, "prefix_lattice")) {
        dd::g_prefix_lattice = value != 0;
        return DD_OK;
    }
    if (!strcmp(name, "polyt_sentinel")) {
        dd::g_polyt_sentinel = value != 0;
        return DD_OK;
    }
    return fail(DD_ERR_ARG, "dd_set_option: unknown option '%s'", name);
}

// ---- K1 ------------------------------------------------------------------------------------------
size_t dd_pack_codes_bytes(size_t max_text_bytes) { return align_up(max_text_bytes / 4 + 64, 256); }
size_t dd_pack_invalid_bytes(size_t max_text_bytes) { return align_up(max_text_bytes / 8 + 64, 256); }
size_t dd_pack_workspace_bytes(size_t chunk_bytes) { return dd::pack_workspace_bytes(chunk_bytes); }

int dd_pack_reset(uint32_t *d_codes, size_t codes_bytes, uint32_t *d_invalid, size_t invalid_bytes,
                  dd_pack_state *d_state, dd_stream stream) {
    if (!d_codes || !d_invalid || !d_state) return fail(DD_ERR_ARG, "dd_pack_reset: null pointer");
    DD_CUDA(dd::pack_reset(d_codes, codes_bytes, d_invalid, invalid_bytes, d_state, S(stream)), "dd_pack_reset");
    return DD_OK;
}

int dd_pack_fasta(const uint8_t *d_text, size_t n_bytes, uint32_t *d_codes, uint32_t *d_invalid, size_t cap_symbols,
                  dd_pack_state *d_state, void *d_ws, size_t ws_bytes, dd_stream stream) {
    if (n_bytes == 0) return DD_OK;
    if (!d_text || !d_codes || !d_invalid || !d_state || !d_ws) return fail(DD_ERR_ARG, "dd_pack_fasta: null pointer");
    if (n_bytes > ((size_t)1 << 36)) return fail(DD_ERR_ARG, "dd_pack_fasta: chunk larger than 64 GiB");
    if (ws_bytes < dd::pack_workspace_bytes(n_bytes))
        return fail(DD_ERR_WORKSPACE, "dd_pack_fasta: workspace %zu < %zu", ws_bytes, dd::pack_workspace_bytes(n_bytes));
    DD_CUDA(dd::pack_fasta(d_text, n_bytes, d_codes, d_invalid, cap_symbols, d_state, d_ws, S(stream)), "dd_pack_fasta");
    return DD_OK;
}

int dd_pack_polyt_sentinel(const uint32_t *d_codes, uint32_t *d_invalid, const dd_pack_state *d_state, uint64_t sym_begin,
                           uint64_t sym_end, size_t max_symbols, dd_stream stream) {
    if (!d_codes || !d_invalid) return fail(DD_ERR_ARG, "dd_pack_polyt_sentinel: null pointer");
    if (!d_state && sym_end < sym_begin) return fail(DD_ERR_ARG, "dd_pack_polyt_sentinel: end < begin");
    DD_CUDA(dd::pack_polyt_sentinel(d_codes, d_invalid, d_state, sym_begin, sym_end, max_symbols, S(stream)),
            "dd_pack_polyt_sentinel");
    return DD_OK;
}

// ---- host-side text helpers (no GPU work) ---------------------------------------------------------
size_t dd_fasta_first_record_host(const uint8_t *h_text, size_t n_bytes) {
    if (!h_text) return 0;
    // kseq looks for '>' or '@' (klib kseq.h: `while ((c = ks_getc(ks)) != -1 && c != '>' && c != '@');`)
    const uint8_t *gt = static_cast<const uint8_t *>(memchr(h_text, '>', n_bytes));
    const size_t lim = gt ? (size_t)(gt - h_text) : n_bytes;   // '@' only matters if it comes first
    const uint8_t *at = static_cast<const uint8_t *>(memchr(h_text, '@', lim));
    return at ? (size_t)(at - h_text) : lim;
}

// The walk of kseq_read() over FASTA/FASTQ text, emitting plain FASTA: ">\n" per record, sequence
// lines verbatim.  One record per iteration of the outer loop.
size_t dd_fastq_to_fasta_host(const uint8_t *h_in, size_t n, uint8_t *h_out) {
    if (!h_in || !h_out) return 0;
    const uint8_t *p = h_in, *const end = h_in + n;
    uint8_t *o = h_out;
    auto line_end = [&](const uint8_t *from) {   // one past the line's '\n', or `end`
        const uint8_t *nl = static_cast<const uint8_t *>(memchr(from, '\n', (size_t)(end - from)));
        return nl ? nl + 1 : end;
    };
    bool marker_taken = false;   // the previous record ended on the next record's marker
    while (true) {
        if (!marker_taken) {
            p += dd_fasta_first_record_host(p, (size_t)(end - p));
            if (p >= end) break;
            ++p;
        }
        marker_taken = false;
        uint8_t *const record_out = o;
        *o++ = '>';
        *o++ = '\n';
        p = line_end(p);   // name and comment
        size_t seq_len = 0;
        int stop = -1;
        while (p < end) {
            const uint8_t c = *p;
            if (c == '>' || c == '@' || c == '+') {
                stop = c;
                ++p;
                break;
            }
            const uint8_t *le = line_end(p);
            for (const uint8_t *q = p; q < le; ++q)
                if (*q != '\n' && *q != '\r') ++seq_len;
            memcpy(o, p, (size_t)(le - p));
            o += le - p;
            p = le;
        }
        if (o > record_out + 2 && o[-1] != '\n') *o++ = '\n';   // text ended without a newline
        if (stop == '>' || stop == '@') {
            marker_taken = true;
            continue;
        }
        if (stop != '+') break;   // end of text
        const uint8_t *le = line_end(p);   // the rest of the '+' line
        if (le == end && (le == p || le[-1] != '\n')) {   // no quality string: kseq_read fails
            o = record_out;
            break;
        }
        p = le;
        size_t qual_len = 0;
        bool first = true;
        while (p < end && (first || qual_len < seq_len)) {
            le = line_end(p);
            for (const uint8_t *q = p; q < le; ++q)
                if (*q != '\n' && *q != '\r') ++qual_len;
            p = le;
            first = false;
        }
        if (qual_len != seq_len) {   // kseq_read returns -2: this record and the rest are not read
            o = record_out;
            break;
        }
    }
    return (size_t)(o - h_out);
}

// ---- K2 ------------------------------------------------------------------------------------------
size_t dd_sketch_workspace_bytes(int nk, int p) { return dd::sketch_workspace_bytes(nk, p); }

int dd_sketch_begin(void *d_ws, size_t ws_bytes, int nk, int p, dd_stream stream) {
    if (!d_ws || nk < 1 || nk > 32 || bad_p(p)) return fail(DD_ERR_ARG, "dd_sketch_begin: bad argument (nk=%d p=%d)", nk, p);
    if (ws_bytes < dd::sketch_workspace_bytes(nk, p)) return fail(DD_ERR_WORKSPACE, "dd_sketch_begin: workspace too small");
    DD_CUDA(dd::sketch_begin(d_ws, nk, p, S(stream)), "dd_sketch_begin");
    return DD_OK;
}

static int sketch_check(const void *c, const void *i, uint32_t kmask, int p, void *ws, size_t ws_bytes, const char *fn) {
    if (!c || !i || !ws) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (kmask == 0) return fail(DD_ERR_ARG, "%s: empty k mask", fn);
    if (bad_p(p)) return fail(DD_ERR_ARG, "%s: p=%d outside [5,26]", fn, p);
    if (ws_bytes < dd::sketch_workspace_bytes(popc(kmask), p)) return fail(DD_ERR_WORKSPACE, "%s: workspace too small", fn);
    return DD_OK;
}

int dd_sketch_update(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state,
                     size_t max_new_symbols, uint32_t kmask, int p, int canon, void *d_ws, size_t ws_bytes,
                     dd_stream stream) {
    if (int rc = sketch_check(d_codes, d_invalid, kmask, p, d_ws, ws_bytes, "dd_sketch_update")) return rc;
    if (!d_state) return fail(DD_ERR_ARG, "dd_sketch_update: null state");
    DD_CUDA(dd::sketch_update(d_codes, d_invalid, d_state, 0, 0, max_new_symbols, kmask, p, canon, d_ws, S(stream)),
            "dd_sketch_update");
    return DD_OK;
}

int dd_sketch_update_range(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end,
                           uint32_t kmask, int p, int canon, void *d_ws, size_t ws_bytes, dd_stream stream) {
    if (int rc = sketch_check(d_codes, d_invalid, kmask, p, d_ws, ws_bytes, "dd_sketch_update_range")) return rc;
    if (sym_end < sym_begin) return fail(DD_ERR_ARG, "dd_sketch_update_range: end < begin");
    DD_CUDA(dd::sketch_update(d_codes, d_invalid, nullptr, sym_begin, sym_end, 0, kmask, p, canon, d_ws, S(stream)),
            "dd_sketch_update_range");
    return DD_OK;
}

int dd_sketch_update_sched(const uint32_t *d_codes, const uint32_t *d_invalid, const dd_pack_state *d_state, uint64_t sym_begin,
                           uint64_t sym_end, size_t max_new_symbols, uint64_t seen_before, uint32_t kmask, int p, int canon,
                           void *d_ws, size_t ws_bytes, dd_stream stream) {
    if (int rc = sketch_check(d_codes, d_invalid, kmask, p, d_ws, ws_bytes, "dd_sketch_update_sched")) return rc;
    if (!d_state && sym_end < sym_begin) return fail(DD_ERR_ARG, "dd_sketch_update_sched: end < begin");
    DD_CUDA(dd::sketch_update_sched(d_codes, d_invalid, d_state, sym_begin, sym_end, max_new_symbols, seen_before, kmask, p, canon,
                                    d_ws, S(stream)),
            "dd_sketch_update_sched");
    return DD_OK;
}

int dd_sketch_refresh_floor(void *d_ws, size_t ws_bytes, uint32_t kmask, int p, dd_stream stream) {
    if (!d_ws || kmask == 0 || bad_p(p)) return fail(DD_ERR_ARG, "dd_sketch_refresh_floor: bad argument");
    if (ws_bytes < dd::sketch_workspace_bytes(popc(kmask), p)) return fail(DD_ERR_WORKSPACE, "dd_sketch_refresh_floor: workspace too small");
    DD_CUDA(dd::sketch_refresh_floor(d_ws, kmask, p, S(stream)), "dd_sketch_refresh_floor");
    return DD_OK;
}

int dd_sketch_end(void *d_ws, size_t ws_bytes, int nk, int p, uint8_t *d_regs, uint32_t *d_hist, double *d_cards,
                  dd_stream stream) {
    if (!d_ws || !d_regs || nk < 1 || nk > 32 || bad_p(p)) return fail(DD_ERR_ARG, "dd_sketch_end: bad argument");
    if (d_cards && !d_hist) return fail(DD_ERR_ARG, "dd_sketch_end: d_cards needs d_hist");
    if (ws_bytes < dd::sketch_workspace_bytes(nk, p)) return fail(DD_ERR_WORKSPACE, "dd_sketch_end: workspace too small");
    DD_CUDA(dd::sketch_end(d_ws, nk, p, d_regs, d_hist, d_cards, S(stream)), "dd_sketch_end");
    return DD_OK;
}

// ---- K4 / K3 / K6 ----------------------------------------------------------------------------------
int dd_card_ertl_mle(const uint8_t *d_regs, int nsk, int p, double *d_cards, uint32_t *d_hist, dd_stream stream) {
    if (nsk == 0) return DD_OK;
    if (!d_regs || !d_cards || !d_hist || nsk < 0 || bad_p(p)) return fail(DD_ERR_ARG, "dd_card_ertl_mle: bad argument");
    DD_CUDA(dd::card_hist(d_regs, nsk, p, d_hist, S(stream)), "dd_card_ertl_mle(hist)");
    DD_CUDA(dd::mle_from_hist(d_hist, nsk, p, d_cards, S(stream)), "dd_card_ertl_mle(mle)");
    return DD_OK;
}

int dd_mle_from_hist(const uint32_t *d_hist, int nsk, int p, double *d_cards, dd_stream stream) {
    if (nsk == 0) return DD_OK;
    if (!d_hist || !d_cards || nsk < 0 || bad_p(p)) return fail(DD_ERR_ARG, "dd_mle_from_hist: bad argument");
    DD_CUDA(dd::mle_from_hist(d_hist, nsk, p, d_cards, S(stream)), "dd_mle_from_hist");
    return DD_OK;
}

int dd_mle_from_hist_f64(const double *d_hist, int nsk, int p, double *d_cards, dd_stream stream) {
    if (nsk == 0) return DD_OK;
    if (!d_hist || !d_cards || nsk < 0 || bad_p(p)) return fail(DD_ERR_ARG, "dd_mle_from_hist_f64: bad argument");
    DD_CUDA(dd::mle_from_hist_f64(d_hist, nsk, p, d_cards, S(stream)), "dd_mle_from_hist_f64");
    return DD_OK;
}

int dd_union_max(const uint8_t *const *d_in, int n_in, size_t len, uint8_t *d_out, dd_stream stream) {
    if (!d_in || !d_out || n_in < 1) return fail(DD_ERR_ARG, "dd_union_max: bad argument");
    if ((reinterpret_cast<uintptr_t>(d_out) & 15) != 0) return fail(DD_ERR_ARG, "dd_union_max: output must be 16-byte aligned");
    DD_CUDA(dd::union_max(d_in, n_in, len, d_out, S(stream)), "dd_union_max");
    return DD_OK;
}

size_t dd_prefix_union_workspace_bytes(int n_ord, int n_steps, int n_genomes, int nk, int p) {
    if (n_ord < 0 || n_steps < 0 || n_genomes < 0 || nk < 0 || bad_p(p)) return 0;
    return dd::prefix_union_workspace_bytes(n_ord, n_steps, n_genomes, nk, p);
}
size_t dd_planes_bytes(int64_t n_sketches, int p) {
    if (n_sketches < 0 || bad_p(p)) return 0;
    return dd::planes_bytes(n_sketches, p);
}

int dd_to_planes(const uint8_t *d_regs, int64_t n_sketches, int p, uint32_t *d_planes, dd_stream stream) {
    if (n_sketches == 0) return DD_OK;
    if (!d_regs || !d_planes || n_sketches < 0 || bad_p(p) || !dd::planes_supported(p))
        return fail(DD_ERR_ARG, "dd_to_planes: bad argument (bit planes need p >= 12)");
    DD_CUDA(dd::to_planes(d_regs, n_sketches, p, d_planes, S(stream)), "dd_to_planes");
    return DD_OK;
}

static int prefix_args_ok(const void *data, const int32_t *d_order, const double *d_cards, const uint32_t *d_hist, int n_ord,
                          int n_steps, int n_genomes, int nk, int p) {
    return data && d_order && d_cards && d_hist && n_ord >= 0 && n_steps >= 0 && n_genomes >= 1 && nk >= 1 && nk <= 65535 &&
           !bad_p(p) && (((size_t)1 << p) + 32767) / 32768 <= 65535;
}

int dd_prefix_union_card(const uint8_t *d_regs, const int32_t *d_order, int n_ord, int n_steps, int n_genomes, int nk,
                         int p, int final_only, double *d_cards, uint32_t *d_hist, uint8_t *d_unions, void *d_ws,
                         size_t ws_bytes, dd_stream stream) {
    if (n_ord == 0 || n_steps == 0) return DD_OK;
    if (!prefix_args_ok(d_regs, d_order, d_cards, d_hist, n_ord, n_steps, n_genomes, nk, p))
        return fail(DD_ERR_ARG, "dd_prefix_union_card: bad argument");
    const size_t rows = (size_t)n_ord * (final_only ? 1 : n_steps) * nk;
    if (rows > 0x7fffffff) return fail(DD_ERR_ARG, "dd_prefix_union_card: too many (ordering, step, k) rows");
    // pairs (two steps, final union only) never use the identical-prefix table: planes alone
    const bool pairs_only = final_only && n_steps == 2;
    if (!d_unions && d_ws && dd::g_prefix_lattice && !pairs_only && dd::lattice_supported(n_genomes, p)) {
        void *base = reinterpret_cast<void *>(align_up(reinterpret_cast<uintptr_t>(d_ws), 256));
        const size_t lost = (size_t)(static_cast<uint8_t *>(base) - static_cast<uint8_t *>(d_ws));
        const size_t need = dd::prefix_lattice_workspace_bytes(n_ord, n_steps, n_genomes, nk);
        if (ws_bytes < lost + need)
            return fail(DD_ERR_WORKSPACE, "dd_prefix_union_card: workspace %zu < %zu", ws_bytes, need + 256);
        DD_CUDA(dd::prefix_union_hist_lattice(d_regs, d_order, n_ord, n_steps, n_genomes, nk, p, final_only, d_hist, base, S(stream)),
                "dd_prefix_union_card(lattice)");
    } else if (!d_unions && d_ws && dd::g_prefix_planes && dd::planes_supported(p)) {
        void *base = reinterpret_cast<void *>(align_up(reinterpret_cast<uintptr_t>(d_ws), 256));
        const size_t lost = (size_t)(static_cast<uint8_t *>(base) - static_cast<uint8_t *>(d_ws));
        const size_t need = dd::prefix_union_workspace_bytes(pairs_only ? 0 : n_ord, pairs_only ? 0 : n_steps, n_genomes, nk, p);
        if (ws_bytes < lost + need - 256)
            return fail(DD_ERR_WORKSPACE, "dd_prefix_union_card: workspace %zu < %zu", ws_bytes, need);
        DD_CUDA(dd::prefix_union_hist_planes(d_regs, d_order, n_ord, n_steps, n_genomes, nk, p, final_only, d_hist, base, S(stream)),
                "dd_prefix_union_card(planes)");
    } else {
        DD_CUDA(dd::prefix_union_hist(d_regs, d_order, n_ord, n_steps, n_genomes, nk, p, final_only, d_hist, d_unions, S(stream)),
                "dd_prefix_union_card(hist)");
    }
    DD_CUDA(dd::mle_from_hist(d_hist, (int)rows, p, d_cards, S(stream)), "dd_prefix_union_card(mle)");
    return DD_OK;
}

int dd_prefix_union_card_planes(const uint32_t *d_planes, const int32_t *d_order, int n_ord, int n_steps, int n_genomes,
                                int nk, int p, int final_only, double *d_cards, uint32_t *d_hist, void *d_ws, size_t ws_bytes,
                                dd_stream stream) {
    if (n_ord == 0 || n_steps == 0) return DD_OK;
    if (!prefix_args_ok(d_planes, d_order, d_cards, d_hist, n_ord, n_steps, n_genomes, nk, p) || !dd::planes_supported(p))
        return fail(DD_ERR_ARG, "dd_prefix_union_card_planes: bad argument (bit planes need p >= 12)");
    const size_t rows = (size_t)n_ord * (final_only ? 1 : n_steps) * nk;
    if (rows > 0x7fffffff) return fail(DD_ERR_ARG, "dd_prefix_union_card_planes: too many (ordering, step, k) rows");
    void *scratch = nullptr;
    if (d_ws) {
        scratch = reinterpret_cast<void *>(align_up(reinterpret_cast<uintptr_t>(d_ws), 256));
        const size_t lost = (size_t)(static_cast<uint8_t *>(scratch) - static_cast<uint8_t *>(d_ws));
        if (ws_bytes < lost + dd::prefix_union_workspace_bytes(n_ord, n_steps, 0, 0, p) - 256)
            return fail(DD_ERR_WORKSPACE, "dd_prefix_union_card_planes: workspace too small");
    }
    DD_CUDA(dd::prefix_union_hist_from_planes(d_planes, d_order, n_ord, n_steps, n_genomes, nk, p, final_only, d_hist, scratch,
                                              S(stream)),
            "dd_prefix_union_card_planes");
    DD_CUDA(dd::mle_from_hist(d_hist, (int)rows, p, d_cards, S(stream)), "dd_prefix_union_card_planes(mle)");
    return DD_OK;
}

int dd_union_sets_card(const uint8_t *const *d_members, int n_sets, int n_steps, int p, int final_only, double *d_cards,
                       uint32_t *d_hist, uint8_t *d_unions, dd_stream stream) {
    if (n_sets == 0 || n_steps == 0) return DD_OK;
    if (!d_members || !d_cards || !d_hist || n_sets < 0 || n_steps < 0 || bad_p(p))
        return fail(DD_ERR_ARG, "dd_union_sets_card: bad argument");
    const size_t rows = (size_t)n_sets * (final_only ? 1 : n_steps);
    if (rows > 0x7fffffff) return fail(DD_ERR_ARG, "dd_union_sets_card: too many (set, step) rows");
    DD_CUDA(dd::union_sets_hist(d_members, n_sets, n_steps, p, final_only, d_hist, d_unions, S(stream)),
            "dd_union_sets_card(hist)");
    DD_CUDA(dd::mle_from_hist(d_hist, (int)rows, p, d_cards, S(stream)), "dd_union_sets_card(mle)");
    return DD_OK;
}

static int pair_count_ok(int64_t n_pairs, int nk) {
    return n_pairs >= 0 && n_pairs <= 0x7fffffff / (2 * (int64_t)(nk > 0 ? nk : 1));
}

int dd_pairwise_union_card(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *d_pairs, int64_t n_pairs,
                           double *d_cards, uint32_t *d_hist, void *d_ws, size_t ws_bytes, dd_stream stream) {
    if (n_pairs == 0) return DD_OK;
    if (!pair_count_ok(n_pairs, nk)) return fail(DD_ERR_ARG, "dd_pairwise_union_card: bad pair count");
    // a pair is a 2-step ordering of which only the full union is estimated
    return dd_prefix_union_card(d_regs, d_pairs, (int)n_pairs, 2, n_genomes, nk, p, /*final_only=*/1, d_cards, d_hist,
                                nullptr, d_ws, ws_bytes, stream);
}

int dd_pairwise_union_card_planes(const uint32_t *d_planes, int n_genomes, int nk, int p, const int32_t *d_pairs,
                                  int64_t n_pairs, double *d_cards, uint32_t *d_hist, dd_stream stream) {
    if (n_pairs == 0) return DD_OK;
    if (!pair_count_ok(n_pairs, nk)) return fail(DD_ERR_ARG, "dd_pairwise_union_card_planes: bad pair count");
    return dd_prefix_union_card_planes(d_planes, d_pairs, (int)n_pairs, 2, n_genomes, nk, p, /*final_only=*/1, d_cards, d_hist,
                                       nullptr, 0, stream);
}

// ---- K10 -----------------------------------------------------------------------------------------
size_t dd_leave_out_workspace_bytes(int n_genomes, int nk) {
    if (n_genomes < 1 || nk < 1) return 0;
    return dd::leave_out_workspace_bytes(n_genomes, nk);
}
int dd_leave_out_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const int32_t *d_group, int n_groups,
                      uint64_t reg_begin, uint64_t reg_end, uint32_t *d_hist, void *d_ws, size_t ws_bytes, dd_stream stream) {
    const char *fn = "dd_leave_out_hist";
    if (!d_regs || !d_group || !d_hist || !d_ws) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (bad_p(p)) return fail(DD_ERR_ARG, "%s: p=%d outside [5,26]", fn, p);
    if (nk < 1 || nk > 65535) return fail(DD_ERR_ARG, "%s: nk=%d outside [1,65535]", fn, nk);
    if (n_genomes < 1 || n_groups < 1 || n_groups > n_genomes || n_groups > 65535)   // group ids are u16 in the kernel
        return fail(DD_ERR_ARG, "%s: need 1 <= n_groups (%d) <= min(n_genomes (%d), 65535)", fn, n_groups, n_genomes);
    if ((int64_t)nk * (1 + (int64_t)n_groups) * DD_HIST_BINS > 0x7fffffffll)
        return fail(DD_ERR_ARG, "%s: too many (k, row) histograms: %d x %d", fn, nk, 1 + n_groups);
    if (reg_begin > reg_end || reg_end > ((uint64_t)1 << p) || (reg_begin & 15) || (reg_end & 15))
        return fail(DD_ERR_ARG, "%s: register range [%llu,%llu) is not 16-aligned within [0,%llu]", fn,
                    (unsigned long long)reg_begin, (unsigned long long)reg_end, (unsigned long long)1 << p);
    if (reinterpret_cast<uintptr_t>(d_regs) & 15) return fail(DD_ERR_ARG, "%s: registers must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(d_ws) & 7) || (reinterpret_cast<uintptr_t>(d_hist) & 3))
        return fail(DD_ERR_ARG, "%s: misaligned workspace or histogram", fn);
    if (ws_bytes < dd::leave_out_workspace_bytes(n_genomes, nk))
        return fail(DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, dd::leave_out_workspace_bytes(n_genomes, nk));
    std::vector<int32_t> group(n_genomes);   // ids index rows and shared counters: checked here, before any launch
    DD_CUDA(cudaMemcpyAsync(group.data(), d_group, group.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, S(stream)), fn);
    DD_CUDA(cudaStreamSynchronize(S(stream)), fn);
    for (int g = 0; g < n_genomes; ++g)
        if (group[g] < 0 || group[g] >= n_groups)
            return fail(DD_ERR_ARG, "%s: genome %d has group %d outside [0,%d)", fn, g, group[g], n_groups);
    DD_CUDA(dd::leave_out_hist(d_regs, n_genomes, nk, p, group.data(), n_groups, reg_begin, reg_end, d_hist, d_ws, S(stream)), fn);
    return DD_OK;
}

// ---- K14 -----------------------------------------------------------------------------------------
size_t dd_register_spectrum_workspace_bytes(int n_genomes, int nk) {
    if (n_genomes < 1 || n_genomes > 65535 || nk < 1 || nk > 65535) return 0;
    return dd::register_spectrum_workspace_bytes(n_genomes, nk);
}
int dd_register_spectrum(const uint8_t *d_regs, int n_genomes, int nk, int p, uint64_t reg_begin, uint64_t reg_end,
                         uint32_t *d_spec, void *d_ws, size_t ws_bytes, dd_stream stream) {
    const char *fn = "dd_register_spectrum";
    if (!d_regs || !d_spec || !d_ws) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (bad_p(p)) return fail(DD_ERR_ARG, "%s: p=%d outside [5,26]", fn, p);
    if (nk < 1 || nk > 65535) return fail(DD_ERR_ARG, "%s: nk=%d outside [1,65535]", fn, nk);
    if (n_genomes < 1 || n_genomes > 65535)   // the value counters are u16
        return fail(DD_ERR_ARG, "%s: n_genomes=%d outside [1,65535]", fn, n_genomes);
    if ((int64_t)nk * DD_HIST_BINS * n_genomes > 0x7fffffffll)
        return fail(DD_ERR_ARG, "%s: too many (k, value, count) cells: %d x 64 x %d", fn, nk, n_genomes);
    if (reg_begin > reg_end || reg_end > ((uint64_t)1 << p) || (reg_begin & 15) || (reg_end & 15))
        return fail(DD_ERR_ARG, "%s: register range [%llu,%llu) is not 16-aligned within [0,%llu]", fn,
                    (unsigned long long)reg_begin, (unsigned long long)reg_end, (unsigned long long)1 << p);
    if (reinterpret_cast<uintptr_t>(d_regs) & 15) return fail(DD_ERR_ARG, "%s: registers must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(d_ws) & 3) || (reinterpret_cast<uintptr_t>(d_spec) & 3))
        return fail(DD_ERR_ARG, "%s: misaligned workspace or table", fn);
    if (ws_bytes < dd::register_spectrum_workspace_bytes(n_genomes, nk))
        return fail(DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, dd::register_spectrum_workspace_bytes(n_genomes, nk));
    DD_CUDA(dd::register_spectrum(d_regs, n_genomes, nk, p, reg_begin, reg_end, d_spec, d_ws, S(stream)), fn);
    return DD_OK;
}

// ---- K11 -----------------------------------------------------------------------------------------
size_t dd_greedy_workspace_bytes(int n_cand) {
    if (n_cand < 1) return 0;
    return dd::greedy_workspace_bytes(n_cand);
}
// The checks every K11 entry shares; the candidates are host values, so no check waits for the device.
static int greedy_check(const char *fn, const void *d_union, int n_genomes, int nk, int p, const int32_t *h_cand,
                        int n_cand, const void *d_ws, size_t ws_bytes) {
    if (!d_union || !h_cand || !d_ws) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (bad_p(p)) return fail(DD_ERR_ARG, "%s: p=%d outside [5,26]", fn, p);
    if (nk < 1 || nk > 65535) return fail(DD_ERR_ARG, "%s: nk=%d outside [1,65535]", fn, nk);
    if (n_genomes < 1 || n_cand < 1) return fail(DD_ERR_ARG, "%s: need n_genomes (%d) >= 1 and n_cand (%d) >= 1", fn, n_genomes, n_cand);
    if ((int64_t)n_cand * nk * DD_HIST_BINS > 0x7fffffffll)
        return fail(DD_ERR_ARG, "%s: too many (candidate, k) histograms: %d x %d", fn, n_cand, nk);
    if (reinterpret_cast<uintptr_t>(d_union) & 15) return fail(DD_ERR_ARG, "%s: the union must be 16-byte aligned", fn);
    if (reinterpret_cast<uintptr_t>(d_ws) & 15) return fail(DD_ERR_ARG, "%s: misaligned workspace", fn);
    if (ws_bytes < dd::greedy_workspace_bytes(n_cand))
        return fail(DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, dd::greedy_workspace_bytes(n_cand));
    std::vector<char> seen(n_genomes, 0);   // a candidate listed twice would compact one segment from two CTAs
    for (int c = 0; c < n_cand; ++c) {
        if (h_cand[c] < 0 || h_cand[c] >= n_genomes)
            return fail(DD_ERR_ARG, "%s: candidate %d is genome %d, outside [0,%d)", fn, c, h_cand[c], n_genomes);
        if (seen[h_cand[c]]++) return fail(DD_ERR_ARG, "%s: genome %d is listed twice", fn, h_cand[c]);
    }
    return DD_OK;
}
int dd_greedy_dense_hist(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union,
                         const uint32_t *d_union_hist, const int32_t *h_cand, int n_cand, uint32_t *d_hist,
                         uint32_t *d_live, void *d_ws, size_t ws_bytes, dd_stream stream) {
    const char *fn = "dd_greedy_dense_hist";
    if (!d_regs || !d_union_hist || !d_hist || !d_live) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (int r = greedy_check(fn, d_union, n_genomes, nk, p, h_cand, n_cand, d_ws, ws_bytes)) return r;
    if (reinterpret_cast<uintptr_t>(d_regs) & 15) return fail(DD_ERR_ARG, "%s: registers must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(d_union_hist) | reinterpret_cast<uintptr_t>(d_hist) | reinterpret_cast<uintptr_t>(d_live)) & 3)
        return fail(DD_ERR_ARG, "%s: misaligned histogram or live counts", fn);
    DD_CUDA(dd::greedy_dense_hist(d_regs, nk, p, d_union, d_union_hist, h_cand, n_cand, d_hist, d_live, d_ws, S(stream)), fn);
    return DD_OK;
}
int dd_greedy_compact(const uint8_t *d_regs, int n_genomes, int nk, int p, const uint8_t *d_union, const int32_t *h_cand,
                      int n_cand, const int64_t *h_seg_off, int64_t *d_seg_off, uint32_t *d_seg_len, uint32_t *d_entries,
                      int64_t n_entries, void *d_ws, size_t ws_bytes, dd_stream stream) {
    const char *fn = "dd_greedy_compact";
    if (!d_regs || !h_seg_off || !d_seg_off || !d_seg_len || (!d_entries && n_entries > 0))
        return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (int r = greedy_check(fn, d_union, n_genomes, nk, p, h_cand, n_cand, d_ws, ws_bytes)) return r;
    if (reinterpret_cast<uintptr_t>(d_regs) & 15) return fail(DD_ERR_ARG, "%s: registers must be 16-byte aligned", fn);
    if ((reinterpret_cast<uintptr_t>(d_seg_off) & 7) || ((reinterpret_cast<uintptr_t>(d_seg_len) | reinterpret_cast<uintptr_t>(d_entries)) & 3))
        return fail(DD_ERR_ARG, "%s: misaligned segment table or entries", fn);
    const size_t n_seg = (size_t)n_genomes * nk;
    if (h_seg_off[0] != 0) return fail(DD_ERR_ARG, "%s: segment offsets must start at 0", fn);
    for (size_t s = 0; s < n_seg; ++s)
        if (h_seg_off[s + 1] < h_seg_off[s]) return fail(DD_ERR_ARG, "%s: segment offsets decrease at %zu", fn, s);
    if (h_seg_off[n_seg] > n_entries)
        return fail(DD_ERR_ARG, "%s: segments need %lld entries, the buffer holds %lld", fn, (long long)h_seg_off[n_seg],
                    (long long)n_entries);
    DD_CUDA(dd::greedy_compact(d_regs, n_genomes, nk, p, d_union, h_cand, n_cand, h_seg_off, d_seg_off, d_seg_len, d_entries,
                               d_ws, S(stream)), fn);
    return DD_OK;
}
int dd_greedy_sparse_hist(uint32_t *d_entries, int64_t n_entries, const int64_t *d_seg_off, uint32_t *d_seg_len,
                          int n_genomes, int nk, int p, const uint8_t *d_union, const uint32_t *d_union_hist,
                          const int32_t *h_cand, int n_cand, uint32_t *d_hist, uint32_t *d_live, void *d_ws,
                          size_t ws_bytes, dd_stream stream) {
    const char *fn = "dd_greedy_sparse_hist";
    if ((!d_entries && n_entries > 0) || n_entries < 0 || !d_seg_off || !d_seg_len || !d_union_hist || !d_hist || !d_live)
        return fail(DD_ERR_ARG, "%s: null pointer or negative entry count", fn);
    if (int r = greedy_check(fn, d_union, n_genomes, nk, p, h_cand, n_cand, d_ws, ws_bytes)) return r;
    if ((reinterpret_cast<uintptr_t>(d_seg_off) & 7) ||
        ((reinterpret_cast<uintptr_t>(d_seg_len) | reinterpret_cast<uintptr_t>(d_entries) | reinterpret_cast<uintptr_t>(d_union_hist) |
          reinterpret_cast<uintptr_t>(d_hist) | reinterpret_cast<uintptr_t>(d_live)) & 3))
        return fail(DD_ERR_ARG, "%s: misaligned segment table, entries, histogram or live counts", fn);
    DD_CUDA(dd::greedy_sparse_hist(d_entries, n_entries, d_seg_off, d_seg_len, nk, p, d_union, d_union_hist, h_cand, n_cand,
                                   d_hist, d_live, d_ws, S(stream)), fn);
    return DD_OK;
}

// ---- K5 ------------------------------------------------------------------------------------------
static int exact_check(int k, uint64_t capacity, const void *ws, size_t ws_bytes, const char *fn) {
    if (!ws) return fail(DD_ERR_ARG, "%s: null workspace", fn);
    if (k < 1 || k > DD_EXACT_MAXK) return fail(DD_ERR_ARG, "%s: k=%d outside [1,%d]", fn, k, DD_EXACT_MAXK);
    if (k > DD_EXACT_BITMAP_MAXK && (capacity < 1024 || (capacity & (capacity - 1))))
        return fail(DD_ERR_ARG, "%s: capacity must be a power of two >= 1024", fn);
    if (ws_bytes < dd::exact_workspace_bytes(k, capacity)) return fail(DD_ERR_WORKSPACE, "%s: workspace too small", fn);
    return DD_OK;
}
size_t dd_exact_workspace_bytes(int k, uint64_t capacity) { return dd::exact_workspace_bytes(k, capacity); }

int dd_exact_begin(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, dd_stream stream) {
    if (int rc = exact_check(k, capacity, d_ws, ws_bytes, "dd_exact_begin")) return rc;
    DD_CUDA(dd::exact_begin(d_ws, k, capacity, S(stream)), "dd_exact_begin");
    return DD_OK;
}
int dd_exact_insert_shard(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                          int canon, void *d_ws, size_t ws_bytes, uint64_t capacity, uint32_t shard_rank,
                          uint32_t shard_world, dd_stream stream) {
    if (!d_codes || !d_invalid) return fail(DD_ERR_ARG, "dd_exact_insert: null pointer");
    if (shard_world < 1 || shard_rank >= shard_world || shard_world > 65536)
        return fail(DD_ERR_ARG, "dd_exact_insert: shard %u of %u", shard_rank, shard_world);
    if (int rc = exact_check(k, capacity, d_ws, ws_bytes, "dd_exact_insert")) return rc;
    DD_CUDA(dd::exact_insert(d_codes, d_invalid, sym_begin, sym_end, k, canon, d_ws, capacity, shard_rank, shard_world,
                             S(stream)),
            "dd_exact_insert");
    return DD_OK;
}
int dd_exact_insert(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                    int canon, void *d_ws, size_t ws_bytes, uint64_t capacity, dd_stream stream) {
    return dd_exact_insert_shard(d_codes, d_invalid, sym_begin, sym_end, k, canon, d_ws, ws_bytes, capacity, 0, 1, stream);
}
int dd_exact_count(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t *d_count, dd_stream stream) {
    if (!d_count) return fail(DD_ERR_ARG, "dd_exact_count: null pointer");
    if (int rc = exact_check(k, capacity, d_ws, ws_bytes, "dd_exact_count")) return rc;
    DD_CUDA(dd::exact_count(d_ws, k, capacity, d_count, S(stream)), "dd_exact_count");
    return DD_OK;
}

// ---- K7 ------------------------------------------------------------------------------------------
static int sm_count_now() {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return 148;
    return sms > 0 ? sms : 148;
}
static int pairs_check(int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams, const void *ws, size_t ws_bytes,
                       const char *fn) {
    if (!ws) return fail(DD_ERR_ARG, "%s: null workspace", fn);
    if (k < 1 || k > DD_EXACT_MAXK) return fail(DD_ERR_ARG, "%s: k=%d outside [1,%d]", fn, k, DD_EXACT_MAXK);
    if (capacity < 1024 || (capacity & (capacity - 1))) return fail(DD_ERR_ARG, "%s: capacity must be a power of two >= 1024", fn);
    if (max_nodes >= 0xFFFFFFFFull) return fail(DD_ERR_ARG, "%s: max_nodes must be below 2^32 - 1", fn);
    if (k > 64 && (max_streams < 1 || max_streams > 65536))   // an entry keeps the stream index in 16 bits
        return fail(DD_ERR_ARG, "%s: k > 64 needs 1 <= max_streams <= 65536", fn);
    if (ws_bytes < dd::exact_pairs_workspace_bytes(k, capacity, max_nodes, max_streams))
        return fail(DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes,
                    dd::exact_pairs_workspace_bytes(k, capacity, max_nodes, max_streams));
    return DD_OK;
}
size_t dd_exact_pairs_workspace_bytes(int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams) {
    return dd::exact_pairs_workspace_bytes(k, capacity, max_nodes, max_streams);
}
int dd_exact_pairs_begin(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                         dd_stream stream) {
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, "dd_exact_pairs_begin")) return rc;
    DD_CUDA(dd::exact_pairs_begin(d_ws, k, capacity, max_streams, S(stream)), "dd_exact_pairs_begin");
    return DD_OK;
}
int dd_exact_pairs_insert_shard(const uint32_t *d_codes, const uint32_t *d_invalid, uint64_t sym_begin, uint64_t sym_end, int k,
                                int canon, uint32_t genome, void *d_ws, size_t ws_bytes, uint64_t capacity, uint64_t max_nodes,
                                uint32_t max_streams, uint32_t shard_rank, uint32_t shard_world, dd_stream stream) {
    if (!d_codes || !d_invalid) return fail(DD_ERR_ARG, "dd_exact_pairs_insert: null pointer");
    if (genome == 0xFFFFFFFFu) return fail(DD_ERR_ARG, "dd_exact_pairs_insert: genome index out of range");
    if (shard_world < 1 || shard_rank >= shard_world || shard_world > 65536)
        return fail(DD_ERR_ARG, "dd_exact_pairs_insert: shard %u of %u", shard_rank, shard_world);
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, "dd_exact_pairs_insert")) return rc;
    DD_CUDA(dd::exact_pairs_insert(d_codes, d_invalid, sym_begin, sym_end, k, canon, genome, d_ws, capacity, max_nodes,
                                   max_streams, shard_rank, shard_world, S(stream)),
            "dd_exact_pairs_insert");
    return DD_OK;
}
int dd_exact_pairs_accumulate(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes,
                              uint32_t max_streams, int64_t n_genomes, uint64_t *d_inter, dd_stream stream) {
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, "dd_exact_pairs_accumulate")) return rc;
    if (n_genomes < 0 || n_genomes > 0xFFFFFFFFll) return fail(DD_ERR_ARG, "dd_exact_pairs_accumulate: n_genomes=%lld", (long long)n_genomes);
    if (n_genomes > 1 && !d_inter) return fail(DD_ERR_ARG, "dd_exact_pairs_accumulate: null output");
    DD_CUDA(dd::exact_pairs_accumulate(d_ws, k, capacity, max_streams, (uint64_t)n_genomes, d_inter, sm_count_now(), S(stream)),
            "dd_exact_pairs_accumulate");
    return DD_OK;
}
// ---- K8 ------------------------------------------------------------------------------------------
int dd_exact_first_rank_hist(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                             int64_t n_genomes, const uint16_t *d_ranks, int64_t n_rows, uint64_t *d_hist, dd_stream stream) {
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, "dd_exact_first_rank_hist")) return rc;
    if (n_genomes < 0 || n_genomes > 0xFFFF)   // ranks are u16 below n_genomes; 0xFFFF means "not in the row"
        return fail(DD_ERR_ARG, "dd_exact_first_rank_hist: n_genomes=%lld outside [0,65535]", (long long)n_genomes);
    if (n_rows < 0 || n_rows > 0x7FFFFFFFll) return fail(DD_ERR_ARG, "dd_exact_first_rank_hist: n_rows=%lld", (long long)n_rows);
    if (n_genomes > 0 && n_rows > 0 && (!d_ranks || !d_hist)) return fail(DD_ERR_ARG, "dd_exact_first_rank_hist: null pointer");
    DD_CUDA(dd::exact_first_rank_hist(d_ws, k, capacity, max_streams, (uint64_t)n_genomes, d_ranks, (uint64_t)n_rows, d_hist,
                                      sm_count_now(), S(stream)),
            "dd_exact_first_rank_hist");
    return DD_OK;
}
// ---- K9 ------------------------------------------------------------------------------------------
int dd_exact_occupancy_hist(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                            int64_t n_genomes, uint64_t *d_hist, uint64_t *d_priv, dd_stream stream) {
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, "dd_exact_occupancy_hist")) return rc;
    if (n_genomes < 1 || n_genomes > 0xFFFFFFFFll)   // genome indices are u32
        return fail(DD_ERR_ARG, "dd_exact_occupancy_hist: n_genomes=%lld outside [1,4294967295]", (long long)n_genomes);
    if (!d_hist) return fail(DD_ERR_ARG, "dd_exact_occupancy_hist: null pointer");
    DD_CUDA(dd::exact_occupancy_hist(d_ws, k, capacity, max_streams, (uint64_t)n_genomes, d_hist, d_priv, sm_count_now(), S(stream)),
            "dd_exact_occupancy_hist");
    return DD_OK;
}
// ---- K13 -----------------------------------------------------------------------------------------
int dd_exact_query_counts(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                          int64_t n_refs, int64_t n_queries, uint64_t *d_inter, uint64_t *d_shared, uint64_t *d_union,
                          dd_stream stream) {
    const char *fn = "dd_exact_query_counts";
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, fn)) return rc;
    if (!d_inter || !d_shared || !d_union) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (n_refs < 1 || n_queries < 1) return fail(DD_ERR_ARG, "%s: n_refs=%lld n_queries=%lld, both must be >= 1", fn,
                                                 (long long)n_refs, (long long)n_queries);
    if (n_refs + n_queries > 0xFFFFFFFFll)   // genome indices are u32, 0xFFFFFFFF is the end of a list
        return fail(DD_ERR_ARG, "%s: n_refs + n_queries=%lld above 4294967295", fn, (long long)(n_refs + n_queries));
    if (n_refs * n_queries > DD_QUERY_MAX_CELLS)
        return fail(DD_ERR_ARG, "%s: n_queries * n_refs=%lld above %lld cells", fn, (long long)(n_refs * n_queries),
                    (long long)DD_QUERY_MAX_CELLS);
    if (k > 64 && n_refs + n_queries > 65536)   // every genome is one stream of the k > 64 key references
        return fail(DD_ERR_ARG, "%s: above k = 64 n_refs + n_queries=%lld above 65536", fn, (long long)(n_refs + n_queries));
    DD_CUDA(dd::exact_query_counts(d_ws, k, capacity, max_streams, (uint32_t)n_refs, (uint32_t)n_queries, d_inter, d_shared,
                                   d_union, sm_count_now(), S(stream)),
            fn);
    return DD_OK;
}
// ---- K12 -----------------------------------------------------------------------------------------
static bool misaligned(const void *p, uintptr_t a) { return reinterpret_cast<uintptr_t>(p) & (a - 1); }
int dd_exact_cover_count(const void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                         uint64_t *d_counts, dd_stream stream) {
    const char *fn = "dd_exact_cover_count";
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, fn)) return rc;
    if (!d_counts) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (misaligned(d_counts, 8)) return fail(DD_ERR_ARG, "%s: misaligned counts", fn);
    DD_CUDA(dd::exact_cover_count(d_ws, k, capacity, max_streams, d_counts, sm_count_now(), S(stream)), fn);
    return DD_OK;
}
int dd_exact_cover_emit(void *d_ws, size_t ws_bytes, int k, uint64_t capacity, uint64_t max_nodes, uint32_t max_streams,
                        int64_t n_genomes, uint64_t n_keys, uint64_t n_nodes, uint32_t *d_offsets, uint16_t *d_holders,
                        uint32_t *d_key_of_node, uint64_t *d_status, dd_stream stream) {
    const char *fn = "dd_exact_cover_emit";
    if (int rc = pairs_check(k, capacity, max_nodes, max_streams, d_ws, ws_bytes, fn)) return rc;
    if (n_genomes < 1 || n_genomes > 0xFFFF)   // holders are u16
        return fail(DD_ERR_ARG, "%s: n_genomes=%lld outside [1,65535]", fn, (long long)n_genomes);
    if (n_keys > 0xFFFFFFFFull) return fail(DD_ERR_ARG, "%s: %llu keys, key ids are u32", fn, (unsigned long long)n_keys);
    if (n_nodes >= 0xFFFFFFFFull) return fail(DD_ERR_ARG, "%s: %llu nodes, offsets are u32", fn, (unsigned long long)n_nodes);
    if (!d_offsets || !d_status || (n_nodes > 0 && (!d_holders || !d_key_of_node))) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (misaligned(d_offsets, 4) || misaligned(d_holders, 2) || misaligned(d_key_of_node, 4) || misaligned(d_status, 8))
        return fail(DD_ERR_ARG, "%s: misaligned offsets, holders, key ids or status", fn);
    DD_CUDA(dd::exact_cover_emit(d_ws, k, capacity, max_streams, (uint32_t)n_genomes, n_keys, n_nodes, d_offsets, d_holders,
                                 d_key_of_node, d_status, sm_count_now(), S(stream)), fn);
    return DD_OK;
}
int dd_exact_cover_step(const dd_cover_part *h_parts, int n_parts, int64_t n_genomes, int64_t genome, void *d_ws,
                        size_t ws_bytes, dd_stream stream) {
    static_assert(sizeof(dd_cover_part) == DD_COVER_PART_BYTES && sizeof(dd::CoverPart) == DD_COVER_PART_BYTES,
                  "cover part descriptors are 64 bytes on both sides");
    const char *fn = "dd_exact_cover_step";
    if (!h_parts || !d_ws) return fail(DD_ERR_ARG, "%s: null pointer", fn);
    if (misaligned(d_ws, 16)) return fail(DD_ERR_ARG, "%s: misaligned workspace", fn);
    if (n_parts < 1 || n_parts > 65535) return fail(DD_ERR_ARG, "%s: n_parts=%d outside [1,65535]", fn, n_parts);
    if (n_genomes < 1 || n_genomes > 0xFFFF) return fail(DD_ERR_ARG, "%s: n_genomes=%lld outside [1,65535]", fn, (long long)n_genomes);
    if (genome < 0 || genome >= n_genomes)
        return fail(DD_ERR_ARG, "%s: genome %lld outside [0,%lld)", fn, (long long)genome, (long long)n_genomes);
    if (ws_bytes < (size_t)n_parts * DD_COVER_PART_BYTES)
        return fail(DD_ERR_WORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, (size_t)n_parts * DD_COVER_PART_BYTES);
    std::vector<dd::CoverPart> parts(n_parts);
    for (int i = 0; i < n_parts; ++i) {
        const dd_cover_part &p = h_parts[i];
        if (!p.d_offsets || !p.d_covered || !p.d_lost || !p.h_node_start || (p.n_nodes > 0 && (!p.d_holders || !p.d_key_of_node)))
            return fail(DD_ERR_ARG, "%s: part %d: null pointer", fn, i);
        if (misaligned(p.d_offsets, 4) || misaligned(p.d_holders, 2) || misaligned(p.d_key_of_node, 4) || misaligned(p.d_lost, 8))
            return fail(DD_ERR_ARG, "%s: part %d: misaligned offsets, holders, key ids or counters", fn, i);
        if (p.n_keys > 0xFFFFFFFFull || p.n_nodes >= 0xFFFFFFFFull)
            return fail(DD_ERR_ARG, "%s: part %d: %llu keys, %llu nodes (key ids and offsets are u32)", fn, i,
                        (unsigned long long)p.n_keys, (unsigned long long)p.n_nodes);
        const uint64_t b = p.h_node_start[genome], e = p.h_node_start[genome + 1];
        if (b > e || e > p.n_nodes)
            return fail(DD_ERR_ARG, "%s: part %d: genome %lld has nodes [%llu,%llu), outside [0,%llu] or decreasing", fn, i,
                        (long long)genome, (unsigned long long)b, (unsigned long long)e, (unsigned long long)p.n_nodes);
        parts[i] = dd::CoverPart{p.d_offsets, p.d_holders, p.d_key_of_node, p.d_covered,
                                 reinterpret_cast<unsigned long long *>(p.d_lost), b, e, 0};
    }
    DD_CUDA(dd::exact_cover_step(parts.data(), n_parts, (uint32_t)n_genomes, d_ws, sm_count_now(), S(stream)), fn);
    return DD_OK;
}

int dd_exact_pairs_node_count(const void *d_ws, size_t ws_bytes, uint64_t *d_out, dd_stream stream) {
    if (!d_ws || !d_out) return fail(DD_ERR_ARG, "dd_exact_pairs_node_count: null pointer");
    if (ws_bytes < sizeof(dd::ExactWsHeader)) return fail(DD_ERR_WORKSPACE, "dd_exact_pairs_node_count: workspace %zu too small", ws_bytes);
    DD_CUDA(dd::exact_pairs_node_count(d_ws, d_out, S(stream)), "dd_exact_pairs_node_count");
    return DD_OK;
}

int dd_exact_pair_popc(const void *d_row_ws, int64_t row0, int nr, const void *d_col_ws, int64_t col0, int nc, size_t ws_stride,
                       int k, int64_t n_genomes, uint64_t *d_inter, dd_stream stream) {
    if (!d_row_ws || !d_col_ws || !d_inter) return fail(DD_ERR_ARG, "dd_exact_pair_popc: null pointer");
    if (k < 1 || k > DD_EXACT_BITMAP_MAXK) return fail(DD_ERR_ARG, "dd_exact_pair_popc: k=%d outside [1,%d]", k, DD_EXACT_BITMAP_MAXK);
    if (ws_stride < dd::exact_workspace_bytes(k, 0) || ws_stride % 16)
        return fail(DD_ERR_WORKSPACE, "dd_exact_pair_popc: stride %zu below the K5 workspace of k=%d or not 16-byte aligned", ws_stride, k);
    if (nr < 0 || nc < 0 || row0 < 0 || col0 < 0 || row0 + nr > n_genomes || col0 + nc > n_genomes)
        return fail(DD_ERR_ARG, "dd_exact_pair_popc: genome block outside [0,%lld)", (long long)n_genomes);
    DD_CUDA(dd::exact_pair_popc(d_row_ws, row0, nr, d_col_ws, col0, nc, ws_stride, k, n_genomes, d_inter, sm_count_now(), S(stream)),
            "dd_exact_pair_popc");
    return DD_OK;
}

// ---- host-buffer path -----------------------------------------------------------------------------
namespace {
constexpr size_t kHostChunk = (size_t)32 << 20;  // text bytes per H2D / pack / sketch round
struct HostWs {
    uint8_t *text;
    uint32_t *codes;
    uint32_t *invalid;
    dd_pack_state *state;
    void *pack_ws;
    void *sketch_ws;
    uint8_t *regs;
    uint32_t *hist;
    double *cards;
    size_t codes_bytes, invalid_bytes, pack_ws_bytes, sketch_ws_bytes, total;
};
HostWs carve(void *base, size_t n_bytes, int nk, int p) {
    HostWs w;
    uint8_t *q = static_cast<uint8_t *>(base);
    auto take = [&](size_t bytes) {
        uint8_t *r = q;
        q += align_up(bytes, 256);
        return r;
    };
    const size_t chunk = n_bytes < kHostChunk ? n_bytes : kHostChunk;
    w.codes_bytes = dd_pack_codes_bytes(n_bytes);
    w.invalid_bytes = dd_pack_invalid_bytes(n_bytes);
    w.pack_ws_bytes = dd::pack_workspace_bytes(chunk);
    w.sketch_ws_bytes = dd::sketch_workspace_bytes(nk, p);
    w.text = take(2 * align_up(chunk + 16, 256));  // double buffer
    w.codes = reinterpret_cast<uint32_t *>(take(w.codes_bytes));
    w.invalid = reinterpret_cast<uint32_t *>(take(w.invalid_bytes));
    w.state = reinterpret_cast<dd_pack_state *>(take(sizeof(dd_pack_state)));
    w.pack_ws = take(w.pack_ws_bytes);
    w.sketch_ws = take(w.sketch_ws_bytes);
    w.regs = take((size_t)nk << p);
    w.hist = reinterpret_cast<uint32_t *>(take((size_t)nk * DD_HIST_BINS * sizeof(uint32_t)));
    w.cards = reinterpret_cast<double *>(take((size_t)nk * sizeof(double)));
    w.total = (size_t)(q - static_cast<uint8_t *>(base));
    return w;
}
}  // namespace

size_t dd_sketch_fasta_host_workspace_bytes(size_t n_bytes, int nk, int p) {
    return carve(nullptr, n_bytes, nk, p).total + 256;
}

// cards <- NaN when the packer saw a line beginning with '+': the registers built from FASTQ text
// without dd_fastq_to_fasta_host are not what kseq would have produced, and an asynchronous caller
// has no other way of learning it.
__global__ void fastq_poison_kernel(const dd_pack_state *st, double *cards, int nk) {
    if ((st->reserved & DD_PACK_FLAG_FASTQ) && threadIdx.x < (unsigned)nk) cards[threadIdx.x] = nan("");
}

static int sketch_fasta_host_impl(const uint8_t *h_text, size_t n_bytes, uint32_t kmask, int p, int canon, uint8_t *h_regs,
                                  double *h_cards, uint8_t *d_regs_or_null, void *d_ws, size_t ws_bytes, dd_stream stream,
                                  bool synchronize) {
    const int nk = popc(kmask);
    if (!h_text || !h_cards || !d_ws || nk == 0 || bad_p(p)) return fail(DD_ERR_ARG, "dd_sketch_fasta_host: bad argument");
    if (ws_bytes < dd_sketch_fasta_host_workspace_bytes(n_bytes, nk, p))
        return fail(DD_ERR_WORKSPACE, "dd_sketch_fasta_host: workspace %zu < %zu", ws_bytes,
                    dd_sketch_fasta_host_workspace_bytes(n_bytes, nk, p));
    void *base = reinterpret_cast<void *>(align_up(reinterpret_cast<uintptr_t>(d_ws), 256));
    HostWs w = carve(base, n_bytes, nk, p);
    uint8_t *d_regs = d_regs_or_null ? d_regs_or_null : w.regs;
    cudaStream_t st = S(stream);

    // kseq ignores everything before the first record marker (SURVEY.md A.1)
    const size_t skip = dd_fasta_first_record_host(h_text, n_bytes);
    const uint8_t *text = h_text + skip;
    const size_t n = n_bytes - skip;

    DD_CUDA(dd::pack_reset(w.codes, w.codes_bytes, w.invalid, w.invalid_bytes, w.state, st), "pack_reset");
    DD_CUDA(dd::sketch_begin(w.sketch_ws, nk, p, st), "sketch_begin");
    const size_t chunk = n_bytes < kHostChunk ? n_bytes : kHostChunk;
    const size_t nchunks = n ? (n + chunk - 1) / chunk : 0;
    // More than one chunk: copies run on their own stream, double-buffered against pack + sketch.
    // The stream and the events are created here and destroyed before returning WITHOUT waiting:
    // CUDA releases a destroyed stream / event once the work already enqueued on it has completed,
    // so the call stays asynchronous however large the file is.
    cudaStream_t cs = st;
    cudaEvent_t copied[2] = {nullptr, nullptr}, freed[2] = {nullptr, nullptr}, entry = nullptr;
    const bool overlap = nchunks > 1;
    int rc = DD_OK;
    auto cleanup = [&]() {
        for (int i = 0; i < 2; ++i) {
            if (copied[i]) cudaEventDestroy(copied[i]);
            if (freed[i]) cudaEventDestroy(freed[i]);
        }
        if (entry) cudaEventDestroy(entry);
        if (overlap && cs != st) cudaStreamDestroy(cs);
    };
#define DD_TRY(call, what)                                   \
    do {                                                     \
        cudaError_t e__ = (call);                            \
        if (e__ != cudaSuccess) { rc = cuda_fail(e__, what); cleanup(); return rc; } \
    } while (0)
    if (overlap) {
        DD_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking), "create copy stream");
        for (int i = 0; i < 2; ++i) {
            DD_TRY(cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming), "event");
            DD_TRY(cudaEventCreateWithFlags(&freed[i], cudaEventDisableTiming), "event");
        }
        DD_TRY(cudaEventCreateWithFlags(&entry, cudaEventDisableTiming), "event");
        DD_TRY(cudaEventRecord(entry, st), "event record");      // workspace may still be in use upstream
        DD_TRY(cudaStreamWaitEvent(cs, entry, 0), "stream wait");
    }
    size_t done = 0;
    for (size_t c = 0; c < nchunks; ++c) {
        const int b = (int)(c & 1);
        const size_t len = n - done < chunk ? n - done : chunk;
        uint8_t *d_text = w.text + (size_t)b * align_up(chunk + 16, 256);
        if (overlap && c >= 2) DD_TRY(cudaStreamWaitEvent(cs, freed[b], 0), "stream wait");
        DD_TRY(cudaMemcpyAsync(d_text, text + done, len, cudaMemcpyHostToDevice, cs), "H2D text");
        if (overlap) {
            DD_TRY(cudaEventRecord(copied[b], cs), "event record");
            DD_TRY(cudaStreamWaitEvent(st, copied[b], 0), "stream wait");
        }
        DD_TRY(dd::pack_fasta(d_text, len, w.codes, w.invalid, n_bytes, w.state, w.pack_ws, st), "pack_fasta");
        if (overlap) DD_TRY(cudaEventRecord(freed[b], st), "event record");
        if (dd::g_polyt_sentinel) DD_TRY(dd::pack_polyt_sentinel(w.codes, w.invalid, w.state, 0, 0, len, st), "polyt_sentinel");
        // (text bytes stand in for symbols in the floor schedule: the cuts move by ~1 %, the result does not)
        DD_TRY(dd::sketch_update_sched(w.codes, w.invalid, w.state, 0, 0, len, done, kmask, p, canon, w.sketch_ws, st),
               "sketch_update");
        done += len;
    }
    cleanup();
#undef DD_TRY
    DD_CUDA(dd::sketch_end(w.sketch_ws, nk, p, d_regs, w.hist, w.cards, st), "sketch_end");
    DD_COUNT_LAUNCH(), fastq_poison_kernel<<<1, 32, 0, st>>>(w.state, w.cards, nk);
    DD_CUDA(cudaGetLastError(), "fastq_poison");
    DD_CUDA(cudaMemcpyAsync(h_cards, w.cards, (size_t)nk * sizeof(double), cudaMemcpyDeviceToHost, st), "D2H cards");
    if (h_regs) DD_CUDA(cudaMemcpyAsync(h_regs, d_regs, (size_t)nk << p, cudaMemcpyDeviceToHost, st), "D2H regs");
    if (synchronize) {
        dd_pack_state hs;
        DD_CUDA(cudaMemcpyAsync(&hs, w.state, sizeof hs, cudaMemcpyDeviceToHost, st), "D2H state");
        DD_CUDA(cudaStreamSynchronize(st), "synchronize");
        if (hs.reserved & DD_PACK_FLAG_FASTQ) return DD_ERR_FORMAT;   // the caller normalises and retries
    }
    return DD_OK;
}

int dd_sketch_fasta_host(const uint8_t *h_text, size_t n_bytes, uint32_t kmask, int p, int canon, uint8_t *h_regs,
                         double *h_cards, uint8_t *d_regs_or_null, void *d_ws, size_t ws_bytes, dd_stream stream) {
    int rc = sketch_fasta_host_impl(h_text, n_bytes, kmask, p, canon, h_regs, h_cards, d_regs_or_null, d_ws, ws_bytes, stream,
                                    true);
    if (rc != DD_ERR_FORMAT) return rc;
    // FASTQ (a line begins with '+'): rewrite to FASTA the way kseq walks it, then sketch that
    std::vector<uint8_t> fasta(n_bytes + 16);
    const size_t m = dd_fastq_to_fasta_host(h_text, n_bytes, fasta.data());
    rc = sketch_fasta_host_impl(fasta.data(), m, kmask, p, canon, h_regs, h_cards, d_regs_or_null, d_ws, ws_bytes, stream,
                                true);
    if (rc == DD_ERR_FORMAT) return fail(DD_ERR_FORMAT, "dd_sketch_fasta_host: text still looks like FASTQ after normalisation");
    return rc;
}

int dd_sketch_fasta_host_async(const uint8_t *h_text, size_t n_bytes, uint32_t kmask, int p, int canon, uint8_t *h_regs,
                               double *h_cards, uint8_t *d_regs_or_null, void *d_ws, size_t ws_bytes, dd_stream stream) {
    return sketch_fasta_host_impl(h_text, n_bytes, kmask, p, canon, h_regs, h_cards, d_regs_or_null, d_ws, ws_bytes, stream,
                                  false);
}

}  // extern "C"
