// Phased VCF output: the body text of a DNM VCF (decoded by csrc/vcf.cu into UnfzVcfRec lines) rewritten with the
// phase of the DNM carriers -- GT 1|0 / 0|1, and the UOPS / UET FORMAT fields of every sample.
//
// The host builds the sparse edit list (one UnfzVcfEdit per phased cell, sorted by line and sample, CSR by line) and
// the header (vcfio.write_phased_vcf).  Two steps, each one __host__ __device__ body per cell / per FORMAT column, with a
// host entry point (engine-less writes, CPU tests) and a device entry point:
//   size   -- one warp per line: tab ballots over 16-byte loads find the sample columns (as vcf_samples_kernel), every
//             lane sizes the cells that start in its chunk; the output length of every line (int64);
//   write  -- the same walk; a warp exclusive scan of the lanes' lengths places each cell, which is then written.
// The line offsets between the steps are unfz_exclusive_scan_i64 of the lengths: the output can exceed 4 GB.
#include "common.cuh"

namespace {

// the FORMAT plan of one line: key count, index of GT / UOPS / UET (-1 absent), key count of the output
struct FmtPlan {
    int32_t nk, gt, uops, uet, nk_out;
};

__host__ __device__ __forceinline__ bool key_eq(const uint8_t* p, const uint8_t* e, const char* k) {
    for (; *k; ++k, ++p)
        if (p >= e || *p != (uint8_t)*k) return false;
    return p == e;
}

__host__ __device__ FmtPlan fmt_plan(const uint8_t* p, const uint8_t* e) {
    FmtPlan pl{0, -1, -1, -1, 0};
    for (;;) {
        const uint8_t* q = p;
        while (q < e && *q != ':') ++q;
        if (key_eq(p, q, "GT") && pl.gt < 0) pl.gt = pl.nk;
        else if (key_eq(p, q, "UOPS") && pl.uops < 0) pl.uops = pl.nk;
        else if (key_eq(p, q, "UET") && pl.uet < 0) pl.uet = pl.nk;
        ++pl.nk;
        if (q >= e) break;
        p = q + 1;
    }
    pl.nk_out = pl.nk;
    if (pl.uops < 0) pl.uops = pl.nk_out++;
    if (pl.uet < 0) pl.uet = pl.nk_out++;
    return pl;
}

// the FORMAT column: the input keys, then ":UOPS" / ":UET" when absent.  Returns the length; writes when dst != null
__host__ __device__ int64_t fmt_out(const uint8_t* p, const uint8_t* e, const FmtPlan& pl, uint8_t* dst) {
    int64_t n = e - p;
    if (dst)
        for (int64_t k = 0; k < n; ++k) dst[k] = p[k];
    const char* add[2] = {pl.uops >= pl.nk ? ":UOPS" : "", pl.uet >= pl.nk ? ":UET" : ""};
    for (int j = 0; j < 2; ++j)
        for (const char* s = add[j]; *s; ++s) {
            if (dst) dst[n] = (uint8_t)*s;
            ++n;
        }
    return n;
}

__host__ __device__ __forceinline__ int put_int(int32_t v, uint8_t* dst) {
    uint8_t t[12];
    int n = 0;
    uint32_t u = v < 0 ? (uint32_t)(-(int64_t)v) : (uint32_t)v;
    do {
        t[n++] = (uint8_t)('0' + u % 10);
        u /= 10;
    } while (u);
    if (v < 0) t[n++] = '-';
    if (dst)
        for (int k = 0; k < n; ++k) dst[k] = t[n - 1 - k];
    return n;
}

// one sample cell [p, e) rewritten: '\t' + the subfields of the output FORMAT.  ed: this cell's edit, or null (UOPS =
// UET = -1, GT kept).  GT of a phase edit: "1|0" / "0|1" then every allele past the second behind '|'.  Subfields the
// cell dropped are '.'.  Returns the length; writes when dst != null; sets status bits (UNFZ_VCFOUT_*).
__host__ __device__ int64_t cell_out(const uint8_t* p, const uint8_t* e, const FmtPlan& pl, const UnfzVcfEdit* ed,
                                     uint8_t* dst, uint8_t* status) {
    int64_t n = 0;
    if (dst) dst[n] = '\t';
    ++n;
    const uint8_t* q = p;                                  // start of input subfield j (null once the cell is exhausted)
    const int phase = ed ? ed->phase : 0;
    for (int j = 0; j < pl.nk_out; ++j) {
        if (j) {
            if (dst) dst[n] = ':';
            ++n;
        }
        const uint8_t* t = nullptr;
        if (q) {
            t = q;
            while (t < e && *t != ':') ++t;
        }
        if (j == pl.uops || j == pl.uet) {
            const int32_t v = ed ? (j == pl.uops ? ed->uops : ed->uet) : -1;
            n += put_int(v, dst ? dst + n : nullptr);
        } else if (!q) {
            if (dst) dst[n] = '.';
            ++n;
        } else if (j == pl.gt && phase) {
            // the first separator ends the first allele; without one the GT is haploid and cannot be phased
            const uint8_t* s = q;
            while (s < t && *s != '/' && *s != '|') ++s;
            if (s >= t) *status |= UNFZ_VCFOUT_HAPLOID;
            const uint8_t* r = s < t ? s + 1 : t;          // past the second allele
            while (r < t && *r != '/' && *r != '|') ++r;
            if (dst) {
                dst[n] = phase == 1 ? '1' : '0';
                dst[n + 1] = '|';
                dst[n + 2] = phase == 1 ? '0' : '1';
            }
            n += 3;
            for (; r < t; ++r, ++n)
                if (dst) dst[n] = (*r == '/') ? '|' : *r;
        } else {
            if (dst)
                for (const uint8_t* r = q; r < t; ++r) dst[n + (r - q)] = *r;
            n += t - q;
        }
        if (q) q = t < e ? t + 1 : nullptr;
        if (q && j == pl.nk - 1) {                         // more subfields than FORMAT keys
            *status |= UNFZ_VCFOUT_FIELDS;
            q = nullptr;
        }
    }
    return n;
}

struct RwArgs {
    const uint8_t* buf;
    const UnfzVcfRec* recs;
    int64_t n_lines;
    const int64_t* edit_off;
    const UnfzVcfEdit* edits;
    int32_t n_samples;
    int64_t* out_len;          // size step
    uint8_t* line_bad;         // size step
    const int64_t* out_off;    // write step
    uint8_t* out;              // write step
};

// the edit of sample column c of line i (bisection of the line's edits, sorted by sample), or null
__host__ __device__ __forceinline__ const UnfzVcfEdit* edit_of(const RwArgs& A, int64_t i, int64_t c) {
    int64_t lo = A.edit_off[i], hi = A.edit_off[i + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (A.edits[mid].sample < c) lo = mid + 1; else hi = mid;
    }
    return (lo < A.edit_off[i + 1] && A.edits[lo].sample == c) ? A.edits + lo : nullptr;
}

// a sample column the line does not have: '.' for every input key, then the values
__host__ __device__ __forceinline__ int64_t missing_out(const RwArgs& A, int64_t i, int64_t c, const FmtPlan& pl,
                                                        uint8_t* dst, uint8_t* status) {
    const uint8_t dot = '.';
    return cell_out(&dot, &dot + 1, pl, edit_of(A, i, c), dst, status);
}

// one line on the host: the same bodies, one column after the other.  dst null: the length only
int64_t line_host(const RwArgs& A, int64_t i, uint8_t* dst, uint8_t* status) {
    const UnfzVcfRec& r = A.recs[i];
    const uint8_t* L = A.buf + r.line_off;
    const int64_t n = r.line_len;
    int64_t o = 0;
    if (r.fmt_off < 0) {
        if (dst) memcpy(dst, L, n);
        o = n;
    } else {
        if (dst) memcpy(dst, L, r.fmt_off);
        o = r.fmt_off;
        const FmtPlan pl = fmt_plan(L + r.fmt_off, L + r.fmt_off + r.fmt_len);
        o += fmt_out(L + r.fmt_off, L + r.fmt_off + r.fmt_len, pl, dst ? dst + o : nullptr);
        int64_t c = 0;
        if (r.fmt_off + r.fmt_len < n) {
            int64_t s = r.fmt_off + r.fmt_len + 1;
            for (;; ++c) {
                int64_t e = s;
                while (e < n && L[e] != '\t') ++e;
                if (c >= A.n_samples) {
                    *status |= UNFZ_VCFOUT_COLUMNS;
                    break;
                }
                o += cell_out(L + s, L + e, pl, edit_of(A, i, c), dst ? dst + o : nullptr, status);
                if (e >= n) {
                    ++c;
                    break;
                }
                s = e + 1;
            }
        }
        for (; c < A.n_samples; ++c) o += missing_out(A, i, c, pl, dst ? dst + o : nullptr, status);
    }
    if (dst) dst[o] = '\n';
    return o + 1;
}

// one warp per line.  WRITE = false: the output length and the status of every line; true: the output bytes at out_off
template <bool WRITE>
__device__ __forceinline__ void rewrite_line(const RwArgs& A) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= A.n_lines) return;
    const UnfzVcfRec r = A.recs[i];
    const uint8_t* L = A.buf + r.line_off;
    const int64_t n = r.line_len;
    uint8_t* D = WRITE ? A.out + A.out_off[i] : nullptr;
    uint8_t st = 0;
    int64_t o;                                             // output bytes before the current step (valid in every lane)
    if (r.fmt_off < 0) {
        if (WRITE)
            for (int64_t k = lane; k < n; k += 32) D[k] = L[k];
        o = n;
    } else {
        if (WRITE)
            for (int64_t k = lane; k < r.fmt_off; k += 32) D[k] = L[k];
        const uint8_t* fs = L + r.fmt_off;
        const uint8_t* fe = fs + r.fmt_len;
        FmtPlan pl{0, -1, -1, -1, 0};
        int64_t head = 0;                                 // FORMAT column and sample 0 (lane 0)
        if (lane == 0) {
            pl = fmt_plan(fs, fe);
            head = fmt_out(fs, fe, pl, WRITE ? D + r.fmt_off : nullptr);
        }
        pl.nk = __shfl_sync(0xffffffffu, pl.nk, 0);
        pl.gt = __shfl_sync(0xffffffffu, pl.gt, 0);
        pl.uops = __shfl_sync(0xffffffffu, pl.uops, 0);
        pl.uet = __shfl_sync(0xffffffffu, pl.uet, 0);
        pl.nk_out = __shfl_sync(0xffffffffu, pl.nk_out, 0);
        int64_t ncol = 0;
        const int64_t s0 = r.fmt_off + r.fmt_len + 1;      // first sample column
        if (s0 <= n) {
            if (lane == 0) {
                if (A.n_samples == 0) {
                    st |= UNFZ_VCFOUT_COLUMNS;
                } else {
                    int64_t e = s0;
                    while (e < n && L[e] != '\t') ++e;
                    head += cell_out(L + s0, L + e, pl, edit_of(A, i, 0), WRITE ? D + r.fmt_off + head : nullptr, &st);
                }
            }
            ncol = 1;
        }
        o = r.fmt_off + __shfl_sync(0xffffffffu, head, 0);
        if (s0 < n) {
            // 16-byte aligned loads (the text buffer is 16-byte aligned and padded by 16 bytes): the first step starts
            // at the boundary at or below s0, and bytes outside [s0, n) are masked
            for (int64_t a = ((r.line_off + s0) & ~(int64_t)15) - r.line_off; a < n; a += 32 * 16) {
                const int64_t b = a + 16 * lane;
                uint8_t w[16];
                if (b < n) {
                    const int4 v = *reinterpret_cast<const int4*>(L + b);
                    memcpy(w, &v, 16);
                } else {
                    memset(w, 0, 16);
                }
                int cnt = 0;
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    if (b + k < s0 || b + k >= n) w[k] = 0;
                    cnt += w[k] == '\t';
                }
                int incl = cnt;
                for (int d = 1; d < 32; d <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += y;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                // this lane's cells: sized, then (WRITE) placed by the warp's exclusive scan of the sizes
                int64_t mine = 0;
                for (int pass = 0; pass < (WRITE ? 2 : 1); ++pass) {
                    int64_t at = 0;
                    if (pass == 1) {
                        int64_t x = mine;
                        for (int d = 1; d < 32; d <<= 1) {
                            const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
                            if (lane >= d) x += y;
                        }
                        at = o + x - mine;
                    }
                    int64_t c = ncol + incl - cnt - 1;
                    for (int k = 0, left = cnt; k < 16 && left; ++k) {
                        if (w[k] != '\t') continue;
                        ++c;                               // the column starting after this tab
                        --left;
                        if (c >= A.n_samples) {
                            st |= UNFZ_VCFOUT_COLUMNS;
                            continue;
                        }
                        const int64_t cs = b + k + 1;
                        int64_t e = cs;
                        while (e < n && L[e] != '\t') ++e;
                        const int64_t len = cell_out(L + cs, L + e, pl, edit_of(A, i, c),
                                                     pass == 1 ? D + at : nullptr, &st);
                        if (pass == 0) mine += len; else at += len;
                    }
                }
                int64_t sum = mine;
                for (int d = 16; d >= 1; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
                o += sum;
                ncol += total;
            }
        }
        // absent trailing columns: lane-strided, each the same missing cell up to its edit, so placed by prefix counts
        const int64_t first_missing = ncol < A.n_samples ? ncol : A.n_samples;
        for (int64_t c0 = first_missing; c0 < A.n_samples; c0 += 32) {
            const int64_t c = c0 + lane;
            int64_t len = 0;
            if (c < A.n_samples) len = missing_out(A, i, c, pl, nullptr, &st);
            int64_t x = len;
            for (int d = 1; d < 32; d <<= 1) {
                const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            if (WRITE && c < A.n_samples) missing_out(A, i, c, pl, D + o + x - len, &st);
            o += __shfl_sync(0xffffffffu, x, 31);
        }
    }
    const unsigned bad = __reduce_or_sync(0xffffffffu, (unsigned)st);
    if (lane == 0) {
        if (WRITE) D[o] = '\n';
        else {
            A.out_len[i] = o + 1;
            A.line_bad[i] = (uint8_t)bad;
        }
    }
}

__global__ void __launch_bounds__(256) vcf_rewrite_size_kernel(RwArgs A) { rewrite_line<false>(A); }

__global__ void __launch_bounds__(256) vcf_rewrite_write_kernel(RwArgs A) { rewrite_line<true>(A); }

}  // namespace

extern "C" int64_t unfz_vcf_rewrite_size_host(const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines,
                                              const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples,
                                              int64_t* out_len, uint8_t* line_bad) {
    RwArgs A{buf, recs, n_lines, edit_off, edits, n_samples, out_len, line_bad, nullptr, nullptr};
    int64_t total = 0;
    for (int64_t i = 0; i < n_lines; ++i) {
        uint8_t st = 0;
        out_len[i] = line_host(A, i, nullptr, &st);
        line_bad[i] = st;
        total += out_len[i];
    }
    return total;
}

extern "C" int unfz_vcf_rewrite_write_host(const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines,
                                           const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples,
                                           const int64_t* out_off, uint8_t* out) {
    RwArgs A{buf, recs, n_lines, edit_off, edits, n_samples, nullptr, nullptr, out_off, out};
    for (int64_t i = 0; i < n_lines; ++i) {
        uint8_t st = 0;
        line_host(A, i, out + out_off[i], &st);
    }
    return 0;
}

extern "C" int unfz_vcf_rewrite_size(UnfzCtx* ctx, const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines,
                                     const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples, int64_t* out_len,
                                     uint8_t* line_bad, void* stream) {
    if (n_lines <= 0) return 0;
    RwArgs A{buf, recs, n_lines, edit_off, edits, n_samples, out_len, line_bad, nullptr, nullptr};
    vcf_rewrite_size_kernel<<<(unsigned)((n_lines * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_vcf_rewrite_write(UnfzCtx* ctx, const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines,
                                      const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples,
                                      const int64_t* out_off, uint8_t* out, void* stream) {
    if (n_lines <= 0) return 0;
    RwArgs A{buf, recs, n_lines, edit_off, edits, n_samples, nullptr, nullptr, out_off, out};
    vcf_rewrite_write_kernel<<<(unsigned)((n_lines * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
