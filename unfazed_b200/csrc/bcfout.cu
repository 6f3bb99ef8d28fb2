// Phased VCF output from a BCF DNM list: every record of the inflated BCF (parsed by csrc/bcf.cu into UnfzBcfRec)
// printed as VCF text, the way htslib's vcf_format prints a binary record, with the phase of the DNM carriers -- GT
// 1|0 / 0|1, and the UOPS / UET FORMAT fields of every sample.
//
// The host builds the sparse edit list (UnfzVcfEdit, CSR by record, as for csrc/vcfout.cu) and the header
// (bcfio.write_phased_vcf).  Two steps, each one __host__ __device__ body for the fixed columns and one per sample cell,
// with a host entry point (engine-less writes, CPU tests) and a device entry point:
//   size   -- one warp per record: lane 0 prints CHROM ... FORMAT, the sample cells are dealt to the lanes (a cell's
//             values are direct loads at field + sample * count * width); the output length of every record (int64);
//   write  -- the same walk; a warp exclusive scan of the cells' lengths places each cell, which is then written.
// The record offsets between the steps are unfz_exclusive_scan_i64 of the lengths: the output can exceed 4 GB.
//
// Floats are printed as C's "%g".  The bodies print a float only when the exact integer path below proves its text;
// any other float marks the record UNFZ_BCFOUT_FLOAT_HOST.  The host bodies then print it with snprintf, and the device
// write step skips the record: its length and text come from the host entry points.
#include "bcf.cuh"

namespace {

// output cursor: counts bytes, and writes them when d != null
struct Out {
    uint8_t* d;
    int64_t n;
    __host__ __device__ __forceinline__ void c(uint8_t x) {
        if (d) d[n] = x;
        ++n;
    }
    __host__ __device__ __forceinline__ void s(const uint8_t* p, int64_t len) {
        if (d)
            for (int64_t k = 0; k < len; ++k) d[n + k] = p[k];
        n += len;
    }
    __host__ __device__ __forceinline__ void z(const char* p) {
        for (; *p; ++p) c((uint8_t)*p);
    }
};

// decimal digits, at least min_digits (zero-padded); written last digit first, so no digit buffer goes to local memory
__host__ __device__ __forceinline__ void put_u64(uint64_t u, Out& o, int min_digits = 1) {
    int nd = 1;
    for (uint64_t t = u; t >= 10; t /= 10) ++nd;
    if (nd < min_digits) nd = min_digits;
    if (o.d)
        for (int k = nd - 1; k >= 0; --k, u /= 10) o.d[o.n + k] = (uint8_t)('0' + u % 10);
    o.n += nd;
}

__host__ __device__ __forceinline__ void put_i64(int64_t v, Out& o) {
    if (v < 0) o.c('-');
    put_u64(v < 0 ? (uint64_t)0 - (uint64_t)v : (uint64_t)v, o);
}

// "%g" of a float32 from integer arithmetic alone: the value is m / 2^s, and 10^5 <= value * 10^k < 10^6 for one k in
// [0, 10] whenever 1e-5 <= |value| < 1e6; then m * 10^k < 2^58 and the six significant digits are that product shifted
// right by s, rounded to nearest with ties to even -- the exact decimal rounding printf performs.  False (nothing
// printed) for a value it does not prove: exponent style (|value| >= 999999.5 or below 1e-4 after rounding),
// subnormals, infinities and NaNs.
__host__ __device__ bool put_g(uint32_t bits, Out& o) {
    const bool neg = bits >> 31;
    const uint32_t ex = (bits >> 23) & 0xFF, fr = bits & 0x7FFFFF;
    if (ex == 0 && fr == 0) {
        if (neg) o.c('-');
        o.c('0');
        return true;
    }
    if (ex == 0 || ex == 0xFF) return false;
    const uint64_t m = fr | 0x800000u;
    const int s = 150 - (int)ex;                         // |value| = m / 2^s
    if (s <= 0) return false;                            // >= 2^24
    uint64_t p10 = 1, n = 0, q = 0;
    int k = 0;
    for (; k <= 10; ++k, p10 *= 10) {
        n = m * p10;
        q = s >= 64 ? 0 : n >> s;
        if (q >= 100000) break;
    }
    if (k > 10 || q >= 1000000) return false;
    const uint64_t rem = n - (q << s), half = 1ull << (s - 1);
    if (rem > half || (rem == half && (q & 1))) ++q;
    int x = 5 - k;                                       // the decimal exponent after rounding
    if (q == 1000000) {
        q = 100000;
        ++x;
    }
    if (x > 5 || x < -4) return false;
    int d = 5 - x;                                       // decimals of the fixed style
    uint64_t pd = 1;
    for (int j = 0; j < d; ++j) pd *= 10;
    uint64_t ip = q / pd, fp = q % pd;
    while (d > 0 && fp % 10 == 0) {
        fp /= 10;
        --d;
    }
    if (neg) o.c('-');
    put_u64(ip, o);
    if (d > 0) {
        o.c('.');
        put_u64(fp, o, d);
    }
    return true;
}

// a float that is not a BCF sentinel: the exact path, else the host's snprintf (the device prints nothing)
__host__ __device__ __forceinline__ void put_float(uint32_t bits, Out& o, uint8_t* st) {
    if (put_g(bits, o)) return;
    *st |= UNFZ_BCFOUT_FLOAT_HOST;
#ifndef __CUDA_ARCH__
    float f;
    memcpy(&f, &bits, 4);
    char t[32];
    const int n = snprintf(t, sizeof(t), "%g", (double)f);
    o.s((const uint8_t*)t, n);
#endif
}

// bytes of a string value up to its first NUL
__host__ __device__ __forceinline__ int64_t str_len(const uint8_t* p, int64_t n) {
    int64_t k = 0;
    while (k < n && p[k]) ++k;
    return k;
}

// a typed vector as bcf_fmt_array prints it: '.' when empty; integers and floats comma-joined up to the end of the
// vector, '.' for a missing value; a string up to its first NUL, with '.' for the missing character 0x07
__host__ __device__ void put_vec(const uint8_t* p, int t, int64_t n, Out& o, uint8_t* st) {
    if (n == 0) {
        o.c('.');
        return;
    }
    if (t == BT_CHAR) {
        for (int64_t j = 0; j < n && p[j]; ++j) o.c(p[j] == 7 ? '.' : p[j]);
    } else if (is_int_type(t)) {
        const int w = type_width(t);
        for (int64_t j = 0; j < n; ++j) {
            int32_t v;
            const int k = ld_int(p + j * w, t, &v);
            if (k == 2) break;
            if (j) o.c(',');
            if (k == 1) o.c('.');
            else put_i64(v, o);
        }
    } else if (t == BT_FLOAT) {
        for (int64_t j = 0; j < n; ++j) {
            const uint32_t b = ld_u32(p + 4 * j);
            if (b == FLOAT_EOV) break;
            if (j) o.c(',');
            if (b == FLOAT_MISSING) o.c('.');
            else put_float(b, o, st);
        }
    } else {
        *st |= UNFZ_BCFOUT_BAD;                          // values of type NULL
    }
}

struct FmtArgs {
    const uint8_t* buf;
    const UnfzBcfRec* recs;
    int64_t n_recs;
    const uint8_t* str_names;
    const int64_t* str_off;
    int32_t n_str;
    const uint8_t* ctg_names;
    const int64_t* ctg_off;
    int32_t n_ctg;
    int32_t gt, uops, uet;                               // string-dictionary ids, -1: not in the header
    const int64_t* edit_off;
    const UnfzVcfEdit* edits;
    int32_t n_samples;
    int64_t* out_len;                                    // size step
    uint8_t* status;                                     // size step: written; write step: records to skip
    const int64_t* out_off;                              // write step
    uint8_t* out;                                        // write step
};

// a dictionary name; an id outside the dictionary (or of an unused index) is malformed
__host__ __device__ __forceinline__ void put_name(const uint8_t* names, const int64_t* off, int32_t n, int32_t id,
                                                  Out& o, uint8_t* st) {
    if (id < 0 || id >= n || off[id + 1] == off[id]) {
        *st |= UNFZ_BCFOUT_BAD;
        return;
    }
    o.s(names + off[id], off[id + 1] - off[id]);
}

// a typed integer key at p (the parse step checked it); p advanced
__host__ __device__ __forceinline__ int32_t rd_key(const uint8_t* b, int64_t& p, int64_t e) {
    int t;
    int64_t n;
    uint8_t why = 0;
    typed_hdr(b, p, e, &t, &n, &why);
    int32_t v = -1;
    if (ld_int(b + p, t, &v) != 0) v = -1;
    p += type_width(t);
    return v;
}

struct RecHead {
    int64_t se, ie;                                      // end of the shared block, end of the record
    int n_info, n_fmt;
};

__host__ __device__ __forceinline__ RecHead rec_head(const uint8_t* b, const UnfzBcfRec& r) {
    const int64_t l_shared = ld_u32(b + r.rec_off), l_indiv = ld_u32(b + r.rec_off + 4);
    RecHead h;
    h.se = r.rec_off + 8 + l_shared;
    h.ie = h.se + l_indiv;
    h.n_info = (int)(ld_u32(b + r.rec_off + 24) & 0xFFFF);
    h.n_fmt = (int)(ld_u32(b + r.rec_off + 28) >> 24);
    return h;
}

// CHROM ... INFO, and with samples '\t' FORMAT (":UOPS" / ":UET" appended unless the record has them)
__host__ __device__ void fixed_out(const FmtArgs& A, const UnfzBcfRec& r, Out& o, uint8_t* st) {
    const uint8_t* b = A.buf;
    const RecHead h = rec_head(b, r);
    uint8_t why = 0;                                     // the parse step validated the layout
    int t;
    int64_t n;
    put_name(A.ctg_names, A.ctg_off, A.n_ctg, r.contig, o, st);
    o.c('\t');
    put_i64((int64_t)r.pos0 + 1, o);
    o.c('\t');
    int64_t p = r.rec_off + 32;
    typed_hdr(b, p, h.se, &t, &n, &why);                 // ID
    if (t != BT_CHAR && n) *st |= UNFZ_BCFOUT_BAD;
    int64_t len = t == BT_CHAR ? str_len(b + p, n) : 0;
    if (len) o.s(b + p, len);
    else o.c('.');
    p += n * type_width(t);
    o.c('\t');
    if (r.n_allele == 0) o.c('.');
    for (int a = 0; a < r.n_allele; ++a) {               // REF, then ALT joined by ','
        typed_hdr(b, p, h.se, &t, &n, &why);
        if (a) o.c(a == 1 ? '\t' : ',');
        o.s(b + p, str_len(b + p, n));
        p += n;
    }
    if (r.n_allele < 2) {
        o.c('\t');
        o.c('.');
    }
    o.c('\t');
    const uint32_t qual = ld_u32(b + r.rec_off + 20);
    if (qual == FLOAT_MISSING || qual == FLOAT_EOV) o.c('.');
    else put_float(qual, o, st);
    o.c('\t');
    typed_hdr(b, p, h.se, &t, &n, &why);                 // FILTER
    if (n == 0) o.c('.');
    else if (!is_int_type(t)) *st |= UNFZ_BCFOUT_BAD;
    else
        for (int64_t j = 0; j < n; ++j) {
            int32_t id;
            if (ld_int(b + p + j * type_width(t), t, &id) != 0) id = -1;
            if (j) o.c(';');
            put_name(A.str_names, A.str_off, A.n_str, id, o, st);
        }
    p += n * type_width(t);
    o.c('\t');
    if (h.n_info == 0) o.c('.');
    for (int k = 0; k < h.n_info; ++k) {                 // INFO: key, or key=value
        const int32_t key = rd_key(b, p, h.se);
        typed_hdr(b, p, h.se, &t, &n, &why);
        if (k) o.c(';');
        put_name(A.str_names, A.str_off, A.n_str, key, o, st);
        if (n) {
            o.c('=');
            put_vec(b + p, t, n, o, st);
        }
        p += n * type_width(t);
    }
    if (A.n_samples == 0) return;
    o.c('\t');
    bool uops = false, uet = false;
    if (h.n_fmt == 0) o.c('.');
    p = h.se;
    for (int k = 0; k < h.n_fmt; ++k) {
        const int32_t key = rd_key(b, p, h.ie);
        typed_hdr(b, p, h.ie, &t, &n, &why);
        if (k) o.c(':');
        put_name(A.str_names, A.str_off, A.n_str, key, o, st);
        uops |= key == A.uops;
        uet |= key == A.uet;
        p += (int64_t)A.n_samples * n * type_width(t);
    }
    if (!uops) o.z(":UOPS");
    if (!uet) o.z(":UET");
}

// one GT allele: '.' for a missing one (allele code 0 or the missing integer); a negative code is malformed
__host__ __device__ __forceinline__ void put_allele(const uint8_t* v, int t, Out& o, uint8_t* st) {
    int32_t x;
    const int k = ld_int(v, t, &x);
    if (k == 1 || (k == 0 && (x >> 1) == 0)) {
        o.c('.');
    } else if (k != 0 || x < 0) {
        *st |= UNFZ_BCFOUT_BAD;
        o.c('.');
    } else {
        put_i64((x >> 1) - 1, o);
    }
}

// GT as bcf_format_gt prints it ("/|"[code & 1] before every allele after the first, '.' when empty); with a phase edit
// "1|0" / "0|1" and every allele past the second behind '|' -- a GT of fewer than two alleles cannot be phased
__host__ __device__ void gt_out(const uint8_t* v, int t, int64_t n, int phase, Out& o, uint8_t* st) {
    if (t != BT_NULL && !is_int_type(t)) {
        *st |= UNFZ_BCFOUT_BAD;
        return;
    }
    const int w = type_width(t);
    int64_t na = 0;                                      // alleles before the end of the vector
    if (w)
        for (int32_t x; na < n && ld_int(v + na * w, t, &x) != 2;) ++na;
    if (phase) {
        if (na < 2) *st |= UNFZ_BCFOUT_HAPLOID;
        o.z(phase == 1 ? "1|0" : "0|1");
        for (int64_t j = 2; j < na; ++j) {
            o.c('|');
            put_allele(v + j * w, t, o, st);
        }
        return;
    }
    if (na == 0) o.c('.');
    for (int64_t j = 0; j < na; ++j) {
        if (j) o.c("/|"[v[j * w] & 1]);
        put_allele(v + j * w, t, o, st);
    }
}

// the edit of sample c of record i (bisection of the record's edits, sorted by sample), or null
__host__ __device__ __forceinline__ const UnfzVcfEdit* edit_of(const FmtArgs& A, int64_t i, int64_t c) {
    int64_t lo = A.edit_off[i], hi = A.edit_off[i + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (A.edits[mid].sample < c) lo = mid + 1; else hi = mid;
    }
    return (lo < A.edit_off[i + 1] && A.edits[lo].sample == c) ? A.edits + lo : nullptr;
}

// sample cell c of record i: '\t' + the values of every FORMAT field (UOPS / UET replaced by the edit's values, -1
// without an edit), then the UOPS / UET the record lacks.  A record without FORMAT fields has the cell "."
__host__ __device__ void cell_out(const FmtArgs& A, const UnfzBcfRec& r, const RecHead& h, int64_t i, int64_t c, Out& o,
                                  uint8_t* st) {
    const uint8_t* b = A.buf;
    const UnfzVcfEdit* ed = edit_of(A, i, c);
    const int32_t uops = ed ? ed->uops : -1, uet = ed ? ed->uet : -1;
    int phase = ed ? ed->phase : 0;
    bool seen_uops = false, seen_uet = false;
    uint8_t why = 0;
    o.c('\t');
    if (h.n_fmt == 0) o.c('.');
    int64_t p = h.se;
    for (int k = 0; k < h.n_fmt; ++k) {
        const int32_t key = rd_key(b, p, h.ie);
        int t;
        int64_t n;
        typed_hdr(b, p, h.ie, &t, &n, &why);
        const int w = type_width(t);
        const uint8_t* v = b + p + c * n * w;
        if (k) o.c(':');
        if (key == A.uops && !seen_uops) {
            put_i64(uops, o);
            seen_uops = true;
        } else if (key == A.uet && !seen_uet) {
            put_i64(uet, o);
            seen_uet = true;
        } else if (key == A.gt) {
            gt_out(v, t, n, phase, o, st);
            phase = 0;                                   // the first GT field takes the edit
        } else {
            put_vec(v, t, n, o, st);
        }
        p += (int64_t)A.n_samples * n * w;
    }
    if (!seen_uops) {
        o.c(':');
        put_i64(uops, o);
    }
    if (!seen_uet) {
        o.c(':');
        put_i64(uet, o);
    }
}

// one record on the host: the same bodies, one cell after the other
int64_t record_host(const FmtArgs& A, int64_t i, uint8_t* dst, uint8_t* st) {
    const UnfzBcfRec& r = A.recs[i];
    const RecHead h = rec_head(A.buf, r);
    Out o{dst, 0};
    fixed_out(A, r, o, st);
    for (int64_t c = 0; c < A.n_samples; ++c) cell_out(A, r, h, i, c, o, st);
    o.c('\n');
    return o.n;
}

// one warp per record.  WRITE = false: the output length and the status of every record; true: the output bytes at
// out_off, except for the records the host prints (UNFZ_BCFOUT_FLOAT_HOST)
template <bool WRITE>
__device__ __forceinline__ void format_record(const FmtArgs& A) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= A.n_recs) return;
    if (WRITE && (A.status[i] & UNFZ_BCFOUT_FLOAT_HOST)) return;
    const UnfzBcfRec r = A.recs[i];
    const RecHead h = rec_head(A.buf, r);
    uint8_t* D = WRITE ? A.out + A.out_off[i] : nullptr;
    uint8_t st = 0;
    int64_t head = 0;
    if (lane == 0) {
        Out o{D, 0};
        fixed_out(A, r, o, &st);
        head = o.n;
    }
    int64_t o = __shfl_sync(0xffffffffu, head, 0);       // output bytes so far (every lane)
    for (int64_t c0 = 0; c0 < A.n_samples; c0 += 32) {
        const int64_t c = c0 + lane;
        int64_t len = 0;
        if (c < A.n_samples) {
            Out t{nullptr, 0};
            cell_out(A, r, h, i, c, t, &st);
            len = t.n;
        }
        int64_t x = len;                                 // inclusive scan of the cells' lengths
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (WRITE && c < A.n_samples) {
            Out t{D + o + x - len, 0};
            cell_out(A, r, h, i, c, t, &st);
        }
        o += __shfl_sync(0xffffffffu, x, 31);
    }
    const unsigned bad = __reduce_or_sync(0xffffffffu, (unsigned)st);
    if (lane == 0) {
        if (WRITE) D[o] = '\n';
        else {
            A.out_len[i] = o + 1;
            A.status[i] = (uint8_t)bad;
        }
    }
}

__global__ void __launch_bounds__(256) bcf_format_size_kernel(FmtArgs A) { format_record<false>(A); }

__global__ void __launch_bounds__(256) bcf_format_write_kernel(FmtArgs A) { format_record<true>(A); }

FmtArgs make_args(const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs, const uint8_t* str_names,
                  const int64_t* str_off, int32_t n_str, const uint8_t* ctg_names, const int64_t* ctg_off, int32_t n_ctg,
                  const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples) {
    return FmtArgs{buf, recs, n_recs, str_names, str_off, n_str, ctg_names, ctg_off, n_ctg, keys[0], keys[1], keys[2],
                   edit_off, edits, n_samples, nullptr, nullptr, nullptr, nullptr};
}

}  // namespace

#define UNFZ_BCFOUT_ARGS buf, recs, n_recs, str_names, str_off, n_str, ctg_names, ctg_off, n_ctg, keys, edit_off, edits, n_samples

extern "C" int64_t unfz_bcf_format_size_host(const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs,
                                             const uint8_t* str_names, const int64_t* str_off, int32_t n_str,
                                             const uint8_t* ctg_names, const int64_t* ctg_off, int32_t n_ctg,
                                             const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                                             int32_t n_samples, int64_t* out_len, uint8_t* status) {
    const FmtArgs A = make_args(UNFZ_BCFOUT_ARGS);
    int64_t total = 0;
    for (int64_t i = 0; i < n_recs; ++i) {
        uint8_t st = 0;
        out_len[i] = record_host(A, i, nullptr, &st);
        status[i] = st;
        total += out_len[i];
    }
    return total;
}

extern "C" int unfz_bcf_format_write_host(const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs,
                                          const uint8_t* str_names, const int64_t* str_off, int32_t n_str,
                                          const uint8_t* ctg_names, const int64_t* ctg_off, int32_t n_ctg,
                                          const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                                          int32_t n_samples, const int64_t* out_off, uint8_t* out) {
    const FmtArgs A = make_args(UNFZ_BCFOUT_ARGS);
    for (int64_t i = 0; i < n_recs; ++i) {
        uint8_t st = 0;
        record_host(A, i, out + out_off[i], &st);
    }
    return 0;
}

extern "C" int unfz_bcf_format_size(UnfzCtx* ctx, const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs,
                                    const uint8_t* str_names, const int64_t* str_off, int32_t n_str,
                                    const uint8_t* ctg_names, const int64_t* ctg_off, int32_t n_ctg, const int32_t* keys,
                                    const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples,
                                    int64_t* out_len, uint8_t* status, void* stream) {
    if (n_recs <= 0) return 0;
    FmtArgs A = make_args(UNFZ_BCFOUT_ARGS);
    A.out_len = out_len;
    A.status = status;
    bcf_format_size_kernel<<<(unsigned)((n_recs * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_bcf_format_write(UnfzCtx* ctx, const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs,
                                     const uint8_t* str_names, const int64_t* str_off, int32_t n_str,
                                     const uint8_t* ctg_names, const int64_t* ctg_off, int32_t n_ctg, const int32_t* keys,
                                     const int64_t* edit_off, const UnfzVcfEdit* edits, int32_t n_samples,
                                     const uint8_t* status, const int64_t* out_off, uint8_t* out, void* stream) {
    if (n_recs <= 0) return 0;
    FmtArgs A = make_args(UNFZ_BCFOUT_ARGS);
    A.status = const_cast<uint8_t*>(status);
    A.out_off = out_off;
    A.out = out;
    bcf_format_write_kernel<<<(unsigned)((n_recs * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
