// VCF text decoding: the inflated text of a tabix region query -> line boundaries, fixed fields per line, and the
// genotype fields of the wanted samples of the selected lines.
//
// The host inflates the BGZF blocks and parses the TBI (vcfio.py).  Three steps, each one __host__ __device__ body with
// a host entry point (engine-less loads, CPU tests) and a device entry point:
//   line boundaries  -- newline count per 16-byte chunk, an exclusive scan (scan.cu), newline positions written out;
//   fixed fields     -- one thread per line: CHROM hash, POS, REF / ALT, INFO END, FORMAT slots (UnfzVcfRec);
//   sample fields    -- one warp per selected line: tab ballots over 16-byte loads find the sample columns, the lanes
//                       that own a wanted column decode GT / GQ / AD (or RO / AO) as cyvcf2 reports them.
#include "common.cuh"

namespace {

constexpr int VCF_CHUNK = 16;                         // bytes per thread of the line-boundary pass

__host__ __device__ __forceinline__ int nl_count16(const uint8_t* buf, int64_t n, int64_t c) {
    const int64_t a = c * VCF_CHUNK;
    const int64_t b = a + VCF_CHUNK < n ? a + VCF_CHUNK : n;
    int k = 0;
    for (int64_t i = a; i < b; ++i) k += buf[i] == '\n';
    return k;
}

__host__ __device__ __forceinline__ void nl_write16(const uint8_t* buf, int64_t n, int64_t c, int64_t at, int64_t* ends) {
    const int64_t a = c * VCF_CHUNK;
    const int64_t b = a + VCF_CHUNK < n ? a + VCF_CHUNK : n;
    for (int64_t i = a; i < b; ++i)
        if (buf[i] == '\n') ends[at++] = i;
}

// non-negative decimal integer of [p, e); false when empty, not all digits, or above `lim`
__host__ __device__ __forceinline__ bool parse_uint(const uint8_t* p, const uint8_t* e, int64_t lim, int64_t* out) {
    if (p >= e) return false;
    int64_t v = 0;
    for (; p < e; ++p) {
        if (*p < '0' || *p > '9') return false;
        v = v * 10 + (*p - '0');
        if (v > lim) return false;
    }
    *out = v;
    return true;
}

__host__ __device__ __forceinline__ bool key_is(const uint8_t* p, const uint8_t* e, const char* k) {
    for (; *k; ++k, ++p)
        if (p >= e || *p != (uint8_t)*k) return false;
    return p == e;
}

// line [s, e) (e: its '\n' or the end of the text)
__host__ __device__ void parse_vcf_line(const uint8_t* buf, int64_t s, int64_t e, UnfzVcfRec* out) {
    UnfzVcfRec r;
    memset(&r, 0, sizeof(r));
    r.line_off = s;
    if (e > s && buf[e - 1] == '\r') --e;               // CRLF line ends
    r.line_len = (int32_t)(e - s);
    r.fmt_off = -1;
    for (int k = 0; k < 5; ++k) r.slot[k] = -1;
    const uint8_t* L = buf + s;
    const int64_t n = e - s;
    // column starts of the first 9 columns (CHROM .. FORMAT)
    int64_t col[10];
    int nc = 1;
    col[0] = 0;
    for (int64_t i = 0; i < n && nc < 10; ++i)
        if (L[i] == '\t') col[nc++] = i + 1;
    if (nc < 8) {
        r.flags = UNFZ_VCF_BAD;
        *out = r;
        return;
    }
    const int64_t col_end8 = nc > 8 ? col[8] - 1 : n;     // INFO ends at the FORMAT tab or the line end
    auto cend = [&](int c) { return c + 1 < nc ? col[c + 1] - 1 : (c == 7 ? col_end8 : n); };
    r.chrom_len = (int32_t)(col[1] - 1);
    uint32_t h = 2166136261u;                            // FNV-1a 32 of CHROM
    for (int64_t i = 0; i < col[1] - 1; ++i) {
        h ^= L[i];
        h *= 16777619u;
    }
    r.chrom_hash = h;
    int64_t pos1;
    if (!parse_uint(L + col[1], L + cend(1), 2147483647LL, &pos1) || pos1 < 1) {
        r.flags = UNFZ_VCF_BAD;
        *out = r;
        return;
    }
    r.pos0 = (int32_t)(pos1 - 1);
    r.ref_off = (int32_t)col[3];
    r.ref_len = (int32_t)(cend(3) - col[3]);
    r.ref0 = r.ref_len > 0 ? L[col[3]] : 0;
    r.alt_off = (int32_t)col[4];
    r.alt_len = (int32_t)(cend(4) - col[4]);
    const uint8_t* a = L + col[4];
    if (r.alt_len == 1 && a[0] == '.') {
        r.n_alt = 0;
    } else {
        r.n_alt = 1;
        for (int i = 0; i < r.alt_len; ++i) r.n_alt += a[i] == ',';
    }
    if (r.n_alt == 1 && r.ref_len == 1 && r.alt_len == 1 && a[0] != '*') r.flags |= UNFZ_VCF_SIMPLE;
    // INFO END (1-based inclusive = 0-based exclusive end), as tabix indexes the record
    int64_t rend = (int64_t)r.pos0 + r.ref_len;
    {
        const uint8_t* p = L + col[7];
        const uint8_t* ie = L + col_end8;
        while (p < ie) {
            const uint8_t* q = p;
            while (q < ie && *q != ';') ++q;
            if (q - p > 4 && p[0] == 'E' && p[1] == 'N' && p[2] == 'D' && p[3] == '=') {
                int64_t v;
                if (parse_uint(p + 4, q, 2147483647LL, &v) && v > r.pos0) rend = v;
                break;
            }
            p = q + 1;
        }
    }
    if (rend > 2147483647LL) {
        r.flags = UNFZ_VCF_BAD;
        *out = r;
        return;
    }
    r.rend = (int32_t)rend;
    if (nc > 8) {
        r.fmt_off = (int32_t)col[8];
        r.fmt_len = (int32_t)((nc > 9 ? col[9] - 1 : n) - col[8]);
        const uint8_t* p = L + col[8];
        const uint8_t* fe = p + r.fmt_len;
        int k = 0;
        while (p <= fe && k < 127) {
            const uint8_t* q = p;
            while (q < fe && *q != ':') ++q;
            if (key_is(p, q, "GT")) r.slot[0] = (int8_t)k;
            else if (key_is(p, q, "GQ")) r.slot[1] = (int8_t)k;
            else if (key_is(p, q, "AD")) r.slot[2] = (int8_t)k;
            else if (key_is(p, q, "RO")) r.slot[3] = (int8_t)k;
            else if (key_is(p, q, "AO")) r.slot[4] = (int8_t)k;
            ++k;
            p = q + 1;
        }
    }
    *out = r;
}

// one allele of GT at p: -1 missing, else its index; *p advanced past it.  false: not a number and not '.'
__host__ __device__ __forceinline__ bool gt_allele(const uint8_t*& p, const uint8_t* e, int64_t* a) {
    if (p < e && *p == '.') {
        ++p;
        *a = -1;
        return true;
    }
    int64_t v = 0;
    const uint8_t* s = p;
    while (p < e && *p >= '0' && *p <= '9') {
        v = v * 10 + (*p - '0');
        if (v > 2147483647LL) return false;
        ++p;
    }
    *a = v;
    return p > s;
}

// cyvcf2's gt_types (gts012=False): the first two alleles; '/' and '|' alike
__host__ __device__ __forceinline__ int decode_gt(const uint8_t* p, const uint8_t* e, bool* bad) {
    int64_t a, b;
    if (!gt_allele(p, e, &a)) { *bad = true; return 2; }
    if (p >= e || (*p != '/' && *p != '|')) {              // haploid
        if (a < 0) return 2;
        return a == 0 ? 0 : (a == 1 ? 3 : 2);
    }
    ++p;
    if (!gt_allele(p, e, &b)) { *bad = true; return 2; }
    if (a < 0 && b < 0) return 2;
    if (a < 0 || b < 0) return (a < 0 ? b : a) == 0 ? 2 : 1;
    if (a != b) return 1;
    return a == 0 ? 0 : 3;
}

// a signed decimal integer [p, e) -> int32; '.' -> missing.  0 ok, 1 missing, 2 malformed / overflow
__host__ __device__ __forceinline__ int parse_int32(const uint8_t* p, const uint8_t* e, int32_t* out) {
    if (e - p == 1 && *p == '.') return 1;
    bool neg = false;
    if (p < e && (*p == '-' || *p == '+')) neg = *p++ == '-';
    int64_t v;
    if (!parse_uint(p, e, 2147483647LL, &v)) return 2;
    *out = (int32_t)(neg ? -v : v);
    return 0;
}

__host__ __device__ __forceinline__ double pow10_exact(int k) {     // 10^k for 0 <= k <= 22, exact in double
    double r = 1.0;
    for (int i = 0; i < k; ++i) r *= 10.0;
    return r;
}

// a float [p, e) on the exact fast path: at most max_digits significant digits (<= 15, so the mantissa is exact in a
// double) and a power of ten of magnitude <= 22 (exact in a double); then m * 10^k or m / 10^-k is the correctly rounded
// double, and the cast to float is what strtod-then-cast gives.  0 ok, 1 missing ('.'), 3 not on the fast path.
__host__ __device__ __forceinline__ int parse_float_fast(const uint8_t* p, const uint8_t* e, int max_digits, float* out) {
    if (e - p == 1 && *p == '.') return 1;
    bool neg = false;
    if (p < e && (*p == '-' || *p == '+')) neg = *p++ == '-';
    int64_t m = 0;
    int nd = 0, ex = 0;
    bool any = false, dot = false;
    for (; p < e; ++p) {
        const uint8_t c = *p;
        if (c >= '0' && c <= '9') {
            any = true;
            if (m == 0 && c == '0') {
                if (dot) --ex;
                continue;                                // leading zeros are not significant
            }
            if (++nd > max_digits) return 3;
            m = m * 10 + (c - '0');
            if (dot) --ex;
        } else if (c == '.' && !dot) {
            dot = true;
        } else {
            break;
        }
    }
    if (!any) return 3;
    if (p < e) {
        if (*p != 'e' && *p != 'E') return 3;
        ++p;
        bool eneg = false;
        if (p < e && (*p == '-' || *p == '+')) eneg = *p++ == '-';
        int64_t x;
        if (!parse_uint(p, e, 1000, &x)) return 3;
        ex += eneg ? -(int)x : (int)x;
    }
    if (ex > 22 || ex < -22) {
        if (m != 0) return 3;
        ex = 0;
    }
    double d = (double)m;
    d = ex >= 0 ? d * pow10_exact(ex) : d / pow10_exact(-ex);
    *out = (float)(neg ? -d : d);
    return 0;
}

// the genotype fields of one sample column [p, e) into cell c
__host__ __device__ __noinline__ void decode_sample(const uint8_t* p, const uint8_t* e, const UnfzVcfRec& r, int gq_float,
                                       int max_digits, int32_t cell_base, int64_t c, uint8_t* gt, float* gq, int32_t* rd,
                                       int32_t* ad, uint8_t* status) {
    // the ranges of the five sub-fields (a dropped trailing sub-field is absent)
    const uint8_t* fs[5];
    const uint8_t* fe[5];
    for (int k = 0; k < 5; ++k) fs[k] = fe[k] = nullptr;
    int k = 0;
    const uint8_t* q = p;
    for (;;) {
        const uint8_t* t = q;
        while (t < e && *t != ':') ++t;
        for (int j = 0; j < 5; ++j)
            if (r.slot[j] == k) { fs[j] = q; fe[j] = t; }
        ++k;
        if (t >= e) break;
        q = t + 1;
    }
    bool bad = false;
    uint8_t st = 0;
    int g = 2;
    if (fs[0]) g = decode_gt(fs[0], fe[0], &bad);
    float qv = -1.0f;
    if (fs[1]) {
        if (gq_float) {
            const int rc = parse_float_fast(fs[1], fe[1], max_digits, &qv);
            if (rc == 1) qv = -1.0f;
            else if (rc == 3) {
                st |= UNFZ_VCF_CELL_HOST;                  // the host re-decodes it: gq holds the value's line offset
                int32_t off = (int32_t)(cell_base + (fs[1] - p));
                memcpy(&qv, &off, 4);
            }
        } else {
            int32_t v;
            const int rc = parse_int32(fs[1], fe[1], &v);
            if (rc == 2) bad = true;
            qv = rc == 0 ? (float)v : -1.0f;
        }
    }
    int32_t ref = -1, alt = -1;
    const int ri = r.slot[2] >= 0 ? 2 : 3;               // AD, or RO / AO without AD
    if (fs[ri]) {
        const uint8_t* t = fs[ri];
        while (t < fe[ri] && *t != ',') ++t;
        int32_t v;
        const int rc = parse_int32(fs[ri], t, &v);
        if (rc == 2) bad = true;
        else if (rc == 0) ref = v;
        if (ri == 2) {
            // alt = the sum of AD[1:]; -1 when an entry is missing or there is only one value
            if (t < fe[2]) {
                int64_t sum = 0;
                bool miss = false;
                while (t < fe[2]) {
                    const uint8_t* u = t + 1;
                    const uint8_t* w = u;
                    while (w < fe[2] && *w != ',') ++w;
                    const int rc2 = parse_int32(u, w, &v);
                    if (rc2 == 2) bad = true;
                    else if (rc2 == 1) miss = true;
                    else sum += v;
                    t = w;
                }
                if (sum > 2147483647LL || sum < -2147483647LL) bad = true;
                alt = miss ? -1 : (int32_t)sum;
            }
        }
    }
    if (ri == 3 && fs[4]) {
        int64_t sum = 0;
        bool miss = false;
        const uint8_t* t = fs[4];
        for (;;) {
            const uint8_t* w = t;
            while (w < fe[4] && *w != ',') ++w;
            int32_t v;
            const int rc = parse_int32(t, w, &v);
            if (rc == 2) bad = true;
            else if (rc == 1) miss = true;
            else sum += v;
            if (w >= fe[4]) break;
            t = w + 1;
        }
        if (sum > 2147483647LL || sum < -2147483647LL) bad = true;
        alt = miss ? -1 : (int32_t)sum;
    }
    if (bad) st |= UNFZ_VCF_CELL_BAD;
    gt[c] = (uint8_t)g;
    gq[c] = qv;
    rd[c] = ref;
    ad[c] = alt;
    status[c] = st;
}

struct SampleArgs {
    const uint8_t* buf;
    const UnfzVcfRec* recs;
    const int64_t* sel;
    int64_t n_sel;
    const int32_t* slot_of;
    int32_t n_samples, n_members, gq_float, max_digits;
    uint8_t* gt;
    float* gq;
    int32_t* rd;
    int32_t* ad;
    uint8_t* status;
    uint8_t* line_bad;
};

__host__ __device__ __forceinline__ void init_cells(const SampleArgs& A, int64_t i, int lane, int step) {
    for (int m = lane; m < A.n_members; m += step) {
        const int64_t c = i * A.n_members + m;
        A.gt[c] = 2;
        A.gq[c] = -1.0f;
        A.rd[c] = -1;
        A.ad[c] = -1;
        A.status[c] = 0;
    }
}

// one warp per selected line: 32 lanes x 16 bytes per step; a lane's tab count and the warp's exclusive scan of the
// counts give the column of every tab, and the lane that owns a tab starting a wanted column decodes that column
__global__ void __launch_bounds__(256) vcf_samples_kernel(SampleArgs A) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= A.n_sel) return;
    init_cells(A, i, lane, 32);
    __syncwarp();
    const UnfzVcfRec r = A.recs[A.sel[i]];
    if (r.fmt_off < 0 || r.fmt_off + r.fmt_len >= r.line_len) {
        if (lane == 0) A.line_bad[i] = 0;
        return;
    }
    const uint8_t* L = A.buf + r.line_off;
    const int64_t s0 = r.fmt_off + r.fmt_len + 1;        // first sample column
    const int64_t n = r.line_len;
    bool bad = false;
    // sample 0 starts at s0
    if (lane == 0) {
        if (A.n_samples == 0) {
            bad = true;
        } else if (A.slot_of[0] >= 0) {
            int64_t e = s0;
            while (e < n && L[e] != '\t') ++e;
            decode_sample(L + s0, L + e, r, A.gq_float, A.max_digits, (int32_t)s0, i * A.n_members + A.slot_of[0],
                          A.gt, A.gq, A.rd, A.ad, A.status);
        }
    }
    int64_t col = 0;                                     // tabs seen before this step
    // 16-byte aligned loads (the text buffer is 16-byte aligned and padded by 16 bytes): the first step starts at the
    // boundary at or below s0, and bytes outside [s0, n) are masked
    int64_t a = ((r.line_off + s0) & ~(int64_t)15) - r.line_off;
    for (; a < n; a += 32 * 16) {
        const int64_t b = a + 16 * lane;
        uint8_t w[16];
        if (b < n) {
            const int4 v = *reinterpret_cast<const int4*>(L + b);
            memcpy(w, &v, 16);
        } else {
            memset(w, 0, 16);
        }
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (b + k < s0 || b + k >= n) w[k] = 0;
        int cnt = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) cnt += w[k] == '\t';
        int incl = cnt;
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        int64_t c = col + incl - cnt;
        for (int k = 0; k < 16 && cnt; ++k) {
            if (w[k] != '\t') continue;
            ++c;                                         // the column starting after this tab
            --cnt;
            if (c >= A.n_samples) { bad = true; continue; }
            const int32_t m = A.slot_of[c];
            if (m < 0) continue;
            const int64_t fs = b + k + 1;
            int64_t e = fs;
            while (e < n && L[e] != '\t') ++e;
            decode_sample(L + fs, L + e, r, A.gq_float, A.max_digits, (int32_t)fs, i * A.n_members + m, A.gt, A.gq,
                          A.rd, A.ad, A.status);
        }
        col += total;
    }
    const bool any_bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) A.line_bad[i] = any_bad ? 1 : 0;
}

// the same decode, one line after the other on the host
void samples_host(const SampleArgs& A) {
    for (int64_t i = 0; i < A.n_sel; ++i) {
        init_cells(A, i, 0, 1);
        A.line_bad[i] = 0;
        const UnfzVcfRec& r = A.recs[A.sel[i]];
        if (r.fmt_off < 0 || r.fmt_off + r.fmt_len >= r.line_len) continue;
        const uint8_t* L = A.buf + r.line_off;
        const int64_t n = r.line_len;
        int64_t s = r.fmt_off + r.fmt_len + 1;
        for (int64_t c = 0;; ++c) {
            int64_t e = s;
            while (e < n && L[e] != '\t') ++e;
            if (c >= A.n_samples) {
                A.line_bad[i] = 1;
                break;
            }
            const int32_t m = A.slot_of[c];
            if (m >= 0)
                decode_sample(L + s, L + e, r, A.gq_float, A.max_digits, (int32_t)s, i * A.n_members + m, A.gt, A.gq,
                              A.rd, A.ad, A.status);
            if (e >= n) break;
            s = e + 1;
        }
    }
}

__global__ void __launch_bounds__(256) vcf_nl_count_kernel(const uint8_t* __restrict__ buf, int64_t n,
                                                            uint32_t* __restrict__ cnt) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c * VCF_CHUNK >= n) return;
    if ((c + 1) * VCF_CHUNK <= n) {
        const int4 v = *reinterpret_cast<const int4*>(buf + c * VCF_CHUNK);
        const uint32_t x[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
        int k = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t t = x[j] ^ 0x0A0A0A0Au;         // zero bytes of t are the newlines
            k += __popc(~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t | 0x7F7F7F7Fu));
        }
        cnt[c] = (uint32_t)k;
    } else {
        cnt[c] = (uint32_t)nl_count16(buf, n, c);
    }
}

__global__ void __launch_bounds__(256) vcf_nl_write_kernel(const uint8_t* __restrict__ buf, int64_t n,
                                                            const uint32_t* __restrict__ at, int64_t* __restrict__ ends) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c * VCF_CHUNK >= n) return;
    if (at[c + 1] != at[c]) nl_write16(buf, n, c, (int64_t)at[c], ends);
}

__global__ void __launch_bounds__(256) vcf_parse_kernel(const uint8_t* __restrict__ buf, const int64_t* __restrict__ ends,
                                                         int64_t n_lines, UnfzVcfRec* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lines) return;
    parse_vcf_line(buf, i ? ends[i - 1] + 1 : 0, ends[i], out + i);
}

}  // namespace

extern "C" int64_t unfz_vcf_line_ends_host(const uint8_t* buf, int64_t n_bytes, int64_t cap, int64_t* ends) {
    int64_t at = 0;
    for (int64_t c = 0; c * VCF_CHUNK < n_bytes; ++c) {
        const int k = nl_count16(buf, n_bytes, c);
        if (at + k > cap) return -1;
        nl_write16(buf, n_bytes, c, at, ends);
        at += k;
    }
    return at;
}

extern "C" int64_t unfz_vcf_parse_host(const uint8_t* buf, const int64_t* ends, int64_t n_lines, UnfzVcfRec* out) {
    int64_t bad = 0;
    for (int64_t i = 0; i < n_lines; ++i) {
        parse_vcf_line(buf, i ? ends[i - 1] + 1 : 0, ends[i], out + i);
        bad += (out[i].flags & UNFZ_VCF_BAD) != 0;
    }
    return bad;
}

extern "C" int unfz_vcf_samples_host(const uint8_t* buf, const UnfzVcfRec* recs, const int64_t* sel, int64_t n_sel,
                                     const int32_t* slot_of, int32_t n_samples, int32_t n_members, int32_t gq_float,
                                     int32_t max_digits, uint8_t* gt, float* gq, int32_t* rd, int32_t* ad, uint8_t* status,
                                     uint8_t* line_bad) {
    SampleArgs A{buf, recs, sel, n_sel, slot_of, n_samples, n_members, gq_float, max_digits < 15 ? max_digits : 15,
                 gt, gq, rd, ad, status, line_bad};
    samples_host(A);
    return 0;
}

extern "C" int64_t unfz_vcf_chunks(int64_t n_bytes) { return (n_bytes + VCF_CHUNK - 1) / VCF_CHUNK; }

extern "C" int unfz_vcf_line_count(UnfzCtx* ctx, const uint8_t* buf, int64_t n_bytes, uint32_t* cnt, void* stream) {
    const int64_t chunks = (n_bytes + VCF_CHUNK - 1) / VCF_CHUNK;
    if (chunks <= 0) return 0;
    vcf_nl_count_kernel<<<(unsigned)((chunks + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, n_bytes, cnt);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_vcf_line_write(UnfzCtx* ctx, const uint8_t* buf, int64_t n_bytes, const uint32_t* at, int64_t* ends,
                                   void* stream) {
    const int64_t chunks = (n_bytes + VCF_CHUNK - 1) / VCF_CHUNK;
    if (chunks <= 0) return 0;
    vcf_nl_write_kernel<<<(unsigned)((chunks + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, n_bytes, at, ends);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_vcf_parse(UnfzCtx* ctx, const uint8_t* buf, const int64_t* ends, int64_t n_lines, UnfzVcfRec* out,
                              void* stream) {
    if (n_lines <= 0) return 0;
    vcf_parse_kernel<<<(unsigned)((n_lines + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, ends, n_lines, out);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_vcf_samples(UnfzCtx* ctx, const uint8_t* buf, const UnfzVcfRec* recs, const int64_t* sel, int64_t n_sel,
                                const int32_t* slot_of, int32_t n_samples, int32_t n_members, int32_t gq_float,
                                int32_t max_digits, uint8_t* gt, float* gq, int32_t* rd, int32_t* ad, uint8_t* status,
                                uint8_t* line_bad, void* stream) {
    if (n_sel <= 0) return 0;
    SampleArgs A{buf, recs, sel, n_sel, slot_of, n_samples, n_members, gq_float, max_digits < 15 ? max_digits : 15,
                 gt, gq, rd, ad, status, line_bad};
    const int64_t threads = n_sel * 32;
    vcf_samples_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
