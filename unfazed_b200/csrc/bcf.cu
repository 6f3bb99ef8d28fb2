// BCF 2.2 decoding: the inflated records of a CSI region query -> record boundaries, fixed fields per record, and the
// genotype fields of the wanted samples of the selected records.
//
// The host inflates the BGZF blocks and parses the CSI (bcfio.py).  Three steps:
//   record boundaries -- l_shared + l_indiv is a sequential chain, so the walk stays on the host
//                        (unfz_bcf_record_offsets, like unfz_bam_record_offsets);
//   fixed fields      -- one thread per record: CHROM, POS, rlen, REF / first ALT, and the value block (offset, type,
//                        per-sample count) of GT / GQ / AD / RO / AO, the other typed values skipped by type and count
//                        (UnfzBcfRec);
//   sample fields     -- one thread per (selected record x member) cell: BCF stores a FORMAT field of all samples at a
//                        fixed stride, so a member's values are a direct load at field + sample * count * width.
// The last two are one __host__ __device__ body each, with a host entry point (engine-less loads, CPU tests) and a
// device entry point.
#include "bcf.cuh"

namespace {

struct Keys {
    int32_t k[5];                                        // string-dictionary index of GT GQ AD RO AO, -1: not declared
};

// a whole typed value: its header, then its count * width bytes
__host__ __device__ __forceinline__ bool skip_typed(const uint8_t* b, int64_t& p, int64_t e, uint8_t* why) {
    int t;
    int64_t n;
    if (!typed_hdr(b, p, e, &t, &n, why)) return false;
    p += n * type_width(t);
    if (p > e) { *why |= UNFZ_BCF_BAD_OVERRUN; return false; }
    return true;
}

// a typed integer of count 1 (a dictionary key)
__host__ __device__ __forceinline__ bool typed_key(const uint8_t* b, int64_t& p, int64_t e, int32_t* key, uint8_t* why) {
    int t;
    int64_t n;
    if (!typed_hdr(b, p, e, &t, &n, why)) return false;
    if (!is_int_type(t) || n != 1) { *why |= UNFZ_BCF_BAD_TYPE; return false; }
    if (p + type_width(t) > e) { *why |= UNFZ_BCF_BAD_OVERRUN; return false; }
    ld_int(b + p, t, key);
    p += type_width(t);
    return true;
}

// record at byte off: l_shared, l_indiv, the shared block, the individual block (bounds checked by the offsets walk)
__host__ __device__ void parse_bcf_record(const uint8_t* b, int64_t off, const Keys& keys, int32_t n_samples,
                                          UnfzBcfRec* out) {
    UnfzBcfRec r;
    memset(&r, 0, sizeof(r));
    r.rec_off = off;
    for (int k = 0; k < 5; ++k) r.fmt_off[k] = -1;
    uint8_t why = 0;
    const int64_t l_shared = ld_u32(b + off), l_indiv = ld_u32(b + off + 4);
    const int64_t s = off + 8, se = s + l_shared, ie = se + l_indiv;
    if (l_shared < 24) {
        r.flags = UNFZ_BCF_BAD | UNFZ_BCF_BAD_OVERRUN;
        *out = r;
        return;
    }
    r.contig = (int32_t)ld_u32(b + s);
    const int64_t pos = (int32_t)ld_u32(b + s + 4), rlen = (int32_t)ld_u32(b + s + 8);
    const uint32_t allele_info = ld_u32(b + s + 16), fmt_sample = ld_u32(b + s + 20);
    const int n_allele = (int)(allele_info >> 16), n_info = (int)(allele_info & 0xFFFF);
    const int n_fmt = (int)(fmt_sample >> 24);
    const int32_t n_sample = (int32_t)(fmt_sample & 0xFFFFFF);
    r.n_allele = (uint16_t)n_allele;
    if (pos < 0 || rlen < 0 || pos + rlen > 2147483647LL) why |= UNFZ_BCF_BAD_POS;
    r.pos0 = (int32_t)pos;
    r.rend = (int32_t)(pos + rlen < 2147483647LL ? pos + rlen : 2147483647LL);
    if (n_sample != n_samples) why |= UNFZ_BCF_BAD_SAMPLES;
    int64_t p = s + 24;
    bool ok = skip_typed(b, p, se, &why);                // ID
    for (int a = 0; ok && a < n_allele; ++a) {           // REF, ALT...
        int t;
        int64_t n;
        ok = typed_hdr(b, p, se, &t, &n, &why);
        if (!ok) break;
        if (t != BT_CHAR && !(t == BT_NULL && n == 0)) { why |= UNFZ_BCF_BAD_TYPE; ok = false; break; }
        if (p + n > se) { why |= UNFZ_BCF_BAD_OVERRUN; ok = false; break; }
        int64_t len = n;
        while (len > 0 && b[p + len - 1] == 0) --len;     // NUL padding
        if (a == 0) {
            r.ref_off = (int32_t)(p - off);
            r.ref_len = (int32_t)len;
            r.ref0 = len > 0 ? b[p] : 0;
        } else if (a == 1) {
            r.alt_off = (int32_t)(p - off);
            r.alt_len = (int32_t)len;
        }
        p += n;
    }
    if (ok) ok = skip_typed(b, p, se, &why);             // FILTER
    for (int k = 0; ok && k < n_info; ++k) {             // INFO: key, value
        int32_t key;
        ok = typed_key(b, p, se, &key, &why) && skip_typed(b, p, se, &why);
    }
    p = se;
    for (int k = 0; ok && k < n_fmt; ++k) {              // FORMAT: key, then n_sample * count values of one type
        int32_t key;
        int t;
        int64_t n;
        ok = typed_key(b, p, ie, &key, &why) && typed_hdr(b, p, ie, &t, &n, &why);
        if (!ok) break;
        if (n >= (1 << 27)) { why |= UNFZ_BCF_BAD_OVERRUN; ok = false; break; }
        const int64_t bytes = (int64_t)n_sample * n * type_width(t);
        if (p + bytes > ie) { why |= UNFZ_BCF_BAD_OVERRUN; ok = false; break; }
        for (int j = 0; j < 5; ++j)
            if (key == keys.k[j] && keys.k[j] >= 0) {
                r.fmt_off[j] = (int32_t)(p - off);
                r.fmt_ct[j] = ((uint32_t)n << 4) | (uint32_t)t;
            }
        p += bytes;
    }
    if (n_allele == 2 && r.ref_len == 1 && r.alt_len == 1 && b[off + r.alt_off] != '*') r.flags |= UNFZ_BCF_SIMPLE;
    if (why) r.flags |= UNFZ_BCF_BAD | why;
    *out = r;
}

// one GT allele value: -2 end of vector, -1 missing, else the allele index
__host__ __device__ __forceinline__ int gt_allele(const uint8_t* p, int t, bool* bad) {
    int32_t v;
    const int k = ld_int(p, t, &v);
    if (k == 2) return -2;
    if (k == 1) return -1;
    if (k == 3 || v < 0) { *bad = true; return -1; }
    return (v >> 1) == 0 ? -1 : (v >> 1) - 1;
}

// the genotype fields of sample s of record r into cell c (the text decoder's contract, vcf.cu decode_sample)
__host__ __device__ __forceinline__ void decode_cell(const uint8_t* buf, const UnfzBcfRec& r, int64_t s, int64_t c,
                                                     uint8_t* gt, float* gq, int32_t* rd, int32_t* ad, uint8_t* status) {
    const uint8_t* R = buf + r.rec_off;
    bool bad = false;
    const uint8_t* v[5];
    int type[5], cnt[5], w[5];
    for (int j = 0; j < 5; ++j) {
        cnt[j] = r.fmt_off[j] >= 0 ? (int)(r.fmt_ct[j] >> 4) : 0;
        type[j] = (int)(r.fmt_ct[j] & 15);
        w[j] = type_width(type[j]);
        if (cnt[j] == 0 || w[j] == 0) {
            cnt[j] = 0;                                  // absent for this record
            v[j] = nullptr;
            continue;
        }
        v[j] = R + r.fmt_off[j] + s * cnt[j] * w[j];
        const bool want_int = j != 1;                    // GQ may be a float
        if (!(is_int_type(type[j]) || (!want_int && type[j] == BT_FLOAT))) {
            bad = true;
            cnt[j] = 0;
        }
    }
    // GT: the first two alleles, as decode_gt reads them from text
    int g = 2;
    if (cnt[0]) {
        const int a = gt_allele(v[0], type[0], &bad);
        const int b = cnt[0] > 1 ? gt_allele(v[0] + w[0], type[0], &bad) : -2;
        if (a == -2) {
            g = 2;
        } else if (b == -2) {                            // haploid
            g = a < 0 ? 2 : (a == 0 ? 0 : (a == 1 ? 3 : 2));
        } else if (a < 0 && b < 0) {
            g = 2;
        } else if (a < 0 || b < 0) {
            g = (a < 0 ? b : a) == 0 ? 2 : 1;
        } else {
            g = a != b ? 1 : (a == 0 ? 0 : 3);
        }
    }
    float q = -1.0f;
    if (cnt[1]) {
        if (type[1] == BT_FLOAT) {
            const uint32_t x = ld_u32(v[1]);
            if (x != FLOAT_MISSING && x != FLOAT_EOV) memcpy(&q, &x, 4);
        } else {
            int32_t x;
            const int k = ld_int(v[1], type[1], &x);
            if (k == 3) bad = true;
            else if (k == 0) q = (float)x;
        }
    }
    int32_t ref = -1, alt = -1;
    const int ri = r.fmt_off[2] >= 0 ? 2 : 3;            // AD, or RO / AO without AD
    if (cnt[ri]) {
        int32_t x;
        const int k = ld_int(v[ri], type[ri], &x);
        if (k == 3) bad = true;
        else if (k == 0) ref = x;
        if (ri == 2 && k != 2) {
            // alt = the sum of AD[1:] up to the end of the vector; -1 when an entry is missing or there is one value
            int64_t sum = 0;
            int n = 0;
            bool miss = false;
            for (int j = 1; j < cnt[2]; ++j) {
                const int kj = ld_int(v[2] + j * w[2], type[2], &x);
                if (kj == 2) break;
                ++n;
                if (kj == 3) bad = true;
                else if (kj == 1) miss = true;
                else sum += x;
            }
            if (sum > 2147483647LL || sum < -2147483647LL) bad = true;
            if (n) alt = miss ? -1 : (int32_t)sum;
        }
    }
    if (ri == 3 && cnt[4]) {
        int64_t sum = 0;
        int n = 0;
        bool miss = false;
        for (int j = 0; j < cnt[4]; ++j) {
            int32_t x;
            const int kj = ld_int(v[4] + j * w[4], type[4], &x);
            if (kj == 2) break;
            ++n;
            if (kj == 3) bad = true;
            else if (kj == 1) miss = true;
            else sum += x;
        }
        if (sum > 2147483647LL || sum < -2147483647LL) bad = true;
        if (n) alt = miss ? -1 : (int32_t)sum;
    }
    gt[c] = (uint8_t)g;
    gq[c] = q;
    rd[c] = ref;
    ad[c] = alt;
    status[c] = bad ? UNFZ_BCF_CELL_BAD : 0;
}

struct SampleArgs {
    const uint8_t* buf;
    const UnfzBcfRec* recs;
    const int64_t* sel;
    int64_t n_sel;
    const int32_t* member_sample;
    int32_t n_members;
    uint8_t* gt;
    float* gq;
    int32_t* rd;
    int32_t* ad;
    uint8_t* status;
};

__host__ __device__ __forceinline__ void sample_cell(const SampleArgs& A, int64_t c) {
    const int64_t i = c / A.n_members;
    const UnfzBcfRec& r = A.recs[A.sel[i]];
    decode_cell(A.buf, r, A.member_sample[c - i * A.n_members], c, A.gt, A.gq, A.rd, A.ad, A.status);
}

__global__ void __launch_bounds__(256) bcf_parse_kernel(const uint8_t* __restrict__ buf, const int64_t* __restrict__ offs,
                                                         int64_t n, Keys keys, int32_t n_samples,
                                                         UnfzBcfRec* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    parse_bcf_record(buf, offs[i], keys, n_samples, out + i);
}

__global__ void __launch_bounds__(256) bcf_samples_kernel(SampleArgs A, int64_t cells) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    sample_cell(A, c);
}

Keys make_keys(const int32_t* k) {
    Keys K;
    for (int j = 0; j < 5; ++j) K.k[j] = k[j];
    return K;
}

}  // namespace

extern "C" int64_t unfz_bcf_record_offsets(const uint8_t* buf, int64_t n_bytes, int64_t max_records, int64_t* offs,
                                           int64_t* end_out) {
    int64_t p = 0, n = 0;
    while (n < max_records && p + 8 <= n_bytes) {
        const int64_t l_shared = ld_u32(buf + p), l_indiv = ld_u32(buf + p + 4);
        if (l_shared < 24) {
            *end_out = p;
            return -1;
        }
        if (p + 8 + l_shared + l_indiv > n_bytes) break;
        offs[n++] = p;
        p += 8 + l_shared + l_indiv;
    }
    *end_out = p;
    return n;
}

extern "C" int64_t unfz_bcf_parse_host(const uint8_t* buf, const int64_t* offs, int64_t n, const int32_t* keys,
                                       int32_t n_samples, UnfzBcfRec* out) {
    const Keys K = make_keys(keys);
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        parse_bcf_record(buf, offs[i], K, n_samples, out + i);
        bad += (out[i].flags & UNFZ_BCF_BAD) != 0;
    }
    return bad;
}

extern "C" int unfz_bcf_samples_host(const uint8_t* buf, const UnfzBcfRec* recs, const int64_t* sel, int64_t n_sel,
                                     const int32_t* member_sample, int32_t n_members, uint8_t* gt, float* gq, int32_t* rd,
                                     int32_t* ad, uint8_t* status) {
    const SampleArgs A{buf, recs, sel, n_sel, member_sample, n_members, gt, gq, rd, ad, status};
    const int64_t cells = n_sel * (int64_t)n_members;
    for (int64_t c = 0; c < cells; ++c) sample_cell(A, c);
    return 0;
}

extern "C" int unfz_bcf_parse(UnfzCtx* ctx, const uint8_t* buf, const int64_t* offs, int64_t n, const int32_t* keys,
                              int32_t n_samples, UnfzBcfRec* out, void* stream) {
    if (n <= 0) return 0;
    bcf_parse_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, offs, n, make_keys(keys),
                                                                                     n_samples, out);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_bcf_samples(UnfzCtx* ctx, const uint8_t* buf, const UnfzBcfRec* recs, const int64_t* sel, int64_t n_sel,
                                const int32_t* member_sample, int32_t n_members, uint8_t* gt, float* gq, int32_t* rd,
                                int32_t* ad, uint8_t* status, void* stream) {
    const int64_t cells = n_sel * (int64_t)n_members;
    if (cells <= 0) return 0;
    const SampleArgs A{buf, recs, sel, n_sel, member_sample, n_members, gt, gq, rd, ad, status};
    bcf_samples_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A, cells);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
