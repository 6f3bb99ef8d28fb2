// BAM record decoding: the inflated record bytes of a region query -> the device read columns (UnfzReadCols).
//
// The host inflates the BGZF blocks (bamio.py) and finds the record boundaries (unfz_bam_record_offsets: block_size is
// a sequential chain, so that walk stays on the host).  unfz_bam_parse reads the fixed fields of every record -- 48 B
// out per record -- from which the host takes the selection (overlap, duplicates between intervals, lone mates, order
// by start) and builds the 32-byte headers.  The bulk of a record -- CIGAR, bases, qualities -- never leaves the device:
// unfz_bam_emit_cigar and unfz_bam_emit_planes write the CIGAR words, 2-bit bases, low-quality plane and non-ACGT
// plane in the layout DeviceReads holds after an upload.
#include "common.cuh"

namespace {

// little-endian loads at any alignment (records are packed back to back)
__host__ __device__ __forceinline__ uint32_t ld_u32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__host__ __device__ __forceinline__ uint16_t ld_u16(const uint8_t* p) { return (uint16_t)(p[0] | (p[1] << 8)); }

// htslib's bam_cigar_type: bit1 consumes the reference (M D N = X)
__host__ __device__ __forceinline__ bool cigar_consumes_ref(uint32_t op) {
    return op == 0u || op == 2u || op == 3u || op == 7u || op == 8u;
}

// bytes of one aux value after its 3-byte tag+type, or -1 when the field is malformed / runs past `end`
__host__ __device__ __forceinline__ int64_t aux_value_bytes(const uint8_t* p, const uint8_t* end, uint8_t type) {
    switch (type) {
        case 'A': case 'c': case 'C': return 1;
        case 's': case 'S': return 2;
        case 'i': case 'I': case 'f': return 4;
        case 'Z': case 'H': {
            const uint8_t* q = p;
            while (q < end && *q) ++q;
            return q < end ? (int64_t)(q - p) + 1 : -1;
        }
        case 'B': {
            if (end - p < 5) return -1;
            const uint8_t sub = p[0];
            const int64_t cnt = (int64_t)ld_u32(p + 1);
            int64_t sz;
            switch (sub) {
                case 'c': case 'C': sz = 1; break;
                case 's': case 'S': sz = 2; break;
                case 'i': case 'I': case 'f': sz = 4; break;
                default: return -1;
            }
            return 5 + cnt * sz;
        }
        default: return -1;
    }
}

__host__ __device__ __forceinline__ void parse_record(const uint8_t* buf, int64_t n_bytes, int64_t off, UnfzBamRec* out) {
    UnfzBamRec r;
    memset(&r, 0, sizeof(r));
    const uint8_t* p = buf + off;
    const int64_t bs = (off + 36 <= n_bytes) ? (int64_t)(int32_t)ld_u32(p) : -1;
    if (bs < 32 || off + 4 + bs > n_bytes) {
        r.aux = UNFZ_BAM_AUX_BAD;
        *out = r;
        return;
    }
    const uint8_t* end = p + 4 + bs;
    r.ref_id = (int32_t)ld_u32(p + 4);
    r.pos = (int32_t)ld_u32(p + 8);
    r.l_name = p[12];
    r.mapq = p[13];
    r.n_cigar = ld_u16(p + 16);
    r.flag = ld_u16(p + 18);
    r.l_seq = (int32_t)ld_u32(p + 20);
    r.next_ref_id = (int32_t)ld_u32(p + 24);
    r.next_pos = (int32_t)ld_u32(p + 28);
    r.tlen = (int32_t)ld_u32(p + 32);
    const uint8_t* name = p + 36;
    const uint8_t* cig = name + r.l_name;
    const uint8_t* seq = cig + 4 * (int64_t)r.n_cigar;
    const uint8_t* aux = seq + (r.l_seq > 0 ? ((int64_t)r.l_seq + 1) / 2 + r.l_seq : 0);
    uint8_t bits = (r.next_ref_id == r.ref_id) ? 1 : 0;
    if (r.l_seq < 0 || r.l_name == 0 || aux > end) {
        r.aux = UNFZ_BAM_AUX_BAD;
        *out = r;
        return;
    }
    uint64_t h = 1469598103934665603ull;                 // FNV-1a 64
    for (int i = 0; i + 1 < r.l_name; ++i) {
        h ^= name[i];
        h *= 1099511628211ull;
    }
    r.name_hash = h;
    int64_t raw = 0;
    for (int i = 0; i < r.n_cigar; ++i) {
        const uint32_t w = ld_u32(cig + 4 * i);
        if (cigar_consumes_ref(w & 15u)) raw += w >> 4;
    }
    const int64_t rlen = (r.flag & 0x4) ? 0 : raw;
    r.end = (int32_t)(r.pos + (rlen ? rlen : 1));
    r.ref_len = (int32_t)raw;
    // every tag, whatever its type: a tag's size depends on the ones before it
    const uint8_t* q = aux;
    while (q < end) {
        if (end - q < 3) { bits |= UNFZ_BAM_AUX_BAD; break; }
        if (q[0] == 'S' && q[1] == 'A') bits |= 2;
        const int64_t nb = aux_value_bytes(q + 3, end, q[2]);
        if (nb < 0 || nb > end - q - 3) { bits |= UNFZ_BAM_AUX_BAD; break; }
        q += 3 + nb;
    }
    r.aux = bits;
    *out = r;
}

__global__ void __launch_bounds__(256) bam_parse_kernel(const uint8_t* __restrict__ buf, int64_t n_bytes,
                                                         const int64_t* __restrict__ offs, int64_t n,
                                                         UnfzBamRec* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    union { UnfzBamRec r; int4 v[3]; } u;
    parse_record(buf, n_bytes, offs[i], &u.r);
    // 48 bytes out as three 16-byte stores (out is 16-byte aligned: 48 B per record from an aligned base)
    int4* d = reinterpret_cast<int4*>(out + i);
    d[0] = u.v[0];
    d[1] = u.v[1];
    d[2] = u.v[2];
}

// one thread per entry of the (block, name hash) order: the mate of read i = order[s] is the first primary read of
// the other segment in i's group (groups are runs of equal key; a stable sort keeps block order inside a group), as
// packers._mate_join defines it.  The name bytes of the joined pair are compared here; a mismatch (a hash collision) or
// a read that is its own candidate (both segment bits) is left to the host: mate = -2.
__global__ void __launch_bounds__(256) bam_mate_join_kernel(const int64_t* __restrict__ order,
                                                             const int64_t* __restrict__ key_hash,
                                                             const int32_t* __restrict__ key_blk,
                                                             const int32_t* __restrict__ flag, int64_t n,
                                                             const uint8_t* __restrict__ buf, const int64_t* __restrict__ src,
                                                             int32_t* __restrict__ mate) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const int64_t i = order[s];
    const int32_t fl = flag[i];
    if (!(fl & 0x1) || (fl & 0x8)) {
        mate[i] = -1;
        return;
    }
    const int64_t h = key_hash[i];
    const int32_t b = key_blk[i];
    int64_t lo = s;
    while (lo > 0 && key_hash[order[lo - 1]] == h && key_blk[order[lo - 1]] == b) --lo;
    const int want = (fl & 0x40) ? 0x80 : 0x40;
    int64_t cand = -1;
    for (int64_t t = lo; t < n; ++t) {
        const int64_t j = order[t];
        if (key_hash[j] != h || key_blk[j] != b) break;
        const int32_t fj = flag[j];
        if ((fj & want) && !(fj & 0x900)) {
            cand = j;
            break;
        }
    }
    if (cand < 0) {
        mate[i] = -1;
        return;
    }
    if (cand == i) {
        mate[i] = -2;
        return;
    }
    const uint8_t* a = buf + src[i];
    const uint8_t* c = buf + src[cand];
    bool same = a[12] == c[12];
    for (int k = 0; same && k < a[12]; ++k) same = a[36 + k] == c[36 + k];
    mate[i] = same ? (int32_t)cand : -2;
}

__global__ void __launch_bounds__(256) bam_emit_cigar_kernel(const UnfzRead* __restrict__ hdr, int64_t n_reads,
                                                              const uint8_t* __restrict__ buf, const int64_t* __restrict__ src,
                                                              uint32_t* __restrict__ cigar) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_reads) return;
    const UnfzRead h = load_read(hdr + r);
    const uint8_t* c = buf + src[r] + 36 + buf[src[r] + 12];
    uint32_t* o = cigar + h.cigar_off;
    for (int j = 0; j < h.n_cigar; ++j) o[j] = ld_u32(c + 4 * j);
}

// 2-bit code and escape bit of a BAM base nibble (=ACMGRSVTWYHKDBN): A C G T -> 0..3; N -> 0 escaped; any other
// letter, '=' included, -> 1 escaped.  Bits 0-1 code, bit 2 escape.
__constant__ uint8_t c_nib[16] = {5, 0, 1, 5, 2, 5, 5, 5, 3, 5, 5, 5, 5, 5, 5, 4};

// one thread per 32 output bases: one lowq word, one nmask word, two seq2 words
__global__ void __launch_bounds__(256) bam_emit_planes_kernel(UnfzRead* __restrict__ hdr, int64_t n_reads, int64_t n_qual,
                                                               const uint8_t* __restrict__ buf, const int64_t* __restrict__ src,
                                                               int32_t min_bq, uint32_t* __restrict__ lowq,
                                                               uint32_t* __restrict__ nmask, uint2* __restrict__ seq2) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t g0 = w * 32;
    if (g0 >= n_qual) return;
    // the read owning base g0: the last read whose first base is at or before it (empty reads share the next offset)
    int64_t lo = 0, hi = n_reads;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (read_qoff(hdr[mid]) <= g0) lo = mid + 1; else hi = mid;
    }
    int64_t r = lo - 1;
    uint32_t lq = 0, nm = 0, s0 = 0, s1 = 0;
    int64_t q0 = 0, l = 0;
    const uint8_t *seq = nullptr, *qual = nullptr;
    bool miss = false, esc = false;
    int64_t cur = -1;
    // aux is byte 29 of the header: bit7 through a word-wide atomic (the neighbours are mapq, qoff_hi, pad), once per
    // read and thread.  The header is read with plain loads: this kernel writes to it
    auto flush = [&]() {
        if (esc) atomicOr(reinterpret_cast<unsigned*>(hdr + cur) + 7, 0x80u << 8);
        esc = false;
    };
    const int64_t g1 = min(g0 + 32, n_qual);
    for (int64_t g = g0; g < g1; ++g) {
        if (r != cur) {
            flush();
            // (re)load the read's layout; advance past reads that end before g (empty reads)
            for (;;) {
                q0 = read_qoff(hdr[r]);
                l = hdr[r].l_seq;
                if (g < q0 + l) break;
                ++r;
            }
            const int64_t s = src[r];
            seq = buf + s + 36 + buf[s + 12] + 4 * (int64_t)hdr[r].n_cigar;
            qual = seq + (l + 1) / 2;
            miss = qual[0] == 0xFF;
            cur = r;
        }
        const int64_t k = g - q0;
        const uint8_t cb = c_nib[(seq[k >> 1] >> ((k & 1) ? 0 : 4)) & 15];
        const uint8_t qv = miss ? 0 : (qual[k] & 0x7F);
        const int b = (int)(g - g0);
        if (qv < min_bq) lq |= 1u << b;
        if (cb & 4) {
            nm |= 1u << b;
            esc = true;
        }
        if (b < 16) s0 |= (uint32_t)(cb & 3) << (2 * b);
        else s1 |= (uint32_t)(cb & 3) << (2 * (b - 16));
        if (g + 1 == q0 + l) ++r;
    }
    flush();
    lowq[w] = lq;
    nmask[w] = nm;
    seq2[w] = make_uint2(s0, s1);
}

}  // namespace

extern "C" int64_t unfz_bam_record_offsets(const uint8_t* buf, int64_t n_bytes, int64_t max_records, int64_t* offs,
                                           int64_t* end_out) {
    int64_t p = 0, n = 0;
    while (n < max_records && p + 4 <= n_bytes) {
        const int64_t bs = (int64_t)(int32_t)ld_u32(buf + p);
        if (bs < 32) {
            *end_out = p;
            return -1;
        }
        if (p + 4 + bs > n_bytes) break;
        offs[n++] = p;
        p += 4 + bs;
    }
    *end_out = p;
    return n;
}

extern "C" int64_t unfz_bam_parse_host(const uint8_t* buf, int64_t n_bytes, const int64_t* offs, int64_t n, UnfzBamRec* out) {
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        parse_record(buf, n_bytes, offs[i], out + i);
        bad += (out[i].aux & UNFZ_BAM_AUX_BAD) != 0;
    }
    return bad;
}

extern "C" int unfz_bam_gather_host(const uint8_t* buf, const int64_t* src, const int64_t* len, int64_t n, uint8_t* dst) {
    for (int64_t i = 0; i < n; ++i) {
        memcpy(dst, buf + src[i], (size_t)len[i]);
        dst += len[i];
    }
    return 0;
}

extern "C" int unfz_bam_parse(UnfzCtx* ctx, const uint8_t* buf, int64_t n_bytes, const int64_t* offs, int64_t n,
                              UnfzBamRec* out, void* stream) {
    if (n <= 0) return 0;
    bam_parse_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(buf, n_bytes, offs, n, out);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_bam_mate_join(UnfzCtx* ctx, const int64_t* order, const int64_t* key_hash, const int32_t* key_blk,
                                  const int32_t* flag, int64_t n, const uint8_t* buf, const int64_t* src, int32_t* mate,
                                  void* stream) {
    if (n <= 0) return 0;
    bam_mate_join_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(order, key_hash, key_blk, flag, n, buf,
                                                                                        src, mate);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_bam_emit_cigar(UnfzCtx* ctx, const UnfzReadCols* reads, const uint8_t* buf, const int64_t* src,
                                   void* stream) {
    if (reads->n_reads <= 0 || reads->n_cigar <= 0) return 0;
    bam_emit_cigar_kernel<<<(unsigned)((reads->n_reads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reads->hdr, reads->n_reads, buf, src, const_cast<uint32_t*>(reads->cigar));
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_bam_emit_planes(UnfzCtx* ctx, const UnfzReadCols* reads, const uint8_t* buf, const int64_t* src,
                                    int32_t min_bq, void* stream) {
    if (reads->n_reads <= 0 || reads->n_qual <= 0) return 0;
    const int64_t words = (reads->n_qual + 31) / 32;
    bam_emit_planes_kernel<<<(unsigned)((words + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        const_cast<UnfzRead*>(reads->hdr), reads->n_reads, reads->n_qual, buf, src, min_bq,
        const_cast<uint32_t*>(reads->lowq), const_cast<uint32_t*>(reads->nmask),
        reinterpret_cast<uint2*>(const_cast<uint8_t*>(reads->seq2)));
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
