// CRAM 3.0 slice decoding: the decompressed blocks of the selected slices -> BAM records (block_size ... aux), the
// bytes bam.cu and bamio.read_regions already consume.
//
// The host (cramio.py) parses the containers, checks the CRC32 of every header and block, decompresses the blocks
// (gzip / bzip2 / lzma through the standard library, rANS 4x8 through unfz_rans4x8_decode_host below) and flattens each
// slice into an UnfzCramSlice: the core block, the external blocks in slice order, a small int32 program holding the
// compression header's encodings (content ids already resolved to the slice's block index) and the tag dictionary, and
// the reference spans the slice may read.  Records of a slice are a sequential chain through the core bit stream and
// the external cursors, so one thread decodes one slice: the size step returns the BAM bytes and CIGAR length of every
// record, unfz_exclusive_scan_i64 turns the bytes into offsets, and the write step decodes again into place and then
// runs the in-slice mate fix-up of attached (NF) mates.  Both steps are one __host__ __device__ body; the host entry
// points run it slice by slice for engine-less loads.
#include "common.cuh"

namespace {

enum { S_BF, S_CF, S_RI, S_RL, S_AP, S_RG, S_RN, S_MF, S_NS, S_NP, S_TS, S_NF, S_TL, S_FN, S_FC, S_FP, S_DL, S_BB,
       S_QQ, S_BS, S_IN, S_RS, S_PD, S_HC, S_SC, S_MQ, S_BA, S_QS };

enum { E_NULL = 0, E_EXTERNAL = 1, E_HUFFMAN = 3, E_BYTE_ARRAY_LEN = 4, E_BYTE_ARRAY_STOP = 5, E_BETA = 6, E_SUBEXP = 7,
       E_GAMMA = 9 };

#define CRAM_ATTACHED (-3)       // scratch marker in next_ref_id during the write step: next_pos holds the mate line

__host__ __device__ __forceinline__ uint32_t ld32(const uint8_t* p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
__host__ __device__ __forceinline__ void st32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24);
}
__host__ __device__ __forceinline__ void st16(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }

// BAM nibble of a base letter (htslib's seq_nt16_table; anything else is N)
__host__ __device__ __forceinline__ uint8_t nt16(uint8_t c) {
    switch (c | 0x20) {
        case '=' | 0x20: return c == '=' ? 0 : 15;
        case 'a': return 1; case 'c': return 2; case 'm': return 3; case 'g': return 4; case 'r': return 5;
        case 's': return 6; case 'v': return 7; case 't': return 8; case 'w': return 9; case 'y': return 10;
        case 'h': return 11; case 'k': return 12; case 'd': return 13; case 'b': return 14;
        default: return 15;
    }
}
__host__ __device__ __forceinline__ int base5(uint8_t c) {
    switch (c) { case 'A': return 0; case 'C': return 1; case 'G': return 2; case 'T': return 3; default: return 4; }
}
__host__ __device__ __forceinline__ uint8_t upper(uint8_t c) { return (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c; }

// htslib's reg2bin for a BAI-style binning (min_shift 14, depth 5)
__host__ __device__ __forceinline__ uint32_t reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (uint32_t)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (uint32_t)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (uint32_t)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (uint32_t)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (uint32_t)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

// One slice's decoder state: the core bit reader, one cursor per external block, the program.
struct Dec {
    const uint8_t* blocks;
    const uint8_t* core;
    int64_t core_len, bitpos;
    const UnfzCramExt* ext;
    int32_t n_ext;
    const int32_t* P;
    int32_t err;
    int64_t cur[UNFZ_CRAM_MAX_EXT];

    __host__ __device__ __forceinline__ void fail(int e) { if (!err) err = e; }

    __host__ __device__ __forceinline__ int bit() {
        if (bitpos >= core_len * 8) { fail(UNFZ_CRAM_OVERRUN); return 0; }
        const int b = (core[bitpos >> 3] >> (7 - (bitpos & 7))) & 1;
        ++bitpos;
        return b;
    }
    __host__ __device__ __forceinline__ uint32_t bits(int n) {
        uint32_t v = 0;
        for (int i = 0; i < n; ++i) v = (v << 1) | (uint32_t)bit();
        return v;
    }
    __host__ __device__ __forceinline__ int ext_byte(int e) {
        if (e < 0 || e >= n_ext) { fail(UNFZ_CRAM_BAD_ENCODING); return -1; }
        if (cur[e] >= ext[e].len) { fail(UNFZ_CRAM_OVERRUN); return -1; }
        return blocks[ext[e].off + cur[e]++];
    }
    __host__ __device__ __forceinline__ int32_t ext_itf8(int e) {
        const int b0 = ext_byte(e);
        if (b0 < 0) return 0;
        if (b0 < 0x80) return b0;
        if (b0 < 0xC0) return ((b0 & 0x3F) << 8) | ext_byte(e);
        if (b0 < 0xE0) { const int b1 = ext_byte(e); return ((b0 & 0x1F) << 16) | (b1 << 8) | ext_byte(e); }
        if (b0 < 0xF0) {
            const int b1 = ext_byte(e), b2 = ext_byte(e);
            return (int32_t)(((uint32_t)(b0 & 0x0F) << 24) | (b1 << 16) | (b2 << 8) | ext_byte(e));
        }
        const int b1 = ext_byte(e), b2 = ext_byte(e), b3 = ext_byte(e), b4 = ext_byte(e);
        return (int32_t)(((uint32_t)(b0 & 0x0F) << 28) | ((uint32_t)b1 << 20) | ((uint32_t)b2 << 12) | ((uint32_t)b3 << 4) |
                         ((uint32_t)b4 & 0x0F));
    }
    __host__ __device__ __forceinline__ const int32_t* enc(int i) const { return P + 4 + 4 * i; }

    // an integer of encoding i; `is_byte`: EXTERNAL reads one raw byte instead of an ITF8
    __host__ __device__ int32_t value(int i, bool is_byte) {
        const int32_t* e = enc(i);
        switch (e[0]) {
            case E_NULL: return 0;
            case E_EXTERNAL: return is_byte ? ext_byte(e[1]) : ext_itf8(e[1]);
            case E_HUFFMAN: {
                const int32_t n = e[1];
                const int32_t* t = P + e[2];                 // (code, length, symbol) sorted by length, then code
                if (n == 1 && t[1] == 0) return t[2];
                uint32_t code = 0;
                int len = 0;
                for (int j = 0; j < n; ++j) {
                    while (len < t[3 * j + 1]) { code = (code << 1) | (uint32_t)bit(); ++len; }
                    if ((uint32_t)t[3 * j] == code && t[3 * j + 1] == len) return t[3 * j + 2];
                    if (err) return 0;
                }
                fail(UNFZ_CRAM_BAD_VALUE);
                return 0;
            }
            case E_BETA: return (int32_t)bits(e[2]) - e[1];
            case E_SUBEXP: {
                int n = 0;
                while (bit() == 1 && !err) ++n;
                const int b = n == 0 ? e[2] : n + e[2] - 1;
                if (b > 31) { fail(UNFZ_CRAM_BAD_VALUE); return 0; }
                uint32_t v = bits(b);
                if (n) v += 1u << b;
                return (int32_t)v - e[1];
            }
            case E_GAMMA: {
                int nz = 0;
                while (bit() == 0 && !err) ++nz;
                if (nz > 31) { fail(UNFZ_CRAM_BAD_VALUE); return 0; }
                const uint32_t v = (1u << nz) | bits(nz);
                return (int32_t)v - e[1];
            }
            default: fail(UNFZ_CRAM_BAD_ENCODING); return 0;
        }
    }
    // a byte array of encoding i written to dst (when non-null); returns its length
    __host__ __device__ int32_t array(int i, uint8_t* dst, int64_t cap) {
        const int32_t* e = enc(i);
        if (e[0] == E_BYTE_ARRAY_LEN) {
            const int32_t n = value(e[1], false);
            if (n < 0 || n > cap) { fail(UNFZ_CRAM_BAD_VALUE); return 0; }
            for (int32_t k = 0; k < n && !err; ++k) {
                const int32_t v = value(e[2], true);
                if (dst) dst[k] = (uint8_t)v;
            }
            return n;
        }
        if (e[0] == E_BYTE_ARRAY_STOP) {
            const int x = e[2];
            if (x < 0 || x >= n_ext) { fail(UNFZ_CRAM_BAD_ENCODING); return 0; }
            const uint8_t* p = blocks + ext[x].off;
            int64_t q = cur[x];
            while (q < ext[x].len && p[q] != (uint8_t)e[1]) ++q;
            if (q >= ext[x].len) { fail(UNFZ_CRAM_OVERRUN); return 0; }
            const int64_t n = q - cur[x];
            if (n > cap) { fail(UNFZ_CRAM_BAD_VALUE); return 0; }
            if (dst) for (int64_t k = 0; k < n; ++k) dst[k] = p[cur[x] + k];
            cur[x] = q + 1;
            return (int32_t)n;
        }
        fail(UNFZ_CRAM_BAD_ENCODING);
        return 0;
    }
};

// the reference base at 0-based position p of reference rid ('N' outside the spans the host uploaded)
__host__ __device__ __forceinline__ uint8_t ref_base(const UnfzCramRef* refs, int32_t n_refs, const uint8_t* rbytes,
                                                     int32_t rid, int64_t p) {
    for (int32_t k = 0; k < n_refs; ++k) {
        const UnfzCramRef& r = refs[k];
        if (r.ref_id == rid && p >= r.start && p < r.start + r.len) return upper(rbytes[r.off + (p - r.start)]);
    }
    return 'N';
}

// The CIGAR as htslib builds it from the features: runs of the same operation merge.
struct Cigar {
    uint8_t* out;          // null in the size step
    int32_t n;
    uint32_t op, len;
    __host__ __device__ __forceinline__ void add(uint32_t o, uint32_t l) {
        if (l == 0) return;
        if (len && o == op) { len += l; return; }
        flush();
        op = o;
        len = l;
    }
    __host__ __device__ __forceinline__ void flush() {
        if (len) {
            if (out) st32(out + 4 * n, (len << 4) | op);
            ++n;
        }
        len = 0;
    }
};

// Decodes every record of slice s.  WRITE = false: rec_len[i] (BAM bytes with block_size) and rec_cig[i] (n_cigar) of
// every record.  WRITE = true: the records at out + rec_off[i], then the mate fix-up.  Returns the slice status.
template <bool WRITE>
__host__ __device__ __forceinline__ int decode_slice(const UnfzCramSlice& s, const uint8_t* blocks, const UnfzCramExt* ext,
                                     const int32_t* prog, const UnfzCramRef* refs, const uint8_t* rbytes,
                                     int64_t* rec_len, int32_t* rec_cig, const int64_t* rec_off, uint8_t* out) {
    Dec d;
    d.blocks = blocks;
    d.core = blocks + s.core_off;
    d.core_len = s.core_len;
    d.bitpos = 0;
    d.ext = ext + s.ext_off;
    d.n_ext = s.n_ext;
    d.P = prog + s.prog_off;
    d.err = 0;
    if (s.n_ext > UNFZ_CRAM_MAX_EXT) return UNFZ_CRAM_BAD_ENCODING;
    for (int k = 0; k < s.n_ext; ++k) d.cur[k] = 0;
    const UnfzCramRef* sref = refs + s.refs_off;
    const int32_t* td = d.P + d.P[1];               // tag dictionary: n_lines, line_off[n_lines + 1], (key, enc) pairs
    const int32_t n_lines = td[0];
    const uint8_t* rg = s.rg_off >= 0 ? blocks + s.rg_off : nullptr;   // n_rg, off[n_rg + 1], "RGZ<id>\0" strings
    // substitution matrix: sub_base[ref][code]
    uint8_t sub_base[5][4];
    const char* acgtn = "ACGTN";
    for (int r = 0; r < 5; ++r) {
        int k = 0;
        for (int a = 0; a < 5; ++a) {
            if (a == r) continue;
            sub_base[r][(s.sub[r] >> (6 - 2 * k)) & 3] = (uint8_t)acgtn[a];
            ++k;
        }
    }
    int64_t prev_ap = s.ap_start;
    for (int32_t i = 0; i < s.n_records && !d.err; ++i) {
        const int64_t gi = s.rec_first + i;
        uint8_t* o = WRITE ? out + rec_off[gi] : nullptr;
        const int32_t bf = d.value(S_BF, false);
        const int32_t cf = d.value(S_CF, false);
        const int32_t rid = s.ref_id == -2 ? d.value(S_RI, false) : s.ref_id;
        const int32_t rl = d.value(S_RL, false);
        int64_t ap = d.value(S_AP, false);
        if (s.flags & UNFZ_CRAM_AP_DELTA) { ap += prev_ap; prev_ap = ap; }
        const int32_t rgi = d.value(S_RG, false);
        if (rl < 0 || rl > (1 << 28) || (bf & ~0xFFFF)) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
        const bool has_seq = !(cf & 8);
        const int64_t l_seq = has_seq ? rl : 0;
        const int64_t n_cig = WRITE ? rec_cig[gi] : 0;
        // read name straight into place
        uint8_t* name = WRITE ? o + 36 : nullptr;
        const int32_t ln = d.array(S_RN, name, 254);
        if (WRITE) name[ln] = 0;
        const int64_t l_name = ln + 1;
        uint8_t* cig = WRITE ? o + 36 + l_name : nullptr;
        uint8_t* seq = WRITE ? cig + 4 * n_cig : nullptr;
        uint8_t* qual = WRITE ? seq + (l_seq + 1) / 2 : nullptr;
        uint8_t* aux = WRITE ? qual + l_seq : nullptr;
        int32_t flag = bf, next_rid = -1, next_pos = -1, tlen = 0;
        if (cf & 2) {                                   // detached mate
            const int32_t mf = d.value(S_MF, false);
            next_rid = d.value(S_NS, false);
            next_pos = d.value(S_NP, false) - 1;
            tlen = d.value(S_TS, false);
            if (mf & 1) flag |= 0x20;
            if (mf & 2) flag |= 0x8;
        } else if (cf & 4) {                            // mate downstream in this slice
            const int32_t nf = d.value(S_NF, false);
            if (nf < 0 || i + 1 + (int64_t)nf >= s.n_records) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
            next_rid = CRAM_ATTACHED;
            next_pos = i + 1 + nf;
            tlen = INT32_MIN;
        } else {
            tlen = INT32_MIN;                           // may be the last fragment of an attached chain
        }
        // tags, in the order of the tag line, then RG
        const int32_t tl = d.value(S_TL, false);
        if (tl < 0 || tl >= n_lines) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
        int64_t l_aux = 0;
        const int32_t* ent = td + 1 + (n_lines + 1);
        for (int32_t k = td[1 + tl]; k < td[1 + tl + 1] && !d.err; ++k) {
            const int32_t key = ent[2 * k], ei = ent[2 * k + 1];
            const uint8_t type = (uint8_t)key;
            uint8_t* v = WRITE ? aux + l_aux : nullptr;
            if (WRITE) { v[0] = (uint8_t)(key >> 16); v[1] = (uint8_t)(key >> 8); v[2] = type; }
            const int32_t n = d.array(ei, WRITE ? v + 3 : nullptr, 1 << 28);
            l_aux += 3 + n;
            if ((type == 'Z' || type == 'H') && d.enc(ei)[0] == E_BYTE_ARRAY_STOP) {
                if (WRITE) v[3 + n] = 0;                 // the stop byte ends the string: the NUL comes back
                ++l_aux;
            }
        }
        if (rgi >= 0) {
            if (!rg || rgi >= (int32_t)ld32(rg)) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
            const int32_t a = (int32_t)ld32(rg + 4 + 4 * rgi), b = (int32_t)ld32(rg + 8 + 4 * rgi);
            if (WRITE) for (int32_t k = 0; k < b - a; ++k) aux[l_aux + k] = rg[a + k];
            l_aux += b - a;
        }
        // bases, qualities and the CIGAR
        Cigar cg;
        cg.out = cig;
        cg.n = 0;
        cg.op = 0;
        cg.len = 0;
        if (WRITE) {
            for (int64_t k = 0; k < (l_seq + 1) / 2; ++k) seq[k] = 0;
            for (int64_t k = 0; k < l_seq; ++k) qual[k] = 0xFF;
        }
        int32_t mapq = 0;
        int64_t ref_len = 0;
        const int64_t pos0 = ap - 1;
        auto put_base = [&](int64_t k, uint8_t c) {
            if (WRITE && has_seq && k >= 0 && k < rl) seq[k >> 1] |= nt16(c) << ((k & 1) ? 0 : 4);
        };
        auto put_qual = [&](int64_t k, int32_t q) {
            if (WRITE && has_seq && k >= 0 && k < rl) qual[k] = (uint8_t)q;
        };
        if (!(bf & 4)) {
            const int32_t fn = d.value(S_FN, false);
            if (fn < 0) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
            int64_t rp = 0, fp = 0, refp = pos0;   // read position (0-based), last feature position, reference position
            auto match = [&](int64_t n) {
                if (n <= 0) return;
                if (WRITE) for (int64_t k = 0; k < n; ++k) put_base(rp + k, ref_base(sref, s.n_refs, rbytes, rid, refp + k));
                cg.add(0, (uint32_t)n);
                rp += n;
                refp += n;
                ref_len += n;
            };
            for (int32_t f = 0; f < fn && !d.err; ++f) {
                const int32_t fc = d.value(S_FC, true);
                fp += d.value(S_FP, false);
                if (fp - 1 < rp || fp - 1 > rl) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
                match(fp - 1 - rp);
                switch (fc) {
                    case 'B': {
                        const int32_t b = d.value(S_BA, true), q = d.value(S_QS, true);
                        put_base(rp, (uint8_t)b);
                        put_qual(rp, q);
                        cg.add(0, 1);
                        ++rp; ++refp; ++ref_len;
                        break;
                    }
                    case 'X': {
                        const int32_t code = d.value(S_BS, true);
                        if (WRITE) put_base(rp, sub_base[base5(ref_base(sref, s.n_refs, rbytes, rid, refp))][code & 3]);
                        cg.add(0, 1);
                        ++rp; ++refp; ++ref_len;
                        break;
                    }
                    case 'I': case 'S': {
                        const int64_t room = rl - rp;
                        // the bases go straight into the nibbles: decode into the quality slot first (same length),
                        // then pack; the qualities of these positions are written later
                        const int32_t n = d.array(fc == 'I' ? S_IN : S_SC, (WRITE && has_seq) ? qual + rp : nullptr, room);
                        if (WRITE && has_seq) for (int32_t k = 0; k < n; ++k) { put_base(rp + k, qual[rp + k]); qual[rp + k] = 0xFF; }
                        cg.add(fc == 'I' ? 1 : 4, (uint32_t)n);
                        rp += n;
                        break;
                    }
                    case 'b': {
                        const int32_t n = d.array(S_BB, (WRITE && has_seq) ? qual + rp : nullptr, rl - rp);
                        if (WRITE && has_seq) for (int32_t k = 0; k < n; ++k) { put_base(rp + k, qual[rp + k]); qual[rp + k] = 0xFF; }
                        cg.add(0, (uint32_t)n);
                        rp += n; refp += n; ref_len += n;
                        break;
                    }
                    case 'q': {
                        d.array(S_QQ, (WRITE && has_seq) ? qual + rp : nullptr, rl - rp);
                        break;
                    }
                    case 'Q': put_qual(rp, d.value(S_QS, true)); break;
                    case 'i': {
                        put_base(rp, (uint8_t)d.value(S_BA, true));
                        cg.add(1, 1);
                        ++rp;
                        break;
                    }
                    case 'D': { const int32_t n = d.value(S_DL, false); if (n < 0) d.fail(UNFZ_CRAM_BAD_VALUE); cg.add(2, (uint32_t)n); refp += n; ref_len += n; break; }
                    case 'N': { const int32_t n = d.value(S_RS, false); if (n < 0) d.fail(UNFZ_CRAM_BAD_VALUE); cg.add(3, (uint32_t)n); refp += n; ref_len += n; break; }
                    case 'P': { const int32_t n = d.value(S_PD, false); if (n < 0) d.fail(UNFZ_CRAM_BAD_VALUE); cg.add(6, (uint32_t)n); break; }
                    case 'H': { const int32_t n = d.value(S_HC, false); if (n < 0) d.fail(UNFZ_CRAM_BAD_VALUE); cg.add(5, (uint32_t)n); break; }
                    default: d.fail(UNFZ_CRAM_BAD_VALUE);
                }
                if (rp > rl) d.fail(UNFZ_CRAM_BAD_VALUE);
            }
            if (d.err) break;
            match(rl - rp);
            mapq = d.value(S_MQ, false);
            if (cf & 1) for (int32_t k = 0; k < rl && !d.err; ++k) put_qual(k, d.value(S_QS, true));
        } else {
            if (has_seq) for (int32_t k = 0; k < rl && !d.err; ++k) put_base(k, (uint8_t)d.value(S_BA, true));
            if (cf & 1) for (int32_t k = 0; k < rl && !d.err; ++k) put_qual(k, d.value(S_QS, true));
        }
        cg.flush();
        if (d.err) break;
        if (!WRITE && (mapq < 0 || mapq > 255 || cg.n > 0xFFFF)) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
        const int64_t size = 36 + l_name + 4 * (int64_t)cg.n + (l_seq + 1) / 2 + l_seq + l_aux;
        if (!WRITE) {
            rec_len[gi] = size;
            rec_cig[gi] = cg.n;
            continue;
        }
        if (cg.n != n_cig || rec_off[gi + 1] - rec_off[gi] != size) { d.fail(UNFZ_CRAM_BAD_VALUE); break; }
        const int64_t end = pos0 + ((bf & 4) || ref_len == 0 ? 1 : ref_len);
        st32(o, (uint32_t)(size - 4));
        st32(o + 4, (uint32_t)rid);
        st32(o + 8, (uint32_t)pos0);
        o[12] = (uint8_t)l_name;
        o[13] = (uint8_t)mapq;
        st16(o + 14, reg2bin(pos0, end));
        st16(o + 16, (uint32_t)cg.n);
        st16(o + 18, (uint32_t)flag);
        st32(o + 20, (uint32_t)l_seq);
        st32(o + 24, (uint32_t)next_rid);
        st32(o + 28, (uint32_t)next_pos);
        st32(o + 32, (uint32_t)tlen);
    }
    if (d.err || !WRITE) return d.err;
    // ---- mate fix-up of attached mates (htslib's cram_decode_slice_xref), on the written records --------------------
    // Scratch while it runs: next_ref_id CRAM_ATTACHED marks a record whose next_pos is its mate line; tlen INT32_MIN is
    // a template length not yet set.  apos / aend are 1-based, aend inclusive (apos for an unmapped read).
    auto R = [&](int32_t i) -> uint8_t* { return out + rec_off[s.rec_first + i]; };
    auto apos = [&](int32_t i) -> int64_t { return (int64_t)(int32_t)ld32(R(i) + 8) + 1; };
    auto aend = [&](int32_t i) -> int64_t {
        const uint8_t* r = R(i);
        if ((r[18] | (r[19] << 8)) & 4) return apos(i);
        const uint8_t* c = r + 36 + r[12];
        int64_t len = 0;
        for (uint32_t k = 0, n = r[16] | (r[17] << 8); k < n; ++k) {
            const uint32_t w = ld32(c + 4 * k), op = w & 15;
            if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) len += w >> 4;
        }
        return apos(i) + (len ? len : 1) - 1;
    };
    auto line = [&](int32_t i) -> int32_t { return (int32_t)ld32(R(i) + 24) == CRAM_ATTACHED ? (int32_t)ld32(R(i) + 28) : -1; };
    auto set_line = [&](int32_t i, int32_t v) { st32(R(i) + 24, (uint32_t)CRAM_ATTACHED); st32(R(i) + 28, (uint32_t)v); };
    auto flag_of = [&](int32_t i) -> uint32_t { return R(i)[18] | (R(i)[19] << 8); };
    auto tlen_of = [&](int32_t i) -> int32_t { return (int32_t)ld32(R(i) + 32); };
    auto set_tlen = [&](int32_t i, int64_t v) { st32(R(i) + 32, (uint32_t)(int32_t)v); };
    for (int32_t rec = 0; rec < s.n_records; ++rec) {
        const int32_t ml = line(rec);
        if (ml < 0) continue;
        if (tlen_of(rec) == INT32_MIN) {
            int32_t id2 = rec;
            int64_t aleft = apos(rec), aright = aend(rec);
            int32_t ref = (int32_t)ld32(R(rec) + 4), left_cnt = 0;
            for (int32_t guard = 0; guard <= s.n_records; ++guard) {
                const int64_t a = apos(id2);
                if (aleft > a) { aleft = a; left_cnt = 1; } else if (aleft == a) ++left_cnt;
                if (aright < aend(id2)) aright = aend(id2);
                const int32_t nx = line(id2);
                if (nx < 0) { set_line(id2, rec); break; }
                if (nx <= id2 || nx >= s.n_records) return UNFZ_CRAM_BAD_VALUE;
                id2 = nx;
                if ((int32_t)ld32(R(id2) + 4) != ref) ref = -1;
            }
            const int64_t tl = aright - aleft + 1;
            int32_t id = rec;
            for (int32_t guard = 0; guard <= s.n_records; ++guard) {
                if (ref == -1) set_tlen(id, 0);
                else if (apos(id) == aleft && (left_cnt == 1 || (flag_of(id) & 0x40))) set_tlen(id, tl);
                else set_tlen(id, -tl);
                id = line(id);
                if (id == rec || id < 0) break;
            }
        }
        const int32_t m = line(rec);
        uint32_t fl = flag_of(rec) | 0x1;
        const uint32_t mfl = flag_of(m);
        if (mfl & 0x4) { fl |= 0x8; set_tlen(rec, 0); }
        if (fl & 0x4) set_tlen(rec, 0);
        if (mfl & 0x10) fl |= 0x20;
        st32(R(rec) + 24, ld32(R(m) + 4));
        st32(R(rec) + 28, (uint32_t)(apos(m) - 1));
        st16(R(rec) + 18, fl);
    }
    for (int32_t rec = 0; rec < s.n_records; ++rec)
        if (tlen_of(rec) == INT32_MIN) set_tlen(rec, 0);
    return 0;
}

__global__ void __maxnreg__(96) cram_slice_size_kernel(const UnfzCramSlice* __restrict__ slices, int64_t n,
                                                               const uint8_t* __restrict__ blocks,
                                                               const UnfzCramExt* __restrict__ ext,
                                                               const int32_t* __restrict__ prog,
                                                               const UnfzCramRef* __restrict__ refs,
                                                               const uint8_t* __restrict__ rbytes, int64_t* rec_len,
                                                               int32_t* rec_cig, int32_t* status) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    status[i] = decode_slice<false>(slices[i], blocks, ext, prog, refs, rbytes, rec_len, rec_cig, nullptr, nullptr);
}

__global__ void __launch_bounds__(128) cram_slice_write_kernel(const UnfzCramSlice* __restrict__ slices, int64_t n,
                                                                const uint8_t* __restrict__ blocks,
                                                                const UnfzCramExt* __restrict__ ext,
                                                                const int32_t* __restrict__ prog,
                                                                const UnfzCramRef* __restrict__ refs,
                                                                const uint8_t* __restrict__ rbytes,
                                                                const int32_t* __restrict__ rec_cig,
                                                                const int64_t* __restrict__ rec_off, uint8_t* out,
                                                                int32_t* status) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || status[i]) return;
    status[i] = decode_slice<true>(slices[i], blocks, ext, prog, refs, rbytes, nullptr, const_cast<int32_t*>(rec_cig),
                                   rec_off, out);
}

}  // namespace

// ---- rANS 4x8 (CRAM 3.0 block method 4), order 0 and order 1 --------------------------------------------------------

namespace {
struct RansIn {
    const uint8_t* p;
    const uint8_t* end;
    bool bad;
    uint8_t get() {
        if (p >= end) { bad = true; return 0; }
        return *p++;
    }
};

// one frequency table (run-length coded symbols, 1- or 2-byte frequencies) into F / C and the slot -> symbol map
bool rans_table(RansIn& in, uint32_t* F, uint32_t* Cf, uint8_t* sym) {
    int rle = 0, x = 0;
    int j = in.get();
    for (int guard = 0; guard < 256; ++guard) {
        uint32_t f = in.get();
        if (f >= 128) f = ((f & 127) << 8) | in.get();
        if (in.bad || x + (int)f > 4096) return false;
        F[j] = f;
        Cf[j] = (uint32_t)x;
        memset(sym + x, j, f);
        x += (int)f;
        if (!rle && in.p < in.end && j + 1 == *in.p) {
            j = in.get();
            rle = in.get();
        } else if (rle) {
            --rle;
            ++j;
        } else {
            j = in.get();
        }
        if (j == 0 || j > 255) break;
    }
    return !in.bad && j == 0;
}
}  // namespace

extern "C" int64_t unfz_rans4x8_decode_host(const uint8_t* in, int64_t in_len, uint8_t* out, int64_t out_cap) {
    if (in_len < 9) return -1;
    const int order = in[0];
    const int64_t comp = ld32(in + 1), raw = ld32(in + 5);
    if (comp + 9 > in_len || raw > out_cap || (order != 0 && order != 1)) return -1;
    if (raw == 0) return 0;
    RansIn r{in + 9, in + 9 + comp, false};
    const uint32_t L = 1u << 23;
    if (order == 0) {
        uint32_t F[256] = {0}, Cf[256] = {0};
        uint8_t* sym = new uint8_t[4096]();
        if (!rans_table(r, F, Cf, sym)) { delete[] sym; return -1; }
        uint32_t R[4];
        for (int k = 0; k < 4; ++k) { R[k] = r.get() | (r.get() << 8) | (r.get() << 16) | ((uint32_t)r.get() << 24); }
        const int64_t out_end = raw & ~(int64_t)3;
        for (int64_t i = 0; i < out_end && !r.bad; i += 4) {
            for (int k = 0; k < 4; ++k) {
                const uint8_t c = sym[R[k] & 4095];
                out[i + k] = c;
                R[k] = F[c] * (R[k] >> 12) + (R[k] & 4095) - Cf[c];
                while (R[k] < L && !r.bad) R[k] = (R[k] << 8) | r.get();
            }
        }
        for (int64_t k = 0; k < (raw & 3); ++k) out[out_end + k] = sym[R[k] & 4095];
        delete[] sym;
        return r.bad ? -1 : raw;
    }
    uint32_t* F = new uint32_t[256 * 256]();
    uint32_t* Cf = new uint32_t[256 * 256]();
    uint8_t* sym = new uint8_t[256 * 4096]();
    bool ok = true;
    int rle_i = 0, i = r.get();
    for (int guard = 0; guard < 256 && ok; ++guard) {
        ok = rans_table(r, F + 256 * i, Cf + 256 * i, sym + 4096 * i);
        if (!rle_i && r.p < r.end && i + 1 == *r.p) {
            i = r.get();
            rle_i = r.get();
        } else if (rle_i) {
            --rle_i;
            ++i;
        } else {
            i = r.get();
        }
        if (i == 0 || i > 255) break;
    }
    int64_t res = -1;
    if (ok && !r.bad && i == 0) {
        uint32_t R[4];
        for (int k = 0; k < 4; ++k) { R[k] = r.get() | (r.get() << 8) | (r.get() << 16) | ((uint32_t)r.get() << 24); }
        const int64_t q = raw >> 2;
        uint8_t l[4] = {0, 0, 0, 0};
        for (int64_t j = 0; j < q && !r.bad; ++j) {
            for (int k = 0; k < 4; ++k) {
                const uint8_t c = sym[4096 * l[k] + (R[k] & 4095)];
                out[j + k * q] = c;
                R[k] = F[256 * l[k] + c] * (R[k] >> 12) + (R[k] & 4095) - Cf[256 * l[k] + c];
                while (R[k] < L && !r.bad) R[k] = (R[k] << 8) | r.get();
                l[k] = c;
            }
        }
        for (int64_t j = 4 * q; j < raw && !r.bad; ++j) {
            const uint8_t c = sym[4096 * l[3] + (R[3] & 4095)];
            out[j] = c;
            R[3] = F[256 * l[3] + c] * (R[3] >> 12) + (R[3] & 4095) - Cf[256 * l[3] + c];
            while (R[3] < L && !r.bad) R[3] = (R[3] << 8) | r.get();
            l[3] = c;
        }
        res = r.bad ? -1 : raw;
    }
    delete[] F;
    delete[] Cf;
    delete[] sym;
    return res;
}

// ---- slice decode entry points ------------------------------------------------------------------------------------

extern "C" int64_t unfz_cram_decode_size_host(const UnfzCramSlice* slices, int64_t n, const uint8_t* blocks,
                                              const UnfzCramExt* ext, const int32_t* prog, const UnfzCramRef* refs,
                                              const uint8_t* rbytes, int64_t* rec_len, int32_t* rec_cig, int32_t* status) {
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        status[i] = decode_slice<false>(slices[i], blocks, ext, prog, refs, rbytes, rec_len, rec_cig, nullptr, nullptr);
        bad += status[i] != 0;
    }
    return bad;
}

extern "C" int64_t unfz_cram_decode_write_host(const UnfzCramSlice* slices, int64_t n, const uint8_t* blocks,
                                               const UnfzCramExt* ext, const int32_t* prog, const UnfzCramRef* refs,
                                               const uint8_t* rbytes, const int32_t* rec_cig, const int64_t* rec_off,
                                               uint8_t* out, int32_t* status) {
    int64_t bad = 0;
    for (int64_t i = 0; i < n; ++i) {
        status[i] = decode_slice<true>(slices[i], blocks, ext, prog, refs, rbytes, nullptr, const_cast<int32_t*>(rec_cig),
                                       rec_off, out);
        bad += status[i] != 0;
    }
    return bad;
}

extern "C" int unfz_cram_decode_size(UnfzCtx* ctx, const UnfzCramSlice* slices, int64_t n, const uint8_t* blocks,
                                     const UnfzCramExt* ext, const int32_t* prog, const UnfzCramRef* refs,
                                     const uint8_t* rbytes, int64_t* rec_len, int32_t* rec_cig, int32_t* status,
                                     void* stream) {
    if (n <= 0) return 0;
    cram_slice_size_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(slices, n, blocks, ext, prog, refs,
                                                                                           rbytes, rec_len, rec_cig, status);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}

extern "C" int unfz_cram_decode_write(UnfzCtx* ctx, const UnfzCramSlice* slices, int64_t n, const uint8_t* blocks,
                                      const UnfzCramExt* ext, const int32_t* prog, const UnfzCramRef* refs,
                                      const uint8_t* rbytes, const int32_t* rec_cig, const int64_t* rec_off, uint8_t* out,
                                      int32_t* status, void* stream) {
    if (n <= 0) return 0;
    cram_slice_write_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        slices, n, blocks, ext, prog, refs, rbytes, rec_cig, rec_off, out, status);
    UNFZ_LAUNCH_CHECK(ctx);
    return 0;
}
