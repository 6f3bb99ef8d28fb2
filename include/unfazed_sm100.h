/*
 * unfazed_sm100.h -- C ABI of libunfazed_sm100.so, the B200 (sm_100a) phasing hot path.
 *
 * The reference (jbelyeu/unfazed) is pure Python and has no FFI: its boundary for this path is the
 * module interface informative_site_finder.find / read_collector.collect_reads_* /
 * site_searcher.match_informative_sites / {snv,sv}_phaser.phase_by_reads / unfazed.summarize_record.
 * Each entry point below names the reference code it replaces (paths relative to the reference
 * repo).  The Python drop-in modules in unfazed_b200/ bind these with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name starts with h_;
 *   - the caller owns all buffers and passes sizes explicitly; nothing is allocated here;
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 = ok, negative = error; text via unfz_last_error();
 *   - no globals: thresholds are passed by value per call (the reference keeps them in module
 *     globals, informative_site_finder.py:187-204, read_collector.py:361-370).
 */
#ifndef UNFAZED_SM100_H
#define UNFAZED_SM100_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNFZ_ABI_VERSION 2

/* ---- class code of one (DNM x site) pair, written by unfz_classify_sites ------------------- */
#define UNFZ_CLS_HET        0x01  /* usable for extended read-backed phasing (het_sites)         */
#define UNFZ_CLS_CAND       0x02  /* informative site (candidate_sites)                          */
#define UNFZ_CLS_ALT_IS_DAD 0x04  /* candidate: alt_parent is the father                         */
#define UNFZ_CLS_KID_ALT    0x08  /* CNV mode: kid_allele == "alt_parent" (else "ref_parent")    */

/* ---- segment modes ------------------------------------------------------------------------- */
#define UNFZ_MODE_READ    0   /* whole_region=False: kid must be HET and high quality            */
#define UNFZ_MODE_CNV_DEL 1   /* whole_region=True, vartype DEL                                  */
#define UNFZ_MODE_CNV_DUP 2   /* whole_region=True, vartype DUP                                  */
#define UNFZ_MODE_CNV_NA  3   /* whole_region=True, any other vartype: never a candidate         */

/* ---- per-read summary flags (UnfzReadSum.flags) -------------------------------------------- */
#define UNFZ_RS_GOOD_CONC 0x01  /* goodread(read)                (read_collector.py:28-53)       */
#define UNFZ_RS_GOOD_DISC 0x02  /* goodread(read, True)                                          */
#define UNFZ_RS_NONE_OK   0x04  /* <= 5 None reference positions (:200, :407)                    */
#define UNFZ_RS_EXT_OK    0x08  /* <= 5 CIGAR ops other than M/= (:190-196)                      */
#define UNFZ_RS_INS_OK    0x10  /* abs(tlen - 2*readlen) <= concordant_upper_len (:181-183,:395) */
#define UNFZ_RS_HAS_MATE  0x20  /* bamfile.mate(read) would not raise                            */

/* ---- DNM kinds for unfz_chain_tally ---------------------------------------------------------- */
#define UNFZ_KIND_SKIP  0   /* nothing to do (autophased, no candidates, no usable REF/ALT)       */
#define UNFZ_KIND_SNV   1   /* len(ref) == len(alt): snv_match_alleles                            */
#define UNFZ_KIND_INDEL 2   /* indel_match_alleles                                               */
#define UNFZ_KIND_SV    3   /* collect_reads_sv seeds                                            */

/* ---- final call codes (UnfzCall.origin) ------------------------------------------------------ */
#define UNFZ_ORIGIN_NONE 0
#define UNFZ_ORIGIN_DAD  1
#define UNFZ_ORIGIN_MOM  2
#define UNFZ_ORIGIN_BOTH 3   /* "dad|mom": AMBIGUOUS_READBACKED                                  */

#define UNFZ_EV_READBACKED        0x01
#define UNFZ_EV_ALLELE_BALANCE    0x02
#define UNFZ_EV_AMBIG_READBACKED  0x04
#define UNFZ_EV_AMBIG_ALLELE_BAL  0x08
#define UNFZ_EV_AMBIG_BOTH        0x10
#define UNFZ_EV_SEX_CHROM         0x20

/* Trio-major site rows on the DEVICE.  The host table (schema.SiteTable) is plain SoA; at upload the
 * genotype fields are packed so that the classifier reads one row with five naturally aligned loads
 * (44 B per row, the "canonical" byte count of SURVEY 8(a)-3):
 *   meta u32      flag | gt_kid<<8 | gt_dad<<16 | gt_mom<<24   (cyvcf2 gt_types 0/1/2/3)        4 B
 *   rec  4 x f32  { pos (int32 bits), gq_kid, gq_dad, gq_mom }                                  16 B
 *   dep  6 x i32  { rd_kid, ad_kid, rd_dad, ad_dad, rd_mom, ad_mom }                            24 B
 * pos / ref / alt are kept as separate columns for the read path and the host. */
typedef struct {
    int64_t         n_rows;
    int32_t         n_blocks;
    int32_t         _pad;
    const int64_t*  blk_off;     /* [n_blocks+1] */
    const int32_t*  pos;
    const uint8_t*  ref;         /* ASCII */
    const uint8_t*  alt;         /* ASCII */
    const uint32_t* meta;        /* bit0 of the low byte: simple biallelic SNV record */
    const float*    rec;         /* [n_rows][4], 16-byte aligned */
    const int32_t*  dep;         /* [n_rows][6],  8-byte aligned */
} UnfzSiteCols;

/* 32-byte read header (schema.READ_HDR).
 * Layout contract of the read columns: reads of a block are sorted by start (BAM file order), and the
 * CIGAR words / quality bytes / bases of consecutive reads are stored back to back in read order
 * (cigar_off and the 40-bit quality offset never decrease with the read index) -- the scan stages the
 * span of 32 consecutive reads with one contiguous copy.  Read and site-row indices fit 31 bits. */
typedef struct {
    int32_t  start;
    int32_t  tlen;
    int32_t  mate;        /* global read index or -1 */
    uint32_t cigar_off;
    uint32_t qoff_lo;
    int32_t  l_seq;
    uint16_t flag;
    uint16_t n_cigar;
    uint8_t  mapq;
    uint8_t  aux;         /* bit0 next_ref==ref, bit1 has SA tag; device only: bit6 the CIGAR is one M/= operation of l_seq bases (set by
                             unfz_read_starts), bit7 a base of the read is not ACGT (set by unfz_expand_nlist or unfz_bam_emit_planes) */
    uint8_t  qoff_hi;
    uint8_t  pad;
} UnfzRead;

typedef struct {
    int64_t         n_reads;
    int32_t         n_blocks;
    int32_t         _pad;
    const int64_t*  blk_off;     /* [n_blocks+1] */
    const int32_t*  blk_sblk;    /* [n_blocks] site block holding this kid's trio on this contig, or -1 */
    const double*   blk_cul;     /* [n_blocks] concordant_upper_len of the kid */
    const UnfzRead* hdr;
    const int32_t*  start;       /* dense copy of hdr[].start (unfz_read_starts): the window searches of the chaining bisect
                                    over it -- 32 starts per 128-byte line instead of 4 */
    const uint32_t* cigar;       /* BAM encoding len<<4|op */
    const uint32_t* lowq;        /* 1 bit per query base (bit i&31 of word i>>5): base quality < --min-gt-qual.
                                    Every use of a base quality on this path is that one comparison (goodread
                                    read_collector.py:44-46, connect_reads :123, indel_match_alleles :281-284), so the
                                    host packs the comparison, not the byte: 8x fewer bytes over PCIe and through the
                                    scan.  16-byte aligned, readable for 48 bytes past ceil(n_qual/8) */
    const uint32_t* nmask;       /* 1 bit per query base: the base is not A/C/G/T (built on the device from the sparse
                                    index list by unfz_expand_nlist; reads that own such a base carry aux bit7) */
    const uint8_t*  seq2;        /* 2-bit bases, base i at bits 2*(i&3) of byte i>>2; a masked base has code 0 for N */
    int64_t         n_qual;      /* number of query bases */
    int64_t         n_cigar;
} UnfzReadCols;

/* per-read summary written by unfz_read_scan: ONE 32-byte sector holds everything the chaining asks about a read
 * (its span, its mate, its filter flags and where its hit words are), so a candidate read costs one sector, not a
 * summary sector plus a header sector */
typedef struct {
    int32_t  end;         /* reference_end (exclusive) */
    int32_t  fmark;       /* number of marked site rows before the first row with pos >= start */
    uint16_t flags;       /* UNFZ_RS_* */
    uint16_t cnt;         /* marked site rows with start <= pos < end */
    uint32_t hoff;        /* first hit word of this read, relative to its scan tile (see unfz_read_scan) */
    int32_t  start;       /* reference_start (copy of the header field) */
    int32_t  mate;        /* mate index or -1 (copy of the header field) */
    int32_t  row_lb;      /* first site row of the read's block with pos >= start (where the allele lookup starts walking) */
    int32_t  _pad;
} UnfzReadSum;

typedef struct {
    double  ab_homref[2];
    double  ab_homalt[2];
    double  ab_het[2];
    double  min_gt_qual;         /* --min-gt-qual; also the minimum base quality */
    int32_t min_depth;
    int32_t min_map_qual;
    int32_t readlen;
    int32_t ext_read_goal;       /* --insert-size-max-sample (Q2) */
    int32_t no_extended;
    int32_t evidence_min_ratio;
    int32_t split_error_margin;
    int32_t _pad;
} UnfzParams;

/* one window of one DNM; produced by the host planner from find()/find_many() semantics */
typedef struct {
    int32_t sblk;         /* site block or -1 */
    int32_t lo_pos;       /* inclusive bounds on the 0-based site position */
    int32_t hi_pos;
    int32_t mult;         /* how many times each site is appended (Q9, find_many duplicates) */
    int32_t dnm;          /* owning DNM entry */
    int32_t excl_lo;      /* small-event rule: skip sites with excl_lo <= pos < excl_hi */
    int32_t excl_hi;
    int32_t mode;         /* UNFZ_MODE_* */
} UnfzSegIn;

typedef struct {
    int32_t pos;          /* denovo["start"] */
    int32_t end;          /* denovo["end"] */
    int32_t rblk;         /* read block or -1 */
    int32_t kind;         /* UNFZ_KIND_* */
    int32_t seg_lo;       /* segments [seg_lo, seg_hi) belong to this DNM entry */
    int32_t seg_hi;
    int32_t ref_off;      /* allele blob offsets / lengths (REF and ALT of the DNM) */
    int32_t ref_len;
    int32_t alt_off;
    int32_t alt_len;
    int32_t cnv_entry;    /* index of the CNV-mode entry of the same DNM, or -1 */
    int32_t flags;        /* bit0: autophased (SEX-CHROM), bit1: autophased on Y, bit2: SV autophase quirk (Q8), bit3: seed fetch window is (pos,pos+1) (Q24) */
} UnfzDnm;

/* per-DNM output of unfz_chain_tally / unfz_summarize */
typedef struct {
    int32_t n_dad_sites, n_mom_sites;   /* unique informative-site positions per parent */
    int32_t n_dad_reads, n_mom_reads;   /* unique read names per parent */
    int32_t cnv_dad, cnv_mom;           /* allele-balance votes (with duplicates) */
    int32_t has_record;                 /* 1: a read-backed record exists (matches non-empty) */
    int32_t status;                     /* 0 ok, >0 capacity / consistency problems */
} UnfzTally;

typedef struct {
    int32_t origin;                     /* UNFZ_ORIGIN_* */
    int32_t evidence_count;
    int32_t evidence_types;             /* UNFZ_EV_* bitmask */
    int32_t emitted;                    /* 0: summarize_record returns None for include_ambiguous=False */
} UnfzCall;

typedef struct UnfzCtx UnfzCtx;

int         unfz_abi_version(void);
int         unfz_ctx_create(int device, UnfzCtx** out);
void        unfz_ctx_destroy(UnfzCtx* ctx);
const char* unfz_last_error(UnfzCtx* ctx);

/* Speculative sizing (no reference counterpart: the reference has no device).  The sizes of the variable
 * outputs -- pairs, hits, chaining scratch -- are only known on the device.  A caller that allocated them
 * from the capacities of an earlier, similar batch calls unfz_check_caps() instead of reading the totals
 * back: it compares up to 8 device-resident int64 totals (h_totals[i] is a device address) with
 * h_caps[i], stores them in actual[0..k) and ORs 1 into *flag when one is exceeded.  While a flag is
 * installed with unfz_ctx_set_guard(), classify_sites / compact_sites / read_scan / chain_size /
 * read_site_alleles / chain_tally return immediately once it is set, so nothing is written out of bounds;
 * the caller then re-runs the batch with exact sizes.  unfz_classify_sites treats n_pairs as the capacity
 * of out_class and reads the batch's own total from seg_pair_off[n_segs].  Pass NULL to remove the guard. */
int unfz_ctx_set_guard(UnfzCtx*, const int32_t* flag);
int unfz_check_caps(UnfzCtx*, int32_t k, const int64_t* const* h_totals, const int64_t* h_caps, int32_t* flag,
                    int64_t* actual, void* stream);

/* Exclusive prefix sums (device-wide).  `work` needs unfz_scan_work_bytes(n) bytes. */
int64_t unfz_scan_work_bytes(int64_t n);
int unfz_exclusive_scan_i64(UnfzCtx*, const int64_t* in, int64_t* out, int64_t n, void* work, void* stream);
int unfz_exclusive_scan_u8_i32(UnfzCtx*, const uint8_t* in, int32_t* out, int64_t n, void* work, void* stream);
int unfz_exclusive_scan_u32(UnfzCtx*, const uint32_t* in, uint32_t* out /* n+1 entries */, int64_t n, int64_t* total_out,
                            void* work, void* stream);
/* n_rows independent rows in one launch: in[n_rows][n] -> out[n_rows][n+1] (last entry = row total) */
int unfz_exclusive_scan_rows_i64(UnfzCtx*, const int64_t* in, int64_t* out, int32_t n_rows, int64_t n, void* stream);

/* Window membership: informative_site_finder.py get_position :10-43 / get_close_vars :399-420.
 * For every segment: seg_row_lo = first row of the block with pos >= lo_pos, seg_count =
 * mult * #rows with lo_pos <= pos <= hi_pos. */
int unfz_window_search(UnfzCtx*, const UnfzSiteCols* sites, const UnfzSegIn* segs, int32_t n_segs,
                       int32_t* seg_row_lo, int64_t* seg_count, void* stream);

/* Informative-site classification of every (DNM x site) pair:
 * is_high_quality_site :46-73, get_kid_allele :76-134, find :252-339 == add_good_candidate_variant
 * :457-542.  seg_pair_off is the exclusive scan of seg_count (n_segs+1 entries). */
int unfz_classify_sites(UnfzCtx*, const UnfzSiteCols* sites, const UnfzSegIn* segs,
                        const int32_t* seg_row_lo, const int64_t* seg_pair_off, int32_t n_segs,
                        int64_t n_pairs, const UnfzParams* h_params, uint8_t* out_class, void* stream);

/* Stable compaction of the class codes into per-DNM het_sites / candidate_sites lists (the sorted
 * lists find() returns, :341-342) + CNV votes (sv_phaser.py phase_by_snvs :71-85) + site marks.
 * Lists live at [seg_pair_off[dnm.seg_lo], ...): het_list[i] = row, cand_list[i] = row |
 * alt_is_dad<<31 | kid_alt<<30.  row_mark[row] = 1 for every het/candidate row of a READ-mode
 * segment. */
int unfz_compact_sites(UnfzCtx*, const UnfzDnm* dnms, int32_t n_dnms, const UnfzSegIn* segs,
                       const int32_t* seg_row_lo, const int64_t* seg_pair_off, const uint8_t* cls,
                       int32_t* het_list, int32_t* n_het, uint32_t* cand_list, int32_t* n_cand,
                       int32_t* cnv_dad, int32_t* cnv_mom, uint8_t* row_mark, void* stream);

/* Device-side completion of the site columns after an upload: the host table is plain SoA (gt / gq / rd / ad as
 * [3][n_rows] member planes, kid dad mom); this writes the packed rows of UnfzSiteCols (meta, rec, dep).  No
 * reference counterpart (cyvcf2 hands out per-record arrays, informative_site_finder.py:240-265). */
int unfz_pack_site_rows(UnfzCtx*, int64_t n_rows, const int32_t* pos, const uint8_t* flag, const uint8_t* gt,
                        const float* gq, const int32_t* rd, const int32_t* ad, uint32_t* meta, float* rec,
                        int32_t* dep, void* stream);

/* Device-side completion of the read columns after an upload: the host ships the positions of the (rare)
 * non-ACGT bases as a sorted list of base indices; this sets their bits in `nmask` (zeroed by the caller,
 * ceil(n_qual/32)+12 words) and bit7 of hdr[].aux of the reads that own them.  No reference counterpart
 * (pysam hands out query_sequence as a string). */
int unfz_expand_nlist(UnfzCtx*, const UnfzReadCols* reads, UnfzRead* hdr_rw, uint32_t* nmask_rw,
                      const int64_t* nidx, int64_t n_idx, void* stream);
/* ... and the dense start column of UnfzReadCols out of the headers.  The same pass marks the reads whose CIGAR is a
 * single M or = operation covering all l_seq bases (bit6 of hdr[].aux, written in place): for those, query index q
 * sits at reference position start + q and the allele lookup and the seed tests skip the CIGAR gather. */
int unfz_read_starts(UnfzCtx*, const UnfzReadCols* reads, int32_t* start_rw, void* stream);

/* Read scan: goodread :28-53, insert-size / None-count / CIGAR-op filters :181-203 :395-408,
 * reference_end and the number of marked site rows each read overlaps.
 * mark_prefix = exclusive scan of row_mark (n_rows+1 entries).
 * Hit slots: reads are processed in tiles of unfz_read_scan_tile_reads(max_l_seq) consecutive
 * reads; UnfzReadSum.hoff is the read's offset INSIDE its tile and tile_tot[tile] the tile's number
 * of hit words.  With tile_base = exclusive scan of tile_tot (unfz_exclusive_scan_u32), the hits of
 * read r live at hits[tile_base[r / tile_reads] + hoff, ... + cnt). */
int32_t unfz_read_scan_tile_reads(int32_t max_l_seq);
int unfz_read_scan(UnfzCtx*, const UnfzReadCols* reads, const UnfzSiteCols* sites,
                   const int32_t* mark_prefix, const UnfzParams* h_params,
                   int32_t max_l_seq /* longest read, 0 = unknown: picks the staging strategy */, UnfzReadSum* out,
                   int32_t* blk_maxspan /* [n_blocks], zeroed by the caller: max(end-start) */,
                   uint32_t* tile_tot /* [ceil(n_reads / tile_reads)] */,
                   uint32_t* tile_info /* [2 * n_tiles] or NULL: per tile {bit i: read i has hits, read block of the
                                          tile's first read}; lets the lookup skip reads without hits unseen */,
                   void* stream);

/* Read-by-site allele lookup: get_reference_positions(full_length=True).index(pos) + base +
 * quality for every (read x marked site) overlap (get_allele_at :56-73, phase_by_reads
 * snv_phaser.py:16-70).  Hit word: bits0-15 query index+1 (0: position not aligned),
 * bit16 base quality < --min-gt-qual, bit23 base is not ACGT, bits24-25 base code, bit26: index+1 < l_seq. */
int unfz_read_site_alleles(UnfzCtx*, const UnfzReadCols* reads, const UnfzSiteCols* sites,
                           const uint8_t* row_mark, const int32_t* mark_prefix,
                           const UnfzReadSum* rsum, const uint32_t* tile_base,
                           int32_t tile_reads, uint32_t* hits, const uint32_t* tile_info /* from unfz_read_scan, or NULL */,
                           void* stream);

/* Sizing pass of unfz_chain_tally: per DNM read window and scratch needs (need[6][n_dnms] int64:
 * window slots, het incidences, seed entries, seed incidences, het sites, candidate sites). */
int unfz_chain_size(UnfzCtx*, const UnfzDnm* dnms, int32_t n_dnms, const UnfzSegIn* segs,
                    const int64_t* seg_pair_off, const UnfzSiteCols* sites,
                    const UnfzReadCols* reads, const UnfzReadSum* rsum, const int32_t* blk_maxspan,
                    const int32_t* het_list, const int32_t* n_het, const uint32_t* cand_list,
                    const int32_t* n_cand, int32_t* win /* [4][n_dnms]: a_lo, a_hi, b_lo, b_hi */,
                    int64_t* need,
                    int32_t* site_lo, int32_t* site_n /* per het-list entry: candidate read range of fetch(pos, pos+1) */,
                    int32_t* seed_win /* [n_dnms][4]: candidate read ranges of the seed fetches */, void* stream);

/* Seed reads (collect_reads_snv :339-432), extended chaining (group_reads_by_haplotype :155-263,
 * connect_reads :76-152), site matching (site_searcher.py:6-78), phase_by_reads and the per-parent
 * evidence tally (snv_phaser.py:168-203).  One CTA per DNM.  slot_label / slot_evid / cand_evid must be
 * zero-filled by the caller (cand_evid padded to a multiple of 4 bytes).
 * off[6][n_dnms+1] are the exclusive scans of need[6][n_dnms] from unfz_chain_size. */
int unfz_chain_tally(UnfzCtx*, const UnfzDnm* dnms, int32_t n_dnms, const UnfzSegIn* segs,
                     const int64_t* seg_pair_off, const UnfzSiteCols* sites,
                     const UnfzReadCols* reads, const UnfzReadSum* rsum, const int32_t* blk_maxspan,
                     const uint32_t* hits, const uint32_t* hit_tile_base, int32_t hit_tile_reads,
                     const int32_t* mark_prefix,
                     const int32_t* het_list, const int32_t* n_het, const uint32_t* cand_list,
                     const int32_t* n_cand, const uint8_t* alleles, const int32_t* win,
                     const int32_t* site_lo, const int32_t* site_n, const int32_t* seed_win, const int64_t* off, const int64_t* h_totals /* off[k][n_dnms], k<6 */,
                     const UnfzParams* h_params, void* scratch, int64_t scratch_bytes,
                     uint8_t* slot_label, uint8_t* slot_evid, uint8_t* cand_evid,
                     UnfzTally* tally,
                     int64_t* ev_need /* [4][n_dnms] or NULL: list lengths for unfz_evidence_lists */,
                     void* stream);

/* The entries behind the tallies, per DNM, per parent and in order: what snv_phaser.py:169-203 puts into the record's
 * dad_reads / mom_reads (read index of the pair's window slot) and dad_sites / mom_sites (0-based position of the
 * informative site; duplicates of a site are kept, the reference builds a set).  ev_off[4][n_dnms+1] = exclusive
 * scans of ev_need (unfz_exclusive_scan_rows_i64), rows: dad pairs, mom pairs, dad sites, mom sites;
 * slot_off = row 0 of unfz_chain_tally's `off`. */
int unfz_evidence_lists(UnfzCtx*, const UnfzDnm* dnms, int32_t n_dnms, const int64_t* seg_pair_off,
                        const UnfzSiteCols* sites, const uint32_t* cand_list, const int32_t* n_cand,
                        const uint8_t* cand_evid, const int32_t* win, const int64_t* slot_off,
                        const uint8_t* slot_evid, const int64_t* ev_off, int32_t* ev_read_dad, int32_t* ev_read_mom,
                        int32_t* ev_pos_dad, int32_t* ev_pos_mom, void* stream);
int64_t unfz_chain_scratch_bytes(int64_t slots, int64_t incs, int64_t seeds, int64_t seed_incs,
                                 int64_t het_sites, int64_t cand_sites, int64_t n_dnms);

/* estimate_concordant_insert_len (read_collector.py:11-25): four order statistics (0-based ranks
 * h_ranks[4], HOST array) of |tlen - 2*readlen| over the reads of n_ranges index ranges
 * [first, first+count) (HOST arrays), selected exactly with a two-level radix histogram.  numpy's
 * percentile interpolates between two adjacent order statistics; the caller asks for the
 * neighbourhood of the 99.5th percentile's virtual index and lets numpy itself interpolate, so the
 * estimate is bit-identical to the reference's.  work: unfz_insert_size_work_bytes() bytes, zeroed
 * by the caller.  out[0..3] (device uint32) receive the values. */
int64_t unfz_insert_size_work_bytes(void);
int unfz_insert_size_order_stats(UnfzCtx*, const UnfzReadCols* reads, const int64_t* h_first, const int64_t* h_count,
                                 int32_t n_ranges, int32_t readlen, const uint64_t* h_ranks, void* work,
                                 uint32_t* out, void* stream);

/* Final call per DNM: unfazed.py summarize_record :190-334 on the tallies (+ autophase :162-187). */
int unfz_summarize(UnfzCtx*, const UnfzDnm* dnms, int32_t n_dnms, const UnfzTally* tally,
                   const int32_t* cnv_dad, const int32_t* cnv_mom, const int32_t* n_cand,
                   const UnfzParams* h_params,
                   UnfzCall* calls_strict, UnfzCall* calls_ambiguous, void* stream);

/* One batch, one call: the sequence window_search -> scan -> check_caps -> classify -> compact -> scan ->
 * [read_scan -> scan -> chain_size -> scan -> check_caps -> read_site_alleles -> chain_tally] -> summarize
 * on buffers the caller allocated from capacities (speculative sizing, see unfz_check_caps).  It exists
 * because a host language pays per call: ~40 ctypes calls cost more than the small kernels they launch.
 * All pointers are device pointers except h_params.  reads == NULL runs the site part only.  The flag
 * `guard` (zeroed by the caller) is installed for the duration of the call; actual[0] receives the pair
 * total, actual[1..6] the chaining totals, actual[7] the hit total. */
typedef struct {
    const UnfzSiteCols* sites;        /* HOST structs, as for the single entry points */
    const UnfzReadCols* reads;
    const UnfzParams*   h_params;
    const UnfzDnm*  dnms;     int32_t n_dnms;  int32_t n_segs;
    const UnfzSegIn* segs;    const uint8_t* alleles;
    int32_t max_l_seq;        int32_t tile_reads;
    int64_t n_tiles;
    int64_t cap_pairs, cap_hits, cap_chain[6];
    /* sized up front */
    int32_t* seg_row_lo;  int64_t* seg_count;  int64_t* seg_pair_off;  void* scan_work;
    uint8_t* row_mark;    int32_t* mark_prefix;
    int32_t* guard;       int64_t* actual;
    int32_t* n_het;  int32_t* n_cand;  int32_t* cnv_dad;  int32_t* cnv_mom;
    UnfzTally* tally;  UnfzCall* calls_strict;  UnfzCall* calls_ambiguous;  int32_t* win;
    int32_t* blk_maxspan;  int64_t* need;  int64_t* off;          /* off: 6*(n_dnms+1) + 1 entries */
    UnfzReadSum* rsum;  uint32_t* tile_tot;  uint32_t* tile_base;  uint32_t* tile_info;
    /* sized by cap_pairs */
    uint8_t* cls;  int32_t* het_list;  uint32_t* cand_list;  int32_t* site_lo;  int32_t* site_n;  int32_t* seed_win;
    uint8_t* cand_evid;
    /* sized by cap_hits / cap_chain */
    uint32_t* hits;  void* scratch;  int64_t scratch_bytes;  uint8_t* slot_label;  uint8_t* slot_evid;
    /* evidence lists (all NULL: not wanted).  ev_need 4*n_dnms, ev_off 4*(n_dnms+1); ev_read_* hold cap_chain[0]
     * entries each, ev_pos_* cap_pairs entries each (upper bounds of what can carry evidence) */
    int64_t* ev_need;  int64_t* ev_off;  int32_t* ev_read_dad;  int32_t* ev_read_mom;  int32_t* ev_pos_dad;  int32_t* ev_pos_mom;
} UnfzBatch;
int unfz_run_batch(UnfzCtx*, const UnfzBatch* h_batch, void* stream);

/* The same batch replayed as one CUDA graph: clears `n_zero` spans (the caller's zero-initialised buffers), runs the
 * sequence of unfz_run_batch and copies `d2h_bytes` from d_src to the (pinned) host address h_dst.  Captured once per
 * distinct set of arguments -- every pointer, capacity and parameter is part of the key -- and cached in the context
 * (8 graphs, least recently used evicted).  `stream` must be a non-default stream.  Asynchronous like everything else:
 * synchronise the stream before reading h_dst. */
typedef struct { void* ptr; int64_t bytes; } UnfzSpan;
int unfz_run_batch_graph(UnfzCtx*, const UnfzBatch* h_batch, const UnfzSpan* h_zero, int32_t n_zero,
                         void* h_dst, const void* d_src, int64_t d2h_bytes, void* stream);
int unfz_batch_struct_bytes(void);      /* sizeof(UnfzBatch), for bindings to check their mirror */

/* ---- BAM record decoding (csrc/bam.cu) ------------------------------------------------------------
 * Input: inflated BAM record bytes (BGZF blocks inflated on the host, records back to back, each starting with its
 * int32 block_size) and the byte offset of every record in that buffer.
 *
 * The fixed part of one record, as the parse step reads it (host and device share the code, so the two agree bit for
 * bit).  end is htslib's bam_endpos: pos + the reference length of the CIGAR, or pos + 1 for an unmapped read or one
 * without a reference-consuming operation.  aux: bit0 next_refID == refID, bit1 an SA tag among the aux fields (full
 * walk over all tag types), bit7 the record is malformed (its fields overrun block_size).  name_hash: 64-bit FNV-1a of
 * the read name without its NUL.  48 bytes. */
#define UNFZ_BAM_AUX_BAD 0x80
typedef struct {
    uint64_t name_hash;
    int32_t  ref_id;
    int32_t  pos;
    int32_t  end;
    int32_t  l_seq;
    int32_t  tlen;
    int32_t  next_ref_id;
    int32_t  next_pos;
    uint16_t flag;
    uint16_t n_cigar;
    uint8_t  mapq;
    uint8_t  aux;
    uint8_t  l_name;      /* read name length including the NUL */
    uint8_t  _pad;
    int32_t  ref_len;     /* sum of the reference-consuming CIGAR lengths, whatever the flag (may be 0) */
} UnfzBamRec;

/* Host only (no device call): the record boundaries of `buf` by walking block_size from byte 0.  Writes at most
 * max_records offsets, stops at a record that does not end inside the buffer and stores where the walk stopped in
 * *end_out.  Returns the number of offsets, or -1 for a block_size below the 32 bytes of the fixed fields. */
int64_t unfz_bam_record_offsets(const uint8_t* buf, int64_t n_bytes, int64_t max_records, int64_t* offs, int64_t* end_out);
/* Host only: the fixed fields of n records (the same function the device parse runs).  Returns the number of malformed
 * records (aux bit7). */
int64_t unfz_bam_parse_host(const uint8_t* buf, int64_t n_bytes, const int64_t* offs, int64_t n, UnfzBamRec* out);
/* Host only: dst <- the byte ranges [src[i], src[i] + len[i]) of buf back to back. */
int unfz_bam_gather_host(const uint8_t* buf, const int64_t* src, const int64_t* len, int64_t n, uint8_t* dst);

/* Device: unfz_bam_parse_host on the GPU, one thread per record (buf, offs, out in device memory). */
int unfz_bam_parse(UnfzCtx*, const uint8_t* buf, int64_t n_bytes, const int64_t* offs, int64_t n, UnfzBamRec* out,
                   void* stream);
/* Device: mate indices of n output reads as packers._mate_join defines them (same name, other segment bit, primary,
 * first in block order; -1 for an unpaired read or one whose mate is unmapped).  order: a stable sort of the reads by
 * (key_blk, key_hash) -- block and 64-bit name hash; flag: SAM flags; buf/src: the records, whose name bytes are compared
 * for every joined pair.  mate[i] = -2 leaves read i to the host: its candidate's name differs (a hash collision) or it
 * is its own candidate (both segment bits set). */
int unfz_bam_mate_join(UnfzCtx*, const int64_t* order, const int64_t* key_hash, const int32_t* key_blk, const int32_t* flag,
                       int64_t n, const uint8_t* buf, const int64_t* src, int32_t* mate, void* stream);
/* Device: the CIGAR words of the output reads.  reads->hdr holds the headers (cigar_off, n_cigar); src[r] is the byte
 * offset in buf of the record output read r is decoded from. */
int unfz_bam_emit_cigar(UnfzCtx*, const UnfzReadCols* reads, const uint8_t* buf, const int64_t* src, void* stream);
/* Device: the base planes of the output reads -- 2-bit bases (seq2), the low-quality plane of quality < min_bq (a
 * quality string starting with 0xFF counts as all zeros), and the non-ACGT plane (nmask) with aux bit7 of the reads that
 * own such a base: the device state unfz_expand_nlist leaves, so run it after unfz_read_starts (which clears aux bit7).
 * One thread per 32 output bases; the planes must be zeroed up to the padding DeviceReads gives them. */
int unfz_bam_emit_planes(UnfzCtx*, const UnfzReadCols* reads, const uint8_t* buf, const int64_t* src, int32_t min_bq,
                         void* stream);

/* ---- VCF text decoding (csrc/vcf.cu) ---------------------------------------------------------------
 * Input: the inflated text of the BGZF chunks of a tabix region query (whole lines, each ending in '\n').
 *
 * The fixed fields of one line, as the parse step reads it.  Offsets and lengths are relative to the line start;
 * line_len excludes the '\n' (and a '\r' before it).  rend is the end tabix indexes the record by: INFO END when it is
 * a number above pos0, else pos0 + ref_len.  n_alt: the ALT count (0 for ALT '.').  slot: the FORMAT index of GT, GQ,
 * AD, RO and AO, or -1.  fmt_off = -1: no FORMAT column.  flags: UNFZ_VCF_SIMPLE (one ALT of one base, REF of one base,
 * ALT not '*'), UNFZ_VCF_BAD (fewer than 8 columns, POS not a positive int32, END overflow).  chrom_hash: 32-bit FNV-1a
 * of CHROM.  64 bytes. */
#define UNFZ_VCF_SIMPLE 0x01
#define UNFZ_VCF_BAD 0x80
/* per-cell status bits of the sample decode */
#define UNFZ_VCF_CELL_HOST 0x01   /* GQ is a float off the exact fast path: gq holds the int32 line offset of its text */
#define UNFZ_VCF_CELL_BAD 0x02    /* a GT / GQ / AD / RO / AO value is malformed or overflows int32 */
typedef struct {
    int64_t  line_off;    /* byte offset of the line in the text */
    int32_t  line_len;
    int32_t  pos0;        /* POS - 1 */
    int32_t  rend;
    int32_t  chrom_len;
    uint32_t chrom_hash;
    int32_t  ref_off, ref_len;
    int32_t  alt_off, alt_len;
    int32_t  fmt_off, fmt_len;
    int32_t  n_alt;
    int8_t   slot[5];     /* GT GQ AD RO AO */
    uint8_t  ref0;        /* first byte of REF (0 when empty) */
    uint8_t  flags;
    uint8_t  _pad;
} UnfzVcfRec;

/* Host only: the positions of the '\n' bytes of buf (at most cap of them).  Returns their number, or -1 when cap is too
 * small.  The same per-16-byte-chunk code as the device pass. */
int64_t unfz_vcf_line_ends_host(const uint8_t* buf, int64_t n_bytes, int64_t cap, int64_t* ends);
/* Host only: the fixed fields of n_lines lines (line i spans ends[i-1] + 1 .. ends[i]).  Returns the number of lines
 * with UNFZ_VCF_BAD. */
int64_t unfz_vcf_parse_host(const uint8_t* buf, const int64_t* ends, int64_t n_lines, UnfzVcfRec* out);
/* Host only: the genotype fields of the selected lines sel[0..n_sel) (indices into recs).  slot_of[s]: the member column
 * of sample s, or -1 (n_samples entries).  Outputs are [n_sel][n_members]: gt (cyvcf2 gt_types), gq (GQ as float32,
 * -1 missing), rd (AD[0], or RO), ad (the sum of AD[1:], or of AO; -1 missing) and status (UNFZ_VCF_CELL_*); cells of
 * members without a column stay missing.  gq_float: the header declares GQ as Float (else Integer).  max_digits (<= 15):
 * significant digits a float may have on the fast path (0 sends every float to the host).  line_bad[i] = 1: line i has
 * more sample columns than n_samples. */
int unfz_vcf_samples_host(const uint8_t* buf, const UnfzVcfRec* recs, const int64_t* sel, int64_t n_sel,
                          const int32_t* slot_of, int32_t n_samples, int32_t n_members, int32_t gq_float, int32_t max_digits,
                          uint8_t* gt, float* gq, int32_t* rd, int32_t* ad, uint8_t* status, uint8_t* line_bad);
/* Number of 16-byte chunks of n_bytes: the length of the newline-count array (and of its scan, plus one). */
int64_t unfz_vcf_chunks(int64_t n_bytes);

/* Device: newline count of every 16-byte chunk of buf (cnt: unfz_vcf_chunks(n_bytes) entries). */
int unfz_vcf_line_count(UnfzCtx*, const uint8_t* buf, int64_t n_bytes, uint32_t* cnt, void* stream);
/* Device: the newline positions; at: the exclusive scan of the counts (unfz_exclusive_scan_u32, chunks + 1 entries). */
int unfz_vcf_line_write(UnfzCtx*, const uint8_t* buf, int64_t n_bytes, const uint32_t* at, int64_t* ends, void* stream);
/* Device: unfz_vcf_parse_host, one thread per line. */
int unfz_vcf_parse(UnfzCtx*, const uint8_t* buf, const int64_t* ends, int64_t n_lines, UnfzVcfRec* out, void* stream);
/* Device: unfz_vcf_samples_host, one warp per selected line.  buf must be 16-byte aligned and readable 16 bytes past
 * its end. */
int unfz_vcf_samples(UnfzCtx*, const uint8_t* buf, const UnfzVcfRec* recs, const int64_t* sel, int64_t n_sel,
                     const int32_t* slot_of, int32_t n_samples, int32_t n_members, int32_t gq_float, int32_t max_digits,
                     uint8_t* gt, float* gq, int32_t* rd, int32_t* ad, uint8_t* status, uint8_t* line_bad, void* stream);

/* ---- phased VCF output (csrc/vcfout.cu) --------------------------------------------------------------
 * Input: the body text and the UnfzVcfRec lines of unfz_vcf_line_ends_host / unfz_vcf_parse (or their device calls),
 * and the sparse edit list of the phased cells: edit_off[n_lines + 1] (CSR by line), edits sorted by (line, sample).
 *
 * Output per line: the text up to FORMAT verbatim; FORMAT with ":UOPS" / ":UET" appended unless present; then for every
 * header sample s, '\t' + the cell: every subfield of the output FORMAT, the cell's own text where it has one, '.'
 * where it dropped it, UOPS / UET = the edit's values (-1 without an edit); an absent trailing column is that of a
 * cell "."; a phase edit writes GT "1|0" (dad) or "0|1" (mom) followed by every allele past the second behind '|'.
 * A line without FORMAT passes through.  Every line ends in '\n' (a '\r' before it is dropped). */
#define UNFZ_VCFOUT_COLUMNS 0x01  /* line status: more sample columns than header samples */
#define UNFZ_VCFOUT_HAPLOID 0x02  /* line status: a phase edit on a GT without a separator */
#define UNFZ_VCFOUT_FIELDS 0x04   /* line status: a cell with more subfields than FORMAT keys */
typedef struct {
    int32_t sample;       /* sample column */
    int32_t phase;        /* 0 keep GT, 1 dad (1|0), 2 mom (0|1) */
    int32_t uops;         /* UOPS value */
    int32_t uet;          /* UET value */
} UnfzVcfEdit;

/* Host only: the output length of every line (int64, '\n' included) and its status (UNFZ_VCFOUT_*).  Returns the sum. */
int64_t unfz_vcf_rewrite_size_host(const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines, const int64_t* edit_off,
                                   const UnfzVcfEdit* edits, int32_t n_samples, int64_t* out_len, uint8_t* line_bad);
/* Host only: the output of every line at out_off[i] (the exclusive scan of out_len). */
int unfz_vcf_rewrite_write_host(const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines, const int64_t* edit_off,
                                const UnfzVcfEdit* edits, int32_t n_samples, const int64_t* out_off, uint8_t* out);
/* Device: unfz_vcf_rewrite_size_host, one warp per line.  buf must be 16-byte aligned and readable 16 bytes past its
 * end. */
int unfz_vcf_rewrite_size(UnfzCtx*, const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines, const int64_t* edit_off,
                          const UnfzVcfEdit* edits, int32_t n_samples, int64_t* out_len, uint8_t* line_bad, void* stream);
/* Device: unfz_vcf_rewrite_write_host, one warp per line (out_off from unfz_exclusive_scan_i64 of out_len). */
int unfz_vcf_rewrite_write(UnfzCtx*, const uint8_t* buf, const UnfzVcfRec* recs, int64_t n_lines, const int64_t* edit_off,
                           const UnfzVcfEdit* edits, int32_t n_samples, const int64_t* out_off, uint8_t* out, void* stream);

/* ---- BCF decoding (csrc/bcf.cu) ----------------------------------------------------------------------
 * Input: the inflated bytes of the BGZF chunks of a CSI region query (whole BCF 2.2 records back to back).
 *
 * The fixed fields of one record, as the parse step reads it.  Offsets are relative to rec_off (the record's l_shared).
 * rend = pos0 + rlen as stored.  ref / alt: the first two allele strings (alt_len 0 when n_allele < 2), NUL padding
 * dropped.  fmt_off: the first value of GT, GQ, AD, RO and AO (FORMAT keys given by the host as string-dictionary
 * indices), -1 when the record has no such field; fmt_ct: values per sample << 4 | BCF type.  Sample s's values of field
 * k start at rec_off + fmt_off[k] + s * count * width.  flags: UNFZ_BCF_SIMPLE (two alleles, REF and ALT of one base,
 * ALT not '*'), UNFZ_BCF_BAD with the reason bits.  80 bytes. */
#define UNFZ_BCF_SIMPLE 0x01
#define UNFZ_BCF_BAD_OVERRUN 0x02   /* a typed value runs past l_shared or l_indiv */
#define UNFZ_BCF_BAD_SAMPLES 0x04   /* n_sample differs from the header's sample count */
#define UNFZ_BCF_BAD_TYPE 0x08      /* a type BCF 2.2 does not define, or a key / count / allele of the wrong type */
#define UNFZ_BCF_BAD_POS 0x10       /* POS or rlen negative, or pos0 + rlen above INT32_MAX */
#define UNFZ_BCF_BAD 0x80
/* per-cell status bit of the sample decode: a reserved integer value, a GT / AD / RO / AO that is not an integer, a GQ
 * that is neither integer nor float, a negative GT value, or an AD / AO sum that overflows int32 */
#define UNFZ_BCF_CELL_BAD 0x02
typedef struct {
    int64_t  rec_off;     /* byte offset of the record in the buffer */
    int32_t  contig;      /* CHROM: index into the contig dictionary */
    int32_t  pos0;
    int32_t  rend;
    int32_t  ref_off, ref_len;
    int32_t  alt_off, alt_len;
    int32_t  fmt_off[5];  /* GT GQ AD RO AO */
    uint32_t fmt_ct[5];
    uint16_t n_allele;
    uint8_t  ref0;        /* first byte of REF (0 when empty) */
    uint8_t  flags;
} UnfzBcfRec;

/* Host only (no device call): the record boundaries of `buf` by walking l_shared + l_indiv from byte 0.  Writes at most
 * max_records offsets, stops at a record that does not end inside the buffer and stores where the walk stopped in
 * *end_out.  Returns the number of offsets, or -1 for an l_shared below the 24 bytes of the fixed fields. */
int64_t unfz_bcf_record_offsets(const uint8_t* buf, int64_t n_bytes, int64_t max_records, int64_t* offs, int64_t* end_out);
/* Host only: the fixed fields of the n records at offs (the same function the device parse runs).  keys: 5 host int32,
 * the string-dictionary indices of GT GQ AD RO AO (-1: not in the header); n_samples: the header's sample count.
 * Returns the number of records with UNFZ_BCF_BAD. */
int64_t unfz_bcf_parse_host(const uint8_t* buf, const int64_t* offs, int64_t n, const int32_t* keys, int32_t n_samples,
                            UnfzBcfRec* out);
/* Host only: the genotype fields of the selected records sel[0..n_sel) (indices into recs) for the member columns;
 * member_sample[m] is the sample of column m.  Outputs are [n_sel][n_members] with the contract of
 * unfz_vcf_samples_host: gt (cyvcf2 gt_types), gq (float32, -1 missing), rd (AD[0], or RO), ad (the sum of AD[1:], or
 * of AO; -1 missing) and status (UNFZ_BCF_CELL_BAD). */
int unfz_bcf_samples_host(const uint8_t* buf, const UnfzBcfRec* recs, const int64_t* sel, int64_t n_sel,
                          const int32_t* member_sample, int32_t n_members, uint8_t* gt, float* gq, int32_t* rd, int32_t* ad,
                          uint8_t* status);

/* Device: unfz_bcf_parse_host, one thread per record (buf, offs, out in device memory; keys in host memory). */
int unfz_bcf_parse(UnfzCtx*, const uint8_t* buf, const int64_t* offs, int64_t n, const int32_t* keys, int32_t n_samples,
                   UnfzBcfRec* out, void* stream);
/* Device: unfz_bcf_samples_host, one thread per (selected record x member) cell. */
int unfz_bcf_samples(UnfzCtx*, const uint8_t* buf, const UnfzBcfRec* recs, const int64_t* sel, int64_t n_sel,
                     const int32_t* member_sample, int32_t n_members, uint8_t* gt, float* gq, int32_t* rd, int32_t* ad,
                     uint8_t* status, void* stream);

/* ---- phased VCF output from BCF (csrc/bcfout.cu) ----------------------------------------------------------
 * Input: the inflated records and their UnfzBcfRec (unfz_bcf_parse_host / unfz_bcf_parse, no record with UNFZ_BCF_BAD);
 * the string and contig dictionaries as names (names + off[id] .. off[id + 1], empty for an unused id); keys: 3 host
 * int32, the string-dictionary ids of GT, UOPS and UET (-1: not in the header); and the sparse edit list of the phased
 * cells, edit_off[n_recs + 1] (CSR by record), edits sorted by (record, sample).
 *
 * Output per record, the VCF line htslib's vcf_format prints: CHROM, POS, ID, REF, ALT, QUAL, FILTER, INFO, and with
 * samples FORMAT (":UOPS" / ":UET" appended unless present; "." without FORMAT fields) and one cell per sample.  In a
 * cell UOPS / UET are the edit's values (-1 without an edit); a phase edit writes GT "1|0" (dad) or "0|1" (mom)
 * followed by every allele past the second behind '|'.  Floats are printed as "%g".  Every record ends in '\n'. */
#define UNFZ_BCFOUT_HAPLOID 0x01     /* record status: a phase edit on a GT of fewer than two alleles */
#define UNFZ_BCFOUT_FLOAT_HOST 0x02  /* record status: a float the device does not print (the host entry points do) */
#define UNFZ_BCFOUT_BAD 0x04         /* record status: an id outside a dictionary, or a value of a type it cannot have */

/* Host only: the output length of every record (int64, '\n' included) and its status (UNFZ_BCFOUT_*).  Returns the
 * sum.  Floats off the exact path are printed with snprintf("%g"). */
int64_t unfz_bcf_format_size_host(const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs, const uint8_t* str_names,
                                  const int64_t* str_off, int32_t n_str, const uint8_t* ctg_names, const int64_t* ctg_off,
                                  int32_t n_ctg, const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                                  int32_t n_samples, int64_t* out_len, uint8_t* status);
/* Host only: the output of every record at out_off[i] (the exclusive scan of out_len). */
int unfz_bcf_format_write_host(const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs, const uint8_t* str_names,
                               const int64_t* str_off, int32_t n_str, const uint8_t* ctg_names, const int64_t* ctg_off,
                               int32_t n_ctg, const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                               int32_t n_samples, const int64_t* out_off, uint8_t* out);
/* Device: unfz_bcf_format_size_host, one warp per record.  The length of a record with UNFZ_BCFOUT_FLOAT_HOST lacks its
 * floats: the caller takes it from the host entry point. */
int unfz_bcf_format_size(UnfzCtx*, const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs, const uint8_t* str_names,
                         const int64_t* str_off, int32_t n_str, const uint8_t* ctg_names, const int64_t* ctg_off,
                         int32_t n_ctg, const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                         int32_t n_samples, int64_t* out_len, uint8_t* status, void* stream);
/* Device: unfz_bcf_format_write_host, one warp per record (out_off from unfz_exclusive_scan_i64 of out_len).  Records
 * whose status (of the size step) has UNFZ_BCFOUT_FLOAT_HOST are skipped: the caller copies in the host's text. */
int unfz_bcf_format_write(UnfzCtx*, const uint8_t* buf, const UnfzBcfRec* recs, int64_t n_recs, const uint8_t* str_names,
                          const int64_t* str_off, int32_t n_str, const uint8_t* ctg_names, const int64_t* ctg_off,
                          int32_t n_ctg, const int32_t* keys, const int64_t* edit_off, const UnfzVcfEdit* edits,
                          int32_t n_samples, const uint8_t* status, const int64_t* out_off, uint8_t* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UNFAZED_SM100_H */
