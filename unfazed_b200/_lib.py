"""ctypes binding of ``libunfazed_sm100.so`` (C ABI declared in ``include/unfazed_sm100.h``).

There is deliberately no fallback: if the shared object is missing or a GPU is not present the
product path raises.  ``build()`` in ``__graft_entry__.py`` (or ``make -C unfazed_b200/csrc``)
produces the library in-tree.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# UNFZ_LIB selects another build of the same library (profiling variants, e.g. -DCH_DEBUG)
LIB_PATH = os.environ.get("UNFZ_LIB") or os.path.join(_HERE, "libunfazed_sm100.so")

c_void_p, c_int32, c_int64, c_double = C.c_void_p, C.c_int32, C.c_int64, C.c_double


class SiteCols(C.Structure):
    _fields_ = [
        ("n_rows", c_int64), ("n_blocks", c_int32), ("_pad", c_int32),
        ("blk_off", c_void_p), ("pos", c_void_p), ("ref", c_void_p), ("alt", c_void_p),
        ("meta", c_void_p), ("rec", c_void_p), ("dep", c_void_p),
    ]


class ReadCols(C.Structure):
    _fields_ = [
        ("n_reads", c_int64), ("n_blocks", c_int32), ("_pad", c_int32),
        ("blk_off", c_void_p), ("blk_sblk", c_void_p), ("blk_cul", c_void_p),
        ("hdr", c_void_p), ("start", c_void_p), ("cigar", c_void_p), ("lowq", c_void_p), ("nmask", c_void_p), ("seq2", c_void_p),
        ("n_qual", c_int64), ("n_cigar", c_int64),
    ]


class Params(C.Structure):
    _fields_ = [
        ("ab_homref", c_double * 2), ("ab_homalt", c_double * 2), ("ab_het", c_double * 2),
        ("min_gt_qual", c_double),
        ("min_depth", c_int32), ("min_map_qual", c_int32), ("readlen", c_int32),
        ("ext_read_goal", c_int32), ("no_extended", c_int32), ("evidence_min_ratio", c_int32),
        ("split_error_margin", c_int32), ("_pad", c_int32),
    ]


class Batch(C.Structure):
    """UnfzBatch of include/unfazed_sm100.h."""
    _fields_ = [
        ("sites", c_void_p), ("reads", c_void_p), ("h_params", c_void_p),
        ("dnms", c_void_p), ("n_dnms", c_int32), ("n_segs", c_int32),
        ("segs", c_void_p), ("alleles", c_void_p),
        ("max_l_seq", c_int32), ("tile_reads", c_int32),
        ("n_tiles", c_int64),
        ("cap_pairs", c_int64), ("cap_hits", c_int64), ("cap_chain", c_int64 * 6),
        ("seg_row_lo", c_void_p), ("seg_count", c_void_p), ("seg_pair_off", c_void_p), ("scan_work", c_void_p),
        ("row_mark", c_void_p), ("mark_prefix", c_void_p),
        ("guard", c_void_p), ("actual", c_void_p),
        ("n_het", c_void_p), ("n_cand", c_void_p), ("cnv_dad", c_void_p), ("cnv_mom", c_void_p),
        ("tally", c_void_p), ("calls_strict", c_void_p), ("calls_ambiguous", c_void_p), ("win", c_void_p),
        ("blk_maxspan", c_void_p), ("need", c_void_p), ("off", c_void_p),
        ("rsum", c_void_p), ("tile_tot", c_void_p), ("tile_base", c_void_p), ("tile_info", c_void_p),
        ("cls", c_void_p), ("het_list", c_void_p), ("cand_list", c_void_p), ("site_lo", c_void_p), ("site_n", c_void_p),
        ("seed_win", c_void_p), ("cand_evid", c_void_p),
        ("hits", c_void_p), ("scratch", c_void_p), ("scratch_bytes", c_int64), ("slot_label", c_void_p), ("slot_evid", c_void_p),
        ("ev_need", c_void_p), ("ev_off", c_void_p), ("ev_read_dad", c_void_p), ("ev_read_mom", c_void_p),
        ("ev_pos_dad", c_void_p), ("ev_pos_mom", c_void_p),
    ]


class Span(C.Structure):
    _fields_ = [("ptr", c_void_p), ("bytes", c_int64)]


SEG_DTYPE = np.dtype([
    ("sblk", "<i4"), ("lo_pos", "<i4"), ("hi_pos", "<i4"), ("mult", "<i4"),
    ("dnm", "<i4"), ("excl_lo", "<i4"), ("excl_hi", "<i4"), ("mode", "<i4"),
])
DNM_DTYPE = np.dtype([
    ("pos", "<i4"), ("end", "<i4"), ("rblk", "<i4"), ("kind", "<i4"), ("seg_lo", "<i4"), ("seg_hi", "<i4"),
    ("ref_off", "<i4"), ("ref_len", "<i4"), ("alt_off", "<i4"), ("alt_len", "<i4"),
    ("cnv_entry", "<i4"), ("flags", "<i4"),
])
TALLY_DTYPE = np.dtype([
    ("n_dad_sites", "<i4"), ("n_mom_sites", "<i4"), ("n_dad_reads", "<i4"), ("n_mom_reads", "<i4"),
    ("cnv_dad", "<i4"), ("cnv_mom", "<i4"), ("has_record", "<i4"), ("status", "<i4"),
])
CALL_DTYPE = np.dtype([("origin", "<i4"), ("evidence_count", "<i4"), ("evidence_types", "<i4"), ("emitted", "<i4")])
RSUM_DTYPE = np.dtype([("end", "<i4"), ("fmark", "<i4"), ("flags", "<u2"), ("cnt", "<u2"), ("hoff", "<u4"),
                       ("start", "<i4"), ("mate", "<i4"), ("row_lb", "<i4"), ("pad", "<i4")])
# UnfzBamRec: the fixed fields of one BAM record (csrc/bam.cu)
BAM_REC_DTYPE = np.dtype([("name_hash", "<u8"), ("ref_id", "<i4"), ("pos", "<i4"), ("end", "<i4"), ("l_seq", "<i4"),
                          ("tlen", "<i4"), ("next_ref_id", "<i4"), ("next_pos", "<i4"), ("flag", "<u2"), ("n_cigar", "<u2"),
                          ("mapq", "u1"), ("aux", "u1"), ("l_name", "u1"), ("_pad", "u1"), ("ref_len", "<i4")])
BAM_AUX_BAD = 0x80
assert BAM_REC_DTYPE.itemsize == 48
# UnfzVcfRec: the fixed fields of one VCF line (csrc/vcf.cu)
VCF_REC_DTYPE = np.dtype([("line_off", "<i8"), ("line_len", "<i4"), ("pos0", "<i4"), ("rend", "<i4"), ("chrom_len", "<i4"),
                          ("chrom_hash", "<u4"), ("ref_off", "<i4"), ("ref_len", "<i4"), ("alt_off", "<i4"),
                          ("alt_len", "<i4"), ("fmt_off", "<i4"), ("fmt_len", "<i4"), ("n_alt", "<i4"), ("slot", "i1", (5,)),
                          ("ref0", "u1"), ("flags", "u1"), ("_pad", "u1")])
VCF_SIMPLE, VCF_BAD, VCF_CELL_HOST, VCF_CELL_BAD = 0x01, 0x80, 0x01, 0x02
assert VCF_REC_DTYPE.itemsize == 64
# UnfzBcfRec: the fixed fields of one BCF record (csrc/bcf.cu)
BCF_REC_DTYPE = np.dtype([("rec_off", "<i8"), ("contig", "<i4"), ("pos0", "<i4"), ("rend", "<i4"), ("ref_off", "<i4"),
                          ("ref_len", "<i4"), ("alt_off", "<i4"), ("alt_len", "<i4"), ("fmt_off", "<i4", (5,)),
                          ("fmt_ct", "<u4", (5,)), ("n_allele", "<u2"), ("ref0", "u1"), ("flags", "u1")])
BCF_SIMPLE, BCF_BAD_OVERRUN, BCF_BAD_SAMPLES, BCF_BAD_TYPE, BCF_BAD_POS, BCF_BAD = 0x01, 0x02, 0x04, 0x08, 0x10, 0x80
BCF_CELL_BAD = 0x02
assert BCF_REC_DTYPE.itemsize == 80
# UnfzVcfEdit: one phased cell of the VCF writer (csrc/vcfout.cu)
VCF_EDIT_DTYPE = np.dtype([("sample", "<i4"), ("phase", "<i4"), ("uops", "<i4"), ("uet", "<i4")])
VCFOUT_COLUMNS, VCFOUT_HAPLOID, VCFOUT_FIELDS = 0x01, 0x02, 0x04
# record status of the BCF -> VCF formatter (csrc/bcfout.cu)
BCFOUT_HAPLOID, BCFOUT_FLOAT_HOST, BCFOUT_BAD = 0x01, 0x02, 0x04
assert VCF_EDIT_DTYPE.itemsize == 16
assert SEG_DTYPE.itemsize == 32 and DNM_DTYPE.itemsize == 48 and RSUM_DTYPE.itemsize == 32

# constants of include/unfazed_sm100.h
CLS_HET, CLS_CAND, CLS_ALT_IS_DAD, CLS_KID_ALT = 1, 2, 4, 8
MODE_READ, MODE_CNV_DEL, MODE_CNV_DUP, MODE_CNV_NA = 0, 1, 2, 3
KIND_SKIP, KIND_SNV, KIND_INDEL, KIND_SV = 0, 1, 2, 3
ORIGIN_NONE, ORIGIN_DAD, ORIGIN_MOM, ORIGIN_BOTH = 0, 1, 2, 3
EV_READBACKED, EV_ALLELE_BALANCE, EV_AMBIG_READBACKED, EV_AMBIG_ALLELE_BAL, EV_AMBIG_BOTH, EV_SEX_CHROM = 1, 2, 4, 8, 16, 32
DNM_AUTOPHASE, DNM_AUTOPHASE_Y, DNM_SV_QUIRK, DNM_FALLBACK_FETCH = 1, 2, 4, 8
ABI_VERSION = 2
RS_GOOD_CONC, RS_GOOD_DISC, RS_NONE_OK, RS_EXT_OK, RS_INS_OK, RS_HAS_MATE = 1, 2, 4, 8, 16, 32

# every symbol the header declares: (name, restype, argtypes)
_P = c_void_p
SYMBOLS = {
    "unfz_abi_version": (C.c_int, []),
    "unfz_ctx_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "unfz_ctx_destroy": (None, [_P]),
    "unfz_last_error": (C.c_char_p, [_P]),
    "unfz_ctx_set_guard": (C.c_int, [_P, _P]),
    "unfz_check_caps": (C.c_int, [_P, c_int32, _P, _P, _P, _P, _P]),
    "unfz_run_batch": (C.c_int, [_P, C.POINTER(Batch), _P]),
    "unfz_run_batch_graph": (C.c_int, [_P, C.POINTER(Batch), _P, c_int32, _P, _P, c_int64, _P]),
    "unfz_batch_struct_bytes": (C.c_int, []),
    "unfz_scan_work_bytes": (c_int64, [c_int64]),
    "unfz_exclusive_scan_i64": (C.c_int, [_P, _P, _P, c_int64, _P, _P]),
    "unfz_exclusive_scan_u8_i32": (C.c_int, [_P, _P, _P, c_int64, _P, _P]),
    "unfz_exclusive_scan_u32": (C.c_int, [_P, _P, _P, c_int64, _P, _P, _P]),
    "unfz_exclusive_scan_rows_i64": (C.c_int, [_P, _P, _P, c_int32, c_int64, _P]),
    "unfz_window_search": (C.c_int, [_P, C.POINTER(SiteCols), _P, c_int32, _P, _P, _P]),
    "unfz_classify_sites": (C.c_int, [_P, C.POINTER(SiteCols), _P, _P, _P, c_int32, c_int64, C.POINTER(Params), _P, _P]),
    "unfz_compact_sites": (C.c_int, [_P, _P, c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "unfz_pack_site_rows": (C.c_int, [_P, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "unfz_expand_nlist": (C.c_int, [_P, C.POINTER(ReadCols), _P, _P, _P, c_int64, _P]),
    "unfz_read_scan_tile_reads": (c_int32, [c_int32]),
    "unfz_read_scan": (C.c_int, [_P, C.POINTER(ReadCols), C.POINTER(SiteCols), _P, C.POINTER(Params), c_int32, _P, _P, _P, _P, _P]),
    "unfz_read_site_alleles": (C.c_int, [_P, C.POINTER(ReadCols), C.POINTER(SiteCols), _P, _P, _P, _P, c_int32, _P, _P, _P]),
    "unfz_read_starts": (C.c_int, [_P, C.POINTER(ReadCols), _P, _P]),
    "unfz_chain_size": (C.c_int, [_P, _P, c_int32, _P, _P, C.POINTER(SiteCols), C.POINTER(ReadCols), _P, _P,
                                  _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "unfz_chain_scratch_bytes": (c_int64, [c_int64] * 7),
    "unfz_chain_tally": (C.c_int, [_P, _P, c_int32, _P, _P, C.POINTER(SiteCols), C.POINTER(ReadCols), _P, _P, _P, _P, c_int32, _P,
                                   _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(Params), _P, c_int64,
                                   _P, _P, _P, _P, _P, _P]),
    "unfz_evidence_lists": (C.c_int, [_P, _P, c_int32, _P, C.POINTER(SiteCols), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "unfz_insert_size_work_bytes": (c_int64, []),
    "unfz_insert_size_order_stats": (C.c_int, [_P, C.POINTER(ReadCols), _P, _P, c_int32, c_int32, _P, _P, _P, _P]),
    "unfz_summarize": (C.c_int, [_P, _P, c_int32, _P, _P, _P, _P, C.POINTER(Params), _P, _P, _P]),
    "unfz_bam_record_offsets": (c_int64, [_P, c_int64, c_int64, _P, _P]),
    "unfz_bam_parse_host": (c_int64, [_P, c_int64, _P, c_int64, _P]),
    "unfz_bam_gather_host": (C.c_int, [_P, _P, _P, c_int64, _P]),
    "unfz_bam_parse": (C.c_int, [_P, _P, c_int64, _P, c_int64, _P, _P]),
    "unfz_bam_mate_join": (C.c_int, [_P, _P, _P, _P, _P, c_int64, _P, _P, _P, _P]),
    "unfz_bam_emit_cigar": (C.c_int, [_P, C.POINTER(ReadCols), _P, _P, _P]),
    "unfz_bam_emit_planes": (C.c_int, [_P, C.POINTER(ReadCols), _P, _P, c_int32, _P]),
    "unfz_vcf_line_ends_host": (c_int64, [_P, c_int64, c_int64, _P]),
    "unfz_vcf_parse_host": (c_int64, [_P, _P, c_int64, _P]),
    "unfz_vcf_samples_host": (C.c_int, [_P, _P, _P, c_int64, _P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, _P]),
    "unfz_vcf_chunks": (c_int64, [c_int64]),
    "unfz_vcf_line_count": (C.c_int, [_P, _P, c_int64, _P, _P]),
    "unfz_vcf_line_write": (C.c_int, [_P, _P, c_int64, _P, _P, _P]),
    "unfz_vcf_parse": (C.c_int, [_P, _P, _P, c_int64, _P, _P]),
    "unfz_vcf_samples": (C.c_int, [_P, _P, _P, _P, c_int64, _P, c_int32, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P, _P,
                                   _P]),
    "unfz_vcf_rewrite_size_host": (c_int64, [_P, _P, c_int64, _P, _P, c_int32, _P, _P]),
    "unfz_vcf_rewrite_write_host": (C.c_int, [_P, _P, c_int64, _P, _P, c_int32, _P, _P]),
    "unfz_vcf_rewrite_size": (C.c_int, [_P, _P, _P, c_int64, _P, _P, c_int32, _P, _P, _P]),
    "unfz_vcf_rewrite_write": (C.c_int, [_P, _P, _P, c_int64, _P, _P, c_int32, _P, _P, _P]),
    "unfz_bcf_record_offsets": (c_int64, [_P, c_int64, c_int64, _P, _P]),
    "unfz_bcf_parse_host": (c_int64, [_P, _P, c_int64, _P, c_int32, _P]),
    "unfz_bcf_samples_host": (C.c_int, [_P, _P, _P, c_int64, _P, c_int32, _P, _P, _P, _P, _P]),
    "unfz_bcf_parse": (C.c_int, [_P, _P, _P, c_int64, _P, c_int32, _P, _P]),
    "unfz_bcf_samples": (C.c_int, [_P, _P, _P, _P, c_int64, _P, c_int32, _P, _P, _P, _P, _P, _P]),
    "unfz_bcf_format_size_host": (c_int64, [_P, _P, c_int64, _P, _P, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, _P, _P]),
    "unfz_bcf_format_write_host": (C.c_int, [_P, _P, c_int64, _P, _P, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, _P, _P]),
    "unfz_bcf_format_size": (C.c_int, [_P, _P, _P, c_int64, _P, _P, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, _P, _P,
                                       _P]),
    "unfz_bcf_format_write": (C.c_int, [_P, _P, _P, c_int64, _P, _P, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, _P, _P,
                                        _P, _P]),
}

_lib = None


class LibraryMissing(RuntimeError):
    pass


def load():
    """Load the shared object (once).  Raises LibraryMissing -- never falls back to a CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C unfazed_b200/csrc`" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.unfz_abi_version() != ABI_VERSION:
        raise LibraryMissing("ABI version mismatch in %s" % LIB_PATH)
    if lib.unfz_batch_struct_bytes() != C.sizeof(Batch):
        raise LibraryMissing("UnfzBatch layout mismatch between %s and _lib.Batch" % LIB_PATH)
    _lib = lib
    return lib
