"""ctypes binding of include/metacov_b200.h.

The product path has no CPU fallback: if the native library is missing this
module raises at import time, and if there is no CUDA device ``mcov_create``
fails and ``McovError`` is raised.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmetacov_b200.so")

MCOV_OK = 0
MCOV_ERR_ARG = -1
MCOV_ERR_STATE = -2
MCOV_ERR_CUDA = -3
MCOV_ERR_NOMEM = -4
MCOV_ERR_IO = -5
MCOV_ERR_RANGE = -6
MCOV_ERR_UNSORTED = -7
MCOV_BEGIN_EXACT_CAP = 1     # mcov_begin_ex: the any-order pass reports the exact cap metric
MEM_HOST = 0
MEM_DEVICE = 1
MCOV_BC_ALL = 0              # mcov_base_counts: pysam's read_callback="all" (skip flags 0x4 | 0x100 | 0x200 | 0x400)
MCOV_BC_NOFILTER = 1         # read_callback="nofilter"

_STATUS_NAMES = {
    MCOV_ERR_ARG: "MCOV_ERR_ARG", MCOV_ERR_STATE: "MCOV_ERR_STATE", MCOV_ERR_CUDA: "MCOV_ERR_CUDA",
    MCOV_ERR_NOMEM: "MCOV_ERR_NOMEM", MCOV_ERR_IO: "MCOV_ERR_IO", MCOV_ERR_RANGE: "MCOV_ERR_RANGE",
    MCOV_ERR_UNSORTED: "MCOV_ERR_UNSORTED",
}


class McovError(RuntimeError):
    def __init__(self, code, message=""):
        self.code = code
        super().__init__("%s (%d): %s" % (_STATUS_NAMES.get(code, "MCOV_ERR"), code, message))


class Filter(C.Structure):
    """mcov_filter: pysam's implicit pileup arguments (SURVEY.md Appendix A-1)."""
    _fields_ = [("flag_filter", C.c_uint16), ("flag_require", C.c_uint16), ("min_mapq", C.c_uint8),
                ("ignore_orphans", C.c_uint8), ("count_del", C.c_uint8), ("reflen0_as_one", C.c_uint8), ("max_depth", C.c_int32)]


class RegionStats(C.Structure):
    _fields_ = [("sum", C.c_int64), ("sumsq", C.c_uint64), ("iq_sum", C.c_int64), ("n_ge1", C.c_int64),
                ("n_geN", C.c_int64), ("min", C.c_int32), ("max", C.c_int32), ("med_lo", C.c_int32),
                ("med_hi", C.c_int32), ("reserved", C.c_int32), ("flags", C.c_int32)]


HIST_BINS = 8192        # MCOV_HIST_BINS

REGION_STATS_DTYPE = np.dtype([
    ("sum", "<i8"), ("sumsq", "<u8"), ("iq_sum", "<i8"), ("n_ge1", "<i8"), ("n_geN", "<i8"),
    ("min", "<i4"), ("max", "<i4"), ("med_lo", "<i4"), ("med_hi", "<i4"), ("reserved", "<i4"), ("flags", "<i4")])
assert REGION_STATS_DTYPE.itemsize == C.sizeof(RegionStats) == 64


class AlleleParams(C.Structure):
    """mcov_allele_params."""
    _fields_ = [("min_coverage", C.c_uint32), ("min_count", C.c_uint32), ("min_freq", C.c_double),
                ("use_reference", C.c_int32), ("pad", C.c_int32)]


ALLELE_STATS_DTYPE = np.dtype([
    ("length", "<i8"), ("covered", "<i8"), ("depth_sum", "<i8"), ("pi_sum", "<f8"), ("snv", "<i8"),
    ("ref_covered", "<i8"), ("sub", "<i8"), ("popsub", "<i8")])
assert ALLELE_STATS_DTYPE.itemsize == 64      # mcov_allele_stats

# mcov_allele_site: the counts as A C G T, ref / consensus as one ASCII letter, kind bits (1 SNV, 2 SUB, 4 POPSUB)
ALLELE_SITE_DTYPE = np.dtype({
    "names": ["tid", "pos", "A", "C", "G", "T", "ref", "consensus", "kind"],
    "formats": ["<i4", "<i4", "<u4", "<u4", "<u4", "<u4", "S1", "S1", "u1"],
    "offsets": [0, 4, 8, 12, 16, 20, 24, 25, 26], "itemsize": 32})
ALLELE_SNV, ALLELE_SUB, ALLELE_POPSUB = 1, 2, 4

COMPARE_STATS_DTYPE = np.dtype([
    ("length", "<i8"), ("covered_a", "<i8"), ("covered_b", "<i8"), ("compared", "<i8"), ("con_snp", "<i8"),
    ("pop_snp", "<i8")])
assert COMPARE_STATS_DTYPE.itemsize == 48     # mcov_compare_stats

# mcov_compare_site: the pair's index, the position, both signature bytes (0x80 covered, bits 4-5 consensus, bits 0-3
# present mask), kind bits (1 con_snp, 2 pop_snp), pad (always 0).  The pad is a field so that every byte of a record
# is defined: numpy leaves the gaps of a structured dtype uninitialised when it copies records (e.g. by a mask), and a
# site list's bytes are then not comparable.
COMPARE_SITE_DTYPE = np.dtype([("pair", "<i4"), ("tid", "<i4"), ("pos", "<i4"), ("sig_a", "u1"), ("sig_b", "u1"),
                               ("kind", "u1"), ("pad", "u1")])
assert COMPARE_SITE_DTYPE.itemsize == 16      # mcov_compare_site
COMPARE_CON_SNP, COMPARE_POP_SNP = 1, 2


class LinkageParams(C.Structure):
    """mcov_linkage_params."""
    _fields_ = [("sites", AlleleParams), ("max_distance", C.c_int32), ("min_reads", C.c_uint32)]


class LinkageInfo(C.Structure):
    """mcov_linkage_info."""
    _fields_ = [("n_sites", C.c_int64), ("n_observations", C.c_int64), ("n_units", C.c_int64), ("n_candidates", C.c_int64)]


# mcov_linkage_pair: the two sites, their major / minor alleles as ASCII letters, the four haplotype counts (upper case
# = the major allele)
LINKAGE_PAIR_DTYPE = np.dtype([("tid", "<i4"), ("pos_a", "<i4"), ("pos_b", "<i4"), ("major_a", "S1"), ("minor_a", "S1"),
                               ("major_b", "S1"), ("minor_b", "S1"), ("n_AB", "<u4"), ("n_Ab", "<u4"), ("n_aB", "<u4"),
                               ("n_ab", "<u4")])
assert LINKAGE_PAIR_DTYPE.itemsize == 32 and C.sizeof(LinkageParams) == 32      # mcov_linkage_pair, mcov_linkage_params

GENE_STATS_DTYPE = np.dtype([(name, "<i8") for name in (
    "length", "codons", "codons_called", "n_sites3", "s_sites3", "snv_n", "snv_s", "snv_m", "sub_n", "sub_s", "sub_m",
    "pad")])
assert GENE_STATS_DTYPE.itemsize == 96        # mcov_gene_stats

# mcov_gene_site: the gene's index, the position, the codon and the position in it (0-2 from the 5' end), the reference
# codon in gene orientation, major / minor allele in genomic orientation, the amino acids, kind bits (1 SNV, 2 SUB), the
# types 'N' 'S' 'M' (b"" where a field does not apply)
GENE_SITE_DTYPE = np.dtype([("gene", "<i8"), ("tid", "<i4"), ("pos", "<i4"), ("codon", "<i4"), ("codon_pos", "u1"),
                            ("ref_codon", "S3"), ("major", "S1"), ("minor", "S1"), ("aa_ref", "S1"), ("aa_major", "S1"),
                            ("aa_minor", "S1"), ("kind", "u1"), ("snv_type", "S1"), ("sub_type", "S1")])
assert GENE_SITE_DTYPE.itemsize == 32         # mcov_gene_site
GENE_SNV, GENE_SUB = 1, 2


class BamGpuStreamInfo(C.Structure):
    _fields_ = [("n_records", C.c_int64), ("n_chunks", C.c_int64), ("n_segments", C.c_int64), ("inflated_bytes", C.c_int64),
                ("file_bytes", C.c_int64), ("max_carry", C.c_int64)]


class BamDev(C.Structure):
    """mcov_bam_dev: device-resident SoA of a BAM decoded on the GPU."""
    _fields_ = [("n_records", C.c_int64), ("n_cigar", C.c_int64), ("inflated_bytes", C.c_int64), ("header_bytes", C.c_int64),
                ("n_segments", C.c_int64), ("n_ref", C.c_int32), ("reserved", C.c_int32),
                ("tid", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("l_seq", C.c_void_p),
                ("isize", C.c_void_p), ("cig_off", C.c_void_p), ("cig", C.c_void_p), ("inflated", C.c_void_p)]


class SamHostCols(C.Structure):
    """mcov_sam_host_cols: columns of the host-compiled SAM rules (test hook mcov_sam_parse_host)."""
    _fields_ = [("n_records", C.c_int64), ("n_cigar", C.c_int64), ("header_bytes", C.c_int64), ("fail_line", C.c_int64),
                ("n_ref", C.c_int32), ("fail_field", C.c_int32), ("k_len", C.c_int32), ("win_bases", C.c_int32),
                ("tid", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("l_seq", C.c_void_p),
                ("isize", C.c_void_p), ("cig_off", C.c_void_p), ("cig", C.c_void_p), ("name_hash", C.c_void_p),
                ("kmer_code", C.c_void_p), ("seq_win", C.c_void_p)]


class BamBatch(C.Structure):
    """mcov_bam_batch: one batch of the streaming host reader (pinned SoA views)."""
    _fields_ = [("n", C.c_int64), ("n_carry", C.c_int64), ("n_cigar", C.c_int64), ("last", C.c_int32), ("reserved", C.c_int32),
                ("tid", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("l_seq", C.c_void_p),
                ("isize", C.c_void_p), ("reflen", C.c_void_p), ("cig_off", C.c_void_p), ("cig", C.c_void_p)]


class PassInfo(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("n_pass", C.c_int64), ("aligned_bases", C.c_int64),
                ("max_depth_seen", C.c_int32), ("cap_metric", C.c_int32), ("sorted", C.c_int32),
                ("cap_contigs", C.c_int32)]


EXP_STATS_DTYPE = np.dtype([
    ("covw_sum", "<f8"), ("cor_sum", "<f8"), ("wnf_sum", "<f8"), ("cov_sum", "<i8"), ("cov2_sum", "<i8"),
    ("n_starts", "<i4"), ("nreads", "<i4"), ("secondary", "<i4"), ("improper", "<i4"), ("no_reflen", "<i4"),
    ("n_pairs", "<i4")])
assert EXP_STATS_DTYPE.itemsize == 64      # mcov_exp_stats


class KernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_int64), ("total_ms", C.c_double)]


class SynthParams(C.Structure):
    """mcov_synth_params (include/mcov_synth.h)."""
    _fields_ = [("seed", C.c_uint64), ("mode", C.c_int32), ("read_len", C.c_int32), ("span_min", C.c_int32),
                ("span_max", C.c_int32), ("margin", C.c_int32), ("reserved", C.c_int32)]


_vp = C.c_void_p
_i32, _i64 = C.c_int32, C.c_int64

# name -> (restype, argtypes); every symbol include/metacov_b200.h declares
SIGNATURES = {
    "mcov_create": (C.c_int, [C.POINTER(_vp), C.c_int, _vp]),
    "mcov_destroy": (None, [_vp]),
    "mcov_last_error": (C.c_char_p, [_vp]),
    "mcov_abi_version": (C.c_int, []),
    "mcov_set_contigs": (C.c_int, [_vp, _i32, _vp]),
    "mcov_n_slots": (_i64, [_vp]),
    "mcov_contig_offset": (_i64, [_vp, _i32]),
    "mcov_bind_depth": (C.c_int, [_vp, _vp, _i64]),
    "mcov_set_filter": (C.c_int, [_vp, C.POINTER(Filter)]),
    "mcov_default_filter": (None, [C.POINTER(Filter)]),
    "mcov_begin": (C.c_int, [_vp]),
    "mcov_begin_ex": (C.c_int, [_vp, C.c_int]),
    "mcov_push_reads": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    "mcov_finalize": (C.c_int, [_vp]),
    "mcov_depth_sorted": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    "mcov_depth_sorted_wide": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "mcov_push_reads_wide": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    "mcov_stream_begin": (C.c_int, [_vp]),
    "mcov_stream_push": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int,
                                   C.POINTER(_i32), C.POINTER(_i32)]),
    "mcov_stream_resend_point": (C.c_int, [_vp, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32)]),
    "mcov_block_bound": (_i64, [_i64, _i64, _i32]),
    "mcov_pack_block": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _i64, C.POINTER(_i64), C.c_int]),
    "mcov_depth_sorted_block": (C.c_int, [_vp, _vp, _i64, C.c_int]),
    "mcov_stream_push_block": (C.c_int, [_vp, _vp, _i64, C.c_int, C.POINTER(_i32), C.POINTER(_i32)]),
    "mcov_block_unpack": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mcov_depth_sorted_async": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int]),
    "mcov_depth_sorted_packed": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, C.c_int]),
    "mcov_depth_sorted_delta": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "mcov_region_stats_run": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp]),
    "mcov_region_stats_submit": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, C.c_int]),
    "mcov_region_stats_collect": (C.c_int, [_vp, C.c_int, _vp]),
    "mcov_sync": (C.c_int, [_vp]),
    "mcov_copy_to_host": (C.c_int, [_vp, _vp, _vp, C.c_int64]),
    "mcov_bam_decode_gpu": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "mcov_bam_decode_gpu_file": (C.c_int, [_vp, C.c_char_p, C.c_int, _vp]),
    "mcov_bam_gpu_names_seq": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, C.c_int]),
    "mcov_bam_gpu_stream_depth": (C.c_int, [_vp, C.c_char_p, _i64, C.c_int, _vp]),
    "mcov_sam_decode_gpu": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, _vp]),
    "mcov_sam_decode_gpu_file": (C.c_int, [_vp, C.c_char_p, C.c_int64, _vp]),
    "mcov_sam_chunk_begin": (C.c_int, [_vp, _vp, C.c_int64, C.POINTER(_i32)]),
    "mcov_sam_chunk_decode": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, C.POINTER(_i64), _vp]),
    "mcov_sam_chunk_longest_line": (_i64, [_vp]),
    "mcov_bam_gpu_mapped": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "mcov_base_counts": (C.c_int, [_vp, C.c_char_p, _i64, _i32, C.c_int]),
    "mcov_copy_base_counts": (C.c_int, [_vp, _i32, _i32, _i32, _vp]),
    "mcov_set_reference": (C.c_int, [_vp, _i32, C.c_char_p, _i32]),
    "mcov_allele_stats_run": (C.c_int, [_vp, _i64, _vp, _vp, _vp, C.POINTER(AlleleParams), _vp]),
    "mcov_allele_sites": (C.c_int, [_vp, C.POINTER(AlleleParams), C.POINTER(_i64)]),
    "mcov_allele_sites_read": (C.c_int, [_vp, _i64, _i64, _vp]),
    "mcov_allele_signature": (C.c_int, [_vp, C.POINTER(AlleleParams), _vp]),
    "mcov_compare_run": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i64, _vp, _vp, _vp, _vp]),
    "mcov_compare_sites": (C.c_int, [_vp, _i32, _vp, _i32, _vp, C.POINTER(_i64)]),
    "mcov_compare_sites_read": (C.c_int, [_vp, _i64, _i64, _vp]),
    "mcov_linkage": (C.c_int, [_vp, C.c_char_p, _i64, C.POINTER(LinkageParams), C.POINTER(_i64), C.POINTER(LinkageInfo)]),
    "mcov_linkage_read": (C.c_int, [_vp, _i64, _i64, _vp]),
    "mcov_gene_run": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, C.POINTER(AlleleParams), _vp, C.POINTER(_i64)]),
    "mcov_gene_sites_read": (C.c_int, [_vp, _i64, _i64, _vp]),
    "mcov_sam_parse_host": (C.c_int, [_vp, C.c_int64, C.POINTER(SamHostCols), C.c_char_p, C.c_int]),
    "mcov_inflate_host": (C.c_int, [_vp, C.c_uint32, _vp, C.c_uint32]),
    "mcov_inflate_host_win": (C.c_int, [_vp, C.c_uint32, _vp, C.c_uint32, C.c_uint32]),
    "mcov_crc32_host": (C.c_uint32, [_vp, C.c_uint32]),
    "mcov_crc32_sliced_host": (C.c_uint32, [_vp, C.c_uint32, C.c_int]),
    "mcov_depth_runs": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "mcov_depth_runs_read": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp]),
    "mcov_region_hist_enqueue": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp, _vp]),
    "mcov_hist_stats_enqueue": (C.c_int, [_vp, C.c_int64, _vp, C.c_int32, _vp]),
    "mcov_region_stats_collect_view": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "mcov_region_stats_enqueue": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp]),
    "mcov_window_means": (C.c_int, [_vp, _i32, _vp, _i64]),
    "mcov_copy_depth": (C.c_int, [_vp, _i32, _i32, _i32, _vp]),
    "mcov_depth_ptr": (_vp, [_vp]),
    "mcov_pass_info_get": (C.c_int, [_vp, C.POINTER(PassInfo)]),
    "mcov_launch_count": (_i64, [_vp]),
    "mcov_region_plan_info": (C.c_int, [_vp, _vp, _vp]),
    "mcov_profile_enable": (C.c_int, [_vp, C.c_int]),
    "mcov_profile_read": (C.c_int, [_vp, C.POINTER(KernelTime), C.c_int]),
    "mcov_isize_hist": (C.c_int, [_vp, _i64, _vp, _vp, C.c_int, _i32, _vp, _i32, _vp, _vp, _vp]),
    "mcov_kmer_hist": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "mcov_kmer_hist_mem": (C.c_int, [_vp, _i64, _vp, _vp, _vp, C.c_int, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "mcov_bam_load_seq": (C.c_int, [_vp]),
    "mcov_bam_seq_windows": (C.c_int, [_vp, _i32, _vp]),
    "mcov_bam_name_hash": (_vp, [_vp]),
    "mcov_bam_qas_kmer": (C.c_int, [_vp, _i32, _vp]),
    "mcov_experimental_run": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp,
                                        _i32, _vp, _vp, _vp, _vp, _vp]),
    "mcov_exp_revsum": (C.c_int, [_vp, _i64, _vp, _i32, _vp, _vp]),
    "mcov_bam_open": (C.c_int, [C.POINTER(_vp), C.c_char_p, C.c_char_p, C.c_int]),
    "mcov_bam_close": (None, [_vp]),
    "mcov_bam_n_ref": (_i32, [_vp]),
    "mcov_bam_ref_name": (C.c_char_p, [_vp, _i32]),
    "mcov_bam_ref_len": (_i32, [_vp, _i32]),
    "mcov_bam_header_text": (C.c_char_p, [_vp]),
    "mcov_bam_index_stats": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "mcov_bai_stats": (C.c_int, [C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "mcov_bam_load": (C.c_int, [_vp, C.c_int]),
    "mcov_bam_n_records": (_i64, [_vp]),
    "mcov_bam_n_cigar": (_i64, [_vp]),
    "mcov_bam_tid": (_vp, [_vp]),
    "mcov_bam_pos": (_vp, [_vp]),
    "mcov_bam_flag": (_vp, [_vp]),
    "mcov_bam_mapq": (_vp, [_vp]),
    "mcov_bam_lseq": (_vp, [_vp]),
    "mcov_bam_isize": (_vp, [_vp]),
    "mcov_bam_cig_off": (_vp, [_vp]),
    "mcov_bam_cig": (_vp, [_vp]),
    "mcov_bam_stream_open": (C.c_int, [C.POINTER(_vp), C.c_char_p, _i64, C.c_int, C.c_char_p, C.c_int]),
    "mcov_bam_stream_close": (None, [_vp]),
    "mcov_bam_stream_n_ref": (_i32, [_vp]),
    "mcov_bam_stream_ref_name": (C.c_char_p, [_vp, _i32]),
    "mcov_bam_stream_ref_len": (_i32, [_vp, _i32]),
    "mcov_bam_stream_header_text": (C.c_char_p, [_vp]),
    "mcov_bam_stream_error": (C.c_char_p, [_vp]),
    "mcov_bam_stream_next": (C.c_int, [_vp, _i32, _i32, C.POINTER(BamBatch)]),
    "mcov_bam_stream_records": (_i64, [_vp]),
    "mcov_bam_stream_next_block": (C.c_int, [_vp, _i32, _i32, C.c_int, C.POINTER(_vp), C.POINTER(_i64), C.POINTER(BamBatch)]),
    "mcov_bam_write": (C.c_int, [C.c_char_p, _i32, C.POINTER(C.c_char_p), _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int]),
    "mcov_synth_gen_ncigar": (C.c_int, [C.POINTER(SynthParams), _i64, _i64, _vp, C.c_int, _vp]),
    "mcov_synth_gen_reads": (C.c_int, [C.POINTER(SynthParams), _i64, _i64, _vp, _vp, _i32, _i32, _vp,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
    "mcov_synth_gen_reads_wide": (C.c_int, [C.POINTER(SynthParams), _i64, _i64, _vp, _vp, _i32, _i32, _vp,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "metacov_b200: native library %s is missing. Build it with "
            "`python metacov_b200/_build.py` (needs nvcc); there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def ptr(a):
    """Raw pointer of a numpy array (host) or a torch tensor (device/host)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()
