"""ctypes mirror of include/simuscop.h (struct layouts only; no logic)."""
import ctypes as C


class ProfileTables(C.Structure):
    _fields_ = [
        ("n_bases", C.c_int32), ("kmer", C.c_int32), ("bins", C.c_int32), ("n_qual", C.c_int32),
        ("min_qual", C.c_int32), ("read_length", C.c_int32), ("paired", C.c_int32), ("use_cdf2", C.c_int32),
        ("fixed_insert_size", C.c_int32), ("min_insert_size", C.c_int32), ("n_isize", C.c_int32),
        ("n_ins", C.c_int32), ("n_del", C.c_int32), ("n_kmer_rows", C.c_int32),
        ("insert_rate", C.c_double), ("del_rate", C.c_double),
        ("bases", C.c_char * 8),
        ("isize_cdf", C.c_void_p), ("ins_cdf", C.c_void_p), ("del_cdf", C.c_void_p),
        ("subs_cdf1", C.c_void_p), ("subs_cdf2", C.c_void_p), ("quality_cdf", C.c_void_p),
    ]


class Bin(C.Structure):
    _fields_ = [
        ("hap_base", C.c_int64), ("contig_end", C.c_int64),
        ("spos", C.c_int32), ("epos", C.c_int32),
        ("segsize", C.c_uint32), ("read_count", C.c_int32),
        ("segment", C.c_int32), ("reserved", C.c_int32),
    ]


class Segment(C.Structure):
    _fields_ = [
        ("first_bin", C.c_int64), ("n_bins", C.c_int64),
        ("name_offset", C.c_int32), ("name_len", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("device_ms", C.c_double), ("launches", C.c_uint64), ("gen_launches", C.c_uint64),
        ("pairs_emitted", C.c_uint64), ("reads_emitted", C.c_uint64), ("bases_emitted", C.c_uint64),
        ("fastq_bytes", C.c_uint64), ("hap_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64),
        ("gen_kernel_ms", C.c_double), ("compact_kernel_ms", C.c_double), ("timed_batches", C.c_uint64),
        ("gz_bytes", C.c_uint64), ("bin_bytes", C.c_uint64), ("mover_kernel_ms", C.c_double),
        ("gen_kernel", C.c_int32), ("gen_nch", C.c_int32), ("gen_qmode", C.c_int32), ("gen_smem_bytes", C.c_int32),
    ]


class ReadArrays(C.Structure):
    _fields_ = [
        ("reads", C.c_void_p), ("length", C.c_void_p), ("pair_id", C.c_void_p),
        ("segment", C.c_void_p), ("pos", C.c_void_p), ("frag", C.c_void_p),
        ("capacity", C.c_int64), ("pitch", C.c_int32),
    ]


SINK_FN =C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int64, C.c_int64)

BIN_DTYPE = [("hap_base", "<i8"), ("contig_end", "<i8"), ("spos", "<i4"), ("epos", "<i4"),
             ("segsize", "<u4"), ("read_count", "<i4"), ("segment", "<i4"), ("reserved", "<i4")]
SEG_DTYPE = [("first_bin", "<i8"), ("n_bins", "<i8"), ("name_offset", "<i4"), ("name_len", "<i4")]
