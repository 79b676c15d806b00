"""ctypes binding of libpanfeed_b200.so (include/panfeed_b200.h).

This is the binding a maintainer of the reference would add next to
`/root/reference/panfeed/panfeed.py` (see INTEGRATION.md).  There is no
fallback: if the shared library is missing or no CUDA device exists the calls
raise.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# PF_LIB_PATH: a differently built library (kernel A/B experiments); default = the in-tree build
LIB_PATH = os.environ.get("PF_LIB_PATH") or os.path.join(HERE, "csrc", "libpanfeed_b200.so")

PF_ABI_VERSION = 2
PF_SEQ_TARGET = 1
PF_SEQ_AMBIGUOUS = 2
AMB_ALPHABET = "ABCDGHKMNRSTVWXY"


class PfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"panfeed_b200 error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("k", C.c_uint32),
                ("n_samples", C.c_uint32), ("canonical", C.c_uint32),
                ("consider_missing", C.c_uint32),
                ("cluster_equal_filter", C.c_uint32),
                ("emit_positions", C.c_uint32), ("sort_bits", C.c_uint32),
                ("mode", C.c_uint32), ("debug_flags", C.c_uint32),
                ("maf", C.c_double)]


SEQ_DTYPE = np.dtype([("base_off", "<u8"), ("len", "<u4"), ("cluster", "<u4"),
                      ("sample", "<u4"), ("flags", "<u4"), ("start", "<i4"),
                      ("end", "<i4"), ("offset", "<i4"), ("strand", "<i4"),
                      ("amb_off", "<u8")])
assert SEQ_DTYPE.itemsize == 48
CLUSTER_DTYPE = np.dtype([("id", "<u4"), ("reserved", "<u4")])


class Batch(C.Structure):
    _fields_ = [("packed_bases", C.c_void_p), ("n_words", C.c_uint64),
                ("seqs", C.c_void_p), ("n_seqs", C.c_uint32),
                ("clusters", C.c_void_p), ("n_clusters", C.c_uint32),
                ("cluster_presence", C.c_void_p),
                ("amb_codes", C.c_void_p), ("n_amb_words", C.c_uint64)]


class BatchResult(C.Structure):
    _fields_ = [("n_rows", C.c_uint64),
                ("row_cluster", C.POINTER(C.c_uint32)),
                ("row_kmer", C.POINTER(C.c_uint64)),
                ("row_count", C.POINTER(C.c_uint32)),
                ("row_pattern", C.POINTER(C.c_uint32)),
                ("n_wide_rows", C.c_uint64),
                ("wide_row_cluster", C.POINTER(C.c_uint32)),
                ("wide_row_kmer", C.POINTER(C.c_uint64)),
                ("wide_row_count", C.POINTER(C.c_uint32)),
                ("wide_row_pattern", C.POINTER(C.c_uint32)),
                ("n_clusters", C.c_uint32),
                ("cluster_pattern", C.POINTER(C.c_uint32)),
                ("kmer_pattern_base", C.c_uint64),
                ("n_new_kmer_patterns", C.c_uint64),
                ("new_kmer_patterns", C.POINTER(C.c_uint32)),
                ("cluster_pattern_base", C.c_uint64),
                ("n_new_cluster_patterns", C.c_uint64),
                ("new_cluster_patterns", C.POINTER(C.c_uint32)),
                ("n_pos", C.c_uint64),
                ("pos_kmer", C.POINTER(C.c_uint64)),
                ("pos_seq", C.POINTER(C.c_uint32)),
                ("pos_contig_start", C.POINTER(C.c_int32)),
                ("pos_gene_start", C.POINTER(C.c_int32)),
                ("pos_flags", C.POINTER(C.c_uint8)),
                ("pos_wide_kmer", C.POINTER(C.c_uint64)),
                ("n_pos_wide", C.c_uint64),
                ("pos_strand_bits", C.POINTER(C.c_uint32)),
                ("n_pos_bit_words", C.c_uint64),
                ("n_xwide_rows", C.c_uint64),
                ("xwide_row_cluster", C.POINTER(C.c_uint32)),
                ("xwide_row_kmer", C.POINTER(C.c_uint64)),
                ("xwide_row_count", C.POINTER(C.c_uint32)),
                ("xwide_row_pattern", C.POINTER(C.c_uint32)),
                ("pos_xwide_kmer", C.POINTER(C.c_uint64)),
                ("n_pos_xwide", C.c_uint64)]


class Stats(C.Structure):
    _fields_ = [("batches", C.c_uint64), ("bases", C.c_uint64),
                ("instances", C.c_uint64), ("unique_kmers", C.c_uint64),
                ("rows", C.c_uint64), ("kmer_patterns", C.c_uint64),
                ("cluster_patterns", C.c_uint64), ("sort_passes", C.c_uint32),
                ("launches", C.c_uint32), ("ms_h2d", C.c_float),
                ("ms_extract", C.c_float), ("ms_hist", C.c_float),
                ("ms_sort", C.c_float), ("ms_mark", C.c_float),
                ("ms_count", C.c_float), ("ms_reduce", C.c_float),
                ("ms_dedup", C.c_float),
                ("ms_d2h", C.c_float), ("ms_total", C.c_float),
                ("total_launches", C.c_uint64), ("engine", C.c_uint32),
                ("block_windows", C.c_uint32), ("block_slots", C.c_uint32),
                ("sub_batches", C.c_uint32), ("partial_rows", C.c_uint64)]


class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_samples", C.c_uint32),
                ("n_clusters", C.c_uint32), ("first_cluster", C.c_uint32),
                ("gene_len", C.c_uint32), ("n_founders", C.c_uint32),
                ("founder_div", C.c_float), ("private_div", C.c_float),
                ("core_fraction", C.c_float), ("paralog_rate", C.c_float),
                ("total_clusters", C.c_uint32), ("all_targets", C.c_uint32)]


class CutResult(C.Structure):
    """pf_cut_result (include/panfeed_b200.h)."""
    _fields_ = [("n_seqs", C.c_uint32),
                ("ascii", C.c_void_p),
                ("seq_off", C.POINTER(C.c_uint64)),
                ("cell", C.POINTER(C.c_uint32)),
                ("feature", C.POINTER(C.c_uint32)),
                ("start", C.POINTER(C.c_int32)),
                ("end", C.POINTER(C.c_int32)),
                ("offset", C.POINTER(C.c_int32)),
                ("strand", C.POINTER(C.c_int32)),
                ("n_missing", C.c_uint32),
                ("missing_cell", C.POINTER(C.c_uint32)),
                ("missing_kind", C.POINTER(C.c_uint8)),
                ("missing_text", C.c_void_p),
                ("missing_off", C.POINTER(C.c_uint64))]


class CutPlanes(C.Structure):
    """pf_cut_planes (include/panfeed_b200.h)."""
    _fields_ = [("packed", C.POINTER(C.c_uint64)), ("n_words", C.c_uint64),
                ("base_off", C.POINTER(C.c_uint64)), ("is_amb", C.POINTER(C.c_uint8)),
                ("amb_plane", C.POINTER(C.c_uint64)), ("n_amb_words", C.c_uint64),
                ("amb_off", C.POINTER(C.c_uint64)), ("bad_symbol", C.c_int32)]


ALL_GATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p)
ALL_TO_ALL_V_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.POINTER(C.c_uint64),
                              C.c_void_p, C.c_void_p)


class Comm(C.Structure):
    """pf_comm: the collectives pf_exchange_run runs over (device buffers, the context's stream)."""
    _fields_ = [("rank", C.c_uint32), ("world", C.c_uint32), ("user", C.c_void_p),
                ("all_gather", ALL_GATHER_FN), ("all_to_all_v", ALL_TO_ALL_V_FN)]


class ExchangeNs(C.Structure):
    """pf_exchange_ns: one namespace of a pf_exchange_run result."""
    _fields_ = [("n_local", C.c_uint64), ("n_global", C.c_uint64), ("n_owned", C.c_uint64),
                ("owned_base", C.c_uint64), ("bytes_sent", C.c_uint64),
                ("local_to_global", C.c_void_p), ("writer", C.c_void_p)]


class ExchangeResult(C.Structure):
    _fields_ = [("cluster", ExchangeNs), ("kmer", ExchangeNs)]


PF_EXCHANGE_WRITER, PF_EXCHANGE_KEEP_UNIQUE, PF_EXCHANGE_NO_PEER = 1, 2, 4


class AssocResult(C.Structure):
    """pf_assoc_result: the device join of one batch against the passing associations."""
    _fields_ = [("n_windows", C.c_uint64), ("window", C.POINTER(C.c_uint64)),
                ("window_assoc", C.POINTER(C.c_uint32)), ("n_clusters", C.c_uint32),
                ("cluster_pass", C.POINTER(C.c_uint8)), ("cluster_assoc", C.POINTER(C.c_uint32)),
                ("n_rows", C.c_uint64), ("row", C.POINTER(C.c_uint32)),
                ("row_assoc", C.POINTER(C.c_uint32)), ("row_seen", C.POINTER(C.c_uint8))]


PF_ASSOC_NONE = 0xFFFFFFFF
PF_ANNOT_ONLY_PASSING, PF_ANNOT_FLOAT_POSITIONS = 1, 2


EXPORTS = ["pf_create", "pf_destroy", "pf_last_error", "pf_abi_version",
           "pf_upload", "pf_execute", "pf_submit", "pf_collect",
           "pf_reset_patterns", "pf_pattern_words", "pf_kmer_pattern_words",
           "pf_maf_window", "pf_patterns_export", "pf_pattern_ids", "pf_stats_get", "pf_struct_size", "pf_stream", "pf_format_positions",
           "pf_format_positions_compact",
           "pf_pack_plan", "pf_pack_2bit", "pf_pack_4bit", "pf_base64_ids", "pf_format_patterns", "pf_format_kmer_rows", "pf_gzip_members",
           "pf_feeder_create", "pf_feeder_destroy", "pf_feeder_last_error", "pf_feeder_add_genome", "pf_feeder_add_genomes",
           "pf_feeder_add_genome_text", "pf_feeder_genome_info", "pf_feeder_feature", "pf_feeder_contig", "pf_feeder_cut",
           "pf_feeder_cut_packed",
           "pf_table_create", "pf_table_destroy", "pf_table_last_error", "pf_table_load", "pf_table_shape",
           "pf_table_names", "pf_table_row_counts", "pf_table_cells",
           "pf_tsv_filter", "pf_free",
           "pf_synth_plan", "pf_synth_fill", "pf_exchange_unique_count", "pf_exchange_unique_export",
           "pf_exchange_run", "pf_exchange_release",
           "pf_comm_local_create", "pf_comm_local_get", "pf_comm_local_abort", "pf_comm_local_destroy",
           "pf_assoc_load", "pf_assoc_collect", "pf_format_annotated"]

_lib = None


def load():
    """Load the CUDA library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PfError(-2, f"{LIB_PATH} is missing: build it with "
                          "`make -C panfeed_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    lib.pf_create.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Params)]
    lib.pf_destroy.argtypes = [vp]
    lib.pf_destroy.restype = None
    lib.pf_last_error.argtypes = [vp]
    lib.pf_last_error.restype = C.c_char_p
    lib.pf_upload.argtypes = [vp, C.POINTER(Batch)]
    lib.pf_execute.argtypes = [vp]
    lib.pf_submit.argtypes = [vp, C.POINTER(Batch)]
    lib.pf_collect.argtypes = [vp, C.POINTER(BatchResult)]
    lib.pf_reset_patterns.argtypes = [vp]
    lib.pf_pattern_words.argtypes = [u32]
    lib.pf_pattern_words.restype = u32
    lib.pf_kmer_pattern_words.argtypes = [vp]
    lib.pf_kmer_pattern_words.restype = u32
    lib.pf_maf_window.argtypes = [C.c_double, u32, C.POINTER(u32), C.POINTER(u32)]
    lib.pf_patterns_export.argtypes = [vp, C.c_int, u64, u64, vp]
    lib.pf_format_patterns.argtypes = [vp, u64, u32, u32, C.c_char_p, vp, u32, C.c_char_p, u64,
                                       C.POINTER(u64), u32]
    lib.pf_format_kmer_rows.argtypes = [C.POINTER(BatchResult), u32, C.c_char_p, vp, vp, u64, vp, u64, vp, u64,
                                        C.POINTER(u64), vp, u32]
    lib.pf_gzip_members.argtypes = [C.c_char_p, u64, C.c_int, u64, vp, u64, C.POINTER(u64), u32]
    lib.pf_feeder_create.argtypes = [C.POINTER(vp)]
    lib.pf_feeder_destroy.argtypes = [vp]
    lib.pf_feeder_destroy.restype = None
    lib.pf_feeder_last_error.argtypes = [vp]
    lib.pf_feeder_last_error.restype = C.c_char_p
    lib.pf_feeder_add_genome.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(u32)]
    lib.pf_feeder_add_genomes.argtypes = [vp, u32, vp, vp, vp, vp, u32]
    lib.pf_feeder_add_genome_text.argtypes = [vp, C.c_char_p, C.c_char_p, u64, C.c_char_p, u64, C.POINTER(u32)]
    lib.pf_feeder_genome_info.argtypes = [vp, u32, C.POINTER(u32), C.POINTER(u32), C.POINTER(u64)]
    lib.pf_feeder_feature.argtypes = [vp, u32, u32, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p),
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
    lib.pf_feeder_contig.argtypes = [vp, u32, u32, C.POINTER(C.c_char_p), C.POINTER(u64), C.POINTER(u32)]
    lib.pf_feeder_cut.argtypes = [vp, u32, vp, C.c_char_p, u64, C.c_int32, C.c_int32, C.c_int32,
                                  C.POINTER(CutResult)]
    lib.pf_feeder_cut_packed.argtypes = [vp, u32, vp, C.c_char_p, u64, C.c_int32, C.c_int32, C.c_int32, u32,
                                         C.POINTER(CutResult), C.POINTER(CutPlanes)]
    lib.pf_table_create.argtypes = [C.POINTER(vp)]
    lib.pf_table_destroy.argtypes = [vp]
    lib.pf_table_destroy.restype = None
    lib.pf_table_last_error.argtypes = [vp]
    lib.pf_table_last_error.restype = C.c_char_p
    lib.pf_table_load.argtypes = [vp, C.c_char_p, C.POINTER(C.c_char_p), u32, C.POINTER(C.c_char_p), u32, u32]
    lib.pf_table_shape.argtypes = [vp, C.POINTER(u64), C.POINTER(u32)]
    lib.pf_table_names.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp)]
    lib.pf_table_row_counts.argtypes = [vp, vp]
    lib.pf_table_cells.argtypes = [vp, vp, u64, vp, vp, vp, u64, C.POINTER(u64), C.POINTER(u64)]
    lib.pf_tsv_filter.argtypes = [C.c_char_p, u32, C.c_char_p, vp, u64, C.c_int, C.POINTER(vp), C.POINTER(u64),
                                  C.POINTER(u64), u32]
    lib.pf_free.argtypes = [vp]
    lib.pf_free.restype = None
    lib.pf_base64_ids.argtypes = [vp, u64, vp, u32]
    lib.pf_pack_plan.argtypes = [vp, u32, vp, C.POINTER(u64)]
    lib.pf_pack_2bit.argtypes = [vp, vp, u32, vp, vp, vp, u32]          # ascii: bytes or a raw address
    lib.pf_pack_4bit.argtypes = [vp, vp, u32, vp, vp, vp, C.POINTER(u64), C.POINTER(C.c_int)]
    lib.pf_format_positions.argtypes = [C.POINTER(BatchResult), u32, C.c_int, u64, u64, C.c_char_p,
                                        C.POINTER(u64), C.POINTER(C.c_int32), C.c_char_p, u64,
                                        C.POINTER(u64), u32]
    lib.pf_format_positions_compact.argtypes = [C.POINTER(Batch), vp, u32, C.c_int, u32, u32, C.c_char_p,
                                                C.POINTER(u64), C.c_char_p, u64, C.POINTER(u64), u32]
    lib.pf_pattern_ids.argtypes = [vp, C.c_int, u64, u64, vp]
    lib.pf_stats_get.argtypes = [vp, C.POINTER(Stats)]
    lib.pf_stream.argtypes = [vp]
    lib.pf_stream.restype = vp
    lib.pf_synth_plan.argtypes = [C.POINTER(SynthParams), C.POINTER(u32), C.POINTER(u64)]
    lib.pf_synth_fill.argtypes = [C.c_int, C.POINTER(SynthParams), vp, vp, vp, vp]
    lib.pf_exchange_unique_count.argtypes = [vp, C.c_int, C.POINTER(u64)]
    lib.pf_exchange_unique_export.argtypes = [vp, C.c_int, vp]
    lib.pf_exchange_run.argtypes = [vp, C.POINTER(Comm), u32, C.POINTER(ExchangeResult)]
    lib.pf_exchange_release.argtypes = [vp, C.POINTER(Comm)]
    lib.pf_comm_local_create.argtypes = [u32, C.POINTER(vp)]
    lib.pf_comm_local_get.argtypes = [vp, u32, C.POINTER(Comm)]
    lib.pf_comm_local_abort.argtypes = [vp]
    lib.pf_comm_local_abort.restype = None
    lib.pf_comm_local_destroy.argtypes = [vp]
    lib.pf_comm_local_destroy.restype = None
    lib.pf_assoc_load.argtypes = [vp, vp, u64]
    lib.pf_assoc_collect.argtypes = [vp, C.POINTER(AssocResult)]
    lib.pf_format_annotated.argtypes = [C.POINTER(Batch), vp, u32, C.c_int, C.POINTER(BatchResult),
                                        C.POINTER(AssocResult), C.c_char_p, vp, C.c_char_p, vp, C.c_char_p, vp,
                                        u64, u32, u32, vp, u64, C.POINTER(u64), u32]
    lib.pf_struct_size.argtypes = [C.c_int]
    lib.pf_struct_size.restype = u32
    if lib.pf_abi_version() != PF_ABI_VERSION:
        raise PfError(-1, "ABI version mismatch")
    _lib = lib
    return lib


def maf_window(maf, n):
    lo, hi = C.c_uint32(), C.c_uint32()
    ok = load().pf_maf_window(maf, n, C.byref(lo), C.byref(hi))
    return (lo.value, hi.value) if ok else None


def pack_sequences(seq_bytes, n_threads=0):
    """Native packer (pf_pack_*): list of upper-case ASCII sequences -> (packed 2-bit plane,
    base_off, is_amb, amb_plane or None, amb_off).  Raises ValueError on a symbol outside
    AMB_ALPHABET."""
    n = len(seq_bytes)
    blob = b"".join(seq_bytes)
    seq_off = np.zeros(n + 1, np.uint64)
    if n:
        np.cumsum(np.fromiter((len(b) for b in seq_bytes), np.uint64, n), out=seq_off[1:])
    return pack_blob(blob, seq_off, n_threads)


def pack_blob(blob, seq_off, n_threads=0):
    """The same from the sequences back to back (`blob`: bytes, or the address of a buffer that
    stays valid during the call, e.g. pf_cut_result.ascii) and their offsets (`seq_off`, uint64
    [n + 1]): what the native feeder hands over."""
    lib = load()
    seq_off = np.ascontiguousarray(seq_off, dtype=np.uint64)
    n = len(seq_off) - 1
    base_off = np.zeros(n, np.uint64)
    n_words = C.c_uint64()
    rc = lib.pf_pack_plan(seq_off.ctypes.data, n, base_off.ctypes.data, C.byref(n_words))
    if rc != 0:
        raise PfError(rc, "pf_pack_plan failed")
    packed = np.zeros(int(n_words.value), np.uint64)
    is_amb = np.zeros(n, np.uint8)
    rc = lib.pf_pack_2bit(blob, seq_off.ctypes.data, n, base_off.ctypes.data, packed.ctypes.data,
                          is_amb.ctypes.data, int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_pack_2bit failed")
    amb_off = np.zeros(n, np.uint64)
    amb_plane = None
    if is_amb.any():
        n_amb = C.c_uint64()
        bad = C.c_int()
        rc = lib.pf_pack_4bit(blob, seq_off.ctypes.data, n, is_amb.ctypes.data, amb_off.ctypes.data, None,
                              C.byref(n_amb), C.byref(bad))
        if rc != 0:
            raise PfError(rc, "pf_pack_4bit (sizing) failed")
        amb_plane = np.zeros(int(n_amb.value), np.uint64)
        rc = lib.pf_pack_4bit(blob, seq_off.ctypes.data, n, is_amb.ctypes.data, amb_off.ctypes.data,
                              amb_plane.ctypes.data, C.byref(n_amb), C.byref(bad))
        if rc == -4:
            raise ValueError(f"unsupported sequence symbol {chr(bad.value)!r}: only "
                             f"{AMB_ALPHABET} (IUPAC, upper case) are accepted")
        if rc != 0:
            raise PfError(rc, "pf_pack_4bit failed")
    return packed, base_off, is_amb.astype(bool), amb_plane, amb_off


_scratch_bufs = {}


def _scratch(name, nbytes):
    """A grow-only uint8 buffer per formatter: the text of one batch is hundreds of MB, and fresh
    memory for every batch costs more (first touch) than formatting into it."""
    buf = _scratch_bufs.get(name)
    if buf is None or buf.size < nbytes:
        buf = _scratch_bufs[name] = np.empty(int(nbytes) + int(nbytes) // 4 + 4096, np.uint8)
    return buf


def format_patterns(words, n_samples, ids, present=None, n_threads=0, raw=False, scratch="patterns"):
    """hashes_to_patterns text (bytes) of the patterns `words` ([n, >= W] uint32) with their
    24-character ids; `present` ([n, >= W] uint32) marks the samples whose cell is not NaN.
    raw=True (all three formatters): a uint8 view of a buffer that the next call of the same
    formatter (here: with the same `scratch` name) reuses, for callers that write the text out
    at once."""
    lib = load()
    words = np.ascontiguousarray(words, dtype=np.uint32)
    n = len(words)
    if n == 0:
        return b""
    if isinstance(ids, np.ndarray) and ids.dtype == np.dtype("S24"):
        idb = np.ascontiguousarray(ids).tobytes()
    else:
        idb = b"".join(x if isinstance(x, bytes) else x.encode() for x in ids)
    assert len(idb) == 24 * n
    pres = None if present is None else np.ascontiguousarray(present, dtype=np.uint32)
    need = C.c_uint64()
    args = (words.ctypes.data, n, words.shape[1], int(n_samples), idb,
            None if pres is None else pres.ctypes.data, 0 if pres is None else pres.shape[1])
    rc = lib.pf_format_patterns(*args, None, 0, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_patterns (sizing) failed")
    out = _scratch(scratch, need.value)
    rc = lib.pf_format_patterns(*args, out.ctypes.data_as(C.c_char_p), out.size, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_patterns failed")
    return out[:int(need.value)] if raw else out[:int(need.value)].tobytes()


def tsv_filter(path, column, keys, skip_header=True, n_threads=0):
    """Lines of the TSV file `path` (header excluded) whose tab-separated field `column` is one of
    `keys` (iterable of str / bytes), in file order: (bytes, number of rows).  pf_tsv_filter,
    library host threads."""
    lib = load()
    kb = [k if isinstance(k, bytes) else str(k).encode() for k in keys]
    blob = b"".join(kb)
    off = np.zeros(len(kb) + 1, np.uint64)
    if kb:
        np.cumsum(np.fromiter((len(k) for k in kb), np.uint64, len(kb)), out=off[1:])
    out, n, rows = C.c_void_p(), C.c_uint64(), C.c_uint64()
    rc = lib.pf_tsv_filter(os.fsencode(path), int(column), blob, off.ctypes.data, len(kb), int(bool(skip_header)),
                           C.byref(out), C.byref(n), C.byref(rows), int(n_threads))
    if rc != 0:
        raise PfError(rc, f"pf_tsv_filter failed on {path}")
    try:
        data = C.string_at(out, n.value) if n.value else b""
    finally:
        if out:
            lib.pf_free(out)
    return data, int(rows.value)


def gzip_members(data, level=9, member_bytes=0, n_threads=0):
    """gzip of `data` (bytes) as a sequence of independently deflated members (pf_gzip_members,
    library host threads): a valid gzip file, or a piece to append to one."""
    lib = load()
    need = C.c_uint64()
    rc = lib.pf_gzip_members(data, len(data), int(level), int(member_bytes), None, 0, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_gzip_members (sizing) failed")
    out = np.empty(int(need.value), np.uint8)
    rc = lib.pf_gzip_members(data, len(data), int(level), int(member_bytes), out.ctypes.data, out.size,
                             C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_gzip_members failed")
    return out[:int(need.value)].tobytes()


def format_kmer_rows(r, k, tags, kmer_ids, cluster_ids, n_threads=0, raw=False):
    """kmers_to_hashes text of the batch result `r` (a dict as returned by Context.collect(), or
    any dict with row_*, wide_row_* (xwide_row_* if present) and cluster_pattern), formatted by
    the library's host threads (pf_format_kmer_rows).  tags[c] = first column of cluster c (bytes);
    kmer_ids / cluster_ids: numpy S24 arrays of all pattern ids numbered so far.  Returns (bytes,
    offsets[n_clusters+1])."""
    lib = load()
    keep = []

    def ptr(a, dtype, ctype):
        a = np.ascontiguousarray(a, dtype=dtype)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(ctype))

    nc = len(r["cluster_pattern"])
    if nc == 0:
        return b"", np.zeros(1, np.uint64)
    res = BatchResult()
    res.n_clusters = nc
    res.cluster_pattern = ptr(r["cluster_pattern"], np.uint32, C.c_uint32)
    res.n_rows = len(r["row_cluster"])
    res.row_cluster = ptr(r["row_cluster"], np.uint32, C.c_uint32)
    res.row_kmer = ptr(r["row_kmer"], np.uint64, C.c_uint64)
    res.row_pattern = ptr(r["row_pattern"], np.uint32, C.c_uint32)
    wide = np.ascontiguousarray(r.get("wide_row_kmer", np.zeros((0, 2), np.uint64)), dtype=np.uint64).reshape(-1)
    res.n_wide_rows = wide.size // 2
    if wide.size:
        res.wide_row_kmer = ptr(wide, np.uint64, C.c_uint64)
        res.wide_row_cluster = ptr(r["wide_row_cluster"], np.uint32, C.c_uint32)
        res.wide_row_pattern = ptr(r["wide_row_pattern"], np.uint32, C.c_uint32)
    xwide = np.ascontiguousarray(r.get("xwide_row_kmer", np.zeros((0, 4), np.uint64)), dtype=np.uint64).reshape(-1)
    res.n_xwide_rows = xwide.size // 4
    if xwide.size:
        res.xwide_row_kmer = ptr(xwide, np.uint64, C.c_uint64)
        res.xwide_row_cluster = ptr(r["xwide_row_cluster"], np.uint32, C.c_uint32)
        res.xwide_row_pattern = ptr(r["xwide_row_pattern"], np.uint32, C.c_uint32)
    blob = b"".join(tags)
    off = np.zeros(nc + 1, np.uint64)
    np.cumsum([len(x) for x in tags], out=off[1:])
    kid = np.ascontiguousarray(kmer_ids, dtype="S24")
    cid = np.ascontiguousarray(cluster_ids, dtype="S24")
    cl_off = np.zeros(nc + 1, np.uint64)
    need = C.c_uint64()
    args = (C.byref(res), int(k), blob, off.ctypes.data, kid.ctypes.data if len(kid) else None, len(kid),
            cid.ctypes.data if len(cid) else None, len(cid))
    rc = lib.pf_format_kmer_rows(*args, None, 0, C.byref(need), cl_off.ctypes.data, int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_kmer_rows (sizing) failed")
    out = _scratch("kmer_rows", need.value)
    rc = lib.pf_format_kmer_rows(*args, out.ctypes.data, out.size, C.byref(need), cl_off.ctypes.data, int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_kmer_rows failed")
    return (out[:int(need.value)] if raw else out[:int(need.value)].tobytes()), cl_off


def format_positions(r, k, canonical, leads, seq_strand, n_threads=0):
    """kmers.tsv text (bytes) of the positional records in `r` (a dict as returned by
    Context.collect(), or any dict with the pos_* arrays), formatted by the library's
    host threads (pf_format_positions).  leads[i] = b"idx\tstrain\tgene_id\tcontig\tstrand\t"
    of sequence i of the batch; seq_strand[i] its Seqinfo.strand."""
    lib = load()
    n = len(r["pos_seq"])
    if n == 0:
        return b""
    keep = {}

    def ptr(a, dtype, ctype):
        a = np.ascontiguousarray(a, dtype=dtype)
        keep[id(a)] = a
        return a.ctypes.data_as(C.POINTER(ctype))

    res = BatchResult()
    res.n_pos = n
    res.pos_kmer = ptr(r["pos_kmer"], np.uint64, C.c_uint64)
    res.pos_seq = ptr(r["pos_seq"], np.uint32, C.c_uint32)
    res.pos_contig_start = ptr(r["pos_contig_start"], np.int32, C.c_int32)
    res.pos_gene_start = ptr(r["pos_gene_start"], np.int32, C.c_int32)
    res.pos_flags = ptr(r["pos_flags"], np.uint8, C.c_uint8)
    wide = np.ascontiguousarray(r.get("pos_wide_kmer", np.zeros((0, 2), np.uint64)), dtype=np.uint64).reshape(-1)
    if wide.size == 0:
        wide = np.zeros(2, np.uint64)
    res.pos_wide_kmer = ptr(wide, np.uint64, C.c_uint64)
    res.n_pos_wide = wide.size // 2
    xwide = np.ascontiguousarray(r.get("pos_xwide_kmer", np.zeros((0, 4), np.uint64)), dtype=np.uint64).reshape(-1)
    if xwide.size:                # (k > 32: positional k-mers holding N/IUPAC symbols, pos_flags bit 2)
        res.pos_xwide_kmer = ptr(xwide, np.uint64, C.c_uint64)
        res.n_pos_xwide = xwide.size // 4
    blob = b"".join(leads)
    off = np.zeros(len(leads) + 1, np.uint64)
    np.cumsum([len(x) for x in leads], out=off[1:])
    strand = np.ascontiguousarray(seq_strand, dtype=np.int32)
    need = C.c_uint64()
    args = (C.byref(res), int(k), int(bool(canonical)), 0, n, blob, off.ctypes.data_as(C.POINTER(C.c_uint64)),
            strand.ctypes.data_as(C.POINTER(C.c_int32)))
    rc = lib.pf_format_positions(*args, None, 0, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_positions (sizing) failed")
    out = np.empty(int(need.value), np.uint8)
    rc = lib.pf_format_positions(*args, out.ctypes.data_as(C.c_char_p), out.size, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_positions failed")
    return out.tobytes()


def format_positions_compact(hb, strand_bits, k, canonical, leads, n_threads=0, raw=False):
    """kmers.tsv text (bytes) of the PF_SEQ_TARGET sequences of the HostBatch `hb` from the compact
    positional form (Context(emit_positions=2)): `strand_bits` = r["pos_strand_bits"] of the
    batch's collect().  leads[i] as in format_positions (may be b"" for non-target sequences)."""
    lib = load()
    n = len(hb.seqs)
    if n == 0:
        return b""
    b = hb.struct()
    blob = b"".join(leads)
    off = np.zeros(n + 1, np.uint64)
    np.cumsum(np.fromiter((len(x) for x in leads), np.uint64, n), out=off[1:])
    bits = None
    if canonical:
        bits = np.ascontiguousarray(strand_bits, dtype=np.uint32)
        if bits.size < hb.packed.size:
            raise ValueError("strand bit plane is shorter than the packed plane")
    need = C.c_uint64()
    args = (C.byref(b), bits.ctypes.data if bits is not None else None, int(k), int(bool(canonical)), 0, n, blob,
            off.ctypes.data_as(C.POINTER(C.c_uint64)))
    rc = lib.pf_format_positions_compact(*args, None, 0, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_positions_compact (sizing) failed")
    out = _scratch("positions", need.value)
    rc = lib.pf_format_positions_compact(*args, out.ctypes.data_as(C.c_char_p), out.size, C.byref(need),
                                         int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_positions_compact failed")
    return out[:int(need.value)] if raw else out[:int(need.value)].tobytes()


def id_digests(ids):
    """Pattern ids (base64(md5)[:24], the first column of an associations file) -> ([n, 16] uint8
    digests, positions in `ids` of the ones that decode).  An id that is not 24 characters of
    base64 for 16 bytes names no pattern and is skipped."""
    import binascii
    out, keep = [], []
    for i, x in enumerate(ids):
        x = x.decode() if isinstance(x, bytes) else str(x)
        if len(x) != 24 or not x.endswith("=="):
            continue
        try:
            d = binascii.a2b_base64(x)
        except (binascii.Error, ValueError):
            continue
        if len(d) != 16 or binascii.b2a_base64(d).decode()[:24] != x:
            continue
        out.append(d)
        keep.append(i)
    return np.frombuffer(b"".join(out), np.uint8).reshape(-1, 16).copy(), np.array(keep, np.int64)


def _blob(parts):
    """bytes joined + uint64 offsets [n + 1]"""
    off = np.zeros(len(parts) + 1, np.uint64)
    if parts:
        np.cumsum(np.fromiter((len(x) for x in parts), np.uint64, len(parts)), out=off[1:])
    return b"".join(parts), off


def format_annotated(hb, strand_bits, k, canonical, r, assoc, tags, leads, snippets, snip_fields, flags,
                     n_threads=0, raw=False):
    """panfeed-get-kmers lines of one batch (pf_format_annotated): hb = the batch's HostBatch, r its
    collect() dict, assoc its Context.assoc_collect() dict, tags[c] = cluster column (bytes) per
    cluster, leads[i] = b"strain\tgene_id\tcontig\t" per sequence, snippets[a] = the hashed_pattern
    and association fields of association row a (bytes, snip_fields fields), flags = PF_ANNOT_*."""
    lib = load()
    keep = []

    def ptr(a, dtype, ctype):
        a = np.ascontiguousarray(a, dtype=dtype)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(ctype))

    b = hb.struct()
    res = BatchResult()
    res.n_clusters = len(hb.clusters)
    res.n_rows = len(r["row_kmer"])
    res.row_cluster = ptr(r["row_cluster"][:res.n_rows], np.uint32, C.c_uint32)
    res.row_kmer = ptr(r["row_kmer"], np.uint64, C.c_uint64)
    res.n_wide_rows = len(r["wide_row_kmer"])
    res.wide_row_cluster = ptr(r["wide_row_cluster"], np.uint32, C.c_uint32)
    res.wide_row_kmer = ptr(r["wide_row_kmer"].reshape(-1), np.uint64, C.c_uint64)
    res.n_xwide_rows = len(r["xwide_row_kmer"])
    res.xwide_row_cluster = ptr(r["xwide_row_cluster"], np.uint32, C.c_uint32)
    res.xwide_row_kmer = ptr(r["xwide_row_kmer"].reshape(-1), np.uint64, C.c_uint64)
    a = AssocResult()
    a.n_windows = len(assoc["window"])
    a.window = ptr(assoc["window"], np.uint64, C.c_uint64)
    a.window_assoc = ptr(assoc["window_assoc"], np.uint32, C.c_uint32)
    a.n_clusters = len(assoc["cluster_pass"])
    a.cluster_pass = ptr(assoc["cluster_pass"], np.uint8, C.c_uint8)
    a.cluster_assoc = ptr(assoc["cluster_assoc"], np.uint32, C.c_uint32)
    a.n_rows = len(assoc["row"])
    a.row = ptr(assoc["row"], np.uint32, C.c_uint32)
    a.row_assoc = ptr(assoc["row_assoc"], np.uint32, C.c_uint32)
    a.row_seen = ptr(assoc["row_seen"], np.uint8, C.c_uint8)
    tag_blob, tag_off = _blob(tags)
    lead_blob, lead_off = _blob(leads)
    snip_blob, snip_off = _blob(snippets)
    bits = None
    if canonical and len(hb.seqs):
        bits = np.ascontiguousarray(strand_bits, dtype=np.uint32)
        if bits.size < hb.packed.size:
            raise ValueError("strand bit plane is shorter than the packed plane")
    need = C.c_uint64()
    args = (C.byref(b), bits.ctypes.data if bits is not None else None, int(k), int(bool(canonical)), C.byref(res),
            C.byref(a), tag_blob, tag_off.ctypes.data, lead_blob, lead_off.ctypes.data, snip_blob,
            snip_off.ctypes.data, len(snippets), int(snip_fields), int(flags))
    rc = lib.pf_format_annotated(*args, None, 0, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_annotated (sizing) failed")
    out = _scratch("annotated", need.value)
    rc = lib.pf_format_annotated(*args, out.ctypes.data, out.size, C.byref(need), int(n_threads))
    if rc != 0:
        raise PfError(rc, "pf_format_annotated failed")
    return out[:int(need.value)] if raw else out[:int(need.value)].tobytes()


def _np(ptr, n, dtype, copy=True):
    if n == 0:
        return np.zeros(0, dtype)
    a = np.ctypeslib.as_array(ptr, shape=(int(n),))
    return a.astype(dtype, copy=True) if copy else a


_B64 = np.frombuffer(b"ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/", np.uint8)


def base64_ids(digests, n_threads=0):
    """[n,16] uint8 MD5 digests -> numpy S24 array of base64 strings (with '=='): pf_base64_ids,
    library host threads (millions of ids per batch)."""
    digests = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 16)
    out = np.empty(len(digests), "S24")
    if len(digests):
        rc = load().pf_base64_ids(digests.ctypes.data, len(digests), out.ctypes.data, int(n_threads))
        if rc != 0:
            raise PfError(rc, "pf_base64_ids failed")
    return out


def base64_ids_numpy(digests):
    """The same with numpy (the tests compare the two)."""
    d = np.zeros((len(digests), 18), np.uint32)
    d[:, :16] = digests
    t = (d[:, 0::3] << 16) | (d[:, 1::3] << 8) | d[:, 2::3]            # [n, 6] 24-bit groups
    sx = np.stack([(t >> 18) & 63, (t >> 12) & 63, (t >> 6) & 63, t & 63], axis=2).reshape(len(d), 24)
    out = _B64[sx]
    out[:, 22:] = ord("=")
    return np.ascontiguousarray(out).view("S24").ravel()


class HostBatch:
    """Numpy-side image of a pf_batch (arrays must stay alive during upload)."""

    def __init__(self, packed, seqs, clusters, presence, amb=None):
        self.packed = np.ascontiguousarray(packed, dtype=np.uint64)
        self.seqs = np.ascontiguousarray(seqs, dtype=SEQ_DTYPE)
        self.clusters = np.ascontiguousarray(clusters, dtype=CLUSTER_DTYPE)
        self.presence = np.ascontiguousarray(presence, dtype=np.uint32)
        self.amb = None if amb is None else np.ascontiguousarray(amb, dtype=np.uint64)

    def struct(self):
        b = Batch()
        b.packed_bases = self.packed.ctypes.data if self.packed.size else None
        b.n_words = self.packed.size
        b.seqs = self.seqs.ctypes.data if self.seqs.size else None
        b.n_seqs = self.seqs.size
        b.clusters = self.clusters.ctypes.data if self.clusters.size else None
        b.n_clusters = self.clusters.size
        b.cluster_presence = self.presence.ctypes.data if self.presence.size else None
        if self.amb is not None and self.amb.size:
            b.amb_codes = self.amb.ctypes.data
            b.n_amb_words = self.amb.size
        return b

    @property
    def n_bases(self):
        return int(self.seqs["len"].sum())


class Context:
    """One pf_ctx: the reference's bound `iter_o` / `func_w` pair for one GPU."""

    def __init__(self, k, n_samples, canonical=True, consider_missing=False,
                 cluster_equal_filter=False, emit_positions=False, maf=0.01,
                 sort_bits=0, device=0, mode=0, debug_flags=0):
        self.lib = load()
        # emit_positions: False / True (21-byte records) / 2 (compact: the used_strand bit plane)
        self.params = Params(PF_ABI_VERSION, k, n_samples, int(canonical),
                             int(consider_missing), int(cluster_equal_filter),
                             int(emit_positions), sort_bits, mode, debug_flags, maf)
        self.h = C.c_void_p()
        rc = self.lib.pf_create(C.byref(self.h), device, C.byref(self.params))
        if rc != 0:
            raise PfError(rc, self.lib.pf_last_error(None).decode())
        self.k, self.S = k, n_samples
        self.W = self.lib.pf_pattern_words(n_samples)
        self.Wk = self.lib.pf_kmer_pattern_words(self.h)
        self.consider_missing = bool(consider_missing)
        self.canonical = bool(canonical)

    def _check(self, rc):
        if rc != 0:
            raise PfError(rc, self.lib.pf_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.lib.pf_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def upload(self, hb):
        s = hb.struct()
        self._check(self.lib.pf_upload(self.h, C.byref(s)))

    def execute(self):
        self._check(self.lib.pf_execute(self.h))

    def submit(self, hb):
        s = hb.struct()
        self._check(self.lib.pf_submit(self.h, C.byref(s)))

    def collect(self, copy=True):
        """Results of the last execution.  copy=False returns views into the
        context's pinned buffers, valid until the next collect()."""
        r = BatchResult()
        self._check(self.lib.pf_collect(self.h, C.byref(r)))
        nr, nw = int(r.n_rows), int(r.n_wide_rows)
        n_rec = int(r.n_pos) if r.pos_seq else 0        # compact positional form: no record arrays
        _np = lambda p, n, d: globals()["_np"](p, n, d, copy)  # noqa: E731
        out = {
            "row_cluster": _np(r.row_cluster, nr, np.uint32),
            "row_kmer": _np(r.row_kmer, nr, np.uint64),
            "row_count": _np(r.row_count, nr, np.uint32),
            "row_pattern": _np(r.row_pattern, nr, np.uint32),
            "wide_row_cluster": _np(r.wide_row_cluster, nw, np.uint32),
            "wide_row_kmer": _np(r.wide_row_kmer, 2 * nw, np.uint64).reshape(-1, 2),
            "wide_row_count": _np(r.wide_row_count, nw, np.uint32),
            "wide_row_pattern": _np(r.wide_row_pattern, nw, np.uint32),
            "cluster_pattern": _np(r.cluster_pattern, r.n_clusters, np.uint32),
            "kmer_pattern_base": int(r.kmer_pattern_base),
            "new_kmer_patterns": _np(r.new_kmer_patterns,
                                     r.n_new_kmer_patterns * self.Wk,
                                     np.uint32).reshape(-1, self.Wk),
            "cluster_pattern_base": int(r.cluster_pattern_base),
            "new_cluster_patterns": _np(r.new_cluster_patterns,
                                        r.n_new_cluster_patterns * self.W,
                                        np.uint32).reshape(-1, self.W),
            "pos_kmer": _np(r.pos_kmer, n_rec, np.uint64),
            "pos_seq": _np(r.pos_seq, n_rec, np.uint32),
            "pos_contig_start": _np(r.pos_contig_start, n_rec, np.int32),
            "pos_gene_start": _np(r.pos_gene_start, n_rec, np.int32),
            "pos_flags": _np(r.pos_flags, n_rec, np.uint8),
            "pos_wide_kmer": _np(r.pos_wide_kmer, 2 * r.n_pos_wide,
                                 np.uint64).reshape(-1, 2),
            "n_pos": int(r.n_pos),
            "pos_strand_bits": _np(r.pos_strand_bits, r.n_pos_bit_words, np.uint32),
            # k > 32: rows / positional k-mers holding N/IUPAC symbols, 4 words (4 bits per symbol)
            "xwide_row_cluster": _np(r.xwide_row_cluster, r.n_xwide_rows, np.uint32),
            "xwide_row_kmer": _np(r.xwide_row_kmer, 4 * r.n_xwide_rows, np.uint64).reshape(-1, 4),
            "xwide_row_count": _np(r.xwide_row_count, r.n_xwide_rows, np.uint32),
            "xwide_row_pattern": _np(r.xwide_row_pattern, r.n_xwide_rows, np.uint32),
            "pos_xwide_kmer": _np(r.pos_xwide_kmer, 4 * r.n_pos_xwide, np.uint64).reshape(-1, 4),
        }
        out["d2h_bytes"] = int(sum(v.nbytes for v in out.values()
                                   if isinstance(v, np.ndarray)))
        return out

    def reset_patterns(self):
        self._check(self.lib.pf_reset_patterns(self.h))

    def stats(self):
        s = Stats()
        self._check(self.lib.pf_stats_get(self.h, C.byref(s)))
        return {f: getattr(s, f) for f, _ in Stats._fields_}

    def export_patterns(self, cluster_namespace, first, count):
        w = self.W if cluster_namespace else self.Wk
        out = np.zeros((count, w), np.uint32)
        self._check(self.lib.pf_patterns_export(self.h, int(cluster_namespace),
                                                first, count, out.ctypes.data))
        return out

    def pattern_ids(self, cluster_namespace, first, count):
        """The reference's id strings (base64(md5(vector bytes))[:24]) of patterns
        [first, first+count), MD5 computed on the device (K5)."""
        if count == 0:
            return np.zeros(0, "S24")
        dig = np.zeros((count, 16), np.uint8)
        self._check(self.lib.pf_pattern_ids(self.h, int(cluster_namespace), first, count,
                                            dig.ctypes.data))
        return base64_ids(dig)

    def assoc_load(self, digests):
        """pf_assoc_load: the passing patterns ([n, 16] uint8 MD5 digests; row i = association row i)."""
        d = np.ascontiguousarray(digests, dtype=np.uint8).reshape(-1, 16)
        self._check(self.lib.pf_assoc_load(self.h, d.ctypes.data if len(d) else None, len(d)))

    def assoc_collect(self):
        """pf_assoc_collect after collect(): the join of the batch, as copies."""
        a = AssocResult()
        self._check(self.lib.pf_assoc_collect(self.h, C.byref(a)))
        return {"window": _np(a.window, a.n_windows, np.uint64),
                "window_assoc": _np(a.window_assoc, a.n_windows, np.uint32),
                "cluster_pass": _np(a.cluster_pass, a.n_clusters, np.uint8),
                "cluster_assoc": _np(a.cluster_assoc, a.n_clusters, np.uint32),
                "row": _np(a.row, a.n_rows, np.uint32),
                "row_assoc": _np(a.row_assoc, a.n_rows, np.uint32),
                "row_seen": _np(a.row_seen, a.n_rows, np.uint8)}

    def stream_handle(self):
        return self.lib.pf_stream(self.h)

    def exchange_run(self, comm, flags=0):
        """pf_exchange_run over `comm` (a Comm, e.g. LocalComm.get(rank)): the global numbering of the
        patterns of every rank.  -> {"cluster": ..., "kmer": ...}, each a dict of the counts and the
        DEVICE addresses of local_to_global (uint32 [n_local]) and writer (uint8 [n_local] or 0),
        owned by the context until its next exchange_run / reset_patterns / close."""
        out = ExchangeResult()
        self._check(self.lib.pf_exchange_run(self.h, C.byref(comm), int(flags), C.byref(out)))
        return {name: {f: (getattr(ns, f) or 0) for f, _ in ExchangeNs._fields_}
                for name, ns in (("cluster", out.cluster), ("kmer", out.kmer))}

    def exchange_release(self, comm):
        """pf_exchange_release: collective, unmaps the peers' receive buffers."""
        self._check(self.lib.pf_exchange_release(self.h, C.byref(comm)))

    def exchange_unique_keys(self, cluster_namespace):
        """The owner-side unique keys of the last exchange (PF_EXCHANGE_KEEP_UNIQUE)."""
        n = C.c_uint64()
        self._check(self.lib.pf_exchange_unique_count(self.h, int(cluster_namespace), C.byref(n)))
        out = np.zeros((n.value, self.W if cluster_namespace else self.Wk), np.uint32)
        self._check(self.lib.pf_exchange_unique_export(self.h, int(cluster_namespace), out.ctypes.data))
        return out


class LocalComm:
    """pf_comm_local: collectives between the threads of this process, one Context per thread (same
    or different devices).  get(rank) is the Comm of one rank."""

    def __init__(self, world):
        self.lib = load()
        self.h = C.c_void_p()
        rc = self.lib.pf_comm_local_create(int(world), C.byref(self.h))
        if rc != 0:
            raise PfError(rc, f"pf_comm_local_create({world}) failed")
        self.world = int(world)

    def get(self, rank):
        c = Comm()
        rc = self.lib.pf_comm_local_get(self.h, int(rank), C.byref(c))
        if rc != 0:
            raise PfError(rc, f"pf_comm_local_get: no rank {rank} in a world of {self.world}")
        return c

    def abort(self):
        """Every rank waiting in (or later entering) a collective returns an error."""
        self.lib.pf_comm_local_abort(self.h)

    def close(self):
        if self.h:
            self.lib.pf_comm_local_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SynthArena:
    """Reusable pinned host buffers for synth_batch (streamed benchmarks generate one batch
    after the other; allocating and pinning ~300 MB per batch would dominate)."""

    def __init__(self):
        self.packed = self.seqs = self.clusters = self.presence = None

    @staticmethod
    def _pinned(nbytes):
        import torch
        return torch.empty(max(8, int(nbytes)), dtype=torch.uint8, pin_memory=True).numpy()

    def take(self, n_words, n_seqs, n_clusters, W):
        def grow(cur, nbytes):
            if cur is None or cur.nbytes < nbytes:
                return self._pinned(nbytes + nbytes // 8)
            return cur
        self.packed = grow(self.packed, n_words * 8)
        self.seqs = grow(self.seqs, n_seqs * SEQ_DTYPE.itemsize)
        self.clusters = grow(self.clusters, n_clusters * CLUSTER_DTYPE.itemsize)
        self.presence = grow(self.presence, n_clusters * W * 4)
        return (self.packed[:n_words * 8].view(np.uint64),
                self.seqs[:n_seqs * SEQ_DTYPE.itemsize].view(SEQ_DTYPE),
                self.clusters[:n_clusters * CLUSTER_DTYPE.itemsize].view(CLUSTER_DTYPE),
                self.presence[:n_clusters * W * 4].view(np.uint32).reshape(n_clusters, W))


def synth_batch(device, seed, n_samples, n_clusters, first_cluster=0,
                total_clusters=None, gene_len=1200, n_founders=8,
                founder_div=0.01, private_div=0.001, core_fraction=0.6,
                paralog_rate=0.01, all_targets=False, pinned=False, arena=None):
    """Deterministic synthetic batch (SURVEY.md §8(d)), bases generated on the
    device and returned in host arrays (pinned, reused, when `arena` is given)."""
    lib = load()
    p = SynthParams(seed, n_samples, n_clusters, first_cluster, gene_len,
                    n_founders, founder_div, private_div, core_fraction,
                    paralog_rate, total_clusters or n_clusters,
                    int(all_targets))
    n_seqs, n_words = C.c_uint32(), C.c_uint64()
    rc = lib.pf_synth_plan(C.byref(p), C.byref(n_seqs), C.byref(n_words))
    if rc != 0:
        raise PfError(rc, "pf_synth_plan failed")
    W = lib.pf_pattern_words(n_samples)
    if arena is not None:
        packed, seqs, clusters, presence = arena.take(n_words.value, n_seqs.value, n_clusters, W)
    else:
        seqs = np.zeros(n_seqs.value, SEQ_DTYPE)
        clusters = np.zeros(n_clusters, CLUSTER_DTYPE)
        presence = np.zeros((n_clusters, W), np.uint32)
        if pinned:
            import torch
            packed = torch.empty(max(1, n_words.value), dtype=torch.int64,
                                 pin_memory=True).numpy().view(np.uint64)[:n_words.value]
        else:
            packed = np.zeros(n_words.value, np.uint64)
    rc = lib.pf_synth_fill(device, C.byref(p), seqs.ctypes.data,
                           clusters.ctypes.data, presence.ctypes.data,
                           packed.ctypes.data)
    if rc != 0:
        raise PfError(rc, lib.pf_last_error(None).decode())
    return HostBatch(packed, seqs, clusters, presence)
