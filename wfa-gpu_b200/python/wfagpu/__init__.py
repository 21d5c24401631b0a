"""Python (ctypes) binding of the B200-native WFA-GPU drop-in library.

Mirrors the reference's C API one to one (lib/aligner.h:49-62): an `Aligner`
owns a `wfagpu_aligner_t`, sequences are added with `add_sequences(query,
target)`, `initialize_parameters(x, o, e)` sets the reference defaults, option
fields are poked directly (`aligner.options.compute_cigar = True`), `align()`
runs on the GPU.  There is no CPU path: without the CUDA library or a GPU the
calls fail loudly.
"""
import ctypes as C
import operator
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WFAGPU_LIB") or os.path.normpath(os.path.join(_HERE, "..", "..", "lib", "libwfagpu.so"))

BAND_NONE = -1


class AffinePenalties(C.Structure):
    _fields_ = [("x", C.c_int), ("o", C.c_int), ("e", C.c_int)]


class SequencePair(C.Structure):
    _fields_ = [("text_offset", C.c_size_t), ("pattern_offset", C.c_size_t),
                ("text_offset_packed", C.c_size_t), ("pattern_offset_packed", C.c_size_t),
                ("text_len", C.c_uint), ("pattern_len", C.c_uint), ("has_N", C.c_bool)]


class Cigar(C.Structure):
    _fields_ = [("buffer", C.c_void_p), ("buffer_size", C.c_size_t), ("last_free_position", C.c_size_t)]


class AlignmentResult(C.Structure):
    _fields_ = [("error", C.c_uint), ("cigar", Cigar)]


class AlignmentOptions(C.Structure):
    _fields_ = [("max_error", C.c_int), ("threads_per_block", C.c_int), ("num_workers", C.c_int),
                ("band", C.c_int), ("batch_size", C.c_size_t), ("num_alignments", C.c_size_t),
                ("penalties", AffinePenalties), ("compute_cigar", C.c_bool)]


class AlignerStruct(C.Structure):
    _fields_ = [("sequences_buffer", C.c_void_p), ("sequences_buffer_len", C.c_size_t),
                ("sequences_metadata", C.POINTER(SequencePair)), ("sequences_metadata_len", C.c_size_t),
                ("num_sequence_pairs", C.c_size_t), ("results", C.POINTER(AlignmentResult)),
                ("last_sequence_pair_idx", C.c_int64), ("alignment_options", AlignmentOptions)]


class RunStats(C.Structure):
    _fields_ = [("wall_s", C.c_double), ("gpu_align_ms", C.c_double), ("gpu_pack_ms", C.c_double),
                ("launches", C.c_uint64), ("redispatched", C.c_uint64), ("ascii_pairs", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("devices", C.c_int), ("staged", C.c_int),
                ("failed_pairs", C.c_uint64), ("checked", C.c_uint64), ("incorrect", C.c_uint64)]


class Step(C.Structure):
    _fields_ = [("row_off", C.c_uint32), ("n", C.c_uint16), ("kind", C.c_uint16)]


class Plan(C.Structure):
    _fields_ = [("x", C.c_int), ("o", C.c_int), ("e", C.c_int), ("max_steps", C.c_int), ("band", C.c_int),
                ("band_width", C.c_int), ("with_cigar", C.c_int), ("threads_hint", C.c_int), ("workers_hint", C.c_int),
                ("o2", C.c_int), ("e2", C.c_int),      # gap-affine 2-piece: second piece; e2 = 0 (default): one piece
                ("with_ends", C.c_int)]                # ends-free score only: also find k_begin (default 0: no)


class PairOut(C.Structure):
    _fields_ = [("distance", C.c_int32), ("status", C.c_uint32), ("ops_off", C.c_uint32), ("n_ops", C.c_uint32)]


class BatchStats(C.Structure):
    _fields_ = [("ms_h2d", C.c_float), ("ms_pack", C.c_float), ("ms_align", C.c_float), ("ms_d2h", C.c_float),
                ("ms_total", C.c_float), ("launches", C.c_uint32), ("redispatched", C.c_uint32),
                ("ascii_pairs", C.c_uint32), ("cells", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("ms_wavefront", C.c_float), ("failed_pairs", C.c_uint32), ("pending_pairs", C.c_uint32),
                ("n_cap", C.c_uint32), ("cta_threads", C.c_uint32), ("ctas", C.c_uint32), ("d_end", C.c_uint32),
                ("reserved1", C.c_uint32)]


class Span(C.Structure):
    """wfagpu_span_t: ends-free span in WFA2-lib's order (pattern begin / end, text begin / end)."""
    _fields_ = [("pattern_begin_free", C.c_int), ("pattern_end_free", C.c_int), ("text_begin_free", C.c_int),
                ("text_end_free", C.c_int)]


class Affine2p(C.Structure):
    """wfagpu_affine2p_t: gap-affine 2-piece penalties; a gap of L bases costs min(o1 + e1 L, o2 + e2 L)."""
    _fields_ = [("x", C.c_int), ("o1", C.c_int), ("e1", C.c_int), ("o2", C.c_int), ("e2", C.c_int)]


class Coords(C.Structure):
    """wfagpu_coords_t: the aligned part, pattern[pattern_begin, pattern_end) against text[text_begin, text_end)."""
    _fields_ = [("pattern_begin", C.c_int), ("pattern_end", C.c_int), ("text_begin", C.c_int), ("text_end", C.c_int)]


class DevPair(C.Structure):
    _fields_ = [("p_ascii", C.c_uint32), ("t_ascii", C.c_uint32), ("p_word", C.c_uint32), ("t_word", C.c_uint32),
                ("plen", C.c_uint32), ("tlen", C.c_uint32), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


EXPORTS = [
    "wfagpu_initialize_aligner", "wfagpu_add_sequences", "wfagpu_initialize_parameters",
    "wfagpu_set_batch_size", "wfagpu_align", "wfagpu_destroy_aligner",
    "launch_alignments", "launch_alignments_distance",
    "initialize_wfa_results", "destroy_wfa_results", "insert_ops",
    "get_num_cuda_devices", "get_cuda_dev_name", "get_cuda_SM_count", "get_cuda_capability",
    "wfagpu_build_step_table", "wfagpu_device_open", "wfagpu_device_close_all", "wfagpu_device_upload",
    "wfagpu_device_align", "wfagpu_device_download", "wfagpu_device_last_stats", "wfagpu_device_sm_count",
    "wfagpu_device_pack_only", "wfagpu_ops_to_cigar", "wfagpu_set_devices", "wfagpu_last_run_stats",
    "wfagpu_synth_add_pairs", "wfagpu_device_wait", "wfagpu_host_register", "wfagpu_host_unregister",
    "wfagpu_pairs_from_metadata", "wfagpu_reset_results", "wfagpu_read_seq_file", "wfagpu_read_fasta_files",
    "wfagpu_check_result", "wfagpu_last_launch_ok", "wfagpu_plan_chunks", "wfagpu_plan_shares", "wfagpu_share_take",
    "check_cigar_edit", "check_affine_distance", "wfagpu_cigar_append", "wfagpu_device_download_text",
    "recover_cigar", "wfagpu_unroll_cigar", "wfagpu_device_release", "wfagpu_device_rescore", "wfagpu_device_staging",
    "wfagpu_host_is_pinned", "wfagpu_host_alloc", "wfagpu_host_free", "wfagpu_reserve", "wfagpu_parse_devices",
    "wfagpu_set_host_threads", "wfagpu_align_span", "wfagpu_launch_alignments_span", "wfagpu_device_align_span",
    "wfagpu_device_download_ends", "wfagpu_device_rescore_span", "wfagpu_ops_to_cigar_span",
    "wfagpu_check_result_span", "wfagpu_build_step_table_span", "wfagpu_align_affine2p",
    "wfagpu_launch_alignments_affine2p", "wfagpu_check_result_affine2p", "wfagpu_build_step_table_affine2p",
    "wfagpu_align_span_coords", "wfagpu_launch_alignments_span_coords", "wfagpu_align_spans",
    "wfagpu_launch_alignments_spans", "wfagpu_device_align_spans", "wfagpu_device_rescore_spans",
]

_lib = None


def load():
    """Load lib/libwfagpu.so (built by wfa-gpu_b200/Makefile). Raises if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make -C wfa-gpu_b200` "
            "(this package has no CPU or PyTorch fallback)")
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    L.wfagpu_initialize_aligner.argtypes = [P(AlignerStruct)]
    L.wfagpu_initialize_aligner.restype = C.c_bool
    L.wfagpu_add_sequences.argtypes = [P(AlignerStruct), C.c_char_p, C.c_char_p]
    L.wfagpu_add_sequences.restype = C.c_bool
    L.wfagpu_initialize_parameters.argtypes = [P(AlignerStruct), AffinePenalties]
    L.wfagpu_initialize_parameters.restype = C.c_bool
    L.wfagpu_set_batch_size.argtypes = [P(AlignerStruct), C.c_size_t]
    L.wfagpu_set_batch_size.restype = C.c_bool
    L.wfagpu_align.argtypes = [P(AlignerStruct)]
    L.wfagpu_align.restype = C.c_bool
    L.wfagpu_destroy_aligner.argtypes = [P(AlignerStruct)]
    L.wfagpu_destroy_aligner.restype = None
    L.wfagpu_set_devices.argtypes = [C.c_char_p]
    L.wfagpu_read_seq_file.argtypes = [P(AlignerStruct), C.c_char_p, C.c_size_t]
    L.wfagpu_read_seq_file.restype = C.c_long
    L.wfagpu_read_fasta_files.argtypes = [P(AlignerStruct), C.c_char_p, C.c_char_p, C.c_size_t]
    L.wfagpu_read_fasta_files.restype = C.c_long
    L.wfagpu_check_result.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, AffinePenalties, C.c_uint, C.c_char_p]
    L.wfagpu_check_result.restype = C.c_bool
    L.wfagpu_plan_chunks.argtypes = [C.c_size_t, C.c_size_t, C.c_int, C.c_size_t, P(C.c_size_t), P(C.c_size_t)]
    L.wfagpu_plan_chunks.restype = None
    L.wfagpu_plan_shares.argtypes = [C.c_size_t, C.c_int, P(C.c_size_t), P(C.c_size_t)]
    L.wfagpu_plan_shares.restype = None
    L.wfagpu_share_take.argtypes = [P(C.c_size_t), P(C.c_size_t), C.c_int, C.c_int, C.c_size_t, C.c_size_t, P(C.c_size_t), P(C.c_size_t)]
    L.wfagpu_share_take.restype = C.c_bool
    L.wfagpu_reset_results.argtypes = [P(AlignerStruct)]
    L.wfagpu_reset_results.restype = None
    L.wfagpu_last_run_stats.argtypes = [P(RunStats)]
    L.wfagpu_synth_add_pairs.argtypes = [P(AlignerStruct), C.c_uint64, C.c_size_t, C.c_int, C.c_double, C.c_double]
    L.wfagpu_synth_add_pairs.restype = C.c_bool
    L.wfagpu_build_step_table.argtypes = [C.c_int] * 6 + [P(Step), P(C.c_uint64)]
    L.wfagpu_ops_to_cigar.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int,
                                      P(C.c_uint32), C.c_uint32, P(Cigar)]
    L.wfagpu_ops_to_cigar.restype = C.c_bool
    L.initialize_wfa_results.argtypes = [P(P(AlignmentResult)), C.c_size_t, C.c_size_t]
    L.initialize_wfa_results.restype = C.c_bool
    L.destroy_wfa_results.argtypes = [P(AlignmentResult), C.c_size_t]
    L.destroy_wfa_results.restype = C.c_bool
    L.get_num_cuda_devices.argtypes = [P(C.c_int)]
    L.get_cuda_SM_count.argtypes = [C.c_int]
    L.get_cuda_dev_name.argtypes = [C.c_int]
    L.get_cuda_dev_name.restype = C.c_void_p
    L.wfagpu_device_open.argtypes = [C.c_int]
    L.wfagpu_device_open.restype = C.c_void_p
    L.wfagpu_device_pack_only.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, P(DevPair), C.c_size_t,
                                          P(C.c_uint32), C.c_size_t]
    L.wfagpu_device_upload.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, P(DevPair), C.c_size_t]
    L.wfagpu_device_align.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), C.c_int]
    L.wfagpu_device_wait.argtypes = [C.c_void_p, C.c_int, P(C.c_float), P(C.c_float)]
    L.wfagpu_device_download.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(PairOut), P(P(C.c_uint32)),
                                         P(C.c_size_t), P(C.c_uint32)]
    L.wfagpu_device_last_stats.argtypes = [C.c_void_p, C.c_int, P(BatchStats)]
    L.wfagpu_device_sm_count.argtypes = [C.c_void_p]
    L.wfagpu_device_release.argtypes = [C.c_void_p]
    L.wfagpu_device_release.restype = None
    L.wfagpu_device_rescore.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), P(C.c_int32)]
    L.wfagpu_host_is_pinned.argtypes = [C.c_void_p]
    L.wfagpu_unroll_cigar.argtypes = [C.c_char_p]
    L.wfagpu_unroll_cigar.restype = C.c_void_p
    L.check_cigar_edit.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_char_p]
    L.check_cigar_edit.restype = C.c_bool
    L.check_affine_distance.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, AffinePenalties, C.c_char_p]
    L.check_affine_distance.restype = C.c_bool
    L.wfagpu_parse_devices.argtypes = [C.c_char_p, C.c_int, P(C.c_int), C.c_int]
    L.launch_alignments.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult), AlignmentOptions, C.c_bool]
    L.launch_alignments.restype = None
    L.launch_alignments_distance.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult), AlignmentOptions, C.c_bool]
    L.launch_alignments_distance.restype = None
    L.wfagpu_host_register.argtypes = [C.c_void_p, C.c_size_t]
    L.wfagpu_host_unregister.argtypes = [C.c_void_p]
    L.wfagpu_pairs_from_metadata.argtypes = [P(SequencePair), C.c_size_t, C.c_size_t, C.c_size_t, P(DevPair),
                                             P(C.c_size_t), P(C.c_size_t)]
    L.wfagpu_align_span.argtypes = [P(AlignerStruct), P(Span)]
    L.wfagpu_align_span.restype = C.c_bool
    L.wfagpu_launch_alignments_span.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult),
                                                AlignmentOptions, C.c_bool, C.c_bool, P(Span)]
    L.wfagpu_launch_alignments_span.restype = None
    L.wfagpu_device_align_span.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), C.c_int, P(Span)]
    L.wfagpu_device_download_ends.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(C.c_int32)]
    L.wfagpu_device_rescore_span.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), P(Span), P(C.c_int32)]
    L.wfagpu_ops_to_cigar_span.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int,
                                           P(C.c_uint32), C.c_uint32, P(Cigar)]
    L.wfagpu_ops_to_cigar_span.restype = C.c_bool
    L.wfagpu_check_result_span.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, AffinePenalties, P(Span),
                                           C.c_uint, C.c_char_p]
    L.wfagpu_check_result_span.restype = C.c_bool
    L.wfagpu_build_step_table_span.argtypes = [C.c_int] * 6 + [P(Step), P(C.c_uint64)]
    L.wfagpu_align_affine2p.argtypes = [P(AlignerStruct), P(Affine2p)]
    L.wfagpu_align_affine2p.restype = C.c_bool
    L.wfagpu_launch_alignments_affine2p.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult),
                                                    AlignmentOptions, C.c_bool, C.c_bool, P(Affine2p)]
    L.wfagpu_launch_alignments_affine2p.restype = None
    L.wfagpu_check_result_affine2p.argtypes = [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, P(Affine2p), C.c_uint,
                                               C.c_char_p]
    L.wfagpu_check_result_affine2p.restype = C.c_bool
    L.wfagpu_build_step_table_affine2p.argtypes = [C.c_int] * 7 + [P(Step), P(C.c_uint64)]
    L.wfagpu_align_span_coords.argtypes = [P(AlignerStruct), P(Span), P(Coords)]
    L.wfagpu_align_span_coords.restype = C.c_bool
    L.wfagpu_launch_alignments_span_coords.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult),
                                                       AlignmentOptions, C.c_bool, C.c_bool, P(Span), P(Coords)]
    L.wfagpu_launch_alignments_span_coords.restype = None
    L.wfagpu_align_spans.argtypes = [P(AlignerStruct), P(Span), P(Coords)]
    L.wfagpu_align_spans.restype = C.c_bool
    L.wfagpu_launch_alignments_spans.argtypes = [C.c_void_p, C.c_size_t, P(SequencePair), P(AlignmentResult),
                                                 AlignmentOptions, C.c_bool, C.c_bool, P(Span), P(Coords)]
    L.wfagpu_launch_alignments_spans.restype = None
    L.wfagpu_device_align_spans.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), C.c_int, P(Span)]
    L.wfagpu_device_rescore_spans.argtypes = [C.c_void_p, C.c_int, C.c_size_t, P(Plan), P(Span), P(C.c_int32)]
    _lib = L
    return L


def span_of(ends_free):
    """A 4-tuple (pattern_begin_free, pattern_end_free, text_begin_free, text_end_free) -> Span (None -> None)."""
    if ends_free is None:
        return None
    vals = tuple(int(v) for v in ends_free)
    if len(vals) != 4:
        raise ValueError("ends_free takes four values: pattern_begin_free, pattern_end_free, text_begin_free, text_end_free")
    return Span(*vals)


def spans_of(ends_free, num_pairs):
    """Per-pair ends-free spans: a sequence of `num_pairs` 4-tuples, or an (num_pairs, 4) array -> a Span array.
    ValueError for another count or shape."""
    try:
        rows = [tuple(operator.index(v) for v in r) for r in ends_free]
    except TypeError:
        raise ValueError("ends_free: give one span of four integers per pair, or a single 4-tuple") from None
    if len(rows) != num_pairs:
        raise ValueError(f"ends_free has {len(rows)} spans for {num_pairs} pairs: give one per pair, or a single 4-tuple")
    if any(len(r) != 4 for r in rows):
        raise ValueError("every per-pair span takes four values: pattern_begin_free, pattern_end_free, "
                         "text_begin_free, text_end_free")
    return (Span * num_pairs)(*(Span(*r) for r in rows))


def _per_pair(ends_free):
    """True when ends_free holds one span per pair (its entries are sequences), False for a single 4-tuple."""
    if ends_free is None or len(ends_free) == 0:
        return ends_free is not None
    try:
        iter(ends_free[0])
    except TypeError:
        return False
    return True


def affine2p_of(pen):
    """A 5-tuple (x, o1, e1, o2, e2) -> Affine2p (None -> None)."""
    if pen is None:
        return None
    vals = tuple(int(v) for v in pen)
    if len(vals) != 5:
        raise ValueError("affine2p takes five values: x, o1, e1, o2, e2")
    return Affine2p(*vals)


def _b(s):
    return s if isinstance(s, bytes) else s.encode()


class Aligner:
    """Drop-in counterpart of the reference's wfagpu_aligner_t workflow."""

    def __init__(self):
        self.L = load()
        self.s = AlignerStruct()
        if not self.L.wfagpu_initialize_aligner(C.byref(self.s)):
            raise RuntimeError("wfagpu_initialize_aligner failed")
        self._alive = True
        self._coords = None

    # -- reference API -------------------------------------------------------
    def add_sequences(self, query, target):
        return bool(self.L.wfagpu_add_sequences(C.byref(self.s), _b(query), _b(target)))

    def initialize_parameters(self, x, o, e):
        return bool(self.L.wfagpu_initialize_parameters(C.byref(self.s), AffinePenalties(x, o, e)))

    def set_batch_size(self, n):
        return bool(self.L.wfagpu_set_batch_size(C.byref(self.s), n))

    @property
    def options(self):
        return self.s.alignment_options

    def align(self, ends_free=None, affine2p=None, coords=False):
        """ends_free: None (global) or (pattern_begin_free, pattern_end_free, text_begin_free, text_end_free),
        WFA2-lib's order: that many leading / trailing bases of either sequence are free (wfagpu_align_span).  Or one
        such span per pair: a sequence of num_pairs 4-tuples or an (num_pairs, 4) array (wfagpu_align_spans); a pair
        whose span is all zero gets its global alignment.
        affine2p: None or (x, o1, e1, o2, e2), gap-affine 2-piece penalties for this call in place of the aligner's
        (wfagpu_align_affine2p); global alignment only.
        coords: also record where every alignment lies, with or without a CIGAR (wfagpu_align_span_coords); read
        them with coords().  Not with affine2p."""
        per_pair = _per_pair(ends_free)
        sp = spans_of(ends_free, self.num_pairs) if per_pair else span_of(ends_free)
        pen2 = affine2p_of(affine2p)
        self._coords = None
        if pen2 is not None:
            if sp is not None:
                raise ValueError("affine2p cannot be combined with ends_free")
            if coords:
                raise ValueError("affine2p cannot be combined with coords")
            if not self.L.wfagpu_align_affine2p(C.byref(self.s), C.byref(pen2)):
                raise RuntimeError("wfagpu_align_affine2p failed (see stderr); there is no CPU fallback")
            return True
        if per_pair:
            cs = (Coords * self.num_pairs)() if coords else None
            if not self.L.wfagpu_align_spans(C.byref(self.s), sp, cs):
                raise RuntimeError("wfagpu_align_spans failed (see stderr); there is no CPU fallback")
            self._coords = cs
            return True
        if coords:
            cs = (Coords * self.num_pairs)()
            if not self.L.wfagpu_align_span_coords(C.byref(self.s), C.byref(sp) if sp is not None else None, cs):
                raise RuntimeError("wfagpu_align_span_coords failed (see stderr); there is no CPU fallback")
            self._coords = cs
            return True
        if sp is None:
            if not self.L.wfagpu_align(C.byref(self.s)):
                raise RuntimeError("wfagpu_align failed (see stderr); there is no CPU fallback")
            return True
        if not self.L.wfagpu_align_span(C.byref(self.s), C.byref(sp)):
            raise RuntimeError("wfagpu_align_span failed (see stderr); there is no CPU fallback")
        return True

    def destroy(self):
        if self._alive:
            self.L.wfagpu_destroy_aligner(C.byref(self.s))
            self._alive = False

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass

    # -- conveniences ----------------------------------------------------------
    @property
    def num_pairs(self):
        return self.s.num_sequence_pairs

    def error(self, i):
        return self.s.results[i].error

    def cigar(self, i):
        buf = self.s.results[i].cigar.buffer
        return C.string_at(buf).decode() if buf else ""

    def errors(self):
        return [self.s.results[i].error for i in range(self.num_pairs)]

    def cigars(self):
        return [self.cigar(i) for i in range(self.num_pairs)]

    def coords(self):
        """(pattern_begin, pattern_end, text_begin, text_end) of every pair of the last align(coords=True): the
        alignment covers pattern[pattern_begin:pattern_end] and text[text_begin:text_end]; all -1 for a pair that
        was not aligned."""
        if self._coords is None:
            raise RuntimeError("no coordinates: call align(..., coords=True) first")
        return [(c.pattern_begin, c.pattern_end, c.text_begin, c.text_end) for c in self._coords]

    def pair(self, i):
        m = self.s.sequences_metadata[i]
        base = self.s.sequences_buffer
        p = C.string_at(base + m.pattern_offset, m.pattern_len)
        t = C.string_at(base + m.text_offset, m.text_len)
        return p.decode(), t.decode()

    def read_seq_file(self, path, max_pairs=0):
        return self.L.wfagpu_read_seq_file(C.byref(self.s), _b(path), max_pairs)

    def read_fasta_files(self, query_path, target_path, max_pairs=0):
        return self.L.wfagpu_read_fasta_files(C.byref(self.s), _b(query_path), _b(target_path), max_pairs)

    def add_synthetic(self, seed, n, length, err_lo, err_hi=None):
        if err_hi is None:
            err_hi = err_lo
        ok = self.L.wfagpu_synth_add_pairs(C.byref(self.s), seed, n, length, err_lo, err_hi)
        if not ok:
            raise RuntimeError("wfagpu_synth_add_pairs failed")

    def reset_results(self):
        self.L.wfagpu_reset_results(C.byref(self.s))

    def host_buffer_pinned(self):
        """True when the sequence buffer is page-locked (wfagpu_initialize_aligner allocates it that way)."""
        return bool(self.L.wfagpu_host_is_pinned(self.s.sequences_buffer))

    def pin_host_buffers(self):
        """Page-lock the sequence buffer so H2D copies are asynchronous DMA (a no-op for the aligner's own buffer)."""
        if self.host_buffer_pinned():
            return True
        return self.L.wfagpu_host_register(self.s.sequences_buffer, self.s.sequences_buffer_len) == 0

    def align_checked(self):
        """launch_alignments* with check_correctness = true; returns (checked, incorrect)."""
        o = self.s.alignment_options
        fn = self.L.launch_alignments if o.compute_cigar else self.L.launch_alignments_distance
        fn(self.s.sequences_buffer, self.s.sequences_buffer_len, self.s.sequences_metadata, self.s.results, o, True)
        st = self.run_stats()
        return st["checked"], st["incorrect"]

    def unpin_host_buffers(self):
        self.L.wfagpu_host_unregister(self.s.sequences_buffer)

    def run_stats(self):
        st = RunStats()
        self.L.wfagpu_last_run_stats(C.byref(st))
        return {k: getattr(st, k) for k, _ in RunStats._fields_}


def set_host_threads(n):
    load().wfagpu_set_host_threads(int(n))


def set_devices(spec):
    load().wfagpu_set_devices(_b(spec) if spec is not None else None)


class ResidentBatch:
    """A batch kept resident in HBM on one device: upload once, re-run the hot path
    (pack + align + traceback kernels) any number of times.  Used by bench.py for the
    device-resident throughput and by the tests to reach the C-ABI device layer."""

    def __init__(self, aligner, device=0, slot=0):
        self.L = load()
        self.a = aligner
        self.slot = slot
        self.dev = self.L.wfagpu_device_open(device)
        if not self.dev:
            raise RuntimeError("no usable CUDA device (and no CPU fallback)")
        n = aligner.num_pairs
        self.n = n
        self.pairs = (DevPair * n)()
        base, nbytes = C.c_size_t(), C.c_size_t()
        if self.L.wfagpu_pairs_from_metadata(aligner.s.sequences_metadata, 0, n, aligner.s.sequences_buffer_len,
                                             self.pairs, C.byref(base), C.byref(nbytes)):
            raise RuntimeError("bad sequence metadata")
        self.base, self.nbytes = base.value, nbytes.value

    def upload(self):
        if self.L.wfagpu_device_upload(self.dev, self.slot, self.a.s.sequences_buffer + self.base, self.nbytes,
                                       self.pairs, self.n):
            raise RuntimeError("upload failed")

    def plan(self, cigar=None):
        o = self.a.options
        return Plan(o.penalties.x, o.penalties.o, o.penalties.e, o.max_error, o.band, o.threads_per_block,
                    int(o.compute_cigar if cigar is None else cigar), o.threads_per_block, o.num_workers)

    def align(self, plan=None):
        plan = plan or self.plan()
        rc = self.L.wfagpu_device_align(self.dev, self.slot, self.n, C.byref(plan), 1)
        if rc:
            raise RuntimeError(f"wfagpu_device_align failed ({rc})")

    def wait(self):
        mp, ma = C.c_float(), C.c_float()
        if self.L.wfagpu_device_wait(self.dev, self.slot, C.byref(mp), C.byref(ma)):
            raise RuntimeError("device wait failed")
        return mp.value, ma.value

    def download(self):
        out = (PairOut * self.n)()
        ops = C.POINTER(C.c_uint32)()
        used = C.c_size_t()
        rc = self.L.wfagpu_device_download(self.dev, self.slot, self.n, out, C.byref(ops), C.byref(used), None)
        if rc:
            raise RuntimeError(f"wfagpu_device_download failed ({rc})")
        return out, ops, used.value

    def stats(self):
        st = BatchStats()
        self.L.wfagpu_device_last_stats(self.dev, self.slot, C.byref(st))
        return {k: getattr(st, k) for k, _ in BatchStats._fields_}

    def sm_count(self):
        return self.L.wfagpu_device_sm_count(self.dev)

    def rescore(self, plan=None):
        """Independent score-only re-computation of the resident batch (the -c path)."""
        plan = plan or self.plan()
        out = (C.c_int32 * self.n)()
        if self.L.wfagpu_device_rescore(self.dev, self.slot, self.n, C.byref(plan), out):
            raise RuntimeError("wfagpu_device_rescore failed")
        return list(out)

    def release(self):
        """Hand the leased device context back to the pool."""
        if self.dev:
            self.L.wfagpu_device_release(self.dev)
            self.dev = None
