"""ctypes binding of the C ABI in include/dmnd_b200.h (the product library diamond_b200/libdmnd_b200.so).

This is a thin harness for tests, bench.py and multi-GPU launch: block images are built with numpy, everything else
happens behind the C ABI.  There is no Python/torch compute path and no CPU fallback: `load()` raises if the CUDA
library is missing, and `Context()` raises if it cannot open a CUDA device.

`load(path)` can also open the test-only oracle build (oracle/_build/libdmnd_oracle.so); only tests/, smoke() and
bench.py's cpu_baseline leg do that.
"""
from __future__ import annotations
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PRODUCT_LIB = os.path.join(HERE, "libdmnd_b200.so")
PADDING = 256
DELIMITER = 31
MAX_SHAPES, MAX_WEIGHT = 64, 12


class Params(C.Structure):
    _fields_ = [("score", C.c_int8 * 1024), ("gap_open", C.c_int32), ("gap_extend", C.c_int32),
                ("reduction", C.c_uint8 * 32), ("map8", C.c_uint8 * 32), ("map8b", C.c_uint8 * 32),
                ("reduction_size", C.c_int32), ("n_shapes", C.c_int32), ("shape_weight", C.c_int32),
                ("shape_len", C.c_int32 * MAX_SHAPES), ("shape_mask", C.c_uint32 * MAX_SHAPES),
                ("shape_pos", (C.c_int32 * MAX_WEIGHT) * MAX_SHAPES), ("hamming_id", C.c_int32),
                ("seedp_bits", C.c_int32), ("index_chunks", C.c_int32), ("seed_cut", C.c_double),
                ("left_most_interval", C.c_int32), ("ungapped_window", C.c_int32), ("ungapped_evalue", C.c_double),
                ("ungapped_cutoff", C.c_int32 * 32), ("short_query_ungapped_cutoff", C.c_int32), ("short_query_max_len", C.c_int32),
                ("gapped_filter_evalue", C.c_double), ("gapped_cutoff1", (C.c_int16 * 32) * 32), ("gapped_cutoff2", (C.c_int16 * 32) * 32),
                ("gapped_filter_diag_score", C.c_int32), ("gapped_filter_window", C.c_int32),
                ("background_scores_f32", C.c_float * 20),
                ("tantan_lr", C.c_float * 1024), ("tantan_d", C.c_float * 50), ("tantan_b2b", C.c_float), ("tantan_f2f", C.c_float),
                ("tantan_p_repeat_end", C.c_float), ("tantan_p_mask", C.c_float), ("max_motif_len", C.c_int32),
                ("query_contexts", C.c_int32), ("ungapped_cutoff_short", C.c_int32 * 32)]


class Hit(C.Structure):
    _fields_ = [("query", C.c_uint32), ("seed_offset", C.c_int32), ("subject_score", C.c_uint64)]


class StageCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("seeds_hit", "seed_hits", "tentative_matches1", "tentative_matches2",
                                          "tentative_matches3", "masked_seeds")]


class DpProblem(C.Structure):
    _fields_ = [("query", C.c_uint32), ("target", C.c_uint32), ("d_begin", C.c_int32), ("d_end", C.c_int32)]


class DpResult(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("score", "q_begin", "q_end", "t_begin", "t_end", "identities", "mismatches",
                                         "gap_openings", "length", "gaps", "positives")] + \
               [("transcript_off", C.c_uint32), ("transcript_len", C.c_uint32), ("status", C.c_int32)]


class Timing(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("seed_ms", "dp_score_ms", "dp_trace_ms", "h2d_ms", "d2h_ms")] + \
               [(n, C.c_uint64) for n in ("launches", "h2d_bytes", "d2h_bytes", "dp_cells_score", "dp_cells_trace", "dp_cells_padded", "dp_overflow_reruns")]


class SearchOpts(C.Structure):
    _fields_ = [("sensitivity", C.c_int32), ("threads", C.c_int32), ("index_chunks", C.c_int32),
                ("comp_based_stats", C.c_int32), ("max_target_seqs", C.c_int32), ("max_evalue", C.c_double),
                ("db_letters", C.c_uint64), ("want_transcript", C.c_int32), ("masking", C.c_int32), ("motif_masking", C.c_int32), ("query_contexts", C.c_int32), ("top_percent", C.c_double),
                ("frame_shift", C.c_int32), ("range_culling", C.c_int32),
                ("min_id", C.c_double), ("query_cover", C.c_double), ("subject_cover", C.c_double), ("min_bit_score", C.c_double), ("approx_min_id", C.c_double), ("self_targets", C.c_void_p), ("range_cover", C.c_double), ("ext_mode", C.c_int32)]


class Match(C.Structure):
    _fields_ = [("query", C.c_uint32), ("target", C.c_uint32), ("score", C.c_int32), ("evalue", C.c_double),
                ("bit_score", C.c_double)] + \
               [(n, C.c_int32) for n in ("q_begin", "q_end", "t_begin", "t_end", "identities", "mismatches",
                                         "gap_openings", "length", "gaps", "positives")] + \
               [("transcript_off", C.c_uint64), ("transcript_len", C.c_uint32), ("reserved", C.c_uint32)]


class RunStats(C.Structure):
    _fields_ = [("seed", StageCounters)] + \
               [(n, C.c_uint64) for n in ("hits", "targets", "dp_problems_round1", "dp_problems_round2", "cells_round1",
                                          "cells_round2", "queries_aligned", "matches", "dp_problems_fused", "targets_extended")] + \
               [(n, C.c_double) for n in ("seed_ms", "host_bridge_ms", "dp1_ms", "dp2_ms", "total_ms")] + \
               [("device", Timing)]


MATCH_DTYPE = np.dtype([("query", "<u4"), ("target", "<u4"), ("score", "<i4"), ("_pad", "<i4"), ("evalue", "<f8"),
                        ("bit_score", "<f8"), ("q_begin", "<i4"), ("q_end", "<i4"), ("t_begin", "<i4"), ("t_end", "<i4"),
                        ("identities", "<i4"), ("mismatches", "<i4"), ("gap_openings", "<i4"), ("length", "<i4"),
                        ("gaps", "<i4"), ("positives", "<i4"), ("transcript_off", "<u8"), ("transcript_len", "<u4"),
                        ("reserved", "<u4")])
assert MATCH_DTYPE.itemsize == C.sizeof(Match), (MATCH_DTYPE.itemsize, C.sizeof(Match))
HIT_DTYPE = np.dtype([("query", "<u4"), ("seed_offset", "<i4"), ("subject_score", "<u8")])
CHAIN_QUERY_DTYPE = np.dtype([("query", "<u4"), ("n_targets", "<u4"), ("n_problems", "<u4"), ("first", "<u4"), ("n_hits", "<u4"), ("flags", "<u4")])
RESULT_DTYPE = np.dtype([(n, "<i4") for n in ("score", "q_begin", "q_end", "t_begin", "t_end", "identities", "mismatches",
                                               "gap_openings", "length", "gaps", "positives")] +
                        [("transcript_off", "<u4"), ("transcript_len", "<u4"), ("status", "<i4")])
SEGMENT_DTYPE = np.dtype([("i", "<i4"), ("j", "<i4"), ("len", "<i4"), ("score", "<i4")])
PROBLEM_DTYPE = np.dtype([("query", "<u4"), ("target", "<u4"), ("d_begin", "<i4"), ("d_end", "<i4")])
FS_RESULT_DTYPE = np.dtype([(n, "<i4") for n in ("score", "q_begin", "q_end", "frame_begin", "frame_end", "t_begin", "t_end", "identities", "mismatches",
                                                  "gap_openings", "length", "gaps", "positives")] +
                           [("transcript_off", "<u4"), ("transcript_len", "<u4"), ("status", "<i4")])  # dmnd_fs_result

# every symbol include/dmnd_b200.h declares (tests/test_abi.py checks the product library exports them all)
SYMBOLS = ["dmnd_last_error", "dmnd_set_last_error", "dmnd_backend", "dmnd_ctx_params", "dmnd_create", "dmnd_destroy", "dmnd_ctx_lane", "dmnd_block_upload",
           "dmnd_block_upload_ranges", "dmnd_block_range_wait", "dmnd_block_compute_bias_range", "dmnd_block_free", "dmnd_block_set_bias", "dmnd_block_download_letters", "dmnd_debug_block_soft", "dmnd_debug_ref_index", "dmnd_debug_left_most", "dmnd_block_build_index", "dmnd_block_compute_bias", "dmnd_block_download_bias", "dmnd_block_download_bias_async", "dmnd_copy_wait", "dmnd_host_alloc", "dmnd_host_free", "dmnd_hits_xdrop", "dmnd_hits_xdrop_sites", "dmnd_block_clear_seed_mask", "dmnd_block_clear_seed_mask_range", "dmnd_block_mask", "dmnd_block_mask_fetch", "dmnd_hits_gapped_filter", "dmnd_comm_unique_id", "dmnd_comm_init", "dmnd_comm_destroy", "dmnd_block_broadcast", "dmnd_block_alloc_empty", "dmnd_block_geometry", "dmnd_block_download_limits", "dmnd_hits_chain", "dmnd_hits_chain_fetch", "dmnd_banded_swipe_chained",
           "dmnd_search_shape", "dmnd_search_shape_range", "dmnd_hits_count", "dmnd_hits_download", "dmnd_hits_free", "dmnd_banded_swipe", "dmnd_banded_3frame_swipe",
           "dmnd_timing_fetch", "dmnd_measure_int_peak", "dmnd_measure_int_peak_packed", "dmnd_search_opts_default", "dmnd_mode_motif_masking", "dmnd_alignment_stats", "dmnd_params_init", "dmnd_blastp", "dmnd_blastp_resident",
           "dmnd_result_matches", "dmnd_result_transcripts", "dmnd_result_stats", "dmnd_result_masked_positions", "dmnd_result_unaligned", "dmnd_result_free"]


def load(path: str | None = None) -> C.CDLL:
    path = path or PRODUCT_LIB
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `make lib` (there is no fallback implementation)")
    lib = C.CDLL(path)
    vp, i8p, i64p = C.c_void_p, C.POINTER(C.c_int8), C.POINTER(C.c_int64)
    lib.dmnd_last_error.restype = C.c_char_p
    lib.dmnd_backend.restype = C.c_char_p
    lib.dmnd_create.argtypes = [C.c_int, C.POINTER(Params), C.POINTER(vp)]
    lib.dmnd_destroy.argtypes = [vp]
    lib.dmnd_destroy.restype = None
    lib.dmnd_block_upload.argtypes = [vp, vp, C.c_size_t, vp, C.c_uint32, C.POINTER(vp)]
    lib.dmnd_block_free.argtypes = [vp, vp]
    lib.dmnd_block_free.restype = None
    lib.dmnd_block_set_bias.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_block_download_letters.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_debug_block_soft.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_debug_ref_index.argtypes = [vp, vp, C.c_int, vp, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.dmnd_debug_left_most.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_uint32, C.c_uint32, vp]
    lib.dmnd_block_mask.argtypes = [vp, vp, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]
    lib.dmnd_block_mask_fetch.argtypes = [vp, vp, C.c_size_t]
    lib.dmnd_comm_unique_id.argtypes = [vp]
    lib.dmnd_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.dmnd_comm_destroy.argtypes = [vp]
    lib.dmnd_comm_destroy.restype = None
    lib.dmnd_block_broadcast.argtypes = [vp, C.c_int, vp, C.POINTER(vp)]
    lib.dmnd_block_alloc_empty.argtypes = [vp, C.c_size_t, C.c_uint32, C.POINTER(vp)]
    lib.dmnd_block_geometry.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_uint32)]
    lib.dmnd_block_download_limits.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_hits_chain.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp]
    lib.dmnd_hits_chain_fetch.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.dmnd_banded_swipe_chained.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, vp, vp, C.c_size_t]
    lib.dmnd_banded_3frame_swipe.argtypes = [vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, vp, vp, C.c_size_t]
    lib.dmnd_hits_gapped_filter.argtypes = [vp, vp, vp, vp, vp, C.c_size_t]
    lib.dmnd_block_clear_seed_mask.argtypes = [vp, vp]
    lib.dmnd_block_build_index.argtypes = [vp, vp, C.c_int]
    lib.dmnd_block_compute_bias.argtypes = [vp, vp, C.c_int]
    lib.dmnd_block_download_bias.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_search_shape.argtypes = [vp, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(StageCounters)]
    lib.dmnd_search_shape_range.argtypes = [vp, vp, vp, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(vp), C.POINTER(StageCounters)]
    lib.dmnd_block_clear_seed_mask_range.argtypes = [vp, vp, C.c_uint32, C.c_uint32]
    lib.dmnd_ctx_lane.argtypes = [vp, C.c_int, C.POINTER(vp)]
    lib.dmnd_hits_count.argtypes = [vp]
    lib.dmnd_hits_count.restype = C.c_size_t
    lib.dmnd_hits_download.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_hits_xdrop.argtypes = [vp, vp, vp, vp, C.c_int, vp, C.c_size_t]
    lib.dmnd_block_download_bias_async.argtypes = [vp, vp, vp, C.c_size_t]
    lib.dmnd_copy_wait.argtypes = [vp]
    lib.dmnd_host_alloc.argtypes = [vp, C.c_size_t]
    lib.dmnd_host_alloc.restype = vp
    lib.dmnd_host_free.argtypes = [vp, vp]
    lib.dmnd_host_free.restype = None
    lib.dmnd_hits_free.argtypes = [vp, vp]
    lib.dmnd_hits_free.restype = None
    lib.dmnd_banded_swipe.argtypes = [vp, vp, vp, vp, C.c_size_t, C.c_int, vp, vp, C.c_size_t]
    lib.dmnd_timing_fetch.argtypes = [vp, C.POINTER(Timing), C.c_int]
    lib.dmnd_measure_int_peak.argtypes = [vp, C.POINTER(C.c_double)]
    lib.dmnd_measure_int_peak_packed.argtypes = [vp, C.POINTER(C.c_double)]
    lib.dmnd_search_opts_default.argtypes = [C.POINTER(SearchOpts)]
    lib.dmnd_search_opts_default.restype = None
    lib.dmnd_params_init.argtypes = [C.POINTER(SearchOpts), C.POINTER(Params)]
    lib.dmnd_blastp.argtypes = [vp, vp, C.c_size_t, vp, C.c_uint32, vp, C.c_size_t, vp, C.c_uint32, C.POINTER(SearchOpts),
                                C.POINTER(vp)]
    lib.dmnd_blastp_resident.argtypes = [vp, vp, vp, vp, vp, C.c_uint32, vp, vp, C.c_uint32, C.POINTER(SearchOpts),
                                         C.POINTER(vp)]
    lib.dmnd_result_matches.argtypes = [vp, C.POINTER(C.c_size_t)]
    lib.dmnd_result_matches.restype = vp
    lib.dmnd_result_transcripts.argtypes = [vp, C.POINTER(C.c_size_t)]
    lib.dmnd_result_transcripts.restype = vp
    lib.dmnd_result_stats.argtypes = [vp]
    lib.dmnd_result_stats.restype = C.POINTER(RunStats)
    lib.dmnd_result_free.argtypes = [vp]
    lib.dmnd_result_free.restype = None
    return lib


class DmndError(RuntimeError):
    pass


def block_image(letters: np.ndarray, offsets: np.ndarray):
    """Flat encoded letters + offsets (n+1) -> the reference's block image (data/string_set.h:26-78):
    256 B of delimiter, each sequence followed by one delimiter, 256 B of delimiter; limits[i] = start of seq i."""
    letters = np.ascontiguousarray(letters, dtype=np.int8)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    lens = np.diff(offsets)
    limits = np.empty(n + 1, dtype=np.int64)
    limits[0] = PADDING
    np.cumsum(lens + 1, out=limits[1:])
    limits[1:] += PADDING
    raw = np.full(int(limits[-1]) + PADDING, DELIMITER, dtype=np.int8)
    dst = np.arange(len(letters), dtype=np.int64) + np.repeat(limits[:-1] - offsets[:-1], lens)
    raw[dst] = letters
    return raw, limits


class Context:
    """One dmnd_ctx on one device."""

    def __init__(self, lib: C.CDLL | None = None, device: int = 0, threads: int = 8, index_chunks: int = 0,
                 comp_based_stats: int = 1, max_target_seqs: int = 25, max_evalue: float = 1e-3, want_transcript: bool = False,
                 masking: int = 0, motif_masking: int = 0, sensitivity: int = 0, query_contexts: int = 1, frame_shift: int = 0, range_culling: int = 0, top_percent: float | None = None,
                 min_id: float = 0.0, query_cover: float = 0.0, subject_cover: float = 0.0, min_bit_score: float = 0.0, approx_min_id: float = 0.0,
                 self_targets: np.ndarray | None = None):
        """masking / motif_masking: the reference's --masking (1 = tantan) and --motif-masking.  This test-harness
        wrapper defaults to the parity-ladder rungs without masking (SURVEY 8c); dmnd_search_opts_default() and the CLI
        default to the reference's own defaults (1, 1)."""
        self.lib = lib or load()
        self.opts = SearchOpts()
        self.lib.dmnd_search_opts_default(C.byref(self.opts))
        self.opts.threads = threads
        self.opts.index_chunks = index_chunks
        self.opts.comp_based_stats = comp_based_stats
        self.opts.max_target_seqs = max_target_seqs
        self.opts.max_evalue = max_evalue
        self.opts.want_transcript = int(want_transcript)
        self.opts.sensitivity = int(sensitivity)  # 0 = --fast, 1 = the reference's default sensitivity
        self.opts.masking = int(masking)
        self.opts.motif_masking = int(motif_masking)
        self.opts.query_contexts = int(query_contexts)  # 6 = blastx: six translated frames per query in the query block
        self.opts.frame_shift = int(frame_shift)        # blastx -F: frameshift alignment mode (needs query_contexts = 6)
        self.opts.range_culling = int(range_culling)    # --range-culling (frameshift mode only)
        self.opts.min_id = float(min_id)                # --id / --query-cover / --subject-cover: report filters inside the extension
        self.opts.query_cover = float(query_cover)
        self.opts.subject_cover = float(subject_cover)
        self.opts.min_bit_score = float(min_bit_score)  # --min-score: replaces the e-value bound
        self.opts.approx_min_id = float(approx_min_id)  # --approx-id
        self._self_targets = None if self_targets is None else np.ascontiguousarray(self_targets, dtype=np.uint32)  # --no-self-hits: per query the target to suppress (0xFFFFFFFF = none)
        self.opts.self_targets = None if self._self_targets is None else self._self_targets.ctypes.data
        if top_percent is not None:
            self.opts.top_percent = float(top_percent)  # --top
        self.params = Params()
        self._check(self.lib.dmnd_params_init(C.byref(self.opts), C.byref(self.params)))
        self.ctx = C.c_void_p()
        self._check(self.lib.dmnd_create(device, C.byref(self.params), C.byref(self.ctx)))

    def _check(self, rc):
        if rc != 0:
            raise DmndError(self.lib.dmnd_last_error().decode())

    def backend(self) -> str:
        return self.lib.dmnd_backend().decode()

    def close(self):
        if self.ctx:
            self.lib.dmnd_destroy(self.ctx)
            self.ctx = C.c_void_p()

    # ---- K layer
    def upload(self, raw: np.ndarray, limits: np.ndarray):
        b = C.c_void_p()
        self._check(self.lib.dmnd_block_upload(self.ctx, raw.ctypes.data, raw.size, limits.ctypes.data, len(limits) - 1, C.byref(b)))
        return b

    def mask_block(self, b, algo: int, s_begin: int, s_end: int) -> np.ndarray:
        """dmnd_block_mask + dmnd_block_mask_fetch: masks sequences [s_begin, s_end) of the resident block in place
        (algo: 1 = tantan hard masking, 4 = motif soft-masking table, 5 = both) and returns the ascending offsets of
        the letters that became X."""
        n = C.c_uint64()
        self._check(self.lib.dmnd_block_mask(self.ctx, b, algo, s_begin, s_end, C.byref(n)))
        pos = np.empty(n.value, dtype=np.uint64)
        if n.value:
            self._check(self.lib.dmnd_block_mask_fetch(self.ctx, pos.ctypes.data, pos.size))
        return pos

    def free_block(self, b):
        self.lib.dmnd_block_free(self.ctx, b)

    def set_bias(self, b, bias: np.ndarray | None, raw_len: int):
        self._check(self.lib.dmnd_block_set_bias(self.ctx, b, bias.ctypes.data if bias is not None else None, raw_len))

    def download_letters(self, b, raw_len: int) -> np.ndarray:
        out = np.empty(raw_len, dtype=np.int8)
        self._check(self.lib.dmnd_block_download_letters(self.ctx, b, out.ctypes.data, raw_len))
        return out

    def debug_block_soft(self, b, raw_len: int) -> np.ndarray:
        """Diagnostics: the block's soft-masking table, one byte per letter."""
        out = np.empty(raw_len, dtype=np.uint8)
        self._check(self.lib.dmnd_debug_block_soft(self.ctx, b, out.ctypes.data, raw_len))
        return out

    def debug_ref_index(self, rb, sid: int, raw_len: int):
        """Diagnostics: (keys, locs) of the reference-side seed index of shape `sid`, in index order."""
        keys, locs, n = np.empty(raw_len, dtype=np.uint64), np.empty(raw_len, dtype=np.uint32), C.c_size_t()
        self._check(self.lib.dmnd_debug_ref_index(self.ctx, rb, sid, keys.ctypes.data, locs.ctypes.data, raw_len, C.byref(n)))
        return keys[:n.value].copy(), locs[:n.value].copy()

    def debug_left_most(self, qb, rb, sid: int, chunk: int, qloc: int, sloc: int) -> np.ndarray:
        """Diagnostics: the left-most filter of one (query location, reference location) pair with its intermediates (30 words)."""
        out = np.zeros(30, dtype=np.uint64)
        self._check(self.lib.dmnd_debug_left_most(self.ctx, qb, rb, sid, chunk, qloc, sloc, out.ctypes.data))
        return out

    def build_index(self, b, sid: int = 0):
        self._check(self.lib.dmnd_block_build_index(self.ctx, b, sid))

    def compute_bias(self, b, mode: int = 1):
        self._check(self.lib.dmnd_block_compute_bias(self.ctx, b, mode))

    def download_bias(self, b, raw_len: int) -> np.ndarray:
        out = np.empty(raw_len, dtype=np.int8)
        self._check(self.lib.dmnd_block_download_bias(self.ctx, b, out.ctypes.data, raw_len))
        return out

    def clear_seed_mask(self, b):
        self._check(self.lib.dmnd_block_clear_seed_mask(self.ctx, b))

    def search_shape(self, qb, rb, sid: int = 0, xdrop: int | None = None, gapped_filter: bool = False):
        """Hits (+ per-hit x-drop segments when `xdrop` is given, + per-hit gapped-filter flags when asked) and the stage counters."""
        h = C.c_void_p()
        cn = StageCounters()
        self._check(self.lib.dmnd_search_shape(self.ctx, qb, rb, sid, C.byref(h), C.byref(cn)))
        n = self.lib.dmnd_hits_count(h)
        hits = np.zeros(n, dtype=HIT_DTYPE)
        if n:
            self._check(self.lib.dmnd_hits_download(self.ctx, h, hits.ctypes.data, n))
        segs = None
        if xdrop is not None:
            segs = np.zeros(n, dtype=SEGMENT_DTYPE)
            self._check(self.lib.dmnd_hits_xdrop(self.ctx, qb, rb, h, xdrop, segs.ctypes.data, n))
        gf = None
        if gapped_filter:
            gf = np.zeros(n, dtype=np.uint8)
            if n:
                self._check(self.lib.dmnd_hits_gapped_filter(self.ctx, qb, rb, h, gf.ctypes.data, n))
        self.lib.dmnd_hits_free(self.ctx, h)
        cnd = {k: getattr(cn, k) for k, _ in StageCounters._fields_}
        if gapped_filter:
            return hits, cnd, gf
        return (hits, cnd) if xdrop is None else (hits, cnd, segs)

    # ---- multi-GPU: NCCL broadcast of the resident reference block (csrc/cuda/comm.cu)
    def comm_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        self._check(self.lib.dmnd_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, rank: int, nranks: int, unique_id: bytes):
        self._check(self.lib.dmnd_comm_init(self.ctx, rank, nranks, C.create_string_buffer(unique_id, 128)))

    def block_broadcast(self, root: int, block=None):
        """Every rank calls it; the root passes its resident block.  Returns (block, raw_len, limits) on every rank."""
        out = C.c_void_p()
        self._check(self.lib.dmnd_block_broadcast(self.ctx, root, block, C.byref(out)))
        raw_len, nseq = C.c_size_t(), C.c_uint32()
        self.lib.dmnd_block_geometry(out, C.byref(raw_len), C.byref(nseq))
        limits = np.empty(nseq.value + 1, dtype=np.int64)
        self._check(self.lib.dmnd_block_download_limits(self.ctx, out, limits.ctypes.data, limits.size))
        return out, raw_len.value, limits

    def hits_chain(self, qb, rb, sid: int = 0, xdrop: int = 0, band_slow: bool = False, max_targets: int = 64, align: bool = False):
        """dmnd_search_shape + dmnd_hits_chain (+ dmnd_banded_swipe_chained with traceback when `align`): per-query records, the DP
        problem list, the hits / segments / sites of the DMND_CHAIN_HOST queries, and the counts."""
        h = C.c_void_p()
        cn = StageCounters()
        self._check(self.lib.dmnd_search_shape(self.ctx, qb, rb, sid, C.byref(h), C.byref(cn)))
        out = (C.c_uint64 * 4)()
        self._check(self.lib.dmnd_hits_chain(self.ctx, qb, rb, h, xdrop, int(band_slow), max_targets, out))
        self.lib.dmnd_hits_free(self.ctx, h)
        nq, npairs, nprob, nhh = (int(x) for x in out)
        q = np.zeros(nq, dtype=CHAIN_QUERY_DTYPE); pr = np.zeros(nprob, dtype=PROBLEM_DTYPE)
        hh = np.zeros(nhh, dtype=HIT_DTYPE); hs = np.zeros(nhh, dtype=SEGMENT_DTYPE); ht = np.zeros(nhh, dtype=np.dtype([("target", "<u4"), ("j", "<i4")]))
        self._check(self.lib.dmnd_hits_chain_fetch(self.ctx, q.ctypes.data, pr.ctypes.data, hh.ctypes.data, hs.ctypes.data, ht.ctypes.data))
        res = None
        if align:
            res = np.zeros(nprob, dtype=RESULT_DTYPE)
            if nprob:
                self._check(self.lib.dmnd_banded_swipe_chained(self.ctx, qb, rb, nprob, 1, res.ctypes.data, None, 0))
        return {"queries": q, "problems": pr, "host_hits": hh, "host_segs": hs, "host_sites": ht, "n_pairs": npairs, "results": res}

    def banded_swipe(self, qb, rb, problems: np.ndarray, traceback: bool, transcript_cap: int = 0):
        problems = np.ascontiguousarray(problems, dtype=PROBLEM_DTYPE)
        res = np.zeros(len(problems), dtype=RESULT_DTYPE)
        tr = np.zeros(transcript_cap, dtype=np.uint8) if transcript_cap else None
        self._check(self.lib.dmnd_banded_swipe(self.ctx, qb, rb, problems.ctypes.data, len(problems), 1 if traceback else 0,
                                               res.ctypes.data, tr.ctypes.data if tr is not None else None, transcript_cap))
        return res, tr

    def banded_3frame_swipe(self, qb, rb, problems: np.ndarray, frame_shift: int, traceback: bool, transcript_cap: int = 0):
        """dmnd_banded_3frame_swipe: problems[k].query = block id of the strand's first frame (6 q or 6 q + 3)."""
        problems = np.ascontiguousarray(problems, dtype=PROBLEM_DTYPE)
        res = np.zeros(len(problems), dtype=FS_RESULT_DTYPE)
        tr = np.zeros(transcript_cap, dtype=np.uint8) if transcript_cap else None
        self._check(self.lib.dmnd_banded_3frame_swipe(self.ctx, qb, rb, problems.ctypes.data, len(problems), int(frame_shift), 1 if traceback else 0,
                                                      res.ctypes.data, tr.ctypes.data if tr is not None else None, transcript_cap))
        return res, tr

    def timing(self, reset: bool = False) -> dict:
        t = Timing()
        self.lib.dmnd_timing_fetch(self.ctx, C.byref(t), int(reset))
        return {k: getattr(t, k) for k, _ in Timing._fields_}

    def int_peak(self, packed: bool = False) -> float:
        """Measured DPX issue rate in T lane-instructions / s (roofline denominator of the DP kernels); packed = VIADDMNMX.S16x2."""
        v = C.c_double()
        self._check((self.lib.dmnd_measure_int_peak_packed if packed else self.lib.dmnd_measure_int_peak)(self.ctx, C.byref(v)))
        return v.value / 1e12

    # ---- P layer
    def _collect(self, res):
        """Zero-copy views of the result arrays; the dmnd_result is freed when the last view dies."""
        lib = self.lib

        class _Owner:
            def __init__(self, h):
                self.h = h

            def __del__(self):
                lib.dmnd_result_free(self.h)

        owner = _Owner(res)
        n = C.c_size_t()
        p = lib.dmnd_result_matches(res, C.byref(n))
        if n.value:
            buf = (C.c_char * (n.value * MATCH_DTYPE.itemsize)).from_address(p)
            buf._owner = owner
            m = np.frombuffer(buf, dtype=MATCH_DTYPE)
        else:
            m = np.zeros(0, dtype=MATCH_DTYPE)
        nt = C.c_size_t()
        tp = lib.dmnd_result_transcripts(res, C.byref(nt))
        if nt.value:
            tbuf = (C.c_char * nt.value).from_address(tp)
            tbuf._owner = owner
            tr = np.frombuffer(tbuf, dtype=np.uint8)
        else:
            tr = np.zeros(0, dtype=np.uint8)
        st = lib.dmnd_result_stats(res).contents
        stats = {}
        for k, _ in RunStats._fields_:
            v = getattr(st, k)
            if isinstance(v, C.Structure):
                stats[k] = {kk: getattr(v, kk) for kk, _ in v._fields_}
            else:
                stats[k] = v
        return m, tr, stats

    def blastp(self, q_raw, q_limits, r_raw, r_limits):
        """Host buffers in, matches out (host<->device copies inside the call)."""
        res = C.c_void_p()
        self._check(self.lib.dmnd_blastp(self.ctx, q_raw.ctypes.data, q_raw.size, q_limits.ctypes.data, len(q_limits) - 1,
                                         r_raw.ctypes.data, r_raw.size, r_limits.ctypes.data, len(r_limits) - 1,
                                         C.byref(self.opts), C.byref(res)))
        return self._collect(res)

    def blastp_resident(self, qb, rb, q_raw, q_limits, r_raw, r_limits):
        """Blocks already resident in HBM (uploaded with `upload`)."""
        res = C.c_void_p()
        self._check(self.lib.dmnd_blastp_resident(self.ctx, qb, rb, q_raw.ctypes.data, q_limits.ctypes.data, len(q_limits) - 1,
                                                  r_raw.ctypes.data, r_limits.ctypes.data, len(r_limits) - 1,
                                                  C.byref(self.opts), C.byref(res)))
        return self._collect(res)


def format_double(x: float) -> str:
    """util/string/string.h:87-92"""
    import math
    if x >= 100.0:
        return str(int(math.floor(x)))
    i = int(math.floor(abs(x) * 10.0 + 0.5)) * (1 if x >= 0 else -1)  # llround
    return f"{i // 10}.{i % 10}"


def fmt6(matches: np.ndarray, q_prefix: str = "q", d_prefix: str = "d") -> str:
    """BLAST tabular lines for synthetic ids (>qI / >dI), output/blast_tab_format.cpp:234-293,652."""
    out = []
    for m in matches:
        ev = "0.0" if m["evalue"] == 0.0 else "%.2e" % m["evalue"]
        out.append("%s%d\t%s%d\t%s\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%s\t%s" % (
            q_prefix, m["query"], d_prefix, m["target"], format_double(float(m["identities"]) * 100.0 / float(m["length"])),
            m["length"], m["mismatches"], m["gap_openings"], m["q_begin"] + 1, m["q_end"], m["t_begin"] + 1, m["t_end"],
            ev, format_double(float(m["bit_score"]))))
    return "\n".join(out) + ("\n" if out else "")


# ---- blastx: the six translated contexts of DNA queries ------------------------------------------------------------------------
_GENCODE1 = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"  # Translator::codes[1], TCAG order (basic/basic.cpp:86-113)
_AA = "ARNDCQEGHILKMFPSTWYVBJZX*_"


def _codon_tables():
    idx, comp = (2, 1, 3, 0), (3, 2, 1, 0)  # A C G T -> position in TCAG; complement
    fwd = np.full((5, 5, 5), 23, dtype=np.int8)
    rev = np.full((5, 5, 5), 23, dtype=np.int8)
    for i in range(4):
        for j in range(4):
            for k in range(4):
                fwd[i, j, k] = _AA.index(_GENCODE1[idx[i] * 16 + idx[j] * 4 + idx[k]])
                rev[i, j, k] = _AA.index(_GENCODE1[idx[comp[i]] * 16 + idx[comp[j]] * 4 + idx[comp[k]]])
            for t in (fwd, rev):  # an N in the last slot is harmless when the other two bases fix the amino acid (basic/basic.cpp:132-138)
                if len(set(t[i, j, :4].tolist())) == 1:
                    t[i, j, 4] = t[i, j, 0]
    return fwd, rev


def translate_reads(reads, frame_shift: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """Flat letters + offsets of the query block of a blastx run: for read s the contexts 6s..6s+5 = frames +1 +2 +3, -1 -2 -3
    (util/sequence/translate.h:58-100), with every stop-to-stop stretch shorter than Config::min_orf_len X-ed out
    (data/block/block.cpp:86-100, util/sequence/sequence.cpp:180-197).  Pass the result to block_image() and run the
    context with query_contexts=6.  frame_shift != 0 (blastx -F): no ORF masking (Config::min_orf_len returns 1, basic/config.h:413-416)."""
    fwd, rev = _codon_tables()
    code = {c: i for i, c in enumerate("ACGTN")}
    code.update({c: 4 for c in "MRWSYKVHDBX"})
    seqs = []
    for r in reads:
        d = np.array([code[c] for c in r.upper()], dtype=np.int64)
        L = len(d)
        fr = [np.zeros(0, dtype=np.int8)] * 6
        if L >= 3:
            fr = []
            for f in range(3):
                n = (L - f) // 3
                p = 3 * np.arange(n) + f
                fr.append(fwd[d[p], d[p + 1], d[p + 2]])
            for f in range(3):
                n = (L - f) // 3
                p = L - 3 - (3 * np.arange(n) + f)
                fr.append(rev[d[p + 2], d[p + 1], d[p]])
        l0 = len(fr[0])
        min_len = 1 if (l0 < 30 or frame_shift) else 20 if l0 < 100 else 40
        for v in fr:
            v = v.copy()
            stops = np.flatnonzero(v == 24).tolist()
            b = 0
            for e in stops + [len(v)]:
                if e - b < min_len:
                    v[b:e] = 23
                b = e + 1
            seqs.append(v)
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum([len(v) for v in seqs], out=off[1:])
    return (np.concatenate(seqs).astype(np.int8) if seqs else np.zeros(0, dtype=np.int8)), off


def translate_codes(codes: np.ndarray, frame_shift: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """translate_reads() for reads of ONE length given as an (n, L) array of nucleotide codes 0..3 (4 = N), vectorised: the same six
    contexts per read in the same order, the same ORF masking (tests/test_blastx.py compares the two)."""
    fwd, rev = _codon_tables()
    d = np.asarray(codes, dtype=np.int64)
    n, L = d.shape
    frames = []
    for f in range(3):
        k = (L - f) // 3
        p = 3 * np.arange(k) + f
        frames.append(fwd[d[:, p], d[:, p + 1], d[:, p + 2]])
    for f in range(3):
        k = (L - f) // 3
        p = L - 3 - (3 * np.arange(k) + f)
        frames.append(rev[d[:, p + 2], d[:, p + 1], d[:, p]])
    l0 = frames[0].shape[1]
    min_len = 1 if (l0 < 30 or frame_shift) else 20 if l0 < 100 else 40
    out = []
    for v in frames:
        v = v.copy()
        k = v.shape[1]
        if k and min_len > 1:
            idx = np.arange(k)[None, :]
            stop = v == 24
            prev = np.maximum.accumulate(np.where(stop, idx, -1), axis=1)          # last stop at or before i
            nxt = np.minimum.accumulate(np.where(stop, idx, k)[:, ::-1], axis=1)[:, ::-1]  # next stop at or after i
            v[(~stop) & ((nxt - prev - 1) < min_len)] = 23
        out.append(v)
    lens = np.array([v.shape[1] for v in out], dtype=np.int64)
    width = int(lens.sum())
    flat = np.concatenate(out, axis=1).reshape(-1).astype(np.int8)  # per read: frame 0 | frame 1 | ... | frame 5
    off = np.zeros(6 * n + 1, dtype=np.int64)
    off[1:] = np.cumsum(np.tile(lens, n))
    assert off[-1] == n * width
    return flat, off


def fmt6_translated(matches: np.ndarray, read_lens, q_prefix: str = "r", d_prefix: str = "d") -> str:
    """fmt6 for a query_contexts=6 run: dmnd_match.query is a context (6 * read + frame) and q_begin / q_end count letters of
    that frame; the reference prints nucleotide coordinates on the read, high end first for the reverse strand
    (TranslatedPosition::absolute_interval, basic/translated_position.h:121-127)."""
    out = []
    for m in matches:
        s, f = divmod(int(m["query"]), 6)
        fe = int(m["reserved"]) - 1 if int(m["reserved"]) else f  # frameshift mode: the frame the alignment ENDS in (Hsp::set_end, basic/hssp.cpp:208-217)
        b, e, L = 3 * int(m["q_begin"]) + f % 3, 3 * int(m["q_end"]) + fe % 3, int(read_lens[s])
        qs, qe = (b + 1, e) if f < 3 else (L - b, L - e + 1)
        ev = "0.0" if m["evalue"] == 0.0 else "%.2e" % m["evalue"]
        out.append("%s%d\t%s%d\t%s\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%s\t%s" % (
            q_prefix, s, d_prefix, m["target"], format_double(float(m["identities"]) * 100.0 / float(m["length"])),
            m["length"], m["mismatches"], m["gap_openings"], qs, qe, m["t_begin"] + 1, m["t_end"],
            ev, format_double(float(m["bit_score"]))))
    return "\n".join(out) + ("\n" if out else "")
