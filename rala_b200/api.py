"""ctypes binding of librala_b200.so (include/rala_b200.h) and the host-side mirror of the two
reference entry points it replaces:

    rala::Graph::construct               /root/reference/src/graph.cpp:427-640
    rala::Graph::remove_transitive_edges /root/reference/src/graph.cpp:1281-1335

There is no CPU fallback: if the shared library is missing, or there is no sm_100 device, every
entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RALA_B200_LIB: another build of the same library (rala_b200/variants/: an experiment's switch turned off, or the
# parent commit's library from profiles/build_prev.sh), to compare its results and times with the product's.
# Never a fallback: the file must exist.
LIB_PATH = os.environ.get("RALA_B200_LIB") or os.path.join(_HERE, "librala_b200.so")
N_STAGES = 9
STAGE_NAMES = ("classify", "retrim", "finalize", "build", "transitive", "k1_classify_kernel", "k1b_fixpoint_kernel",
               "k3_transitive_kernels", "k1_survivors_kernel")

KX, KA, KB, KAB, KBA, REJECTED = 0, 1, 2, 3, 4, 255


class RalaB200Error(RuntimeError):
    pass


class Counts(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_overlaps", C.c_uint64), ("n_internals", C.c_uint64),
                ("n_candidates", C.c_uint64), ("n_rounds", C.c_uint32), ("n_piles", C.c_uint32),
                ("n_alive_piles", C.c_uint32), ("n_nodes", C.c_uint32), ("n_edges", C.c_uint64),
                ("n_two_hop", C.c_uint64), ("n_transitive_pairs", C.c_uint64), ("n_heavy_items", C.c_uint32),
                ("n_final_rounds", C.c_uint32), ("n_final_candidates", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class PafStats(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_unresolved", C.c_uint64), ("n_length_mismatch", C.c_uint64),
                ("first_length_mismatch", C.c_uint64), ("n_bytes", C.c_uint64), ("n_chunks", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class MhapStats(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_length_mismatch", C.c_uint64), ("first_length_mismatch", C.c_uint64),
                ("n_query_rc", C.c_uint64), ("n_bytes", C.c_uint64), ("n_chunks", C.c_uint64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class ReadsStats(C.Structure):
    _fields_ = [("format", C.c_uint32), ("n_reads", C.c_uint32), ("n_lines", C.c_uint64), ("n_bases", C.c_uint64),
                ("name_bytes", C.c_uint64), ("max_len", C.c_uint32), ("n_described", C.c_uint32), ("n_bytes", C.c_uint64),
                ("n_chunks", C.c_uint64), ("device_ms", C.c_float)]

    def as_dict(self):
        return {k: (float(getattr(self, k)) if k == "device_ms" else int(getattr(self, k))) for k, _ in self._fields_}


class BgzfStats(C.Structure):
    _fields_ = [("n_blocks", C.c_uint64), ("n_compressed", C.c_uint64), ("n_bytes", C.c_uint64), ("inflate_ms", C.c_float)]

    def as_dict(self):
        return {k: (float(getattr(self, k)) if k == "inflate_ms" else int(getattr(self, k))) for k, _ in self._fields_}


GZIP_STAGES = ("finder", "counting", "symbols", "chain", "resolve_crc")


class GzipStats(C.Structure):
    _fields_ = [("n_members", C.c_uint64), ("n_compressed", C.c_uint64), ("n_bytes", C.c_uint64), ("n_chunks", C.c_uint64),
                ("n_corrected", C.c_uint64), ("chunk_bytes", C.c_uint64), ("rounds", C.c_uint32), ("bgzf", C.c_uint32),
                ("inflate_ms", C.c_float), ("stage_ms", C.c_float * 5)]

    def as_dict(self):
        d = {k: int(getattr(self, k)) for k, _ in self._fields_[:8]}
        d["inflate_ms"] = float(self.inflate_ms)
        d["stage_ms"] = {name: float(v) for name, v in zip(GZIP_STAGES, self.stage_ms)}
        return d


PAF_CHUNK_BYTES = 32 << 20   # RALA_B200_PAF_CHUNK_BYTES (the MHAP reader uses the same chunks)


class PileStats(C.Structure):
    _fields_ = [("n_counted", C.c_uint64), ("n_runs", C.c_uint64), ("max_coverage", C.c_uint32), ("n_live", C.c_uint32),
                ("n_tied", C.c_uint32), ("n_exact_min", C.c_uint32)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


def _text(text):
    """PAF / MHAP / FASTA / FASTQ text as bytes, a uint8 numpy array or a contiguous uint8 CPU tensor (pinned: uploaded in place)."""
    if isinstance(text, (bytes, bytearray, memoryview)):
        text = np.frombuffer(text, np.uint8)
    if hasattr(text, "data_ptr"):
        if not text.is_contiguous() or text.device.type != "cpu" or text.element_size() != 1:
            raise RalaB200Error("text must be a contiguous uint8 CPU tensor")
        return text, int(text.numel())
    text = np.ascontiguousarray(text, dtype=np.uint8).reshape(-1)
    return text, int(text.shape[0])


def _names(names, read_len):
    """Read names as a list of bytes, or as (blob, name_end) -> (blob uint8, name_end uint64, read_len uint32)."""
    if isinstance(names, tuple):
        blob, ends = names
        blob = np.frombuffer(bytes(blob), np.uint8) if isinstance(blob, (bytes, bytearray)) else np.ascontiguousarray(blob, np.uint8)
        ends = np.ascontiguousarray(ends, np.uint64)
    else:
        blob = np.frombuffer(b"".join(names), np.uint8)
        ends = np.cumsum(np.fromiter((len(n) for n in names), np.uint64, len(names)), dtype=np.uint64)
    rl = np.ascontiguousarray(read_len, np.uint32)
    if rl.shape[0] != ends.shape[0]:
        raise RalaB200Error("one read length per read name")
    if blob.size == 0:
        blob = np.zeros(1, np.uint8)
    return blob, ends, rl


EXPORTS = [
    "rala_b200_abi_version", "rala_b200_create", "rala_b200_destroy", "rala_b200_last_error",
    "rala_b200_launch_count", "rala_b200_event_record", "rala_b200_event_elapsed_ms", "rala_b200_synchronize",
    "rala_b200_trim_classify", "rala_b200_transitive_reduce", "rala_b200_filter_duplicates",
    "rala_b200_parse_paf", "rala_b200_graph_set_reads", "rala_b200_graph_set_overlaps_paf",
    "rala_b200_parse_mhap", "rala_b200_graph_set_overlaps_mhap", "rala_b200_graph_set_reads_text", "rala_b200_graph_get_reads",
    "rala_b200_build_piles", "rala_b200_graph_build_piles", "rala_b200_graph_get_medians", "rala_b200_graph_get_coverage_runs",
    "rala_b200_graph_create", "rala_b200_graph_destroy", "rala_b200_graph_set_overlaps",
    "rala_b200_graph_set_piles", "rala_b200_graph_set_hills", "rala_b200_graph_classify",
    "rala_b200_graph_retrim", "rala_b200_graph_retrim_promote", "rala_b200_graph_finalize",
    "rala_b200_graph_build", "rala_b200_graph_transitive", "rala_b200_graph_run", "rala_b200_graph_counts",
    "rala_b200_graph_get_hill_coverage", "rala_b200_graph_get_piles", "rala_b200_graph_get_connections",
    "rala_b200_graph_get_lists", "rala_b200_graph_get_seq_to_node", "rala_b200_graph_get_edges",
    "rala_b200_graph_get_marked", "rala_b200_graph_stage_ms", "rala_b200_graph_set_kept_overlaps",
    "rala_b200_graph_use_cuda_graph", "rala_b200_graph_set_overlaps_columns", "rala_b200_graph_set_outputs",
    "rala_b200_graph_set_overlaps_packed", "rala_b200_multi_set_overlaps_packed", "rala_b200_graph_get_adjacency",
    "rala_b200_graph_get_csr", "rala_b200_inflate_bgzf", "rala_b200_graph_set_reads_bgzf", "rala_b200_graph_set_overlaps_paf_bgzf",
    "rala_b200_graph_set_overlaps_mhap_bgzf", "rala_b200_inflate_gzip", "rala_b200_graph_set_reads_gzip",
    "rala_b200_graph_set_overlaps_paf_gzip", "rala_b200_graph_set_overlaps_mhap_gzip",
    # multi-GPU phases
    "rala_b200_create_on_stream", "rala_b200_graph_set_shard", "rala_b200_graph_phase_events",
    "rala_b200_graph_phase_resolve", "rala_b200_graph_phase_survivors", "rala_b200_graph_phase_emit_edges",
    "rala_b200_graph_phase_csr", "rala_b200_graph_phase_transitive",
    "rala_b200_graph_export_marks", "rala_b200_graph_phase_marks",
    "rala_b200_graph_export_padded", "rala_b200_graph_import_gathered", "rala_b200_graph_export_list_counts",
    "rala_b200_graph_phase_final_events_gathered", "rala_b200_exchange_block_words",
    # multi-GPU session (orchestration inside the library, exchanges over peer memory)
    "rala_b200_multi_create", "rala_b200_multi_destroy", "rala_b200_multi_last_error", "rala_b200_multi_set_piles",
    "rala_b200_multi_set_overlaps", "rala_b200_multi_set_overlaps_columns", "rala_b200_multi_default_caps",
    "rala_b200_multi_reserve", "rala_b200_multi_export_handle", "rala_b200_multi_import_handles", "rala_b200_multi_run",
    "rala_b200_multi_use_cuda_graph", "rala_b200_multi_synchronize", "rala_b200_multi_demand", "rala_b200_multi_plan",
    "rala_b200_multi_counts", "rala_b200_multi_edge_range", "rala_b200_multi_get_edges", "rala_b200_multi_get_marked",
    "rala_b200_multi_get_seq_to_node", "rala_b200_multi_get_piles", "rala_b200_multi_event_record",
    "rala_b200_multi_event_elapsed_ms", "rala_b200_multi_launch_count", "rala_b200_multi_stage_ms",
    "rala_b200_multi_set_outputs", "rala_b200_multi_set_barrier_timeout_ms", "rala_b200_multi_set_rounds", "rala_b200_multi_barrier_log", "rala_b200_multi_sweep_log",
    # multi-GPU staged construct (pile tables that change between the passes)
    "rala_b200_multi_set_hills", "rala_b200_multi_classify", "rala_b200_multi_retrim", "rala_b200_multi_retrim_promote",
    "rala_b200_multi_finish", "rala_b200_multi_get_hill_coverage", "rala_b200_multi_get_lists", "rala_b200_multi_edge_runs",
]
MAX_SEGMENTS = 64

_LIB = None


def load_path(path: str):
    """Load one build of the CUDA extension; raises (never falls back) when the file is missing."""
    if not os.path.exists(path):
        raise RalaB200Error(f"{path} is missing: run `python -m rala_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(path)
    lib.rala_b200_last_error.restype = C.c_char_p
    lib.rala_b200_launch_count.restype = C.c_uint64
    lib.rala_b200_exchange_block_words.restype = C.c_uint64
    lib.rala_b200_destroy.restype = None
    lib.rala_b200_graph_destroy.restype = None
    lib.rala_b200_multi_destroy.restype = None
    lib.rala_b200_multi_last_error.restype = C.c_char_p
    lib.rala_b200_multi_launch_count.restype = C.c_uint64
    return lib


def load():
    """The product library (LIB_PATH), loaded once."""
    global _LIB
    if _LIB is None:
        _LIB = load_path(LIB_PATH)
    return _LIB


def _ptr(a):
    """Raw address of a numpy array or a (CPU, possibly pinned) torch tensor."""
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(a.ctypes.data)


def _np(a, dtype, cols=None):
    if hasattr(a, "data_ptr"):   # torch tensor: must already be contiguous and of the right dtype
        if not a.is_contiguous() or a.device.type != "cpu":
            raise RalaB200Error("host buffers must be contiguous CPU tensors")
        return a
    a = np.ascontiguousarray(a, dtype=dtype)
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


def records_to_columns(records) -> np.ndarray:
    """rala_ovl_t rows (n, 7) -> the six columns of rala_b200_graph_set_overlaps_columns as one contiguous (6, n)
    array: bit 31 of a_id = invalid record (or an id >= 2^31), bit 31 of b_id = orientation."""
    r = np.ascontiguousarray(records, dtype=np.uint32).reshape(-1, 7)
    cols = np.empty((6, r.shape[0]), dtype=np.uint32)
    top = np.uint32(0x80000000)
    bad = ((r[:, 6] & 2) != 0) | ((r[:, 0] & top) != 0) | ((r[:, 1] & top) != 0)
    cols[0] = (r[:, 0] & ~top) | np.where(bad, top, np.uint32(0))
    cols[1] = (r[:, 1] & ~top) | ((r[:, 6] & 1) << 31)
    cols[2:6] = r[:, 2:6].T
    return cols


class PackedRecords:
    """Host form of rala_b200_graph_set_overlaps_packed: 12 bytes per record (+ 8 per query group) instead of 24."""

    def __init__(self, query_id, group_end, b_id, a_span, b_span):
        self.query_id, self.group_end, self.b_id, self.a_span, self.b_span = query_id, group_end, b_id, a_span, b_span

    @property
    def n(self) -> int:
        return int(self.b_id.shape[0])

    @property
    def nbytes(self) -> int:
        return sum(int(x.numel() * x.element_size()) if hasattr(x, "numel") else int(x.nbytes)
                   for x in (self.query_id, self.group_end, self.b_id, self.a_span, self.b_span))

    def pin(self):
        """The same arrays in pinned host memory (torch), for asynchronous uploads."""
        import torch
        return PackedRecords(*[torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in
                               (self.query_id, self.group_end, self.b_id, self.a_span, self.b_span)])


def records_to_packed(records):
    """rala_ovl_t rows (n, 7), grouped by query as a PAF lists them -> PackedRecords, or None when a coordinate does not fit
    16 bits or an id needs bit 31 (use records_to_columns then).  Invalid records travel with both spans 0."""
    r = np.ascontiguousarray(records, dtype=np.uint32).reshape(-1, 7)
    n = r.shape[0]
    if n == 0:
        return None
    bad = ((r[:, 6] & 2) != 0) | (r[:, 0] >= 0x80000000) | (r[:, 1] >= 0x80000000)
    if (r[~bad, 2:6] >= 65536).any():
        return None
    a = np.where(bad, np.uint32(0), r[:, 0])          # an invalid record joins whatever group it sits in: id 0 is as good as any
    a = a.copy()
    # keep the grouping tight: an invalid record takes the id of its predecessor (it is rejected whatever its ids are)
    if bad.any():
        idx = np.where(~bad, np.arange(n), 0)
        np.maximum.accumulate(idx, out=idx)
        a = r[idx, 0] * (~bad[idx]).astype(np.uint32)
    change = np.nonzero(a[1:] != a[:-1])[0] + 1
    group_end = np.concatenate([change, [n]]).astype(np.uint32)
    query_id = a[np.concatenate([[0], change])].astype(np.uint32)
    span = lambda lo, hi: np.where(bad, np.uint32(0), lo | (hi << 16)).astype(np.uint32)   # noqa: E731
    b_id = np.where(bad, np.uint32(0), r[:, 1] | ((r[:, 6] & 1) << 31)).astype(np.uint32)
    return PackedRecords(query_id, group_end, b_id, span(r[:, 2], r[:, 3]), span(r[:, 4], r[:, 5]))


class Context:
    """One CUDA device + stream (rala_b200_ctx)."""

    def __init__(self, device: int = 0, lib=None):
        self.lib = lib or load()   # lib: another build of the same library (bench.py --ab)
        self.handle = C.c_void_p()
        rc = self.lib.rala_b200_create(C.byref(self.handle), C.c_int(device))
        if rc != 0:
            raise RalaB200Error(f"rala_b200_create(device={device}) failed with status {rc}: "
                                "an sm_100 (B200) device is required, there is no CPU fallback")
        self.device = device
        self._graphs = []   # weak references: sessions are destroyed before their context (rala_b200_graph holds a ctx pointer)

    def check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.rala_b200_last_error(self.handle)
            raise RalaB200Error(f"{what}: status {rc}: {msg.decode() if msg else ''}")

    @property
    def launch_count(self) -> int:
        return int(self.lib.rala_b200_launch_count(self.handle))

    def event_record(self, which: int):
        self.check(self.lib.rala_b200_event_record(self.handle, C.c_int(which)), "event_record")

    def event_elapsed_ms(self) -> float:
        ms = C.c_float(0)
        self.check(self.lib.rala_b200_event_elapsed_ms(self.handle, C.byref(ms)), "event_elapsed_ms")
        return float(ms.value)

    def synchronize(self):
        self.check(self.lib.rala_b200_synchronize(self.handle), "synchronize")

    def close(self):
        if self.handle:
            for ref in getattr(self, "_graphs", []):
                g = ref()
                if g is not None:
                    g.close()
            self._graphs = []
            self.lib.rala_b200_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- stateless stages -------------------------------------------------------------------
    def trim_classify(self, records, piles):
        """Overlap::trim + Overlap::type (overlap.cpp:117-259) -> (trimmed records, types)."""
        rec = np.array(records, dtype=np.uint32, copy=True).reshape(-1, 7)
        piles = _np(piles, np.uint32, 2)
        types = np.zeros(rec.shape[0], dtype=np.uint8)
        self.check(self.lib.rala_b200_trim_classify(self.handle, _ptr(rec), C.c_uint64(rec.shape[0]), _ptr(piles),
                                                    C.c_uint32(piles.shape[0]), _ptr(types)), "trim_classify")
        return rec, types

    def transitive_reduce(self, n_nodes: int, edges):
        """Graph::remove_transitive_edges (graph.cpp:1281-1318) on an injected edge list -> (marked, n_pairs)."""
        edges = _np(edges, np.uint32, 3)
        marked = np.zeros(edges.shape[0], dtype=np.uint8)
        n_pairs = C.c_uint64(0)
        self.check(self.lib.rala_b200_transitive_reduce(self.handle, C.c_uint32(n_nodes), C.c_uint64(edges.shape[0]),
                                                        _ptr(edges), _ptr(marked), C.byref(n_pairs)), "transitive_reduce")
        return marked, int(n_pairs.value)

    def filter_duplicates(self, a_id, b_id, length, with_time: bool = False):
        """Graph::initialize's duplicate filter (graph.cpp:273-303, grouping :340-361) -> is_valid_overlap_ as bytes.
        a_id with bit 31 set = unresolved record; length = Overlap::length() as parsed."""
        a, b, ln = _np(a_id, np.uint32), _np(b_id, np.uint32), _np(length, np.uint32)
        if not (a.shape == b.shape == ln.shape):
            raise ValueError("filter_duplicates: the three columns must have one length")
        valid = np.zeros(a.shape[0], dtype=np.uint8)
        ms = C.c_float(0.0)
        self.check(self.lib.rala_b200_filter_duplicates(self.handle, _ptr(a), _ptr(b), _ptr(ln), C.c_uint64(a.shape[0]),
                                                        _ptr(valid), C.byref(ms)), "filter_duplicates")
        return (valid, float(ms.value)) if with_time else valid

    def parse_paf(self, text, names, read_len, with_time: bool = False):
        """PAF text -> (columns (7, n) uint32: a_id | invalid << 31, b_id | orientation << 31, a_begin, a_end, b_begin,
        b_end, length (column 11); stats dict) with the reads' names resolved on the device (no duplicate filter)."""
        buf, n_bytes = _text(text)
        blob, ends, rl = _names(names, read_len)
        cap = n_bytes // 19 + 2
        cols = np.zeros((7, cap), dtype=np.uint32)
        st, ms = PafStats(), C.c_float(0.0)
        self.check(self.lib.rala_b200_parse_paf(self.handle, _ptr(blob), _ptr(ends), _ptr(rl), C.c_uint32(ends.shape[0]), _ptr(buf),
                                                C.c_uint64(n_bytes), _ptr(cols), C.c_uint64(cap), C.byref(st), C.byref(ms)), "parse_paf")
        stats = st.as_dict()
        out = np.ascontiguousarray(cols[:, :stats["n_records"]])
        return (out, stats, float(ms.value)) if with_time else (out, stats)

    def parse_mhap(self, text, read_len, with_time: bool = False):
        """MHAP text -> (columns (7, n) uint32: a_id, b_id | orientation << 31, a_begin, a_end, b_begin, b_end, length
        (the longer span); stats dict).  Ids are 1-based in the text, checked against len(read_len); no duplicate filter."""
        buf, n_bytes = _text(text)
        rl = _np(read_len, np.uint32)
        cap = n_bytes // 22 + 2
        cols = np.zeros((7, cap), dtype=np.uint32)
        st, ms = MhapStats(), C.c_float(0.0)
        self.check(self.lib.rala_b200_parse_mhap(self.handle, _ptr(rl), C.c_uint32(rl.shape[0]), _ptr(buf), C.c_uint64(n_bytes),
                                                 _ptr(cols), C.c_uint64(cap), C.byref(st), C.byref(ms)), "parse_mhap")
        stats = st.as_dict()
        out = np.ascontiguousarray(cols[:, :stats["n_records"]])
        return (out, stats, float(ms.value)) if with_time else (out, stats)

    def inflate_bgzf(self, data) -> tuple:
        """A BGZF file (bytes, uint8 array or pinned CPU tensor) inflated on the device -> (text as a uint8 array, stats dict:
        blocks, compressed bytes, inflated bytes, inflate_ms)."""
        buf, n = _text(data)
        st = BgzfStats()
        self.check(self.lib.rala_b200_inflate_bgzf(self.handle, _ptr(buf), C.c_uint64(n), None, C.c_uint64(0), C.byref(st)),
                   "inflate_bgzf")
        out = np.zeros(max(int(st.n_bytes), 1), np.uint8)
        self.check(self.lib.rala_b200_inflate_bgzf(self.handle, _ptr(buf), C.c_uint64(n), _ptr(out), C.c_uint64(int(st.n_bytes)),
                                                   C.byref(st)), "inflate_bgzf")
        return out[:int(st.n_bytes)], st.as_dict()

    def inflate_gzip(self, data) -> tuple:
        """A gzip file of one or more members (bytes, uint8 array or pinned CPU tensor) inflated on the device -> (text as a
        uint8 array, stats dict: members, compressed and inflated bytes, chunks, corrected chunk decodes, chunk bytes,
        rounds, bgzf (1: the BGZF path ran), inflate_ms and its stage_ms)."""
        buf, n = _text(data)
        st = GzipStats()
        self.check(self.lib.rala_b200_inflate_gzip(self.handle, _ptr(buf), C.c_uint64(n), None, C.c_uint64(0), C.byref(st)),
                   "inflate_gzip")
        out = np.zeros(max(int(st.n_bytes), 1), np.uint8)
        self.check(self.lib.rala_b200_inflate_gzip(self.handle, _ptr(buf), C.c_uint64(n), _ptr(out), C.c_uint64(int(st.n_bytes)),
                                                   C.byref(st)), "inflate_gzip")
        return out[:int(st.n_bytes)], st.as_dict()

    def build_piles(self, columns, read_len, with_time: bool = False):
        """Graph::initialize's coverage half on the device: six host columns in the set_overlaps_columns layout (bit 31 of
        a_id = unresolved record; records the duplicate filter drops still count) + the read lengths -> (piles (n_reads, 2)
        uint32, dead = 0 0; medians (n_reads,) uint16, 0 = dead; stats dict)."""
        cols = [_np(c, np.uint32) for c in columns]
        n = cols[0].shape[0]
        if len(cols) != 6 or any(c.shape[0] != n for c in cols):
            raise RalaB200Error("build_piles needs six columns of equal length")
        rl = _np(read_len, np.uint32)
        piles = np.zeros((rl.shape[0], 2), dtype=np.uint32)
        med = np.zeros(rl.shape[0], dtype=np.uint16)
        st, ms = PileStats(), C.c_float(0.0)
        self.check(self.lib.rala_b200_build_piles(self.handle, *[_ptr(c) for c in cols], C.c_uint64(n), _ptr(rl), C.c_uint32(rl.shape[0]),
                                                  _ptr(piles), _ptr(med), C.byref(st), C.byref(ms)), "build_piles")
        return (piles, med, st.as_dict(), float(ms.value)) if with_time else (piles, med, st.as_dict())


class Graph:
    """Host-side mirror of rala::Graph for the hot path (graph.hpp:37-60).

    `construct()` is Graph::construct's hot half (graph.cpp:443-632) on numeric inputs — what the
    unchanged Graph::initialize leaves behind: overlap records in file order with their validity
    bit, the pile table with flags, the chimeric hills.  `remove_transitive_edges()` is
    graph.cpp:1281-1335 including the host-side tail (transitive_edges_, stable adjacency compaction).
    """

    def __init__(self, ctx: Context | None = None, device: int = 0):
        self.ctx = ctx or Context(device)
        self.lib = self.ctx.lib
        self.handle = C.c_void_p()
        self.ctx.check(self.lib.rala_b200_graph_create(self.ctx.handle, C.byref(self.handle)), "graph_create")
        if hasattr(self.ctx, "_graphs"):
            import weakref
            self.ctx._graphs.append(weakref.ref(self))
        self.n_piles = 0
        self.n_hills = 0
        self._keep = []   # host buffers referenced by in-flight async copies
        self.transitive_edges = None

    def close(self):
        if self.handle:
            self.lib.rala_b200_graph_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, name, *args):
        self.ctx.check(getattr(self.lib, name)(self.handle, *args), name)

    # ---- inputs ------------------------------------------------------------------------------
    def set_overlaps(self, records):
        rec = _np(records, np.uint32, 7)
        n = rec.shape[0]
        self._keep = [rec]
        self._call("rala_b200_graph_set_overlaps", _ptr(rec), C.c_uint64(n))
        return self

    def set_overlaps_columns(self, columns):
        """Six host columns (a_id | invalid << 31, b_id | orientation << 31, a_begin, a_end, b_begin, b_end), e.g. the
        rows of a contiguous (6, n) array: 24 B per record cross PCIe and land in the device layout."""
        cols = [_np(c, np.uint32) for c in columns]
        n = cols[0].shape[0]
        if len(cols) != 6 or any(c.shape[0] != n for c in cols):
            raise RalaB200Error("set_overlaps_columns needs six columns of equal length")
        self._keep = list(cols)
        self._call("rala_b200_graph_set_overlaps_columns", *[_ptr(c) for c in cols], C.c_uint64(n))
        return self

    def set_overlaps_packed(self, p: PackedRecords):
        """The compact upload (records_to_packed): 12 B per record cross PCIe, expanded on the device."""
        self._keep = [p]
        self._call("rala_b200_graph_set_overlaps_packed", _ptr(p.query_id), _ptr(p.group_end), C.c_uint32(int(p.query_id.shape[0])),
                   _ptr(p.b_id), _ptr(p.a_span), _ptr(p.b_span), C.c_uint64(p.n))
        return self

    def set_reads(self, names, read_len):
        """Read names (list of bytes, or (blob, name_end)) and sequence lengths the PAF text is resolved against; MHAP text
        uses the lengths and their order (id k + 1 = read k)."""
        blob, ends, rl = _names(names, read_len)
        self._call("rala_b200_graph_set_reads", _ptr(blob), _ptr(ends), _ptr(rl), C.c_uint32(ends.shape[0]))
        self._n_reads = int(ends.shape[0])
        return self

    def set_reads_text(self, text) -> dict:
        """FASTA or FASTQ text (bytes, uint8 array or pinned CPU tensor) -> the read names and lengths, parsed on the device;
        afterwards the session is as after set_reads with them.  Returns the stats (format, reads, lines, bases, name
        bytes, longest read, headers with a description, bytes, upload chunks, device_ms)."""
        buf, n_bytes = _text(text)
        st = ReadsStats()
        self._call("rala_b200_graph_set_reads_text", _ptr(buf), C.c_uint64(n_bytes), C.byref(st))
        self._n_reads = int(st.n_reads)
        return st.as_dict()

    def set_reads_bgzf(self, data) -> tuple:
        """set_reads_text on a BGZF file, inflated on the device -> (reads stats dict, BGZF stats dict)."""
        buf, n = _text(data)
        st, z = ReadsStats(), BgzfStats()
        self._call("rala_b200_graph_set_reads_bgzf", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        self._n_reads = int(st.n_reads)
        return st.as_dict(), z.as_dict()

    def set_reads_gzip(self, data) -> tuple:
        """set_reads_text on a gzip file (BGZF included), inflated on the device -> (reads stats dict, gzip stats dict)."""
        buf, n = _text(data)
        st, z = ReadsStats(), GzipStats()
        self._call("rala_b200_graph_set_reads_gzip", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        self._n_reads = int(st.n_reads)
        return st.as_dict(), z.as_dict()

    def reads(self):
        """The session's reads as set_reads holds them: (names blob uint8, name_end uint64, read_len uint32)."""
        n, nb = C.c_uint32(0), C.c_uint64(0)
        self._call("rala_b200_graph_get_reads", None, None, None, C.byref(n), C.byref(nb))
        blob = np.zeros(max(int(nb.value), 1), np.uint8)
        ends = np.zeros(int(n.value), np.uint64)
        rl = np.zeros(int(n.value), np.uint32)
        self._call("rala_b200_graph_get_reads", _ptr(blob), _ptr(ends), _ptr(rl), None, None)
        return blob[:int(nb.value)], ends, rl

    def set_overlaps_paf(self, text) -> dict:
        """PAF text in file order -> the session's records (parse, name lookup, duplicate filter on the device); returns
        the stats (records, unresolved names, read-length mismatches, bytes, upload chunks)."""
        buf, n_bytes = _text(text)
        st = PafStats()
        self._call("rala_b200_graph_set_overlaps_paf", _ptr(buf), C.c_uint64(n_bytes), C.byref(st))
        return st.as_dict()

    def set_overlaps_mhap(self, text) -> dict:
        """MHAP text in file order -> the session's records (parse, id check, duplicate filter on the device); returns the
        stats (records, read-length mismatches, records with a_rc = 1, bytes, upload chunks)."""
        buf, n_bytes = _text(text)
        st = MhapStats()
        self._call("rala_b200_graph_set_overlaps_mhap", _ptr(buf), C.c_uint64(n_bytes), C.byref(st))
        return st.as_dict()

    def set_overlaps_paf_bgzf(self, data) -> tuple:
        """set_overlaps_paf on a BGZF file, inflated on the device -> (PAF stats dict, BGZF stats dict)."""
        buf, n = _text(data)
        st, z = PafStats(), BgzfStats()
        self._call("rala_b200_graph_set_overlaps_paf_bgzf", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        return st.as_dict(), z.as_dict()

    def set_overlaps_mhap_bgzf(self, data) -> tuple:
        """set_overlaps_mhap on a BGZF file, inflated on the device -> (MHAP stats dict, BGZF stats dict)."""
        buf, n = _text(data)
        st, z = MhapStats(), BgzfStats()
        self._call("rala_b200_graph_set_overlaps_mhap_bgzf", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        return st.as_dict(), z.as_dict()

    def set_overlaps_paf_gzip(self, data) -> tuple:
        """set_overlaps_paf on a gzip file (BGZF included), inflated on the device -> (PAF stats dict, gzip stats dict)."""
        buf, n = _text(data)
        st, z = PafStats(), GzipStats()
        self._call("rala_b200_graph_set_overlaps_paf_gzip", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        return st.as_dict(), z.as_dict()

    def set_overlaps_mhap_gzip(self, data) -> tuple:
        """set_overlaps_mhap on a gzip file (BGZF included), inflated on the device -> (MHAP stats dict, gzip stats dict)."""
        buf, n = _text(data)
        st, z = MhapStats(), GzipStats()
        self._call("rala_b200_graph_set_overlaps_mhap_gzip", _ptr(buf), C.c_uint64(n), C.byref(st), C.byref(z))
        return st.as_dict(), z.as_dict()

    def build_piles(self) -> dict:
        """The pile table from the records of the last set_overlaps_paf / _mhap, built on the device and installed as
        set_piles(piles) would (flags 0, hills untouched); returns the stats."""
        st = PileStats()
        self._call("rala_b200_graph_build_piles", C.byref(st))
        self.n_piles = self._built_piles = self._n_reads
        return st.as_dict()

    def medians(self):
        """After build_piles: Pile::find_median of every pile (uint16, 0 = dead)."""
        out = np.zeros(getattr(self, "_built_piles", 0), dtype=np.uint16)
        self._call("rala_b200_graph_get_medians", _ptr(out))
        return out

    def coverage_runs(self):
        """After build_piles: (run_off (n_piles + 1), run_begin, run_cov uint16) — the maximal constant-coverage runs of
        every read over [0, read_len); read r's runs are [run_off[r], run_off[r + 1])."""
        off = np.zeros(getattr(self, "_built_piles", 0) + 1, dtype=np.uint32)
        self._call("rala_b200_graph_get_coverage_runs", _ptr(off), None, None, C.c_uint64(0))
        total = int(off[-1])
        begin = np.zeros(max(total, 1), dtype=np.uint32)
        cov = np.zeros(max(total, 1), dtype=np.uint16)
        self._call("rala_b200_graph_get_coverage_runs", _ptr(off), _ptr(begin), _ptr(cov), C.c_uint64(total))
        return off, begin[:total], cov[:total]

    def set_outputs(self, edges_out=None, marked_out=None):
        """Pinned host (or device-visible) buffers the run writes its edge rows and marks into directly."""
        e_cap = 0 if edges_out is None else int(edges_out.shape[0])
        m_cap = 0 if marked_out is None else int(marked_out.shape[0])
        self._outputs = (edges_out, marked_out)
        self._call("rala_b200_graph_set_outputs", _ptr(edges_out), C.c_uint64(e_cap), _ptr(marked_out), C.c_uint64(m_cap))
        return self

    def set_piles(self, piles, flags=None):
        p = _np(piles, np.uint32, 2)
        f = None if flags is None else _np(flags, np.uint8)
        self.n_piles = p.shape[0]
        self._keep += [p, f]
        self._call("rala_b200_graph_set_piles", _ptr(p), _ptr(f), C.c_uint32(self.n_piles))
        return self

    def set_hills(self, hills):
        h = _np(np.zeros((0, 3)) if hills is None else hills, np.uint32, 3)
        self.n_hills = h.shape[0]
        self._call("rala_b200_graph_set_hills", _ptr(h), C.c_uint32(self.n_hills))
        return self

    # ---- stages (same boundaries as the reference's construct) ---------------------------------
    def classify(self):
        self._call("rala_b200_graph_classify")
        return self

    def retrim(self):
        self._call("rala_b200_graph_retrim")
        return self

    def retrim_promote(self) -> bool:
        changed = C.c_int(0)
        self._call("rala_b200_graph_retrim_promote", C.byref(changed))
        return bool(changed.value)

    def finalize(self):
        self._call("rala_b200_graph_finalize")
        return self

    def build(self):
        self._call("rala_b200_graph_build")
        return self

    def transitive(self):
        self._call("rala_b200_graph_transitive")
        return self

    def run(self):
        """classify .. transitive with the pile table frozen; no host synchronisation inside."""
        self._call("rala_b200_graph_run")
        return self

    # ---- outputs -----------------------------------------------------------------------------
    def use_cuda_graph(self, enabled: bool):
        """run() replays a captured CUDA graph by default; stage_ms() needs the eager chain (enabled=False)."""
        self._call("rala_b200_graph_use_cuda_graph", C.c_int(1 if enabled else 0))
        return self

    def counts(self) -> dict:
        c = Counts()
        self._call("rala_b200_graph_counts", C.byref(c))
        return c.as_dict()

    def hill_coverage(self):
        out = np.zeros(self.n_hills, dtype=np.uint32)
        self._call("rala_b200_graph_get_hill_coverage", _ptr(out))
        return out

    def piles(self):
        out = np.zeros((self.n_piles, 2), dtype=np.uint32)
        self._call("rala_b200_graph_get_piles", _ptr(out))
        return out

    def connections(self):
        n = self.counts()["n_overlaps"]
        out = np.zeros((n, 2), dtype=np.uint32)
        self._call("rala_b200_graph_get_connections", _ptr(out))
        return out

    def lists(self):
        c = self.counts()
        ovl = np.zeros((c["n_overlaps"], 7), dtype=np.uint32)
        inl = np.zeros((c["n_internals"], 7), dtype=np.uint32)
        self._call("rala_b200_graph_get_lists", _ptr(ovl), _ptr(inl))
        return ovl, inl

    def set_kept_overlaps(self, kept):
        """graph.cpp:523: replace `overlaps` by the host-filtered list (the -s repeat filter only drops entries)"""
        k = _np(kept, np.uint32, 7)
        self._call("rala_b200_graph_set_kept_overlaps", _ptr(k), C.c_uint64(k.shape[0]))
        return self

    def seq_to_node(self):
        out = np.zeros(self.n_piles, dtype=np.uint32)
        self._call("rala_b200_graph_get_seq_to_node", _ptr(out))
        return out

    def edges(self, out=None):
        n = self.counts()["n_edges"]
        if out is None:
            out = np.zeros((n, 3), dtype=np.uint32)
        self._call("rala_b200_graph_get_edges", _ptr(out))
        return out

    def marked(self, out=None):
        n = self.counts()["n_edges"]
        if out is None:
            out = np.zeros(n, dtype=np.uint8)
        self._call("rala_b200_graph_get_marked", _ptr(out))
        return out

    def adjacency(self, which: int = 0, skip_marked: bool = False):
        """(off, ids): per node the ids of its out- (which = 0) or in-edges (which = 1) in ascending edge id, built on the
        device; skip_marked: without the removed edges (what Graph::remove_marked_objects leaves, graph.cpp:2118-2151)."""
        c = self.counts()
        off = np.zeros(c["n_nodes"] + 1, dtype=np.uint32)
        ids = np.zeros(max(c["n_edges"], 1), dtype=np.uint32)
        n = C.c_uint64(0)
        self._call("rala_b200_graph_get_adjacency", C.c_int(which), C.c_int(1 if skip_marked else 0), _ptr(off), _ptr(ids), C.byref(n))
        return off, ids[:int(n.value)]

    def csr(self):
        """(row_ptr (n_nodes + 1), col (n_edges, 2) = (destination, length), col_eid (n_edges)): the CSR rows build wrote
        for the transitive pass; slot order inside a row is arbitrary."""
        c = self.counts()
        row_ptr = np.zeros(c["n_nodes"] + 1, dtype=np.uint32)
        col = np.zeros((max(c["n_edges"], 1), 2), dtype=np.uint32)
        col_eid = np.zeros(max(c["n_edges"], 1), dtype=np.uint32)
        self._call("rala_b200_graph_get_csr", _ptr(row_ptr), _ptr(col), _ptr(col_eid))
        return row_ptr, col[:c["n_edges"]], col_eid[:c["n_edges"]]

    def stage_ms(self) -> dict:
        ms = (C.c_float * N_STAGES)()
        self._call("rala_b200_graph_stage_ms", ms)
        return dict(zip(STAGE_NAMES, [float(x) for x in ms]))

    # ---- the reference's two entry points ------------------------------------------------------
    def construct(self, records, piles, flags=None, hills=None, pile_ops=None):
        """Graph::construct's hot half.  `pile_ops` stands for the host-side Pile calls the reference
        makes between the passes (they stay on the host, SURVEY.md 8b):
            pile_ops.break_over_chimeric_hills(hill_coverage) -> (piles, flags) | None   graph.cpp:704-720
            pile_ops.break_over_chimeric_pits(connections)    -> (piles, flags) | None   graph.cpp:740-797
        With pile_ops=None the pile table is frozen (clean data)."""
        self.set_piles(piles, flags).set_hills(hills).set_overlaps(records)
        self.classify()
        if pile_ops is not None:
            upd = pile_ops.break_over_chimeric_hills(self.hill_coverage())
            if upd is not None:
                self.set_piles(*upd)
        self.retrim()
        while True:
            if pile_ops is not None:
                upd = pile_ops.break_over_chimeric_pits(self.connections())
                if upd is not None:
                    self.set_piles(*upd)
            if not self.retrim_promote():
                break
        self.finalize().build()
        c = self.counts()
        self.n_nodes, self.n_edges = c["n_nodes"], c["n_edges"]
        return self

    def remove_transitive_edges(self) -> int:
        """graph.cpp:1281-1335.  Device: marks.  Host tail: transitive_edges_ (:1320-1330)."""
        self.transitive()
        c = self.counts()
        marked = self.marked()
        e = self.edges()
        odd = np.nonzero(marked[1::2])[0] * 2 + 1
        s, d = e[odd, 0] & ~np.uint32(1), e[odd, 1] & ~np.uint32(1)
        pairs = np.concatenate([np.stack([s, d], 1), np.stack([d, s], 1)])
        order = np.lexsort((pairs[:, 1], pairs[:, 0]))
        self.transitive_edges = pairs[order]
        self.removed = marked
        return c["n_transitive_pairs"]


N_CAPS = 6
CAP_NAMES = ("events_per_pair", "edges_per_pair", "slice_edges", "max_sweeps", "max_final_sweeps", "local_edges")


def _by_position(parts):
    """[(rows, global positions), ...] -> the rows in position order"""
    rows = np.concatenate([r for r, _ in parts]) if parts else np.zeros((0, 7), np.uint32)
    pos = np.concatenate([p for _, p in parts]) if parts else np.zeros(0, np.uint64)
    return np.ascontiguousarray(rows[np.argsort(pos, kind="stable")])


class MultiCounts(C.Structure):
    _fields_ = [("world", C.c_int), ("n_local", C.c_int), ("n_records", C.c_uint64), ("n_piles", C.c_uint32),
                ("n_alive_piles", C.c_uint32), ("n_nodes", C.c_uint32), ("n_edges", C.c_uint64), ("n_local_edges", C.c_uint64),
                ("n_candidates", C.c_uint64), ("n_final_candidates", C.c_uint64), ("n_rounds", C.c_uint32),
                ("n_final_rounds", C.c_uint32), ("n_two_hop", C.c_uint64), ("n_transitive_pairs", C.c_uint64),
                ("n_heavy_items", C.c_uint32), ("fabric_error", C.c_uint32)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class Multi:
    """The multi-GPU session (rala_b200_multi): ranks [first_rank, first_rank + len(devices)) of `world` live in this
    process, one per entry of `devices` (an id may repeat: several ranks on one GPU, which is how the parity tests
    cover world > 1 on a one-GPU box).  Graph::construct's hot half + remove_transitive_edges with the pile table
    frozen (run), or changed by the host between the passes (the staged calls classify .. finish, construct),
    bit-identical to the single-GPU session on the concatenation of the shards."""

    def __init__(self, devices, first_rank: int = 0, world: int | None = None, lib=None):
        self.lib = lib or load()
        self.devices = list(devices)
        self.n_local = len(self.devices)
        self.world = self.n_local if world is None else world
        self.first_rank = first_rank
        self.handle = C.c_void_p()
        dev = (C.c_int * self.n_local)(*self.devices)
        rc = self.lib.rala_b200_multi_create(C.byref(self.handle), dev, C.c_int(self.n_local), C.c_int(first_rank), C.c_int(self.world))
        if rc != 0:
            raise RalaB200Error(f"rala_b200_multi_create(devices={self.devices}) failed with status {rc}: "
                                "sm_100 (B200) devices are required, there is no CPU fallback")
        self.n_piles = 0
        self.n_hills = 0
        self._keep = {}
        if len(set(self.devices)) < self.n_local:
            # ranks sharing a GPU wait for each other INSIDE kernels: every stream needs a hardware queue of its own
            # (3 streams per rank), or work of one rank queues up behind another rank's waiting barrier
            if int(os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "8")) < 3 * self.n_local + 3:
                raise RalaB200Error("several ranks on one device need CUDA_DEVICE_MAX_CONNECTIONS=32 in the environment "
                                    "before CUDA is initialised (tests/conftest.py sets it)")

    def _call(self, name, *args):
        rc = getattr(self.lib, name)(self.handle, *args)
        if rc != 0:
            msg = self.lib.rala_b200_multi_last_error(self.handle)
            raise RalaB200Error(f"{name}: status {rc}: {msg.decode() if msg else ''}")

    def close(self):
        if self.handle:
            self.lib.rala_b200_multi_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- inputs ------------------------------------------------------------------------------
    def set_piles(self, piles, flags=None):
        p = _np(piles, np.uint32, 2)
        f = None if flags is None else _np(flags, np.uint8)
        self.n_piles = p.shape[0]
        self._keep["piles"] = (p, f)
        self._call("rala_b200_multi_set_piles", _ptr(p), _ptr(f), C.c_uint32(self.n_piles))
        return self

    def set_hills(self, hills):
        """Replicated hill rows (grouped by ascending pile id); only the staged classify counts them."""
        h = _np(np.zeros((0, 3)) if hills is None else hills, np.uint32, 3)
        self.n_hills = h.shape[0]
        self._keep["hills"] = h
        self._call("rala_b200_multi_set_hills", _ptr(h), C.c_uint32(self.n_hills))
        return self

    def set_overlaps(self, k: int, records, t0: int):
        """Shard of local rank k: records [t0, t0 + n) of the file, in file order."""
        rec = _np(records, np.uint32, 7)
        self._keep[("rec", k)] = rec
        self._call("rala_b200_multi_set_overlaps", C.c_int(k), _ptr(rec), C.c_uint64(rec.shape[0]), C.c_uint64(t0))
        return self

    def set_overlaps_columns(self, k: int, columns, t0: int):
        cols = [_np(c, np.uint32) for c in columns]
        n = cols[0].shape[0]
        if len(cols) != 6 or any(c.shape[0] != n for c in cols):
            raise RalaB200Error("set_overlaps_columns needs six columns of equal length")
        self._keep[("rec", k)] = cols
        self._call("rala_b200_multi_set_overlaps_columns", C.c_int(k), *[_ptr(c) for c in cols], C.c_uint64(n), C.c_uint64(t0))
        return self

    def set_overlaps_packed(self, k: int, p: PackedRecords, t0: int):
        self._keep[("rec", k)] = p
        self._call("rala_b200_multi_set_overlaps_packed", C.c_int(k), _ptr(p.query_id), _ptr(p.group_end),
                   C.c_uint32(int(p.query_id.shape[0])), _ptr(p.b_id), _ptr(p.a_span), _ptr(p.b_span), C.c_uint64(p.n), C.c_uint64(t0))
        return self

    def set_outputs(self, k: int, edges_out=None, marked_out=None):
        """Pinned host buffers local rank k writes the rows of the edges it emitted, and their marks, into directly."""
        e_cap = 0 if edges_out is None else int(edges_out.shape[0])
        m_cap = 0 if marked_out is None else int(marked_out.shape[0])
        self._keep[("out", k)] = (edges_out, marked_out)
        self._call("rala_b200_multi_set_outputs", C.c_int(k), _ptr(edges_out), C.c_uint64(e_cap), _ptr(marked_out), C.c_uint64(m_cap))
        return self

    def set_shards(self, records, bounds=None):
        """All ranks local: cut the record list into `world` contiguous file ranges (equal record counts, 4-record aligned)."""
        rec = _np(records, np.uint32, 7)
        n = rec.shape[0]
        if bounds is None:
            per = ((n + self.world - 1) // self.world + 3) // 4 * 4
            bounds = [(min(n, r * per), min(n, (r + 1) * per)) for r in range(self.world)]
        for k, (b, e) in enumerate(bounds):
            self.set_overlaps(k, rec[b:e], b)
        return self

    # ---- exchange buffers ----------------------------------------------------------------------
    def default_caps(self):
        caps = np.zeros(N_CAPS, dtype=np.uint64)
        self._call("rala_b200_multi_default_caps", _ptr(caps))
        return caps

    def reserve(self, caps):
        caps = np.ascontiguousarray(caps, dtype=np.uint64)
        self._call("rala_b200_multi_reserve", _ptr(caps))
        self.caps = caps.copy()
        return self

    def set_rounds(self, rounds: int, final_rounds: int):
        self._call("rala_b200_multi_set_rounds", C.c_uint32(rounds), C.c_uint32(final_rounds))
        if hasattr(self, "caps"):   # only reserve() keeps a copy here: plan() sizes the buffers inside the library
            self.caps[3], self.caps[4] = rounds, final_rounds
        return self

    def export_handle(self, k: int = 0) -> bytes:
        buf = C.create_string_buffer(64)
        self._call("rala_b200_multi_export_handle", C.c_int(k), buf)
        return buf.raw

    def import_handles(self, handles: bytes):
        if len(handles) != 64 * self.world:
            raise RalaB200Error("import_handles needs one 64-byte handle per rank")
        self._call("rala_b200_multi_import_handles", C.c_char_p(handles))
        return self

    def plan(self):
        """All ranks local: size the exchange buffers from a first step (grows what did not fit)."""
        self._call("rala_b200_multi_plan")
        return self

    # ---- step ------------------------------------------------------------------------------------
    def run(self):
        self._call("rala_b200_multi_run")
        return self

    def use_cuda_graph(self, enabled: bool):
        self._call("rala_b200_multi_use_cuda_graph", C.c_int(1 if enabled else 0))
        return self

    def synchronize(self):
        self._call("rala_b200_multi_synchronize")
        return self

    def set_barrier_timeout_ms(self, ms: int):
        self._call("rala_b200_multi_set_barrier_timeout_ms", C.c_uint32(ms))
        return self

    def demand(self):
        need = np.zeros(N_CAPS, dtype=np.uint64)
        fits = C.c_int(0)
        self._call("rala_b200_multi_demand", _ptr(need), C.byref(fits))
        return need, bool(fits.value)

    def counts(self) -> dict:
        c = MultiCounts()
        self._call("rala_b200_multi_counts", C.byref(c))
        return c.as_dict()

    # ---- staged construct (pile tables that change between the passes) ---------------------------
    def classify(self):
        self._call("rala_b200_multi_classify")
        return self

    def retrim(self):
        self._call("rala_b200_multi_retrim")
        return self

    def retrim_promote(self) -> bool:
        changed = C.c_int(0)
        self._call("rala_b200_multi_retrim_promote", C.byref(changed))
        return bool(changed.value)

    def finish(self):
        """graph.cpp:831-877, 552-632 and 1281-1318 on the staged lists."""
        self._call("rala_b200_multi_finish")
        return self

    def hill_coverage(self, k: int = 0):
        """Hill counters of the first pass summed over all ranks, as local rank k holds them."""
        out = np.zeros(self.n_hills, dtype=np.uint32)
        self._call("rala_b200_multi_get_hill_coverage", C.c_int(k), _ptr(out))
        return out

    def local_lists(self, k: int):
        """(overlaps, their global positions, internals, their global positions) of local rank k."""
        n = np.zeros(2, dtype=np.uint64)
        self._call("rala_b200_multi_get_lists", C.c_int(k), None, None, None, None, _ptr(n))
        ovl, inl = np.zeros((int(n[0]), 7), np.uint32), np.zeros((int(n[1]), 7), np.uint32)
        opos, ipos = np.zeros(int(n[0]), np.uint64), np.zeros(int(n[1]), np.uint64)
        self._call("rala_b200_multi_get_lists", C.c_int(k), _ptr(ovl), _ptr(opos), _ptr(inl), _ptr(ipos), _ptr(n))
        return ovl, opos, inl, ipos

    def lists(self):
        """`overlaps` and `internals` in the reference's order, rebuilt from every local rank's entries and global positions
        (the whole lists when every rank is local)."""
        parts = [self.local_lists(k) for k in range(self.n_local)]
        return _by_position([(p[0], p[1]) for p in parts]), _by_position([(p[2], p[3]) for p in parts])

    def connections(self):
        """(a_id, b_id) of every entry of `overlaps` in list order: the input of the host's pit loop (graph.cpp:740-744)."""
        return np.ascontiguousarray(self.lists()[0][:, :2])

    def construct(self, records, piles, flags=None, hills=None, pile_ops=None):
        """Graph::construct's hot half and remove_transitive_edges on all ranks, with the same `pile_ops` contract as
        Graph.construct (pile_ops=None: the pile table is frozen, but the staged calls still run).  Every rank local: the
        records are cut with set_shards and plan() sizes the exchange buffers first."""
        self.set_piles(piles, flags).set_hills(hills).set_shards(records)
        self.plan()
        self.classify()
        if pile_ops is not None:
            upd = pile_ops.break_over_chimeric_hills(self.hill_coverage())
            if upd is not None:
                self.set_piles(*upd)
        self.retrim()
        while True:
            if pile_ops is not None:
                upd = pile_ops.break_over_chimeric_pits(self.connections())
                if upd is not None:
                    self.set_piles(*upd)
            if not self.retrim_promote():
                break
        self.finish()
        need, fits = self.demand()
        if not fits:   # plan() sized the buffers from a frozen step; the staged passes may need more
            raise RalaB200Error(f"construct: the staged passes did not fit the exchange buffers (need {need.tolist()}): "
                                "reserve() with larger capacities and construct again")
        c = self.counts()
        self.n_nodes, self.n_edges = c["n_nodes"], c["n_edges"]
        return self

    # ---- results -----------------------------------------------------------------------------------
    def edge_range(self, k: int):
        first, n = C.c_uint64(0), C.c_uint64(0)
        self._call("rala_b200_multi_edge_range", C.c_int(k), C.byref(first), C.byref(n))
        return int(first.value), int(n.value)

    def edge_runs(self, k: int):
        """(n, 2) array of (first global edge id, count): the ids of the rows edges(k) returns, in that order."""
        out = np.zeros((MAX_SEGMENTS, 2), dtype=np.uint64)
        n = C.c_uint32(0)
        self._call("rala_b200_multi_edge_runs", C.c_int(k), _ptr(out), C.byref(n))
        return out[:int(n.value)]

    def edge_ids(self, k: int):
        """Global id of every row edges(k) returns."""
        runs = self.edge_runs(k)
        if runs.shape[0] == 0:
            return np.zeros(0, dtype=np.int64)
        return np.concatenate([np.arange(int(f), int(f) + int(c), dtype=np.int64) for f, c in runs])

    def edges(self, k: int, out=None):
        n = int(self.edge_runs(k)[:, 1].sum())
        if out is None:
            out = np.zeros((n, 3), dtype=np.uint32)
        if n:
            self._call("rala_b200_multi_get_edges", C.c_int(k), _ptr(out))
        return out

    def marked(self, k: int, out=None):
        n = int(self.edge_runs(k)[:, 1].sum())
        if out is None:
            out = np.zeros(n, dtype=np.uint8)
        if n:
            self._call("rala_b200_multi_get_marked", C.c_int(k), _ptr(out))
        return out

    def all_edges(self):
        """Edge rows and marks of the local ranks in edge-id order (the whole graph when every rank is local)."""
        ids = [self.edge_ids(k) for k in range(self.n_local)]
        e = np.concatenate([self.edges(k) for k in range(self.n_local)])
        m = np.concatenate([self.marked(k) for k in range(self.n_local)])
        order = np.argsort(np.concatenate(ids), kind="stable")
        return e[order], m[order]

    def seq_to_node(self):
        out = np.zeros(self.n_piles, dtype=np.uint32)
        self._call("rala_b200_multi_get_seq_to_node", _ptr(out))
        return out

    def piles(self):
        out = np.zeros((self.n_piles, 2), dtype=np.uint32)
        self._call("rala_b200_multi_get_piles", _ptr(out))
        return out

    # ---- timing ------------------------------------------------------------------------------------
    def event_record(self, which: int):
        self._call("rala_b200_multi_event_record", C.c_int(which))

    def event_elapsed_ms(self) -> float:
        ms = C.c_float(0)
        self._call("rala_b200_multi_event_elapsed_ms", C.byref(ms))
        return float(ms.value)

    @property
    def launch_count(self) -> int:
        return int(self.lib.rala_b200_multi_launch_count(self.handle))

    def barrier_log(self, k: int = 0):
        """(n, 2) device timestamps in ns of the last barriers of local rank k: kernel started, all peers arrived."""
        out = np.zeros((128, 2), dtype=np.uint64)
        n = C.c_uint32(0)
        self._call("rala_b200_multi_barrier_log", C.c_int(k), _ptr(out), C.byref(n))
        return out[:int(n.value)]

    def sweep_log(self, k: int = 0, which_pass: int = 0):
        """(n, 2): per sweep of the last containment resolution, open victims at its start and ns since the kernel started."""
        out = np.zeros((48, 2), dtype=np.uint64)
        n = C.c_uint32(0)
        self._call("rala_b200_multi_sweep_log", C.c_int(k), C.c_int(which_pass), _ptr(out), C.byref(n))
        return out[:int(n.value)]

    BARRIERS_PER_STEP = 6   # events routed, list counts, final events routed, edges routed, slices pushed, marks routed

    def stage_ms(self, k: int = 0) -> dict:
        ms = (C.c_float * N_STAGES)()
        self._call("rala_b200_multi_stage_ms", C.c_int(k), ms)
        return dict(zip(STAGE_NAMES, [float(x) for x in ms]))
