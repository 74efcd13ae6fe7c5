"""ctypes binding of oracle/liboracle.so — TEST INFRASTRUCTURE.

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs may import this module; the product package ``rala_b200`` never does.  Parity status of the
underlying C code: pinned against the compiled reference (see rala_oracle.h).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

KX, KA, KB, KAB, KBA, REJECT = 0, 1, 2, 3, 4, 255


def build() -> str:
    """Compile liboracle.so (and oracle/_ref when /root/reference is present)."""
    subprocess.run(["make", "-s", "-C", _HERE, "all"], check=True)
    return os.path.join(_HERE, "liboracle.so")


def lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "liboracle.so")
        if not os.path.exists(path):
            subprocess.run(["make", "-s", "-C", _HERE, "liboracle.so"], check=True)
        _LIB = C.CDLL(path)
        _LIB.ora_transitive.restype = C.c_uint64
        _LIB.ora_transitive_pairs.restype = C.c_uint64
        _LIB.ora_retrim.restype = C.c_uint64
    return _LIB


def _p(a, t=C.c_uint32):
    return a.ctypes.data_as(C.POINTER(t))


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def comparable(a: int, b: int) -> bool:
    return bool(lib().ora_comparable(C.c_uint32(a), C.c_uint32(b)))


def trim_type(rec, pa, pb):
    """rec: 7 u32 (a_id/b_id ignored); pa/pb: (begin, end).  -> (ok, trimmed rec, type)"""
    r = _u32(rec).copy()
    r[0], r[1] = 0, 1
    piles = _u32([pa[0], pa[1], pb[0], pb[1]])
    ok = lib().ora_trim(_p(r), _p(piles), C.c_uint32(2))
    t = lib().ora_type(_p(r), _p(piles)) if ok else REJECT
    return bool(ok), r, t


def trim_type_batch(rec, piles):
    """rec (n,7), piles (n_piles,2) -> (trimmed (n,7), type (n,) uint8 with 255 = rejected)."""
    r = _u32(rec).reshape(-1, 7).copy()
    piles = _u32(piles).reshape(-1, 2)
    types = np.full(r.shape[0], REJECT, dtype=np.uint8)
    if r.shape[0]:
        lib().ora_trim_type_batch(_p(r), C.c_uint64(r.shape[0]), _p(piles), C.c_uint32(piles.shape[0]), _p(types, C.c_uint8))
    return r, types


class Pipeline:
    """The hot path, stage by stage, on numpy arrays (same stage boundaries as the CUDA session)."""

    def __init__(self, records, piles, pflags=None, hills=None):
        self.records = _u32(records).reshape(-1, 7)
        self.piles = _u32(piles).reshape(-1, 2).copy()
        self.n_piles = self.piles.shape[0]
        self.pflags = (np.zeros(self.n_piles, dtype=np.uint8) if pflags is None
                       else np.ascontiguousarray(pflags, dtype=np.uint8))
        self.hills = _u32(np.zeros((0, 3)) if hills is None else hills).reshape(-1, 3)
        self.hill_cov = np.zeros(self.hills.shape[0], dtype=np.uint32)
        self.ovl = np.zeros((0, 7), dtype=np.uint32)
        self.int = np.zeros((0, 7), dtype=np.uint32)

    def classify(self):
        n = self.records.shape[0]
        ovl = np.zeros((max(n, 1), 7), dtype=np.uint32)
        inl = np.zeros((max(n, 1), 7), dtype=np.uint32)
        n_ovl, n_int = C.c_uint64(0), C.c_uint64(0)
        hills = self.hills if self.hills.shape[0] else np.zeros((1, 3), dtype=np.uint32)
        cov = self.hill_cov if self.hill_cov.shape[0] else np.zeros(1, dtype=np.uint32)
        lib().ora_classify(_p(self.records), C.c_uint64(n), _p(self.piles), _p(self.pflags, C.c_uint8),
                           C.c_uint32(self.n_piles), _p(hills), C.c_uint32(self.hills.shape[0]), _p(cov),
                           _p(ovl), C.byref(n_ovl), _p(inl), C.byref(n_int))
        self.ovl = ovl[:n_ovl.value].copy()
        self.int = inl[:n_int.value].copy()
        return self

    def set_piles(self, piles):
        self.piles = _u32(piles).reshape(-1, 2).copy()
        return self

    def _retrim(self, lst):
        lst = np.ascontiguousarray(lst)
        n = C.c_uint64(lst.shape[0])
        dropped = lib().ora_retrim(_p(lst), C.byref(n), _p(self.piles), C.c_uint32(self.n_piles))
        return lst[:n.value].copy(), int(dropped)

    def retrim(self):
        """graph.cpp:722-736"""
        self.ovl, _ = self._retrim(self.ovl)
        self.int, _ = self._retrim(self.int)
        return self

    def retrim_promote(self) -> bool:
        """graph.cpp:801-824; returns is_changed"""
        self.ovl, dropped = self._retrim(self.ovl)
        n_o, n_i = self.ovl.shape[0], self.int.shape[0]
        ovl = np.zeros((n_o + n_i + 1, 7), dtype=np.uint32)
        ovl[:n_o] = self.ovl
        inl = np.ascontiguousarray(self.int) if n_i else np.zeros((1, 7), dtype=np.uint32)
        c_o, c_i = C.c_uint64(n_o), C.c_uint64(n_i)
        lib().ora_retrim_promote(_p(inl), C.byref(c_i), _p(ovl), C.byref(c_o), _p(self.piles),
                                 C.c_uint32(self.n_piles))
        self.ovl = ovl[:c_o.value].copy()
        self.int = inl[:c_i.value].copy()
        return dropped > 0

    def final_containment(self):
        ovl = np.ascontiguousarray(self.ovl) if self.ovl.shape[0] else np.zeros((1, 7), dtype=np.uint32)
        inl = np.ascontiguousarray(self.int) if self.int.shape[0] else np.zeros((1, 7), dtype=np.uint32)
        c_o, c_i = C.c_uint64(self.ovl.shape[0]), C.c_uint64(self.int.shape[0])
        lib().ora_final_containment(_p(ovl), C.byref(c_o), _p(inl), C.byref(c_i), _p(self.piles),
                                    C.c_uint32(self.n_piles))
        self.ovl = ovl[:c_o.value].copy()
        self.int = inl[:c_i.value].copy()
        return self

    def build_edges(self):
        n = self.ovl.shape[0]
        s2n = np.zeros(self.n_piles, dtype=np.uint32)
        edges = np.zeros((2 * n + 1, 3), dtype=np.uint32)
        n_nodes, n_edges = C.c_uint32(0), C.c_uint64(0)
        ovl = np.ascontiguousarray(self.ovl) if n else np.zeros((1, 7), dtype=np.uint32)
        lib().ora_build_edges(_p(ovl), C.c_uint64(n), _p(self.piles), C.c_uint32(self.n_piles), _p(s2n),
                              C.byref(n_nodes), _p(edges), C.byref(n_edges))
        self.seq_to_node = s2n
        self.n_nodes = n_nodes.value
        self.edges = edges[:n_edges.value].copy()
        return self

    def transitive(self):
        self.marked, self.n_pairs = transitive(self.n_nodes, self.edges)
        return self

    def run(self):
        """Frozen pile table (no host pile breaking between the passes)."""
        self.classify().retrim()
        while self.retrim_promote():
            pass
        return self.final_containment().build_edges().transitive()


def transitive(n_nodes: int, edges):
    edges = _u32(edges).reshape(-1, 3)
    marked = np.zeros(max(edges.shape[0], 1), dtype=np.uint8)
    e = edges if edges.shape[0] else np.zeros((1, 3), dtype=np.uint32)
    n_pairs = lib().ora_transitive(C.c_uint32(n_nodes), C.c_uint64(edges.shape[0]), _p(e), _p(marked, C.c_uint8))
    return marked[:edges.shape[0]], int(n_pairs)


def transitive_pairs(edges, marked):
    edges = _u32(edges).reshape(-1, 3)
    marked = np.ascontiguousarray(marked, dtype=np.uint8)
    out = np.zeros((max(int(marked.sum()), 1), 2), dtype=np.uint32)
    n = lib().ora_transitive_pairs(C.c_uint64(edges.shape[0]), _p(edges), _p(marked, C.c_uint8), _p(out))
    return out[:n]


def adjacency(n_nodes: int, edges, marked=None, which: int = 0):
    edges = _u32(edges).reshape(-1, 3)
    off = np.zeros(n_nodes + 1, dtype=np.uint32)
    ids = np.zeros(max(edges.shape[0], 1), dtype=np.uint32)
    m = None if marked is None else np.ascontiguousarray(marked, dtype=np.uint8)
    lib().ora_adjacency(C.c_uint32(n_nodes), C.c_uint64(edges.shape[0]), _p(edges),
                        None if m is None else _p(m, C.c_uint8), C.c_int(which), _p(off), _p(ids))
    return off, ids[:off[-1]]


# ---------------------------------------------------------------------------------------------
# oracle/_ref (the compiled, unmodified reference + harness) — present when built in this container
# ---------------------------------------------------------------------------------------------
REF_BIN = os.path.join(_HERE, "_ref", "rala_ref")


def filter_duplicates(a, b, length):
    """is_valid_overlap_ after Graph::initialize's overlap pass (graph.cpp:273-303); a with bit 31 = unknown record."""
    a, b, length = _u32(a), _u32(b), _u32(length)
    valid = np.zeros(a.shape[0], dtype=np.uint8)
    lib().ora_filter_duplicates(_p(a), _p(b), _p(length), C.c_uint64(a.shape[0]), _p(valid, C.c_uint8))
    return valid


def have_ref() -> bool:
    return os.path.exists(REF_BIN) and os.access(REF_BIN, os.X_OK)


def load_u32(path: str, cols: int | None = None):
    a = np.fromfile(path, dtype=np.uint32)
    return a if cols is None else a.reshape(-1, cols)


def ref_run(args, stdin: str | None = None) -> str:
    out = subprocess.run([REF_BIN] + [str(a) for a in args], input=stdin, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError(f"rala_ref {args[0]} failed ({out.returncode}): {out.stderr[-2000:]}")
    return out.stdout


def write_hotpath_inputs(prefix: str, records, piles, pflags=None, hills=None, read_len=None, medians=None):
    """Files in the layout `rala_ref hotpath` reads."""
    records = _u32(records).reshape(-1, 7)
    piles = _u32(piles).reshape(-1, 2)
    n = piles.shape[0]
    p4 = np.zeros((n, 4), dtype=np.uint32)
    p4[:, :2] = piles
    if pflags is not None:
        p4[:, 2] = np.asarray(pflags, dtype=np.uint32)
    if medians is not None:
        p4[:, 3] = np.asarray(medians, dtype=np.uint32)
    records.tofile(prefix + ".in.records.u32")
    p4.tofile(prefix + ".in.piles.u32")
    h = np.zeros((0, 4), dtype=np.uint32) if hills is None else np.concatenate(
        [_u32(hills).reshape(-1, 3), np.zeros((len(hills), 1), dtype=np.uint32)], axis=1)
    h.tofile(prefix + ".in.hills.u32")
    if read_len is None:
        read_len = piles[:, 1] + 15
    _u32(read_len).tofile(prefix + ".in.read_len.u32")
