"""The plain-C restatement of Graph::initialize's coverage half (tests/piles_oracle.c), compiled with the system C compiler
into a temporary directory the first time it is needed (the repository tree stays untouched).

`build_piles(cols, read_len)` -> dict with piles (n_reads, 2), medians, runs (run_off, run_begin, run_cov) and stats, or
raises Refused(record, kind) / CoverageLimit."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
KIND = {1: "id", 2: "self", 3: "a_empty", 4: "a_beyond", 5: "b_empty", 6: "b_beyond"}
STATS = ("n_counted", "n_runs", "max_coverage", "n_live", "n_tied", "n_exact_min")
_LIB = None


class Refused(ValueError):
    def __init__(self, record: int, kind: str):
        super().__init__(f"record {record}: {kind}")
        self.record, self.kind = record, kind


class CoverageLimit(ValueError):
    pass


def lib():
    global _LIB
    if _LIB is None:
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        assert cc, "a C compiler is needed for the pile oracle"
        tmp = tempfile.mkdtemp(prefix="piles_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libpiles_oracle.so")
        subprocess.run([cc, "-O2", "-std=c11", "-Wall", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "piles_oracle.c")],
                       check=True, capture_output=True)
        _LIB = C.CDLL(so)
        _LIB.ora_build_piles.restype = C.c_int
    return _LIB


def columns(records) -> np.ndarray:
    """rala_ovl_t rows (n, 7) as the golden front end dumps them (unresolved = a_id 0xFFFFFFFF) -> the six columns (6, n),
    bit 31 of a_id = unresolved; the INVALID flag (duplicate filter) is NOT carried: those records count."""
    r = np.ascontiguousarray(records, np.uint32).reshape(-1, 7)
    cols = np.empty((6, r.shape[0]), np.uint32)
    cols[0] = np.where(r[:, 0] == 0xFFFFFFFF, np.uint32(0xFFFFFFFF), r[:, 0])
    cols[1] = (r[:, 1] & 0x7FFFFFFF) | ((r[:, 6] & 1) << 31)
    cols[2:6] = r[:, 2:6].T
    return cols


def build_piles(cols, read_len, runs: bool = True) -> dict:
    cols = np.ascontiguousarray(cols, np.uint32).reshape(6, -1)
    rl = np.ascontiguousarray(read_len, np.uint32)
    n, n_reads = cols.shape[1], rl.shape[0]
    piles = np.zeros((n_reads, 2), np.uint32)
    med = np.zeros(n_reads, np.uint16)
    stats = np.zeros(6, np.uint64)
    err = np.zeros(2, np.uint64)
    cap = 4 * n + n_reads if runs else 0
    off = np.zeros(n_reads + 1, np.uint32) if runs else None
    rb = np.zeros(max(cap, 1), np.uint32) if runs else None
    rc_ = np.zeros(max(cap, 1), np.uint16) if runs else None
    p = lambda a: None if a is None else C.c_void_p(a.ctypes.data)   # noqa: E731
    rc = lib().ora_build_piles(p(cols) if n else C.c_void_p(0), C.c_uint64(n), p(rl) if n_reads else C.c_void_p(0), C.c_uint32(n_reads),
                               p(piles), p(med), p(stats), p(off), p(rb), p(rc_), C.c_uint64(cap), p(err))
    if rc == -1:
        raise Refused(int(err[0]), KIND[int(err[1])])
    if rc == -2:
        raise CoverageLimit(f"coverage {int(err[0])} >= 65536")
    assert rc == 0, rc
    out = {"piles": piles, "medians": med, "stats": {k: int(v) for k, v in zip(STATS, stats)}}
    if runs:
        t = int(off[-1])
        out["runs"] = (off, rb[:t].copy(), rc_[:t].copy())
    return out


def expand_runs(run_off, run_begin, run_cov, read_len, r: int) -> np.ndarray:
    """Per-base coverage of read r from its runs."""
    a, b = int(run_off[r]), int(run_off[r + 1])
    ends = np.append(run_begin[a + 1:b], read_len[r]).astype(np.int64)
    return np.repeat(run_cov[a:b].astype(np.int64), ends - run_begin[a:b].astype(np.int64))


def coverage(cols, read_len, r: int) -> np.ndarray:
    """Per-base coverage of read r straight from the rule, in numpy (difference array)."""
    cols = np.asarray(cols, np.int64).reshape(6, -1)
    ok = (cols[0] >> 31) == 0
    a, b = cols[0], cols[1] & 0x7FFFFFFF
    d = np.zeros(int(read_len[r]) + 1, np.int64)
    for ids, lo, hi in ((a, cols[2], cols[3]), (b, cols[4], cols[5])):
        m = ok & (ids == r)
        np.add.at(d, lo[m] + 15, 1)
        np.add.at(d, hi[m] - 15, -1)
    return np.cumsum(d)[:-1]
