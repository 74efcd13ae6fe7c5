"""The plain-C PAF reader (tests/paf_oracle.c) and a short Python restatement of the same text contract.

`parse(text, names, read_len)` runs the C reader: compiled with the system C compiler into a temporary directory the
first time it is needed (the repository tree stays untouched).  `restate(...)` is the contract in a dozen lines of Python,
slow, for small adversarial inputs.  Both return (cols (7, n) uint32, stats dict) or raise PafRefused(line, kind, column)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
KIND = {1: "fields", 2: "empty", 3: "digit", 4: "overflow"}
UNKNOWN = 0x7FFFFFFF
_LIB = None


class PafRefused(ValueError):
    def __init__(self, line: int, kind: str, column: int):
        super().__init__(f"line {line} column {column}: {kind}")
        self.line, self.kind, self.column = line, kind, column


class DuplicateName(ValueError):
    pass


def lib():
    global _LIB
    if _LIB is None:
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        assert cc, "a C compiler is needed for the PAF oracle"
        tmp = tempfile.mkdtemp(prefix="paf_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libpaf_oracle.so")
        subprocess.run([cc, "-O2", "-std=c11", "-Wall", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "paf_oracle.c")],
                       check=True, capture_output=True)
        _LIB = C.CDLL(so)
        _LIB.ora_parse_paf.restype = C.c_int
    return _LIB


def name_blob(names):
    """list of bytes -> (blob uint8, ends uint64); a (blob, ends) pair passes through."""
    if isinstance(names, tuple):
        return np.frombuffer(bytes(names[0]), np.uint8) if not isinstance(names[0], np.ndarray) else names[0], \
            np.ascontiguousarray(names[1], np.uint64)
    blob = b"".join(names)
    ends = np.cumsum([len(n) for n in names], dtype=np.uint64) if names else np.zeros(0, np.uint64)
    return np.frombuffer(blob, np.uint8), ends


def parse(text: bytes, names, read_len):
    blob, ends = name_blob(names)
    rl = np.ascontiguousarray(read_len, np.uint32)
    cap = len(text) // 19 + 2
    cols = np.zeros((7, cap), np.uint32)
    stats = np.zeros(4, np.uint64)
    err = np.zeros(3, np.uint64)
    buf = np.frombuffer(text, np.uint8) if len(text) else np.zeros(1, np.uint8)
    rc = lib().ora_parse_paf(C.c_void_p(blob.ctypes.data if blob.size else 0), C.c_void_p(ends.ctypes.data), C.c_void_p(rl.ctypes.data),
                             C.c_uint32(ends.shape[0]), C.c_void_p(buf.ctypes.data), C.c_uint64(len(text)),
                             C.c_void_p(cols.ctypes.data), C.c_uint64(cap), C.c_void_p(stats.ctypes.data), C.c_void_p(err.ctypes.data))
    if rc == -1:
        raise PafRefused(int(err[0]), KIND[int(err[1])], int(err[2]))
    if rc == -2:
        raise DuplicateName(f"reads {int(err[1])} and {int(err[0])} have the same name")
    assert rc == 0, rc
    n = int(stats[0])
    return np.ascontiguousarray(cols[:, :n]), {"n_records": n, "n_unresolved": int(stats[1]), "n_length_mismatch": int(stats[2]),
                                               "first_length_mismatch": int(stats[3])}


def restate(text: bytes, names, read_len):
    """The contract of include/rala_b200.h, line by line."""
    ids = {}
    for i, nm in enumerate(names):
        if nm in ids:
            raise DuplicateName(nm)
        ids[nm] = i
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                        # the text ended with '\n'
    rows, unresolved, mism, first = [], 0, 0, 2**64 - 1
    for no, ln in enumerate(lines, 1):
        if ln == b"":
            raise PafRefused(no, "empty", 1)
        f = ln.split(b"\t", 12)[:12]
        if len(f) < 12:
            raise PafRefused(no, "fields", len(f))
        num = {}
        for c in (1, 2, 3, 6, 7, 8, 10):
            if not f[c]:
                raise PafRefused(no, "digit", c + 1)
            v = 0
            for ch in f[c]:                # left to right: whichever comes first, a non-digit or the 33rd bit
                if not 48 <= ch <= 57:
                    raise PafRefused(no, "digit", c + 1)
                v = v * 10 + ch - 48
                if v >= 2**32:
                    raise PafRefused(no, "overflow", c + 1)
            num[c] = v
        a, b = ids.get(f[0], UNKNOWN), ids.get(f[5], UNKNOWN)
        known = a != UNKNOWN and b != UNKNOWN
        ori = 0 if f[4][:1] == b"+" else 1
        rows.append([a | (0 if known else 0x80000000), b | ori << 31, num[2], num[3], num[7], num[8], num[10]])
        unresolved += not known
        if (a != UNKNOWN and num[1] != int(read_len[a])) or (b != UNKNOWN and num[6] != int(read_len[b])):
            first = min(first, no - 1)
            mism += 1
    cols = np.asarray(rows, np.uint32).reshape(-1, 7).T.copy()
    return cols, {"n_records": len(rows), "n_unresolved": unresolved, "n_length_mismatch": mism, "first_length_mismatch": first}
