"""The plain-C MHAP reader (tests/mhap_oracle.c) and a short Python restatement of the same text contract.

`parse(text, read_len)` runs the C reader, compiled as tests/paf_oracle.py compiles its reader (into a temporary
directory, the repository tree stays untouched).  `restate(...)` is the contract in a dozen lines of Python, slow, for
small adversarial inputs.  Both return (cols (7, n) uint32, stats dict) or raise MhapRefused(line, kind, field)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from tests.paf_oracle import PafRefused

HERE = os.path.dirname(os.path.abspath(__file__))
KIND = {1: "fields", 2: "empty", 3: "digit", 4: "overflow", 5: "read id", 6: "strand"}
_LIB = None


class MhapRefused(PafRefused):
    """A refused line: .line (1-based), .kind, .column (= the 1-based field; fields found for "fields")."""

    @property
    def field(self) -> int:
        return self.column


def lib():
    global _LIB
    if _LIB is None:
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        assert cc, "a C compiler is needed for the MHAP oracle"
        tmp = tempfile.mkdtemp(prefix="mhap_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libmhap_oracle.so")
        subprocess.run([cc, "-O2", "-std=c11", "-Wall", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "mhap_oracle.c")],
                       check=True, capture_output=True)
        _LIB = C.CDLL(so)
        _LIB.ora_parse_mhap.restype = C.c_int
    return _LIB


def parse(text: bytes, read_len):
    rl = np.ascontiguousarray(read_len, np.uint32)
    if rl.size == 0:
        rl = np.zeros(1, np.uint32)[:0]
    cap = len(text) // 22 + 2
    cols = np.zeros((7, cap), np.uint32)
    stats = np.zeros(4, np.uint64)
    err = np.zeros(3, np.uint64)
    buf = np.frombuffer(text, np.uint8) if len(text) else np.zeros(1, np.uint8)
    rc = lib().ora_parse_mhap(C.c_void_p(rl.ctypes.data), C.c_uint32(rl.shape[0]), C.c_void_p(buf.ctypes.data),
                              C.c_uint64(len(text)), C.c_void_p(cols.ctypes.data), C.c_uint64(cap), C.c_void_p(stats.ctypes.data),
                              C.c_void_p(err.ctypes.data))
    if rc == -1:
        raise MhapRefused(int(err[0]), KIND[int(err[1])], int(err[2]))
    assert rc == 0, rc
    n = int(stats[0])
    return np.ascontiguousarray(cols[:, :n]), {"n_records": n, "n_length_mismatch": int(stats[1]),
                                               "first_length_mismatch": int(stats[2]), "n_query_rc": int(stats[3])}


def restate(text: bytes, read_len):
    """The contract of include/rala_b200.h, line by line."""
    lines = text.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()                        # the text ended with '\n'
    rows, mism, first, qrc = [], 0, 2**64 - 1, 0
    for no, ln in enumerate(lines, 1):
        if ln == b"":
            raise MhapRefused(no, "empty", 1)
        f = ln.split(b" ", 12)
        if len(f) < 12:
            raise MhapRefused(no, "fields", len(f))
        if len(f) == 12 and f[11].endswith(b"\r"):
            f[11] = f[11][:-1]             # CRLF
        v = {}
        for c in (0, 1, 4, 5, 6, 7, 8, 9, 10, 11):
            if c in (4, 8):
                if f[c] not in (b"0", b"1"):
                    raise MhapRefused(no, "strand", c + 1)
                v[c] = int(f[c])
                continue
            if not f[c]:
                raise MhapRefused(no, "digit", c + 1)
            x = 0
            for ch in f[c]:                # left to right: whichever comes first, a non-digit or the 33rd bit
                if not 48 <= ch <= 57:
                    raise MhapRefused(no, "digit", c + 1)
                x = x * 10 + ch - 48
                if x >= 2**32:
                    raise MhapRefused(no, "overflow", c + 1)
            v[c] = x
            if c < 2 and not 1 <= v[c] <= len(read_len):
                raise MhapRefused(no, "read id", c + 1)
        a, b = v[0] - 1, v[1] - 1
        length = max((v[6] - v[5]) % 2**32, (v[10] - v[9]) % 2**32)
        rows.append([a, b | (v[4] ^ v[8]) << 31, v[5], v[6], v[9], v[10], length])
        qrc += v[4]
        if v[7] != int(read_len[a]) or v[11] != int(read_len[b]):
            first = min(first, no - 1)
            mism += 1
    cols = np.asarray(rows, np.uint32).reshape(-1, 7).T.copy()
    return cols, {"n_records": len(rows), "n_length_mismatch": mism, "first_length_mismatch": first, "n_query_rc": qrc}
