"""The plain-C FASTA / FASTQ reader (tests/reads_oracle.c) and a short Python restatement of the same text contract.

`read(text)` runs the C reader: compiled with the system C compiler into a temporary directory the first time it is needed
(the repository tree stays untouched).  `restate(text)` is the contract in plain Python, slow, for small adversarial inputs.
Both return (blob bytes, name_end uint64, read_len uint32, stats dict) or raise ReadsRefused(line, kind, column) /
DuplicateName(earlier, later)."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
KINDS = ["empty", "cr", "header", "name_empty", "name_byte", "seq_byte", "plus", "qual_len", "truncated", "no_seq", "too_long",
         "too_many", "format"]
KIND = {i + 1: k for i, k in enumerate(KINDS)}
RANK = {k: i + 1 for i, k in enumerate(KINDS)}
STATS = ["format", "n_reads", "n_lines", "n_bases", "name_bytes", "max_len", "n_described"]
_LIB = None


class ReadsRefused(ValueError):
    def __init__(self, line: int, kind: str, column: int):
        super().__init__(f"line {line} column {column}: {kind}")
        self.line, self.kind, self.column = line, kind, column


class DuplicateName(ValueError):
    def __init__(self, earlier: int, later: int):
        super().__init__(f"reads {earlier} and {later} have the same name")
        self.earlier, self.later = earlier, later


def lib():
    global _LIB
    if _LIB is None:
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        assert cc, "a C compiler is needed for the FASTA / FASTQ oracle"
        tmp = tempfile.mkdtemp(prefix="reads_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libreads_oracle.so")
        subprocess.run([cc, "-O2", "-std=c11", "-Wall", "-fPIC", "-shared", "-o", so, os.path.join(HERE, "reads_oracle.c")],
                       check=True, capture_output=True)
        _LIB = C.CDLL(so)
        _LIB.ora_read_seq.restype = C.c_int
    return _LIB


def read(text, cap: int | None = None):
    """text: bytes or a uint8 array; cap: reads to make room for (default: as many as the text could hold)."""
    n = len(text)
    cap = n // 2 + 2 if cap is None else cap
    buf = np.frombuffer(text, np.uint8) if n else np.zeros(1, np.uint8)
    blob = np.zeros(n + 1, np.uint8)
    ends = np.zeros(cap, np.uint64)
    lens = np.zeros(cap, np.uint32)
    stats = np.zeros(7, np.uint64)
    err = np.zeros(3, np.uint64)
    rc = lib().ora_read_seq(C.c_void_p(buf.ctypes.data), C.c_uint64(n), C.c_void_p(blob.ctypes.data), C.c_void_p(ends.ctypes.data),
                            C.c_void_p(lens.ctypes.data), C.c_uint64(cap), C.c_void_p(stats.ctypes.data), C.c_void_p(err.ctypes.data))
    if rc == -1:
        raise ReadsRefused(int(err[0]), KIND[int(err[2])], int(err[1]))
    if rc == -2:
        raise DuplicateName(int(err[0]), int(err[1]))
    assert rc == 0, rc
    st = {k: int(v) for k, v in zip(STATS, stats)}
    r = st["n_reads"]
    return blob[:st["name_bytes"]].tobytes(), ends[:r].copy(), lens[:r].copy(), st


def restate(text: bytes):
    """The contract of include/rala_b200.h, line by line; refusals collected and the smallest (line, column, kind) raised."""
    if not text:
        return b"", np.zeros(0, np.uint64), np.zeros(0, np.uint32), dict.fromkeys(STATS, 0)
    if text[:1] not in (b">", b"@"):
        raise ReadsRefused(1, "format", 1)
    fastq = text[:1] == b"@"
    lines = text.split(b"\n")
    if lines[-1] == b"":
        lines.pop()                                            # the text ended with '\n'
    bad = []
    names, hdr_line, length, described = [], [], [], 0
    for no, ln in enumerate(lines, 1):
        role = (no - 1) % 4
        hdr = role == 0 if fastq else ln[:1] == b">"
        seq = role == 1 if fastq else not hdr
        if not ln:
            bad.append((no, 1, "empty"))
        for col, ch in enumerate(ln, 1):
            if ch == 13 or (seq and not 0x21 <= ch <= 0x7E):
                bad.append((no, col, "cr" if ch == 13 else "seq_byte"))
                break
        if hdr:
            name = b""
            if ln:
                if fastq and ln[:1] != b"@":
                    bad.append((no, 1, "header"))
                cut = [i for i in (ln.find(b" ", 1), ln.find(b"\t", 1)) if i > 0]
                end = min(cut) if cut else len(ln)
                described += bool(cut)
                name = ln[1:end]
                if not name:
                    bad.append((no, 2, "name_empty"))
                ctl = [i for i, ch in enumerate(name) if (ch < 0x20 and ch != 13) or ch == 0x7F]
                if ctl:
                    bad.append((no, ctl[0] + 2, "name_byte"))
            names.append(name)
            hdr_line.append(no)
            length.append(0)
        elif ln:
            if not fastq:
                length[-1] += len(ln)
            elif role == 1:
                length[-1] = len(ln)
            elif role == 2:
                if ln[:1] != b"+":
                    bad.append((no, 1, "plus"))
            elif len(ln) != length[-1]:
                bad.append((no, min(len(ln), length[-1]) + 1, "qual_len"))
    if fastq and len(lines) % 4:
        bad.append((len(lines) // 4 * 4 + 1, 1, "truncated"))
    for no, ln in zip(hdr_line, length):
        if ln == 0:
            bad.append((no, 1, "no_seq"))
        if ln >= 2**32:
            bad.append((no, 1, "too_long"))
    if bad:
        no, col, kind = min(bad, key=lambda b: (b[0], b[1], RANK[b[2]]))
        raise ReadsRefused(no, kind, col)
    seen = {}
    for i, nm in enumerate(names):
        if nm in seen:
            raise DuplicateName(seen[nm], i)
        seen[nm] = i
    ends = np.cumsum([len(nm) for nm in names], dtype=np.uint64)
    st = {"format": 2 if fastq else 1, "n_reads": len(names), "n_lines": len(lines), "n_bases": sum(length),
          "name_bytes": int(ends[-1]) if len(ends) else 0, "max_len": max(length, default=0), "n_described": described}
    return b"".join(names), ends, np.asarray(length, np.uint32), st
