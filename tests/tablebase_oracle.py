"""ctypes binding of the tablebase oracle (tests/tablebase_oracle.cpp, TEST INFRASTRUCTURE: the CPU restatement of onb_tb_*). The
library is compiled on first use into the temporary directory, keyed by the hash of its sources, so the repository tree is never
written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "tablebase_oracle.cpp"), os.path.join(ROOT, "oracle", "onb_oracle.cpp")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]
NONE = -32768
THREADS = os.cpu_count() or 1

_lib = None
_solved = {}


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_tablebase_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, out)  # atomic: concurrent builders never load a half-written library
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        P = C.c_void_p
        L.orc_tb_entries.restype = C.c_uint64
        L.orc_tb_entries.argtypes = [C.c_int, C.c_int]
        L.orc_tb_solve.argtypes = [P, C.c_int, C.c_int, P, P]
        L.orc_tb_check_local.restype = C.c_int64
        L.orc_tb_check_local.argtypes = [P, C.c_int, P, C.c_int, P, C.c_int64, C.c_int, P, C.c_int64]
        L.orc_tb_check_swap.restype = C.c_int64
        L.orc_tb_check_swap.argtypes = [P, C.c_int, P, C.c_int, P, C.c_int64, C.c_int]
        L.orc_tb_probe.argtypes = [P, C.c_int, P, P, C.c_int64, P]
        L.orc_tb_best.argtypes = [P, C.c_int, P, P, C.c_int64, C.c_int, P]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def entries(p, q):
    return int(lib().orc_tb_entries(p, q))


def _cards(cards):
    return np.ascontiguousarray(cards, dtype=np.uint8).reshape(5)


def _ptrs(tables):
    """{(p, q): int16 array} -> 25 pointers"""
    arr = (C.c_void_p * 25)()
    for (p, q), t in tables.items():
        assert t.dtype == np.int16 and t.flags.c_contiguous and len(t) == entries(p, q)
        arr[5 * p + q] = t.ctypes.data
    return arr


def solve(cards, max_pawns):
    """{(p, q): int16 table} and {(p, q): dict(iterations, max_win, max_loss)}; memoised per process"""
    key = (tuple(sorted(int(c) for c in cards)), max_pawns)
    if key not in _solved:
        tables = {(p, q): np.zeros(entries(p, q), np.int16) for p in range(5) for q in range(5) if p + q <= max_pawns}
        stats = np.zeros((25, 4), np.int32)
        rc = lib().orc_tb_solve(_p(_cards(cards)), max_pawns, THREADS, _ptrs(tables), _p(stats))
        assert rc == 0
        info = {(k // 5, k % 5): dict(iterations=int(stats[k, 0]), max_win=int(stats[k, 1]), max_loss=int(stats[k, 2]))
                for k in range(25) if stats[k, 3]}
        _solved[key] = (tables, info)
    return _solved[key]


def check_local(cards, max_pawns, tables, p, q, idx=None, cap=16):
    """(number of entries of class (p, q) that differ from the rule applied to their children, the first offenders)"""
    i = None if idx is None else np.ascontiguousarray(idx, dtype=np.int64)
    bad = np.zeros(cap, np.int64)
    nb = lib().orc_tb_check_local(_p(_cards(cards)), max_pawns, _ptrs(tables), 5 * p + q, _p(i), 0 if i is None else len(i), THREADS,
                                  _p(bad), cap)
    return int(nb), bad[:min(nb, cap)]


def check_swap(cards, max_pawns, tables, p, q, idx=None):
    i = None if idx is None else np.ascontiguousarray(idx, dtype=np.int64)
    return int(lib().orc_tb_check_swap(_p(_cards(cards)), max_pawns, _ptrs(tables), 5 * p + q, _p(i), 0 if i is None else len(i), THREADS))


def probe(cards, max_pawns, tables, states):
    s = np.ascontiguousarray(states)
    out = np.zeros(len(s), np.int16)
    lib().orc_tb_probe(_p(_cards(cards)), max_pawns, _ptrs(tables), _p(s), len(s), _p(out))
    return out


def best(cards, max_pawns, tables, states):
    s = np.ascontiguousarray(states)
    out = np.zeros(len(s), np.uint16)
    lib().orc_tb_best(_p(_cards(cards)), max_pawns, _ptrs(tables), _p(s), len(s), THREADS, _p(out))
    return out
