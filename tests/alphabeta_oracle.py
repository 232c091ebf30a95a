"""ctypes binding of the alpha-beta oracle (tests/alphabeta_oracle.cpp, TEST INFRASTRUCTURE: the CPU restatement of
ONB_AGENT_ALPHABETA). The library is compiled on first use into the temporary directory, keyed by the hash of its sources, so
the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "alphabeta_oracle.cpp"), os.path.join(ROOT, "oracle", "onb_oracle.cpp")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]
WIN = 1000000

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_alphabeta_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, out)  # atomic: concurrent builders never load a half-written library
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        for name in ("orc_alphabeta_batch", "orc_minimax_batch"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_ab_eval.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _batch(fn, roots, depth, threads):
    roots = np.ascontiguousarray(roots)
    assert roots.dtype.itemsize == 24
    n = len(roots)
    best = np.zeros(n, dtype=np.uint16)
    score = np.zeros(n, dtype=np.int32)
    nodes = np.zeros(n, dtype=np.uint64)
    fn(_p(roots), n, depth, threads, _p(best), _p(score), _p(nodes))
    return dict(best=best, score=score, nodes=nodes)


def alphabeta_batch(roots, depth, threads=None):
    """the defined search (fail-hard alpha-beta) per root: dict(best, score, nodes)"""
    return _batch(lib().orc_alphabeta_batch, roots, depth, threads or os.cpu_count() or 1)


def minimax_batch(roots, depth, threads=None):
    """the same tree without pruning"""
    return _batch(lib().orc_minimax_batch, roots, depth, threads or os.cpu_count() or 1)


def evaluate(states):
    """eval of each position from the view of its side to move"""
    s = np.ascontiguousarray(states)
    out = np.zeros(len(s), dtype=np.int32)
    lib().orc_ab_eval(_p(s), len(s), _p(out))
    return out
