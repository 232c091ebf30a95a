"""ctypes binding of the Gumbel MuZero oracle (tests/gumbel_interior_oracle.cpp, TEST INFRASTRUCTURE): the Gumbel-search oracle with
interior selection below the root (onb_gumbel_config.interior) and the per-node rule on given nodes. The library is compiled on first
use into the temporary directory, keyed by the hash of its sources, so the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import gumbel_oracle as GO
from oracle_lib import EVAL_CB, TreeDump

SOURCES = [os.path.join(GO.HERE, "gumbel_interior_oracle.cpp")] + GO.SOURCES

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(GO.CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_gumbel_interior_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + GO.CXXFLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, out)  # atomic: concurrent builders never load a half-written library
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.orc_gumbel_interior_search_batch.argtypes = ([C.c_void_p, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                                        C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32, C.c_uint64] +
                                                       [C.c_void_p] * 7 + [C.c_int64, C.c_void_p, C.c_int64, C.c_int])
        L.orc_gumbel_interior_choice.argtypes = [C.c_int64] + [C.c_void_p] * 5 + [C.c_double, C.c_double, C.c_void_p]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def choice(off, P, N, Q, rx, c_visit=50.0, c_scale=0.1):
    """the oracle's interior choice for nodes i = 0 .. len(rx): children [off[i], off[i + 1]) of P / N / Q"""
    off, P, N, Q, rx = (np.ascontiguousarray(off, np.int64), np.ascontiguousarray(P, np.float64), np.ascontiguousarray(N, np.uint32),
                        np.ascontiguousarray(Q, np.float64), np.ascontiguousarray(rx, np.float64))
    out = np.zeros(len(rx), np.int64)
    lib().orc_gumbel_interior_choice(len(rx), _p(off), _p(P), _p(N), _p(Q), _p(rx), c_visit, c_scale, _p(out))
    return out


def search(roots, c_puct, sims, evaluator=0, m=16, c_visit=50.0, c_scale=0.1, gumbel_scale=1.0, seed=0, step=0, game0=0, callback=None,
           dump_tree=-1, threads=None, interior=1):
    """gumbel_oracle.search with interior selection below the root (interior=0: the root-only search through this library's loop)"""
    s = np.ascontiguousarray(roots)
    assert s.dtype.itemsize == 24
    n = len(s)
    out = dict(best=np.zeros(n, np.uint16), pi=np.zeros((n, 2, 25), np.float32), root_visits=np.zeros(n, np.uint32), root_q=np.zeros(n, np.float64),
               child_visits=np.zeros((n, 40), np.uint32), n_nodes=np.zeros(n, np.int64), r0=np.zeros(n, np.float64))
    cb = None
    if callback is not None:
        def _cb(planes_p, pol_p, val_p, _user):
            planes = np.ctypeslib.as_array(planes_p, shape=(525,)).copy()
            pol, val = callback(planes)
            np.ctypeslib.as_array(pol_p, shape=(50,))[:] = np.asarray(pol, dtype=np.float32).reshape(50)
            val_p[0] = float(val)
        cb = EVAL_CB(_cb)
        evaluator = 2
    cap = 1 + 40 * max(sims, 1) + 2
    arrs = dict(visits=np.zeros(cap, np.uint32), reward=np.zeros(cap, np.float64), winrate=np.zeros(cap, np.float64), prior=np.zeros(cap, np.float64),
                action=np.zeros(cap, np.uint16), parent=np.zeros(cap, np.int32), first_child=np.zeros(cap, np.uint32), n_child=np.zeros(cap, np.uint32),
                flags=np.zeros(cap, np.uint8))
    td = TreeDump(*[_p(arrs[k]) for k, _ in TreeDump._fields_]) if dump_tree >= 0 else None
    lib().orc_gumbel_interior_search_batch(_p(s), n, c_puct, sims, evaluator, C.cast(cb, C.c_void_p) if cb else None, None,
                                           threads or os.cpu_count() or 1, m, c_visit, c_scale, gumbel_scale, seed, step, game0,
                                           *[_p(out[k]) for k in ("best", "pi", "root_visits", "root_q", "child_visits", "n_nodes", "r0")],
                                           dump_tree, C.byref(td) if td is not None else None, cap, int(interior))
    if dump_tree >= 0:
        nn = int(out["n_nodes"][dump_tree])
        out["tree"] = {k: v[:nn].copy() for k, v in arrs.items()}
    return out
