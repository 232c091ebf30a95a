"""ctypes binding of the Gumbel-search oracle (tests/gumbel_oracle.cpp, TEST INFRASTRUCTURE: the CPU restatement of
onb_mcts_set_gumbel on top of the CPU oracle's MctsArena, and the host build of onb_gumbel.cuh's onb_log / onb_exp /
sequential-halving table). The library is compiled on first use into the temporary directory, keyed by the hash of its sources,
so the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle_lib import EVAL_CB, TreeDump

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "gumbel_oracle.cpp"), os.path.join(ROOT, "oracle", "onb_oracle.cpp"),
           os.path.join(ROOT, "onitama_alphazero_b200", "csrc", "onb_gumbel.cuh")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_gumbel_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, out)  # atomic: concurrent builders never load a half-written library
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.orc_gumbel_log.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        L.orc_gumbel_exp.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        L.orc_gumbel_seq.argtypes = [C.c_uint32, C.c_uint32, C.c_void_p]
        L.orc_gumbel_search_batch.argtypes = ([C.c_void_p, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_uint32,
                                               C.c_double, C.c_double, C.c_double, C.c_uint64, C.c_uint32, C.c_uint64] + [C.c_void_p] * 7 +
                                              [C.c_int64, C.c_void_p, C.c_int64])
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def onb_log(x):
    x = np.ascontiguousarray(x, np.float64)
    out = np.empty_like(x)
    lib().orc_gumbel_log(_p(x), x.size, _p(out))
    return out


def onb_exp(x):
    x = np.ascontiguousarray(x, np.float64)
    out = np.empty_like(x)
    lib().orc_gumbel_exp(_p(x), x.size, _p(out))
    return out


def seq(m, n):
    out = np.zeros(n, np.uint32)
    lib().orc_gumbel_seq(m, n, _p(out))
    return out


def search(roots, c_puct, sims, evaluator=0, m=16, c_visit=50.0, c_scale=0.1, gumbel_scale=1.0, seed=0, step=0, game0=0, callback=None,
           dump_tree=-1, threads=None):
    """Gumbel searches of every root (tree i = global game game0 + i). callback(planes[525]) -> (policy[50], value) replaces the
    evaluator (single-threaded). Returns dict(best, pi [n,2,25], root_visits, root_q, child_visits [n,40], n_nodes, r0) and, with
    dump_tree >= 0, 'tree': that tree's arena as orc_mcts_search dumps it."""
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
    lib().orc_gumbel_search_batch(_p(s), n, c_puct, sims, evaluator, C.cast(cb, C.c_void_p) if cb else None, None, threads or os.cpu_count() or 1,
                                  m, c_visit, c_scale, gumbel_scale, seed, step, game0,
                                  *[_p(out[k]) for k in ("best", "pi", "root_visits", "root_q", "child_visits", "n_nodes", "r0")],
                                  dump_tree, C.byref(td) if td is not None else None, cap)
    if dump_tree >= 0:
        nn = int(out["n_nodes"][dump_tree])
        out["tree"] = {k: v[:nn].copy() for k, v in arrs.items()}
    return out
