"""ctypes binding of the MCTS-solver oracle (tests/solver_oracle.cpp, TEST INFRASTRUCTURE): PUCT searches on the CPU oracle's MctsArena
with the solver on or off, optionally with tablebase leaves probed through tests/tablebase_oracle.cpp's orc_tb_probe, and the
propagation rule on hand-built trees. The library is compiled on first use into the temporary directory, keyed by the hash of its
sources, so the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import tablebase_oracle as TBO
from oracle_lib import TreeDump

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "solver_oracle.cpp"), os.path.join(HERE, "tb_search_oracle.cpp"), os.path.join(HERE, "vl_oracle.cpp"),
           os.path.join(ROOT, "oracle", "onb_oracle.cpp")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]
WIN, LOSS = 8, 16

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_solver_oracle_%s.so" % h.hexdigest()[:16])
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
        L.orc_sol_search_batch.argtypes = ([P, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int, P, P]
                                           + [P] * 7 + [C.c_int64, P, C.c_int64])
        L.orc_sol_propagate.argtypes = [C.c_int64, P, P, P, P, C.c_uint32]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def search(roots, c_puct, sims, solver=True, evaluator=0, table=None, dump_tree=-1, threads=None):
    """searches of every root; table: None, or (cards, max_pawns, {(p, q): int16 array}) for tablebase leaves. Returns dict(best,
    pi [n,2,25], root_visits, root_q, child_visits [n,40], n_nodes, proof [n] int8) and, with dump_tree >= 0, 'tree': that tree's
    arena with the proof bits in its flags."""
    s = np.ascontiguousarray(roots)
    assert s.dtype.itemsize == 24
    n = len(s)
    out = dict(best=np.zeros(n, np.uint16), pi=np.zeros((n, 2, 25), np.float32), root_visits=np.zeros(n, np.uint32), root_q=np.zeros(n, np.float64),
               child_visits=np.zeros((n, 40), np.uint32), n_nodes=np.zeros(n, np.int64), proof=np.zeros(n, np.int8))
    cap = 1 + 40 * max(sims, 1) + 2
    arrs = dict(visits=np.zeros(cap, np.uint32), reward=np.zeros(cap, np.float64), winrate=np.zeros(cap, np.float64), prior=np.zeros(cap, np.float64),
                action=np.zeros(cap, np.uint16), parent=np.zeros(cap, np.int32), first_child=np.zeros(cap, np.uint32), n_child=np.zeros(cap, np.uint32),
                flags=np.zeros(cap, np.uint8))
    td = TreeDump(*[_p(arrs[k]) for k, _ in TreeDump._fields_]) if dump_tree >= 0 else None
    if table is not None:
        cards, max_pawns, tables = table
        keep = (TBO._cards(cards), TBO._ptrs(tables))
        cards_p, ptrs, probe = _p(keep[0]), keep[1], C.cast(TBO.lib().orc_tb_probe, C.c_void_p)
    else:
        max_pawns, cards_p, ptrs, probe = 0, None, None, None
    lib().orc_sol_search_batch(_p(s), n, c_puct, sims, evaluator, threads or os.cpu_count() or 1, int(bool(solver)), int(table is not None), cards_p,
                               max_pawns, ptrs, probe, *[_p(out[k]) for k in ("best", "pi", "root_visits", "root_q", "child_visits", "n_nodes", "proof")],
                               dump_tree, C.byref(td) if td is not None else None, cap)
    if dump_tree >= 0:
        nn = int(out["n_nodes"][dump_tree])
        out["tree"] = {k: v[:nn].copy() for k, v in arrs.items()}
    return out


def propagate(parent, first_child, n_child, proof, x):
    """the propagation rule on a hand-built tree from node x (proof[x] already set); returns the updated proof array"""
    par = np.ascontiguousarray(parent, np.int32)
    fc = np.ascontiguousarray(first_child, np.uint32)
    nc = np.ascontiguousarray(n_child, np.uint32)
    pr = np.array(proof, np.uint8)
    lib().orc_sol_propagate(len(par), _p(par), _p(fc), _p(nc), _p(pr), int(x))
    return pr
