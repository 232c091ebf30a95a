"""ctypes binding of the tablebase-leaf oracle (tests/tb_search_oracle.cpp, TEST INFRASTRUCTURE): PUCT searches on the CPU oracle's
MctsArena that probe a table at their leaves, with one descent per simulation or in virtual-loss rounds, and the rule's reward of one
leaf. The table is probed through tests/tablebase_oracle.cpp's orc_tb_probe. The library is compiled on first use into the
temporary directory, keyed by the hash of its sources, so the repository tree is never written."""
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
SOURCES = [os.path.join(HERE, "tb_search_oracle.cpp"), os.path.join(HERE, "vl_oracle.cpp"), os.path.join(ROOT, "oracle", "onb_oracle.cpp")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_tb_search_oracle_%s.so" % h.hexdigest()[:16])
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
        L.orc_tbs_search_batch.argtypes = ([P, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_int, C.c_uint32, C.c_double, P, C.c_int, P, P]
                                           + [P] * 6 + [C.c_int64, P, C.c_int64])
        L.orc_tbs_reward.restype = C.c_double
        L.orc_tbs_reward.argtypes = [C.c_int16, C.c_int, C.c_int]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def reward(v, depth, leaf_color):
    """the reward a leaf of table value v (!= TB_NONE) backs up at `depth`, leaf_color the side to move at the leaf"""
    return float(lib().orc_tbs_reward(int(v), int(depth), int(leaf_color)))


def search(roots, c_puct, sims, cards, max_pawns, tables, leaves=1, vl=1.0, evaluator=0, dump_tree=-1, threads=None):
    """searches of every root with tablebase leaves; tables: {(p, q): int16 array} of the set `cards` (tablebase_oracle.solve or a
    copy of the device's). leaves >= 2: virtual-loss rounds of that many descents. Returns dict(best, pi [n,2,25], root_visits,
    root_q, child_visits [n,40], n_nodes) and, with dump_tree >= 0, 'tree': that tree's arena as orc_mcts_search dumps it."""
    s = np.ascontiguousarray(roots)
    assert s.dtype.itemsize == 24
    n = len(s)
    out = dict(best=np.zeros(n, np.uint16), pi=np.zeros((n, 2, 25), np.float32), root_visits=np.zeros(n, np.uint32), root_q=np.zeros(n, np.float64),
               child_visits=np.zeros((n, 40), np.uint32), n_nodes=np.zeros(n, np.int64))
    cap = 1 + 40 * max(sims, 1) + 2
    arrs = dict(visits=np.zeros(cap, np.uint32), reward=np.zeros(cap, np.float64), winrate=np.zeros(cap, np.float64), prior=np.zeros(cap, np.float64),
                action=np.zeros(cap, np.uint16), parent=np.zeros(cap, np.int32), first_child=np.zeros(cap, np.uint32), n_child=np.zeros(cap, np.uint32),
                flags=np.zeros(cap, np.uint8))
    td = TreeDump(*[_p(arrs[k]) for k, _ in TreeDump._fields_]) if dump_tree >= 0 else None
    ptrs = TBO._ptrs(tables)
    probe = C.cast(TBO.lib().orc_tb_probe, C.c_void_p)
    lib().orc_tbs_search_batch(_p(s), n, c_puct, sims, evaluator, threads or os.cpu_count() or 1, leaves, vl, _p(TBO._cards(cards)), max_pawns,
                               ptrs, probe, *[_p(out[k]) for k in ("best", "pi", "root_visits", "root_q", "child_visits", "n_nodes")],
                               dump_tree, C.byref(td) if td is not None else None, cap)
    if dump_tree >= 0:
        nn = int(out["n_nodes"][dump_tree])
        out["tree"] = {k: v[:nn].copy() for k, v in arrs.items()}
    return out
