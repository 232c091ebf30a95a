"""ctypes binding of the tree-reuse oracle (tests/reuse_oracle.cpp, TEST INFRASTRUCTURE: the CPU restatement of
onb_mcts_set_reuse on top of the CPU oracle's MctsArena). The library is compiled on first use into the temporary directory, keyed
by the hash of its sources, so the repository tree is never written."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle_lib import EVAL_CB, TreeDump

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SOURCES = [os.path.join(HERE, "reuse_oracle.cpp"), os.path.join(ROOT, "oracle", "onb_oracle.cpp")]
CXXFLAGS = ["-O3", "-march=x86-64-v3", "-std=c++17", "-fPIC", "-shared", "-pthread", "-ffp-contract=off", "-fno-fast-math"]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    out = os.path.join(tempfile.gettempdir(), "onb_reuse_oracle_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(out):
        tmp = "%s.%d.tmp" % (out, os.getpid())
        subprocess.check_call([os.environ.get("CXX", "g++")] + CXXFLAGS + ["-o", tmp, SOURCES[0]])
        os.replace(tmp, out)  # atomic: concurrent builders never load a half-written library
    return out


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.orc_reuse_new.restype = C.c_void_p
        L.orc_reuse_new.argtypes = [C.c_int64]
        L.orc_reuse_free.argtypes = [C.c_void_p]
        L.orc_reuse_search.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 8
        L.orc_reuse_dump.restype = C.c_int64
        L.orc_reuse_dump.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
        L.orc_reuse_play_games.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_uint32, C.c_int, C.c_uint32, C.c_int, C.c_int] + [C.c_void_p] * 5
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class ReuseSet:
    """one remembered search tree per game, like a context's pools with reuse on"""

    def __init__(self, n):
        self.n = n
        self._h = lib().orc_reuse_new(n)

    def close(self):
        if self._h:
            lib().orc_reuse_free(self._h)
            self._h = None

    def __del__(self):
        self.close()

    def search(self, states, c_puct, sims, evaluator=0, callback=None, threads=None):
        """every game: keep the matching child's subtree (or start fresh), search to `sims` root visits. callback(planes[525]) ->
        (policy[50], value) replaces the evaluator (single-threaded)."""
        s = np.ascontiguousarray(states)
        assert len(s) == self.n and s.dtype.itemsize == 24
        n = self.n
        out = dict(best=np.zeros(n, np.uint16), pi=np.zeros((n, 2, 25), np.float32), root_visits=np.zeros(n, np.uint32),
                   root_q=np.zeros(n, np.float64), child_visits=np.zeros((n, 40), np.uint32), n_nodes=np.zeros(n, np.int64),
                   kept=np.zeros(n, np.int32), sims_run=np.zeros(n, np.uint32))
        cb = None
        if callback is not None:
            def _cb(planes_p, pol_p, val_p, _user):
                planes = np.ctypeslib.as_array(planes_p, shape=(525,)).copy()
                pol, val = callback(planes)
                np.ctypeslib.as_array(pol_p, shape=(50,))[:] = np.asarray(pol, dtype=np.float32).reshape(50)
                val_p[0] = float(val)
            cb = EVAL_CB(_cb)
            evaluator, threads = 2, 1
        lib().orc_reuse_search(self._h, _p(s), n, c_puct, sims, evaluator, C.cast(cb, C.c_void_p) if cb else None, None,
                               threads or os.cpu_count() or 1, *[_p(out[k]) for k in ("best", "pi", "root_visits", "root_q", "child_visits",
                                                                                       "n_nodes", "kept", "sims_run")])
        return out

    def dump(self, i, cap=None):
        """the tree of game i as orc_mcts_search dumps it (None: no tree)"""
        nn = lib().orc_reuse_dump(self._h, i, None, 0)
        if nn == 0:
            return None
        cap = cap or nn
        arrs = dict(visits=np.zeros(cap, np.uint32), reward=np.zeros(cap, np.float64), winrate=np.zeros(cap, np.float64),
                    prior=np.zeros(cap, np.float64), action=np.zeros(cap, np.uint16), parent=np.zeros(cap, np.int32),
                    first_child=np.zeros(cap, np.uint32), n_child=np.zeros(cap, np.uint32), flags=np.zeros(cap, np.uint8))
        td = TreeDump(*[_p(arrs[k]) for k, _ in TreeDump._fields_])
        lib().orc_reuse_dump(self._h, i, C.byref(td), cap)
        return {k: v[:nn].copy() for k, v in arrs.items()}


def filter_tree(tree, keep):
    """the arena-order filter in numpy: node `keep` and its descendants, renumbered in order (parent / first_child remapped, the new
    root without a parent, a node without children keeps first_child 0)"""
    n = len(tree["parent"])
    member = np.zeros(n, bool)
    member[keep] = True
    for i in range(keep + 1, n):
        p = tree["parent"][i]
        member[i] = p >= keep and member[p]
    idx = np.nonzero(member)[0]
    new = np.full(n, -1, np.int64)
    new[idx] = np.arange(len(idx))
    out = {k: v[idx].copy() for k, v in tree.items()}
    par = tree["parent"][idx]
    out["parent"] = np.where(idx == keep, -1, new[np.maximum(par, 0)]).astype(np.int32)
    fc = tree["first_child"][idx]
    out["first_child"] = np.where(out["n_child"] > 0, new[fc], fc).astype(np.uint32)
    return out


def play_games(starts, c_puct, sims, evaluator=0, max_plies=150, reuse=True, threads=None):
    """whole games with one search per ply (reuse on or off) and the best move played; dict(pi [n, max_plies + 2, 2, 25],
    color [n, max_plies + 2], plies [n], result [n], sims [n] simulations run)"""
    s = np.ascontiguousarray(starts)
    n, stride = len(s), max_plies + 2
    out = dict(pi=np.zeros((n, stride, 2, 25), np.float32), color=np.zeros((n, stride), np.uint8), plies=np.zeros(n, np.int32),
               result=np.zeros(n, np.uint8), sims=np.zeros(n, np.uint64))
    lib().orc_reuse_play_games(_p(s), n, c_puct, sims, evaluator, max_plies, int(bool(reuse)), threads or os.cpu_count() or 1,
                               *[_p(out[k]) for k in ("pi", "color", "plies", "result", "sims")])
    return out
