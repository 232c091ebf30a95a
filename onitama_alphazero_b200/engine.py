"""Thin Python host layer over the C ABI (include/onb.h). One `Context` per GPU; every method is a direct call
into libonb.so. numpy is used for host staging only; device buffers can be wrapped zero-copy as torch tensors
(`Context.tensor`) so a torch module can read the leaf planes and write policy/value in place."""
import ctypes as C

import numpy as np

from . import _lib as L
from ._lib import STATE_DTYPE, OnbError


class _DevBuf:
    """Minimal __cuda_array_interface__ carrier so torch.as_tensor() wraps a borrowed device pointer without a copy."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3,
                                         "strides": None}


class Context:
    """Owns one onb_ctx (all device memory of `n_games` games / search trees on one GPU and one stream)."""

    def __init__(self, n_games, seed=0, device=0, game_id_base=0, stream=0, mcts_max_sims=0, mcts_node_cap=0, planes=True):
        self._lib = L.load()
        cfg = L.Config(device=device, flags=0, n_games=n_games, game_id_base=game_id_base, seed=seed, stream=stream or None,
                       mcts_max_sims=mcts_max_sims, mcts_node_cap=mcts_node_cap, alloc_planes=1 if planes else 0, reserved=0)
        h = C.c_void_p()
        rc = self._lib.onb_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise OnbError(rc, self._lib.onb_last_error(None).decode())
        self._h = h
        self.n = int(n_games)
        self.device = device
        self.seed = seed
        self.game_id_base = game_id_base
        self.mcts_max_sims = mcts_max_sims
        self.tb_leaves = False  # the tablebase-leaf switch (set_tablebase)
        self.solver = False     # the MCTS solver switch (set_solver)
        self._tb_serial = 0     # raised by every tb_solve / tb_free: the table a captured search round was given

    # ------------------------------------------------------------------ plumbing
    def _ck(self, rc):
        if rc != 0:
            raise OnbError(rc, self._lib.onb_last_error(self._h).decode())

    def close(self):
        self.__dict__.pop("_graphs", None)   # captured simulation rounds reference this context's buffers
        if getattr(self, "_h", None):
            self._lib.onb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def sync(self):
        self._ck(self._lib.onb_sync(self._h))

    def stream_handle(self):
        p = C.c_void_p()
        self._ck(self._lib.onb_get_stream(self._h, C.byref(p)))
        return p.value or 0

    def torch_stream(self):
        """The context's CUDA stream as a torch stream: run torch ops that touch its buffers under
        `with torch.cuda.stream(ctx.torch_stream())` so they are ordered with the kernels."""
        import torch
        if getattr(self, "_tstream", None) is None:
            self._tstream = torch.cuda.ExternalStream(self.stream_handle(), device="cuda:%d" % self.device)
        return self._tstream

    def buffer(self, which):
        p, b = C.c_void_p(), C.c_int64()
        self._ck(self._lib.onb_buffer(self._h, which, C.byref(p), C.byref(b)))
        return p.value, b.value

    def tensor(self, which):
        """Zero-copy torch view of a device buffer (the network reads LEAF_PLANES and writes POLICY / VALUE in place)."""
        import torch
        p, nbytes = self.buffer(which)
        n = self.n
        if which in (L.BUF_VL_PLANES, L.BUF_VL_POLICY, L.BUF_VL_VALUE):  # every allocated row (a search with K uses the first n K)
            row = {L.BUF_VL_PLANES: (21, 5, 5), L.BUF_VL_POLICY: (2, 25), L.BUF_VL_VALUE: ()}[which]
            rows = nbytes // (4 * int(np.prod(row, dtype=np.int64)))
            return torch.as_tensor(_DevBuf(p, (rows,) + row, "<f4"), device="cuda:%d" % self.device)
        spec = {L.BUF_MASKS: ((n, 2), "<u4", torch.int32), L.BUF_PLANES: ((n, 21, 5, 5), "<f4", None),
                L.BUF_ACTIONS: ((n,), "<i2", None), L.BUF_LEAF_PLANES: ((n, 21, 5, 5), "<f4", None),
                L.BUF_POLICY: ((n, 2, 25), "<f4", None), L.BUF_VALUE: ((n,), "<f4", None), L.BUF_PI: ((n, 2, 25), "<f4", None),
                L.BUF_BEST: ((n,), "<i2", None), L.BUF_STATES: ((n, 4), "<i4", None), L.BUF_STATS: ((L.STAT_COUNT,), "<i8", None),
                L.BUF_ROOT_M: ((n,), "<f8", None), L.BUF_ROOT_PROOF: ((n,), "|i1", None)}[which]
        shape, typestr, _ = spec
        if typestr == "<u4":
            typestr = "<i4"
        return torch.as_tensor(_DevBuf(p, shape, typestr), device="cuda:%d" % self.device)

    # ------------------------------------------------------------------ env
    def reset(self, decks=None, epoch=0):
        """decks: None (deal from the RNG), one deck of 5 card ids, or [n,5]."""
        if decks is None:
            self._ck(self._lib.onb_env_reset(self._h, None, 0, epoch))
            return
        d = np.ascontiguousarray(decks, dtype=np.uint8).reshape(-1, 5)
        self._ck(self._lib.onb_env_reset(self._h, L.ptr(d), len(d), epoch))

    def reset_games(self, mask=None, epoch=0):
        """onb_env_reset_games: restart the games selected by mask (uint8/bool [n]); None restarts every finished game. Returns the count."""
        cnt = C.c_int64(0)
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        self._ck(self._lib.onb_env_reset_games(self._h, None if m is None else L.ptr(m), epoch, C.byref(cnt)))
        return int(cnt.value)

    def set_states(self, states, first=0):
        s = np.ascontiguousarray(states, dtype=STATE_DTYPE)
        self._ck(self._lib.onb_env_set_states(self._h, L.ptr(s), first, len(s)))

    def get_states(self, first=0, n=None):
        n = self.n - first if n is None else n
        out = np.zeros(n, dtype=STATE_DTYPE)
        self._ck(self._lib.onb_env_get_states(self._h, L.ptr(out), first, n))
        return out

    def legal_moves(self):
        moves = np.zeros((self.n, 40), dtype=np.uint16)
        counts = np.zeros(self.n, dtype=np.uint8)
        self._ck(self._lib.onb_env_legal_moves(self._h, L.ptr(moves), L.ptr(counts)))
        return moves, counts

    def legal_masks(self, to_host=True):
        out = np.zeros((self.n, 2), dtype=np.uint32) if to_host else None
        self._ck(self._lib.onb_env_legal_masks(self._h, L.ptr(out)))
        return out

    def encode(self, to_host=True):
        out = np.zeros((self.n, 21, 5, 5), dtype=np.float32) if to_host else None
        self._ck(self._lib.onb_env_encode(self._h, L.ptr(out)))
        return out

    def step(self, actions=None, out_flags=0, step=0, auto_reset=False):
        a = None if actions is None else np.ascontiguousarray(actions, dtype=np.uint16)
        self._ck(self._lib.onb_env_step(self._h, L.ptr(a), step, int(auto_reset), out_flags))

    def step_from_host_ptr(self, host_ptr, step=0, auto_reset=False, out_flags=0):
        """onb_env_step with a raw host pointer (e.g. pinned memory owned by the caller)."""
        self._ck(self._lib.onb_env_step(self._h, C.c_void_p(host_ptr), step, int(auto_reset), out_flags))

    def step_random(self, step, policy=L.POLICY_UNIFORM, auto_reset=False, out_flags=0):
        self._ck(self._lib.onb_env_step_random(self._h, step, policy, int(auto_reset), out_flags))

    def choose_random(self, step, policy=L.POLICY_UNIFORM):
        self._ck(self._lib.onb_env_choose_random(self._h, step, policy))

    def run_random(self, step0, n_steps, policy=L.POLICY_UNIFORM, auto_reset=False, out_flags=0):
        self._ck(self._lib.onb_env_run_random(self._h, step0, n_steps, policy, int(auto_reset), out_flags))

    def playout(self, step0=0, max_plies=1 << 30, policy=L.POLICY_UNIFORM, want_plies=True, want_trace=True):
        plies = np.zeros(self.n, dtype=np.uint32) if want_plies else None
        trace = np.zeros(self.n, dtype=np.uint64) if want_trace else None
        self._ck(self._lib.onb_env_playout(self._h, step0, min(max_plies, 0xFFFFFFFF), policy, L.ptr(plies), L.ptr(trace)))
        return plies, trace

    def stats(self, clear=False):
        out = np.zeros(L.STAT_COUNT, dtype=np.uint64)
        self._ck(self._lib.onb_env_stats(self._h, L.ptr(out), int(clear)))
        return out

    def read(self, which, dtype, shape):
        """Copy a device buffer to the host (test helper; uses torch for the D2H copy)."""
        import torch
        with torch.cuda.stream(self.torch_stream()):
            return self.tensor(which).cpu().numpy().view(dtype).reshape(shape)

    def write(self, which, array):
        """onb_write_buffer: host array -> device buffer (the whole buffer or a prefix of it)"""
        a = np.ascontiguousarray(array)
        self._ck(self._lib.onb_write_buffer(self._h, which, L.ptr(a), a.nbytes))

    # ------------------------------------------------------------------ perft
    def perft(self, roots, depth):
        r = np.ascontiguousarray(roots, dtype=STATE_DTYPE)
        nodes = np.zeros((len(r), depth), dtype=np.uint64)
        wins = np.zeros((len(r), depth), dtype=np.uint64)
        zero = np.zeros((len(r), depth), dtype=np.uint64)
        self._ck(self._lib.onb_perft(self._h, L.ptr(r), len(r), depth, L.ptr(nodes), L.ptr(wins), L.ptr(zero)))
        return nodes, wins, zero

    # ------------------------------------------------------------------ mcts
    def mcts_begin(self, c_puct, sims):
        self._ck(self._lib.onb_mcts_begin(self._h, float(c_puct), sims))
        if getattr(self, "gumbel", None) is not None:
            self.gumbel_step += 1  # the library's serial: the step of the next Gumbel search

    def mcts_set_noise(self, enabled, epsilon=0.25, alpha=0.03, seed=0):
        """train mode: root exploration noise (AlphaZeroMctsConfig::train); statistical parity only."""
        self._ck(self._lib.onb_mcts_set_noise(self._h, int(bool(enabled)), float(epsilon), float(alpha), int(seed)))
        # the select kernel's launch parameters include the noise settings: a captured simulation round is only valid for them
        self._noise = (bool(enabled), float(epsilon), float(alpha), int(seed)) if enabled else (False,)

    def set_reuse(self, enabled):
        """onb_mcts_set_reuse: keep the played child's subtree between moves (mcts_begin, self_play_native). `sims` then counts root
        visits, kept ones included; switching off forgets the remembered trees. See include/onb.h."""
        self._ck(self._lib.onb_mcts_set_reuse(self._h, int(bool(enabled))))
        self.reuse = bool(enabled)

    def reuse_stats(self, clear=False):
        """onb_mcts_reuse_stats: dict(trees, kept, kept_visits, sims) summed over the reuse-enabled searches since the last clear"""
        out = np.zeros(4, np.uint64)
        self._ck(self._lib.onb_mcts_reuse_stats(self._h, L.ptr(out), int(bool(clear))))
        return dict(trees=int(out[0]), kept=int(out[1]), kept_visits=int(out[2]), sims=int(out[3]))

    def set_gumbel(self, enabled, m=16, c_visit=50.0, c_scale=0.1, gumbel_scale=1.0, seed=0, step0=0, interior=False):
        """onb_mcts_set_gumbel: the Gumbel root search (sequential halving over m Gumbel-Top-k samples at the root, improved-policy
        targets in mcts_finish's pi). The step of the next search becomes step0; every search begun afterwards takes the next step.
        interior=True: Gumbel MuZero's interior selection below the root instead of PUCT. See include/onb.h and DESIGN.md §5f."""
        cfg = L.GumbelConfig(int(bool(enabled)), int(m), float(c_visit), float(c_scale), float(gumbel_scale), int(seed), int(step0),
                             int(bool(interior)))
        self._ck(self._lib.onb_mcts_set_gumbel(self._h, C.byref(cfg)))
        # interior appends a sixth entry, so that a root-only setting keeps its five-entry tuple
        self.gumbel = (int(m), float(c_visit), float(c_scale), float(gumbel_scale), int(seed)) + ((True,) if interior else ()) if enabled else None
        self.gumbel_step = int(step0)  # self_play_native and fight_native leave the library's serial as they found it

    def set_virtual_loss(self, leaves, virtual_loss=1.0):
        """onb_mcts_set_virtual_loss: leaf parallelism with virtual loss for the searches begun afterwards -- rounds of `leaves` (K, 2 ..
        32) descents per tree, each pending descent counting as a lost visit of `virtual_loss` for the next; leaves <= 1 switches it
        off. See include/onb.h and DESIGN.md §5h."""
        self._ck(self._lib.onb_mcts_set_virtual_loss(self._h, int(leaves), float(virtual_loss)))
        self.vl = (int(leaves), float(virtual_loss)) if leaves > 1 else None

    def set_tablebase(self, enabled):
        """onb_mcts_set_tablebase: tablebase leaves for the searches begun afterwards -- a leaf below the root whose position the
        resident table holds is not expanded and backs up the table's exact value (needs tb_solve first; tb_free and tb_solve switch it
        off). See include/onb.h and DESIGN.md §5i."""
        self._ck(self._lib.onb_mcts_set_tablebase(self._h, int(bool(enabled))))
        self.tb_leaves = bool(enabled)

    def set_solver(self, enabled):
        """onb_mcts_set_solver: the MCTS solver for the searches begun afterwards -- immediate wins are marked at expansion, proofs
        (ONB_NODE_WIN / ONB_NODE_LOSS in the tree dump) are propagated to the root, descents stop at proven nodes and skip children
        proven lost, and mcts_finish plays a proven win. See include/onb.h and DESIGN.md §5k."""
        self._ck(self._lib.onb_mcts_set_solver(self._h, int(bool(enabled))))
        self.solver = bool(enabled)

    def _use_solver(self, solver):
        """the solver= argument of the search drivers: None leaves the solver switch, True / False sets it"""
        if solver is not None and bool(solver) != self.solver:
            self.set_solver(solver)

    def root_proof(self):
        """ONB_BUF_ROOT_PROOF after mcts_finish of a solver search: int8 [n], +1 the side to move wins with best play, -1 it loses,
        0 unproven (game order)"""
        return self.read(L.BUF_ROOT_PROOF, np.int8, (self.n,))

    def _use_tb(self, tb):
        """the tb= argument of the search drivers: None leaves the tablebase-leaf switch, True / False sets it"""
        if tb is not None and bool(tb) != self.tb_leaves:
            self.set_tablebase(tb)

    def _tb_graph_key(self):
        """what a captured round with tablebase leaves bakes in: the table the expand/backup launch was given"""
        return self._tb_serial if self.tb_leaves else None

    def _use_vl(self, vl):
        """the vl= argument of the search drivers: None leaves the switch, K (virtual loss 1) or (K, virtual_loss) sets it, K <= 1 or
        False switches it off"""
        if vl is None:
            return
        k, loss = (vl, 1.0) if not isinstance(vl, (tuple, list)) else vl
        want = (int(k), float(loss)) if int(k) > 1 else None
        if want != getattr(self, "vl", None):
            self.set_virtual_loss(int(k), float(loss))

    def _vl_rows(self):
        """zero-copy views (planes, policy, value) of the n K rows of the switch as it is; None without virtual loss"""
        k = getattr(self, "vl", None)
        if k is None:
            return None
        rows = self.n * k[0]
        return self.tensor(L.BUF_VL_PLANES)[:rows], self.tensor(L.BUF_VL_POLICY)[:rows], self.tensor(L.BUF_VL_VALUE)[:rows]

    def vl_rounds(self, sims):
        """rounds of a search of `sims` simulations begun with the switch as it is: 1 + ceil((sims - 1) / K) with virtual loss"""
        k = getattr(self, "vl", None)
        if k is None or sims == 0:
            return sims
        return 1 + (sims - 1 + k[0] - 1) // k[0]

    def _use_gumbel(self, gumbel):
        """the gumbel= argument of the search drivers: None leaves the switch, False switches it off, True (the defaults) or a dict of
        set_gumbel keywords switches it on unless that setting is already on (so consecutive searches keep advancing the step)"""
        if gumbel is None:
            return
        if not gumbel:
            if getattr(self, "gumbel", None) is not None:
                self.set_gumbel(False)
            return
        kw = dict(gumbel) if isinstance(gumbel, dict) else {}
        want = (int(kw.get("m", 16)), float(kw.get("c_visit", 50.0)), float(kw.get("c_scale", 0.1)), float(kw.get("gumbel_scale", 1.0)),
                int(kw.get("seed", 0))) + ((True,) if kw.get("interior", False) else ())
        if getattr(self, "gumbel", None) != want or "step0" in kw:
            self.set_gumbel(True, **kw)

    def set_selfplay_protocol(self, protocol):
        """onb_self_play_set_protocol: AlphaZero's self-play move protocol for the onb_self_play runs started afterwards. protocol: None /
        False / {} switches it off, else a dict with the keys of selfplay_protocol() -- temp_plies (T: the first T plies of a game
        sample their move in proportion to N^(1/temperature)), temperature, resign (the side to move resigns when max(v_root, q_best) <
        resign_below), resign_below, resign_holdout (fraction of games that never resign and are recorded for calibration) and seed.
        See include/onb.h and DESIGN.md §5j."""
        p = selfplay_protocol(**protocol) if protocol else None
        cfg = L.SelfPlayProtocol(p["temp_plies"], int(p["resign"]), p["temperature"], p["resign_below"], p["resign_holdout"], p["seed"]) if p else None
        self._ck(self._lib.onb_self_play_set_protocol(self._h, C.byref(cfg) if p else None))
        self.selfplay_protocol = p

    def selfplay_protocol_stats(self):
        """onb_self_play_protocol_stats after self_play_native: dict(resigned, held_out=dict(serial, result, min_m)) with torch copies of
        the held-out records (result 0 draw, 1 Red, 2 Blue; min_m [G, 2] over Red's and Blue's searches)"""
        import torch
        st = L.SelfPlayProtocolStats()
        self._ck(self._lib.onb_self_play_protocol_stats(self._h, C.byref(st)))
        g, dev = int(st.held_out), "cuda:%d" % self.device
        with torch.cuda.stream(self.torch_stream()):
            if g == 0:
                rec = dict(serial=torch.zeros(0, dtype=torch.int64, device=dev), result=torch.zeros(0, dtype=torch.uint8, device=dev),
                           min_m=torch.zeros((0, 2), dtype=torch.float64, device=dev))
            else:
                rec = dict(serial=torch.as_tensor(_DevBuf(st.serial, (g,), "<i8"), device=dev).clone(),
                           result=torch.as_tensor(_DevBuf(st.result, (g,), "|u1"), device=dev).clone(),
                           min_m=torch.as_tensor(_DevBuf(st.min_m, (g, 2), "<f8"), device=dev).clone())
        return dict(resigned=int(st.resigned), held_out=rec)

    def mcts_choose(self, seed, step, temperature=1.0, sample_mask=None):
        """onb_mcts_choose after mcts_finish: the self-play protocol's move of every searched game into BUF_ACTIONS and m = max(v_root,
        q_best) into BUF_ROOT_M; games with sample_mask[i] != 0 sample at `temperature` (draw onb_rand_u32(seed, game_id_base + i,
        step, 0x20000)), the others play best"""
        m = None if sample_mask is None else np.ascontiguousarray(sample_mask, dtype=np.uint8).reshape(self.n)
        self._ck(self._lib.onb_mcts_choose(self._h, int(seed), int(step), float(temperature), L.ptr(m)))

    def mcts_select(self):
        self._ck(self._lib.onb_mcts_select(self._h))

    def mcts_eval(self, evaluator):
        self._ck(self._lib.onb_mcts_eval(self._h, evaluator))

    def mcts_expand_backup(self):
        self._ck(self._lib.onb_mcts_expand_backup(self._h))

    def mcts_run(self, evaluator, sims):
        self._ck(self._lib.onb_mcts_run(self._h, evaluator, sims))

    def self_play_native(self, c_puct, sims, n_games, max_plies=150, evaluator=L.EVAL_UNIFORM, train=False, noise_seed=0, sample_cap=None,
                         reuse=None, gumbel=None, protocol=None):
        """onb_self_play: the whole self-play loop inside the library (search, recording, moves, z, restart of finished slots).
        Returns torch tensors of the completed games' samples (gathered from the context's device buffers) like
        selfplay.self_play_continuous. reuse: True / False sets the tree-reuse switch first (set_reuse), None leaves it. gumbel: as for
        search_device (the Gumbel step of ply p is p; pi is then the improved policy). protocol: None leaves the self-play protocol as
        it is, False switches it off, a dict sets it (set_selfplay_protocol); with it on the result also has `resigned` and `held_out`
        (selfplay_protocol_stats)."""
        import torch
        if reuse is not None:
            self.set_reuse(reuse)
        self._use_gumbel(gumbel)
        if protocol is not None:
            self.set_selfplay_protocol(protocol)
        if sample_cap is None:
            sample_cap = self.n * (max_plies + 2) * max(2, 2 * (n_games + self.n - 1) // self.n)
        cfg = L.SelfPlayConfig(c_puct, sims, evaluator, n_games, max_plies, int(bool(train)), noise_seed, sample_cap)
        res = L.SelfPlayResult()
        self._ck(self._lib.onb_self_play(self._h, C.byref(cfg), C.byref(res)))
        with torch.cuda.stream(self.torch_stream()):
            m = int(res.n_samples)

            def view(ptr, shape, typestr, dtype):
                if m == 0 or not ptr:
                    return torch.zeros(shape, dtype=dtype, device="cuda:%d" % self.device)
                return torch.as_tensor(_DevBuf(ptr, shape, typestr), device="cuda:%d" % self.device)

            idx = view(res.valid_idx, (int(res.n_valid),), "<i8", torch.int64)
            out = dict(planes=view(res.planes, (m, 21, 5, 5), "<f4", torch.float32)[idx], pi=view(res.pi, (m, 2, 25), "<f4", torch.float32)[idx],
                       z=view(res.z, (m,), "<f4", torch.float32)[idx], color=view(res.color, (m,), "|u1", torch.uint8)[idx].to(torch.int8),
                       serial=view(res.serial, (m,), "<i8", torch.int64)[idx], games=int(res.n_games), plies_run=int(res.plies_run),
                       truncated=bool(res.truncated))
        if getattr(self, "selfplay_protocol", None):
            out.update(self.selfplay_protocol_stats())
        return out

    @staticmethod
    def agent_random():
        return L.Agent(L.AGENT_RANDOM, 0, 0, 0, 0.0, 0, 0)

    @staticmethod
    def agent_puct(sims, c_puct=2.0, evaluator=L.EVAL_UNIFORM, net_slot=0, leaves=1, tablebase=False, solver=False):
        """AlphaZeroMcts as an arena agent; leaves > 1: ONB_AGENT_PUCT_VL, rounds of `leaves` descents with virtual loss 1;
        tablebase=True: ONB_AGENT_PUCT_TB, the table's move in the games of the resident table and a search with tablebase leaves in
        the others (no agent kind combines it with leaves > 1); solver=True: ONB_AGENT_PUCT_SOLVER, a search with the MCTS solver
        playing its best move (no agent kind combines it with leaves > 1 or tablebase=True)"""
        if tablebase and leaves > 1:
            raise ValueError("agent_puct: tablebase=True does not combine with leaves > 1 (no agent kind covers both)")
        if solver and (leaves > 1 or tablebase):
            raise ValueError("agent_puct: solver=True does not combine with leaves > 1 or tablebase=True (no agent kind covers both)")
        if solver:
            return L.Agent(L.AGENT_PUCT_SOLVER, evaluator, net_slot, sims, c_puct, 0, 0)
        if tablebase:
            return L.Agent(L.AGENT_PUCT_TB, evaluator, net_slot, sims, c_puct, 0, 0)
        if leaves > 1:
            return L.Agent(L.AGENT_PUCT_VL, evaluator, net_slot, sims, c_puct, int(leaves), 0)
        return L.Agent(L.AGENT_PUCT, evaluator, net_slot, sims, c_puct, 0, 0)

    @staticmethod
    def agent_uct(playouts, exploration_c=2.0 ** 0.5, min_node_visits=5):
        return L.Agent(L.AGENT_UCT, 0, 0, playouts, exploration_c, min_node_visits, 0)

    @staticmethod
    def agent_gumbel(sims, m=16, c_scale=0.1, evaluator=L.EVAL_UNIFORM, net_slot=0, interior=False):
        """the Gumbel root search as an arena agent (c_visit 50, gumbel_scale 1, seed = the context's seed, step = ply);
        interior=True: Gumbel MuZero (ONB_AGENT_GUMBEL_MUZERO, interior selection below the root)"""
        return L.Agent(L.AGENT_GUMBEL_MUZERO if interior else L.AGENT_GUMBEL, evaluator, net_slot, sims, c_scale, m, 0)

    @staticmethod
    def agent_alphabeta(depth):
        """the `AlphaBeta` agent: fixed-depth alpha-beta search to `depth` plies (1 .. 8), see Context.alphabeta"""
        return L.Agent(L.AGENT_ALPHABETA, 0, 0, depth, 0.0, 0, 0)

    @staticmethod
    def agent_tablebase():
        """the perfect endgame agent: plays Context.tb_best in the games in which it is to move (needs a solved table that holds every
        undecided game)"""
        return L.Agent(L.AGENT_TABLEBASE, 0, 0, 0, 0.0, 0, 0)

    def fight_native(self, agent_a, agent_b, a_is_red, max_plies=150):
        """onb_fight: the arena loop inside the library. Returns (a_wins, b_wins, draws, per-game results [n] uint8)."""
        mask = np.ascontiguousarray(np.asarray(a_is_red), dtype=np.uint8)
        res = L.FightResult()
        results = np.zeros(self.n, dtype=np.uint8)
        self._ck(self._lib.onb_fight(self._h, C.byref(agent_a), C.byref(agent_b), L.ptr(mask), max_plies, C.byref(res), L.ptr(results)))
        self.last_fight_results = results
        self.last_fight_moves_chosen = int(res.moves_chosen)
        self.last_fight_plies = int(res.plies_run)
        return int(res.a_wins), int(res.b_wins), int(res.draws), results

    def fight_stats(self, rating_a=800.0, rating_b=800.0, history=False):
        """onb_fight_stats: FightStatistics of the last fight_native (W/L/D overall and per colour of agent A, win rates, sequential Elo
        updates), folded on the device in game order. Returns a dict; history=True adds the [n, 4] rating changes
        (before_a, after_a, before_b, after_b)."""
        st = L.FightStats()
        hist = np.zeros((self.n, 4), dtype=np.float64) if history else None
        self._ck(self._lib.onb_fight_stats(self._h, float(rating_a), float(rating_b), C.byref(st), L.ptr(hist)))
        out = dict(n_games=int(st.n_games), general=dict(wins=int(st.wins), loses=int(st.loses), draws=int(st.draws)),
                   color=[dict(wins=int(st.color_wins[k]), loses=int(st.color_loses[k]), draws=int(st.color_draws[k])) for k in range(2)],
                   winrate=float(st.winrate), color_winrate=[float(st.color_winrate[0]), float(st.color_winrate[1])],
                   rating_a=float(st.rating_a), rating_b=float(st.rating_b))
        if history:
            out["rating_change_history"] = hist
        return out

    def uct_search(self, exploration_c=2.0 ** 0.5, min_node_visits=5, playouts=5000, to_host=True):
        """The reference's `Mcts` agent for every game at once: plain UCT with random rollouts (ai/mcts/mcts_arena.rs)."""
        self.mcts_begin(0.0, playouts)
        self._ck(self._lib.onb_uct_run(self._h, exploration_c, min_node_visits, playouts))
        return self.mcts_finish(to_host=to_host)

    def alphabeta(self, depth, to_host=True):
        """onb_alphabeta_run: a fixed-depth alpha-beta search (negamax, fail-hard; DESIGN.md §5d) from every game's current position,
        one game per GPU thread. The chosen actions stay in BUF_ACTIONS (ACTION_NONE for decided games), so step(None) plays them.
        Returns dict(best [n] uint16, score [n] int32 from the side to move's view, nodes [n] uint64 positions entered), or None
        with to_host=False."""
        if not to_host:
            self._ck(self._lib.onb_alphabeta_run(self._h, depth, None, None, None))
            return None
        out = dict(best=np.zeros(self.n, np.uint16), score=np.zeros(self.n, np.int32), nodes=np.zeros(self.n, np.uint64))
        self._ck(self._lib.onb_alphabeta_run(self._h, depth, L.ptr(out["best"]), L.ptr(out["score"]), L.ptr(out["nodes"])))
        return out

    # ------------------------------------------------------------------ endgame tablebase (DESIGN.md §5g)
    def tb_solve(self, cards, max_pawns=3):
        """onb_tb_solve: solves every class with p + q <= max_pawns of the five-card set `cards` on the device; the table stays in the
        context. Returns {(p, q): dict(entries, wins, losses, draws, invalid, max_win, max_loss, iterations, examined)}."""
        c = np.ascontiguousarray(cards, dtype=np.uint8).reshape(5)
        out = (L.TbClass * 25)()
        self.tb_leaves = False  # the solve switches tablebase leaves off, whether it succeeds or not
        self._tb_serial += 1
        self._ck(self._lib.onb_tb_solve(self._h, L.ptr(c), int(max_pawns), out))
        return {(k // 5, k % 5): {f: int(getattr(out[k], f)) for f, _ in L.TbClass._fields_ if f != "solved"}
                for k in range(25) if out[k].solved}

    def tb_free(self):
        self._ck(self._lib.onb_tb_free(self._h))
        self.tb_leaves = False
        self._tb_serial += 1

    def tb_table(self, p, q):
        """zero-copy torch int16 view of the solved class (p, q) on the device (valid until the next solve / tb_free)"""
        import torch
        ptr, n = C.c_void_p(), C.c_int64()
        self._ck(self._lib.onb_tb_table(self._h, int(p), int(q), C.byref(ptr), C.byref(n)))
        return torch.as_tensor(_DevBuf(ptr.value, (n.value,), "<i2"), device="cuda:%d" % self.device)

    def tb_probe(self):
        """onb_tb_probe: the game value of every game [n] np.int16 (TB_NONE outside the table)"""
        out = np.zeros(self.n, dtype=np.int16)
        self._ck(self._lib.onb_tb_probe(self._h, L.ptr(out)))
        return out

    def tb_best(self, to_host=True):
        """onb_tb_best: the table's move for every game (ACTION_NONE outside it); the moves also stay in BUF_ACTIONS"""
        out = np.zeros(self.n, dtype=np.uint16) if to_host else None
        self._ck(self._lib.onb_tb_best(self._h, L.ptr(out)))
        return out

    def mcts_finish(self, to_host=True, out=None):
        """out: optional dict of preallocated arrays (e.g. views of pinned memory) with the keys below; reused across calls."""
        if not to_host:
            self._ck(self._lib.onb_mcts_finish(self._h, None, None, None, None, None))
            return None
        n = self.n
        if out is None:
            out = dict(best=np.zeros(n, np.uint16), pi=np.zeros((n, 2, 25), np.float32), root_visits=np.zeros(n, np.uint32),
                       root_q=np.zeros(n, np.float64), child_visits=np.zeros((n, 40), np.uint32))
        self._ck(self._lib.onb_mcts_finish(self._h, L.ptr(out["best"]), L.ptr(out["pi"]), L.ptr(out["root_visits"]), L.ptr(out["root_q"]),
                                           L.ptr(out["child_visits"])))
        return out

    def mcts_play_best(self, out_flags=0):
        self._ck(self._lib.onb_mcts_play_best(self._h, out_flags))

    def net_select(self, slot):
        """onb_net_select: which of the two resident networks net_load fills and net_forward / EVAL_NET evaluate"""
        self._ck(self._lib.onb_net_select(self._h, slot))

    def net_load(self, params, tf32=False, precision=None):
        """onb_net_load: params = a torch module / state_dict / dict name -> array with the reference's VarStore names
        (net.rs:118-213; '.' or '|' separators). Folds BatchNorm, lays the weights out for the tensor cores, uploads them.
        precision: "f32" = f32-faithful split-operand arithmetic (ONB_NET_F32: |dp|, |dv| <= 1e-5 vs the reference's f32 CPU
        forward), "f16" (default) = the fast mode, operands rounded to f16's 11-bit significand, "tf32" = tf32 operands (cuDNN's
        default conv arithmetic); tf32=True is the older spelling of precision="tf32"."""
        mode = {"f16": L.NET_F16, "tf32": L.NET_TF32, "f32": L.NET_F32}[precision or ("tf32" if tf32 else "f16")]
        self._ck(self._lib.onb_net_precision(self._h, mode))
        if hasattr(params, "state_dict"):
            params = params.state_dict()
        names, arrays = [], []
        for k, v in params.items():
            if k.endswith("num_batches_tracked"):
                continue
            if hasattr(v, "detach"):
                v = v.detach().float().cpu().numpy()
            names.append(k.encode())
            arrays.append(np.ascontiguousarray(v, dtype=np.float32))
        n = len(names)
        c_names = (C.c_char_p * n)(*names)
        c_data = (C.c_void_p * n)(*[a.ctypes.data for a in arrays])
        c_numel = (C.c_int64 * n)(*[a.size for a in arrays])
        self._ck(self._lib.onb_net_load(self._h, n, c_names, c_data, c_numel))

    def net_forward(self, planes_buffer=L.BUF_LEAF_PLANES):
        """onb_net_forward: planes buffer -> ONB_BUF_POLICY / ONB_BUF_VALUE on the device (async on the context's stream)"""
        self._ck(self._lib.onb_net_forward(self._h, planes_buffer))

    def selftest(self, which=0):
        """onb_selftest: number of results that differ from the IEEE answer (0 on a correct build)"""
        bad = C.c_uint64(0)
        self._ck(self._lib.onb_selftest(self._h, which, C.byref(bad)))
        return int(bad.value)

    def mcts_tree_info(self):
        nn = np.zeros(self.n, np.uint32)
        fl = np.zeros(self.n, np.uint8)
        self._ck(self._lib.onb_mcts_tree_info(self._h, L.ptr(nn), L.ptr(fl)))
        return nn, fl

    def mcts_dump_tree(self, tree, cap=None):
        cap = cap or (1 + 40 * self.mcts_max_sims + 2)
        arrs = dict(visits=np.zeros(cap, np.uint32), reward=np.zeros(cap, np.float64), prior=np.zeros(cap, np.float64),
                    action=np.zeros(cap, np.uint16), parent=np.zeros(cap, np.int32), first_child=np.zeros(cap, np.uint32),
                    n_child=np.zeros(cap, np.uint32), flags=np.zeros(cap, np.uint8))
        td = L.TreeDump(*[L.ptr(arrs[k]) for k, _ in L.TreeDump._fields_])
        nn = C.c_int64()
        self._ck(self._lib.onb_mcts_dump_tree(self._h, tree, cap, C.byref(td), C.byref(nn)))
        return {k: v[:nn.value].copy() for k, v in arrs.items()}

    def search(self, c_puct, sims, evaluator=L.EVAL_UNIFORM, fused=True, net=None, vl=None, tb=None, solver=None):
        """MctsArena::search for every game at once. net: callable(leaf_planes tensor [n,21,5,5]) -> (policy [n,2,25], value [n])
        running on this context's stream; it reads/writes the device buffers zero-copy. vl: None leaves the virtual-loss switch, K or
        (K, virtual_loss) sets it, 1 switches it off (set_virtual_loss); with it on, `net` gets the n K rows of ONB_BUF_VL_PLANES and
        the split phase runs vl_rounds(sims) rounds. tb: None leaves the tablebase-leaf switch, True / False sets it (set_tablebase).
        solver: None leaves the MCTS solver switch, True / False sets it (set_solver); root_proof() reads the proofs afterwards."""
        self._use_vl(vl)
        self._use_tb(tb)
        self._use_solver(solver)
        self.mcts_begin(c_puct, sims)
        if net is None and fused:
            self.mcts_run(evaluator, sims)
        elif net is None:
            for _ in range(self.vl_rounds(sims)):
                self.mcts_select()
                self.mcts_eval(evaluator)
                self.mcts_expand_backup()
        else:
            import torch
            with torch.cuda.stream(self.torch_stream()):
                planes, pol, val = self._vl_rows() or (self.tensor(L.BUF_LEAF_PLANES), self.tensor(L.BUF_POLICY), self.tensor(L.BUF_VALUE))
                for _ in range(self.vl_rounds(sims)):
                    self.mcts_select()
                    p, v = net(planes)
                    pol.copy_(p.reshape(pol.shape))
                    val.copy_(v.reshape(val.shape))
                    self.mcts_expand_backup()
        return self.mcts_finish()


class Actor:
    """onb_actor_*: host-acted stepping of a context, pipelined over `n_sub` sub-batches inside the library (own streams, pinned host
    staging, one event per sub-batch). views[j] holds numpy views of the library's pinned buffers: actions [count] u16 (optional staging
    for the host's actions), masks [count, 2] u32, done [count/32, 2] u32 (bit j of [w, 0] / [w, 1]: game first+32w+j was won by Red / Blue
    in the step), stats [STAT_COUNT] u64 -- valid after wait(j)."""

    def __init__(self, ctx, n_sub=4, out_flags=0, host_flags=L.HOST_DONE):
        self.ctx, self._lib, self.n_sub = ctx, ctx._lib, n_sub
        h = C.c_void_p()
        ctx._ck(self._lib.onb_actor_create(ctx._h, n_sub, out_flags, host_flags, C.byref(h)))
        self._h = h
        self.views = []
        for j in range(n_sub):
            v = L.ActorView()
            ctx._ck(self._lib.onb_actor_get_view(self._h, j, C.byref(v)))
            cnt = int(v.count)

            def arr(ptr, ctype, shape, dtype):
                if not ptr or cnt == 0:
                    return None
                n = int(np.prod(shape))
                return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(n,)).view(dtype).reshape(shape)

            self.views.append(dict(first=int(v.first), count=cnt, actions=arr(v.actions, C.c_uint16, (cnt,), np.uint16),
                                   masks=arr(v.masks, C.c_uint32, (cnt, 2), np.uint32), done=arr(v.done, C.c_uint32, ((cnt + 31) // 32, 2), np.uint32),
                                   stats=arr(v.stats, C.c_uint64, (L.STAT_COUNT,), np.uint64)))

    def submit(self, sub, actions=None, step=0, auto_reset=False):
        """actions: None (the sub-batch's pinned staging, views[sub]['actions']), a raw host address (int), or a uint16 array of the
        sub-batch's `count` actions -- it must stay alive and untouched until wait(sub)."""
        if actions is None or isinstance(actions, int):
            p = C.c_void_p(actions) if actions else None
        else:
            assert actions.dtype == np.uint16 and actions.flags["C_CONTIGUOUS"] and actions.size == self.views[sub]["count"]
            p = L.ptr(actions)
        self.ctx._ck(self._lib.onb_actor_submit(self._h, sub, p, step, int(auto_reset)))

    def wait(self, sub):
        self.ctx._ck(self._lib.onb_actor_wait(self._h, sub))

    def join(self):
        self.ctx._ck(self._lib.onb_actor_join(self._h))

    def replay(self, trace, step0=0, auto_reset=False):
        """trace: uint16 [n_steps, stride >= n] array or (address, stride, n_steps) of pinned host memory"""
        if isinstance(trace, tuple):
            addr, stride, steps = trace
        else:
            assert trace.dtype == np.uint16 and trace.ndim == 2 and trace.flags["C_CONTIGUOUS"]
            addr, stride, steps = trace.ctypes.data, trace.shape[1], trace.shape[0]
        self.ctx._ck(self._lib.onb_actor_replay(self._h, C.c_void_p(addr), stride, step0, steps, int(auto_reset)))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.onb_actor_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _search_device(self, c_puct, sims, evaluator=L.EVAL_UNIFORM, net=None, use_graph=False, reuse=None, gumbel=None, vl=None, tb=None,
                   solver=None):
    """Context.search without copying the results to the host (PI / BEST stay in their device buffers).
    use_graph: capture one simulation round (select -> network -> expand/backup) in a CUDA graph on the context's stream and
    replay it; the round is launch-bound otherwise (~40 small network kernels per round).
    reuse: True / False sets the tree-reuse switch first (set_reuse), None leaves it. Reuse needs a device evaluator (a torch `net`
    drives the split phase, which a reuse search refuses).
    gumbel: None leaves the Gumbel switch as it is, False switches it off, True or a dict of set_gumbel keywords switches it on (only
    when that setting is not on already, so that consecutive searches take consecutive steps).
    vl: as for search. With virtual loss a torch `net` gets the n K rows, and use_graph runs round 0 eagerly and replays one captured
    round for the others: the kernels take a round's descents from the root's visit count, so the short last round replays too.
    tb: as for search. A captured round with tablebase leaves bakes in the table, so a new tb_solve captures anew.
    solver: as for search; a captured round bakes in the solver's kernels, so the switch is part of the graph key."""
    if reuse is not None and bool(reuse) != getattr(self, "reuse", False):
        self.set_reuse(reuse)
    self._use_gumbel(gumbel)
    self._use_vl(vl)
    self._use_tb(tb)
    self._use_solver(solver)
    if net is not None and getattr(self, "reuse", False):
        raise ValueError("search_device: tree reuse needs a device evaluator (EVAL_UNIFORM / EVAL_HASH / EVAL_NET), not a torch net")
    self.mcts_begin(c_puct, sims)
    if net is None:
        self.mcts_run(evaluator, sims)
    else:
        import torch
        ts = self.torch_stream()
        with torch.cuda.stream(ts):
            vl_rows = self._vl_rows()
            planes, pol, val = vl_rows or (self.tensor(L.BUF_LEAF_PLANES), self.tensor(L.BUF_POLICY), self.tensor(L.BUF_VALUE))
            rounds = self.vl_rounds(sims)

            def one_round():
                self.mcts_select()
                p, v = net(planes)
                pol.copy_(p.reshape(pol.shape))
                val.copy_(v.reshape(val.shape))
                self.mcts_expand_backup()

            if not use_graph or rounds < 3:
                for _ in range(rounds):
                    one_round()
            elif vl_rows is not None:
                # the captured round bakes in K, vl, the round target (the begin's sims) and the row buffers (reallocated by a larger K)
                key = (id(net), float(c_puct), self.vl, int(sims), self.buffer(L.BUF_VL_PLANES)[0], self._tb_graph_key())
                cache = self.__dict__.setdefault("_graphs", {})
                one_round()  # round 0 (one descent), eagerly: also the warm-up before a capture
                if key not in cache:
                    ts.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=ts):
                        one_round()  # captured, not executed
                    cache[key] = (g, net)
                g = cache[key][0]
                for _ in range(rounds - 1):
                    g.replay()
            else:
                # a captured round bakes in everything the launches were given: the evaluator, c_puct AND the root-noise settings
                # (ADVICE r01: switching train mode after a capture must not replay the old setting). The cache holds a strong
                # reference to `net`, so its id cannot be recycled for another module while the graph lives; close() drops it.
                key = (id(net), float(c_puct), getattr(self, "_noise", (False,)), getattr(self, "gumbel", None), self._tb_graph_key(), self.solver)
                cache = self.__dict__.setdefault("_graphs", {})
                done = 0
                if key not in cache:
                    one_round()  # eager warm-up round (lazy cuDNN/cuBLAS initialisation must not happen during capture)
                    done = 1
                    ts.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=ts):
                        one_round()  # captured, not executed
                    cache[key] = (g, net)
                g = cache[key][0]
                for _ in range(sims - done):
                    g.replay()
    self.mcts_finish(to_host=False)


Context.search_device = _search_device


def selfplay_protocol(temp_plies=0, temperature=1.0, resign=False, resign_below=-1.0, resign_holdout=0.1, seed=0):
    """the self-play protocol setting (onb_selfplay_protocol) as a dict with every key; see Context.set_selfplay_protocol"""
    return dict(temp_plies=int(temp_plies), temperature=float(temperature), resign=bool(resign), resign_below=float(resign_below),
                resign_holdout=float(resign_holdout), seed=int(seed))


def tb_index(cards, states):
    """onb_tb_index: (class id 5 p + q, entry) of each state for the card set `cards`; -1, -1 for states outside the classes"""
    c = np.ascontiguousarray(cards, dtype=np.uint8).reshape(5)
    s = np.ascontiguousarray(states, dtype=STATE_DTYPE).reshape(-1)
    cls, idx = np.zeros(len(s), np.int32), np.zeros(len(s), np.int64)
    rc = L.load().onb_tb_index(L.ptr(c), L.ptr(s), len(s), L.ptr(cls), L.ptr(idx))
    if rc != 0:
        raise OnbError(rc, "onb_tb_index: invalid card set")
    return cls, idx


def tb_states(cards, cls, idx):
    """onb_tb_state: the states of entries idx of class cls (hands in ascending card order, then the neutral card)"""
    c = np.ascontiguousarray(cards, dtype=np.uint8).reshape(5)
    i = np.ascontiguousarray(idx, dtype=np.int64).reshape(-1)
    out = np.zeros(len(i), dtype=STATE_DTYPE)
    rc = L.load().onb_tb_state(L.ptr(c), int(cls), L.ptr(i), len(i), L.ptr(out))
    if rc != 0:
        raise OnbError(rc, "onb_tb_state: invalid card set, class or entry")
    return out


def start_states(decks):
    d = np.ascontiguousarray(decks, dtype=np.uint8).reshape(-1, 5)
    out = np.zeros(len(d), dtype=STATE_DTYPE)
    rc = L.load().onb_start_states(L.ptr(d), len(d), L.ptr(out))
    if rc != 0:
        raise OnbError(rc, "onb_start_states: invalid deck")
    return out
