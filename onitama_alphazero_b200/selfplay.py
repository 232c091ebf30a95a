"""Lockstep batched self-play and arena loops on top of one Context (host glue; all game/search work is in libonb.so).

self_play  <- alphazero-training/src/train.rs:35-98   (per ply: search -> record (pi, planes, colour) -> play best -> flip;
              stop on a win or after max_plies+2 plies (check-then-decrement, Q15); z = reward(final, sample colour))
fight      <- alphazero-training/src/evaluator.rs:355-399 (two move sources alternate by side; W/L/D counted per colour)
"""
import numpy as np
import torch

from . import _lib as L


class EloRating:
    """elo_rating.rs:53-70 (K = 32, 1/400 scale)"""
    K = 32.0
    C_ELO = 2.5e-3

    @staticmethod
    def elo_change(ra, rb, is_a_win):
        ea = 1.0 / (1.0 + 10.0 ** (EloRating.C_ELO * (rb - ra)))
        eb = 1.0 / (1.0 + 10.0 ** (EloRating.C_ELO * (ra - rb)))
        sa = 1.0 if is_a_win else 0.0
        sb = 1.0 - sa
        return ra + EloRating.K * (sa - ea), rb + EloRating.K * (sb - eb)


class FightStatistics:
    """evaluator.rs:38-110: W/L/D in total and per colour of agent A, win rates, sequential Elo updates game by game."""

    def __init__(self, rating_a=800.0, rating_b=800.0):
        self.general = dict(wins=0, loses=0, draws=0)
        self.color = [dict(wins=0, loses=0, draws=0), dict(wins=0, loses=0, draws=0)]
        self.winrate = 0.0
        self.color_winrate = [0.0, 0.0]
        self.rating_a, self.rating_b = rating_a, rating_b
        self.rating_change_history = []

    def update(self, result, player_color):
        """result: 0 none/draw, 1 RedWin, 2 BlueWin; player_color: colour agent A played (0 Red, 1 Blue)"""
        before = (self.rating_a, self.rating_b)
        if result in (1, 2):
            a_won = (result - 1) == player_color
            self.rating_a, self.rating_b = EloRating.elo_change(self.rating_a, self.rating_b, a_won)
            key = "wins" if a_won else "loses"
        else:
            key = "draws"
        self.rating_change_history.append((before[0], self.rating_a, before[1], self.rating_b))
        self.general[key] += 1
        self.color[player_color][key] += 1
        tot = sum(self.general.values())
        self.winrate = self.general["wins"] / tot
        for c in (0, 1):
            t = sum(self.color[c].values())
            self.color_winrate[c] = self.color[c]["wins"] / t if t else float("nan")


def fight_statistics(results, a_is_red, rating_a=800.0, rating_b=800.0):
    """Fold the per-game results of a lockstep arena (game order = the reference's sequential order) into FightStatistics."""
    st = FightStatistics(rating_a, rating_b)
    for r, red in zip(results, a_is_red):
        st.update(int(r), 0 if red else 1)
    return st


def self_play(ctx, c_puct, sims, max_plies=150, evaluator=L.EVAL_UNIFORM, net=None, decks=None):
    with torch.cuda.stream(ctx.torch_stream()):  # torch ops ordered with the context's kernels
        return _self_play(ctx, c_puct, sims, max_plies, evaluator, net, decks)


def _self_play(ctx, c_puct, sims, max_plies, evaluator, net, decks):
    """Plays every game of `ctx` to the end with MCTS moves. Returns device tensors (planes [m,21,5,5], pi [m,2,25], z [m],
    colour [m], game [m]) for all recorded samples, in ply-major order."""
    ctx.reset(decks=decks)
    n = ctx.n
    dev = "cuda:%d" % ctx.device
    planes_buf, pi_buf, color_buf, game_buf = [], [], [], []
    plies_left = max_plies
    states_t = ctx.tensor(L.BUF_STATES)
    while True:
        st = states_t.clone()
        result = (st[:, 2] >> 29) & 3
        live = result == 0
        if not bool(live.any()):
            break
        ctx.encode(to_host=False)  # create_tensor_from_state of the position the search starts from (train.rs:58)
        planes = ctx.tensor(L.BUF_PLANES)
        ctx.search_device(c_puct, sims, evaluator=evaluator, net=net)
        pi = ctx.tensor(L.BUF_PI)
        idx = live.nonzero(as_tuple=True)[0]
        planes_buf.append(planes[idx].clone())
        pi_buf.append(pi[idx].clone())
        color_buf.append(((st[idx, 1] >> 30) & 1).to(torch.int8))
        game_buf.append(idx)
        ctx.mcts_play_best()
        if plies_left < 0:  # train.rs:74-79: checked AFTER the move, then decremented
            break
        plies_left -= 1
    final = states_t.clone()
    result = ((final[:, 2] >> 29) & 3)  # 0 none, 1 Red won, 2 Blue won
    planes = torch.cat(planes_buf) if planes_buf else torch.zeros((0, 21, 5, 5), device=dev)
    pi = torch.cat(pi_buf) if pi_buf else torch.zeros((0, 2, 25), device=dev)
    color = torch.cat(color_buf) if color_buf else torch.zeros((0,), dtype=torch.int8, device=dev)
    game = torch.cat(game_buf) if game_buf else torch.zeros((0,), dtype=torch.int64, device=dev)
    r = result[game]
    # reward(progress, s.player_color), alphazero_mcts/mod.rs:45-53
    z = torch.where(r == 0, 0.0, torch.where((r - 1) == color.to(r.dtype), 1.0, -1.0)).to(torch.float32)
    return dict(planes=planes, pi=pi, z=z, color=color, game=game)


def self_play_continuous(ctx, c_puct, sims, n_games, max_plies=150, evaluator=L.EVAL_UNIFORM, net=None, train=False, noise_seed=0, reuse=False,
                         gumbel=None, protocol=None):
    """self_play for at least n_games games with every slot of the context kept busy: a slot whose game ends (or hits the ply cap)
    is re-dealt at once (onb_env_reset_games), the way a worker thread of the reference starts its next game as soon as one is over
    (train.rs:218-245 around :44-98). Lockstep self_play instead searches finished slots until the longest game ends -- with game
    lengths between ~10 and 152 plies that wastes most of the work. Only completed games are returned; sample order is ply-major.
    Extra keys: `serial` [m] (slot + n * generation: samples with the same serial belong to one game), `games` (completed games).
    reuse=True keeps the played child's subtree between plies (Context.set_reuse; device evaluators only), as
    onb_self_play does with the switch on; the switch is left as it was.
    gumbel=True or a dict of Context.set_gumbel keywords: the Gumbel root search with step = ply (set_gumbel(step0=0) at the start, one
    search per ply), pi = its improved policy, as onb_self_play does with the switch on; the switch is left as it was.
    protocol: a dict of Context.set_selfplay_protocol keys -- the self-play move protocol as onb_self_play plays it with that setting
    (DESIGN.md §5j): Context.mcts_choose picks the moves and m, resignation and the held-out records are restated here. The result then
    also has `resigned`, `held_out` (dict(serial, result, min_m), as Context.selfplay_protocol_stats) and `m` (each sample's search's
    max(v_root, q_best)). The context's own protocol
    setting is not used and left as it was."""
    if reuse and net is not None:
        raise ValueError("self_play_continuous: reuse=True needs a device evaluator, not a torch net")
    from .engine import selfplay_protocol
    protocol = selfplay_protocol(**protocol) if protocol else None
    if protocol and protocol["temp_plies"] and gumbel:
        raise ValueError("self_play_continuous: the Gumbel root search plays its sequential-halving winner; temp_plies must be 0")
    was = getattr(ctx, "reuse", False)
    gb_was, step_was = getattr(ctx, "gumbel", None), getattr(ctx, "gumbel_step", 0)
    if reuse:
        ctx.set_reuse(False)   # forget trees of earlier searches: every game starts from a fresh tree
        ctx.set_reuse(True)
    if gumbel:
        ctx.set_gumbel(True, **dict(dict(gumbel) if isinstance(gumbel, dict) else {}, step0=0))
    try:
        return _self_play_continuous(ctx, c_puct, sims, n_games, max_plies, evaluator, net, train, noise_seed, bool(reuse), protocol)
    finally:
        if getattr(ctx, "reuse", False) != was:
            ctx.set_reuse(was)
        if gumbel:
            if gb_was is None:
                ctx.set_gumbel(False)
            else:
                m, c_visit, c_scale, scale, seed = gb_was[:5]
                ctx.set_gumbel(True, m, c_visit, c_scale, scale, seed, step0=step_was, interior=len(gb_was) > 5)  # the setting and its step as they were


def _held_out(ctx, protocol, slots, generation):
    """onb_rand_u32(seed, g, gen, 0x20001) < floor(h 2^32) for the games (slot, generation): the held-out games never resign"""
    lib, below = L.load(), int(np.floor(protocol["resign_holdout"] * 4294967296.0)) if protocol["resign"] else 0
    return [lib.onb_rand_u32(protocol["seed"], ctx.game_id_base + s, g, 0x20001) < below for s, g in zip(slots, generation)]


def _self_play_continuous(ctx, c_puct, sims, n_games, max_plies, evaluator, net, train, noise_seed, reuse, protocol):
    with torch.cuda.stream(ctx.torch_stream()):
        n = ctx.n
        dev = "cuda:%d" % ctx.device
        ctx.reset()
        ctx.mcts_set_noise(bool(train), 0.25, 0.03, noise_seed)
        states_t = ctx.tensor(L.BUF_STATES)
        generation = torch.zeros(n, dtype=torch.int64, device=dev)   # games already finished in this slot
        plies = torch.zeros(n, dtype=torch.int64, device=dev)        # plies played in the slot's current game
        slots = torch.arange(n, device=dev)
        rec = {"planes": [], "pi": [], "color": [], "serial": []}
        winners = {}   # serial -> 0 draw (ply cap), 1 Red, 2 Blue
        done, tick = 0, 0   # tick = plies played so far; a slot restarted after ply `tick` is dealt at epoch tick + 1 (as onb_self_play does)
        # exactly max(n_games, slots) games are started and ALL of them are played to the end (dropping the games still running when a
        # quota is reached would drop the long ones and bias z / pi): a finished slot starts its next game while games remain to be
        # started -- slots in ascending order, as onb_self_play does -- and goes idle afterwards
        target, started = max(int(n_games), n), n
        idle = torch.zeros(n, dtype=torch.bool, device=dev)
        acts_t, best_t = ctx.tensor(L.BUF_ACTIONS), ctx.tensor(L.BUF_BEST)
        rec["live"] = []
        if protocol:   # per slot: held out, min m over Red's / Blue's searches; the records of the completed held-out games
            held = torch.tensor(_held_out(ctx, protocol, range(n), [0] * n), dtype=torch.bool, device=dev)
            mmin = torch.full((n, 2), float("inf"), dtype=torch.float64, device=dev)
            records = {"serial": [], "result": [], "min_m": []}
            n_resigned = 0
            m_t = ctx.tensor(L.BUF_ROOT_M)
            rec["m"] = []
        while not bool(idle.all()):
            st = states_t.clone()
            ctx.encode(to_host=False)                       # create_tensor_from_state of the searched position (train.rs:58)
            ctx.search_device(c_puct, sims, evaluator=evaluator, net=net, reuse=reuse)   # (this driver searches idle slots too and ignores them)
            side = ((st[:, 1] >> 30) & 1).long()
            rec["planes"].append(ctx.tensor(L.BUF_PLANES).clone())
            rec["pi"].append(ctx.tensor(L.BUF_PI).clone())
            rec["color"].append(side.to(torch.int8))
            rec["serial"].append(slots + n * generation)
            rec["live"].append(~idle)
            resigned = torch.zeros(n, dtype=torch.bool, device=dev)
            if protocol:
                t_plies = protocol["temp_plies"]
                mask = ((~idle) & (plies < t_plies)).to(torch.uint8).cpu().numpy() if t_plies else None
                ctx.mcts_choose(protocol["seed"], tick, protocol["temperature"] if t_plies else 1.0, mask)   # the move into ACTIONS, m
                m = m_t.clone()
                rec["m"].append(m)
                live_ = ~idle
                cur = mmin[slots, side]
                mmin[slots, side] = torch.where(live_ & (m < cur), m, cur)
                if protocol["resign"]:
                    resigned = live_ & ~held & (m < protocol["resign_below"])
                    n_resigned += int(resigned.sum())
                    acts_t[resigned] = -1                    # a resigning side plays no move
            else:
                acts_t.copy_(best_t)
            acts_t[idle] = -1                                # ONB_ACTION_NONE: an idle slot (e.g. a game cut at the ply cap) is not stepped
            ctx.step(None)
            plies += (~idle).to(plies.dtype)
            result = (states_t.clone()[:, 2] >> 29) & 3
            result = torch.where(resigned, (side ^ 1) + 1, result.long())   # the side to move resigned: the opponent wins
            # train.rs:74-79: the cap is checked after the move with max_plies counting down from 150 -> a game has at most max_plies + 2 plies
            over = ~idle & (resigned | (result != 0) | (plies >= max_plies + 2))
            if bool(over.any()):
                idx = over.nonzero(as_tuple=True)[0]
                ser = (idx + n * generation[idx]).tolist()
                for s_, r_ in zip(ser, result[idx].tolist()):
                    winners[s_] = r_
                if protocol:
                    h = idx[held[idx]]
                    records["serial"].append(h + n * generation[h])
                    records["result"].append(result[h].to(torch.uint8))
                    records["min_m"].append(mmin[h].clone())
                done += len(ser)
                k = min(len(ser), target - started)
                again, stop = idx[:k], idx[k:]
                if k:
                    mask = torch.zeros(n, dtype=torch.uint8, device=dev)
                    mask[again] = 1
                    ctx.reset_games(mask.cpu().numpy(), epoch=tick + 1)
                    generation[again] += 1
                    started += k
                    if protocol:
                        held[again] = torch.tensor(_held_out(ctx, protocol, again.tolist(), generation[again].tolist()), dtype=torch.bool, device=dev)
                        mmin[again] = float("inf")
                idle[stop] = True
                plies[idx] = 0
            tick += 1
        live = torch.cat(rec["live"])
        planes = torch.cat(rec["planes"])
        pi = torch.cat(rec["pi"])
        color = torch.cat(rec["color"])
        serial = torch.cat(rec["serial"])
        table = torch.full((int(serial.max()) + 1,), -1, dtype=torch.int64, device=dev)
        keys = torch.tensor(list(winners.keys()), dtype=torch.int64, device=dev)
        table[keys] = torch.tensor(list(winners.values()), dtype=torch.int64, device=dev)
        r = table[serial]
        keep = (r >= 0) & live                                # every started game was completed; rows of idle slots are not samples
        r, color_k = r[keep], color[keep]
        z = torch.where(r == 0, 0.0, torch.where((r - 1) == color_k.to(r.dtype), 1.0, -1.0)).to(torch.float32)
        ctx.mcts_set_noise(False)
        out = dict(planes=planes[keep], pi=pi[keep], z=z, color=color_k, serial=serial[keep], games=done)
        if protocol:
            out["m"] = torch.cat(rec["m"])[keep]   # the m of each sample's search
            out["resigned"] = n_resigned
            out["held_out"] = {k: (torch.cat(v) if v else torch.zeros((0, 2) if k == "min_m" else (0,), dtype=torch.float64 if k == "min_m" else
                                                                        (torch.int64 if k == "serial" else torch.uint8), device=dev))
                               for k, v in records.items()}
        return out


def resign_threshold(records, fp=0.05):
    """AlphaGo Zero's resignation threshold from the held-out games of a self-play run (records: the `held_out` dict of self_play_native /
    self_play_continuous, or any dict with `result` [G] (0 draw, 1 Red, 2 Blue) and `min_m` [G, 2]). A held-out game would have been a
    false positive at v if a side that did not lose (the winner, either side of a draw) has min m < v. Returns the (floor(fp G) + 1)-th
    smallest such non-loser minimum (+inf when there are fewer): resigning below it, at most floor(fp G) of the G held-out games would
    have been false positives."""
    result = np.asarray(records["result"].cpu() if hasattr(records["result"], "cpu") else records["result"]).astype(np.int64).reshape(-1)
    min_m = np.asarray(records["min_m"].cpu() if hasattr(records["min_m"], "cpu") else records["min_m"], dtype=np.float64).reshape(-1, 2)
    k = int(np.floor(fp * len(result)))
    vals = np.sort(np.concatenate([min_m[result != 2, 0], min_m[result != 1, 1]]))   # Red did not lose, Blue did not lose
    return float(vals[k]) if k < len(vals) else float("inf")


def fight(ctx, move_fn_a, move_fn_b, a_is_red, max_plies=150):
    with torch.cuda.stream(ctx.torch_stream()):
        return _fight(ctx, move_fn_a, move_fn_b, a_is_red, max_plies)


def _fight(ctx, move_fn_a, move_fn_b, a_is_red, max_plies):
    """Arena loop over all games of ctx in lockstep. move_fn_x(ctx) must leave actions for every game in ONB_BUF_ACTIONS
    (e.g. a search followed by a copy of BEST, or a random policy). a_is_red: bool tensor/array [n], which games agent A
    plays as Red. Returns (a_wins, b_wins, draws)."""
    n = ctx.n
    a_is_red = torch.as_tensor(np.asarray(a_is_red), device="cuda:%d" % ctx.device).bool()
    states_t = ctx.tensor(L.BUF_STATES)
    acts = ctx.tensor(L.BUF_ACTIONS)
    plies_left = max_plies
    while True:
        st = states_t.clone()
        live = ((st[:, 2] >> 29) & 3) == 0
        if not bool(live.any()):
            break
        side = (st[:, 1] >> 30) & 1
        a_to_move = (side == 0) == a_is_red
        move_fn_a(ctx)
        act_a = acts.clone()
        move_fn_b(ctx)
        act_b = acts.clone()
        acts.copy_(torch.where(a_to_move, act_a, act_b))
        ctx.step(None)
        if plies_left < 0:
            break
        plies_left -= 1
    res = (states_t.clone()[:, 2] >> 29) & 3
    red_won, blue_won = res == 1, res == 2
    a_wins = int((red_won & a_is_red).sum() + (blue_won & ~a_is_red).sum())
    b_wins = int((red_won & ~a_is_red).sum() + (blue_won & a_is_red).sum())
    ctx.last_fight_results = res.cpu().numpy()  # per-game results for fight_statistics()
    return a_wins, b_wins, int(n - a_wins - b_wins)


def puct_tb_move(sims, c_puct=2.0, evaluator=L.EVAL_UNIFORM):
    """ONB_AGENT_PUCT_TB as a move function of fight(): an eval-mode PUCT search with tablebase leaves (tb=True) over every game,
    then the table's move (tb_best) in the games of the resident table. The context's tablebase-leaf switch is left as it was."""
    def move(ctx):
        was = ctx.tb_leaves
        ctx.search_device(c_puct, sims, evaluator=evaluator, tb=True)
        ctx._use_tb(was)
        best = ctx.tensor(L.BUF_BEST).clone()
        ctx.tb_best(to_host=False)  # the table's moves into ACTIONS, ACTION_NONE (-1 as int16) outside the table
        acts = ctx.tensor(L.BUF_ACTIONS)
        acts.copy_(torch.where(acts != -1, acts, best))
    return move


def puct_solver_move(sims, c_puct=2.0, evaluator=L.EVAL_UNIFORM):
    """ONB_AGENT_PUCT_SOLVER as a move function of fight(): an eval-mode PUCT search with the MCTS solver (solver=True) over every game,
    playing the solver's best move. The context's solver switch is left as it was; ctx.last_root_proof keeps the root proofs."""
    def move(ctx):
        was = ctx.solver
        ctx.search_device(c_puct, sims, evaluator=evaluator, solver=True)
        ctx.last_root_proof = ctx.root_proof()
        ctx._use_solver(was)
        ctx.tensor(L.BUF_ACTIONS).copy_(ctx.tensor(L.BUF_BEST))
    return move


class ReplayBuffer:
    """Fixed-capacity ring buffer of self-play samples on one device (train.rs:213,241-245 keeps `data_buffer =
    Vec::with_capacity(buffer_size)` and only ever extends it; the ring bounds it: the newest samples overwrite the oldest).
    2 304 B per sample. `NativeReplayBuffer` below is the same thing behind the C ABI (onb_replay_*)."""

    def __init__(self, capacity, device="cpu"):
        self.capacity = int(capacity)
        self.planes = torch.zeros((self.capacity, 21, 5, 5), dtype=torch.float32, device=device)
        self.pi = torch.zeros((self.capacity, 2, 25), dtype=torch.float32, device=device)
        self.z = torch.zeros((self.capacity,), dtype=torch.float32, device=device)
        self.size = 0
        self.head = 0  # next write position

    def add(self, planes, pi, z):
        """Append m samples (newest overwrite the oldest once full). Accepts the dict fields returned by self_play()."""
        m = int(planes.shape[0])
        if m == 0:
            return
        if m >= self.capacity:  # keep only the newest `capacity` samples
            planes, pi, z = planes[-self.capacity:], pi[-self.capacity:], z[-self.capacity:]
            m = self.capacity
        idx = (self.head + torch.arange(m, device=self.planes.device)) % self.capacity
        self.planes[idx] = planes.to(self.planes.device)
        self.pi[idx] = pi.to(self.pi.device)
        self.z[idx] = z.to(self.z.device)
        self.head = (self.head + m) % self.capacity
        self.size = min(self.capacity, self.size + m)

    def sample(self, batch_size, generator=None):
        """train.rs:280-283: `choose_multiple` -> batch_size distinct samples, uniformly at random."""
        b = min(int(batch_size), self.size)
        idx = torch.randperm(self.size, generator=generator, device="cpu")[:b].to(self.planes.device)
        return self.planes[idx], self.pi[idx], self.z[idx].unsqueeze(1)


class NativeReplayBuffer:
    """onb_replay_*: the replay ring and the choose_multiple minibatch gather inside the library (device memory of the context), for
    hosts without torch. add() takes device tensors; sample() returns zero-copy views of the ring's minibatch buffers (valid until the
    next sample())."""

    def __init__(self, ctx, capacity):
        import ctypes as C
        self.ctx = ctx
        h = C.c_void_p()
        ctx._ck(ctx._lib.onb_replay_create(ctx._h, int(capacity), C.byref(h)))
        self._h = h
        self.capacity = int(capacity)

    @property
    def size(self):
        import ctypes as C
        n = C.c_int64(0)
        self.ctx._ck(self.ctx._lib.onb_replay_size(self._h, C.byref(n), None))
        return int(n.value)

    def add(self, planes, pi, z):
        with torch.cuda.stream(self.ctx.torch_stream()):
            planes, pi, z = planes.contiguous().float(), pi.contiguous().float(), z.contiguous().float()
            self.ctx._ck(self.ctx._lib.onb_replay_add(self._h, planes.data_ptr(), pi.data_ptr(), z.data_ptr(), int(planes.shape[0])))
            self.ctx.sync()   # the source tensors may be freed by the caller afterwards

    def sample(self, batch_size, seed=0):
        import ctypes as C
        from .engine import _DevBuf
        p, q, z, m = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_int64(0)
        self.ctx._ck(self.ctx._lib.onb_replay_sample(self._h, int(batch_size), int(seed), C.byref(p), C.byref(q), C.byref(z), C.byref(m)))
        b = int(m.value)
        dev = "cuda:%d" % self.ctx.device
        if b == 0:
            return (torch.zeros((0, 21, 5, 5), device=dev), torch.zeros((0, 2, 25), device=dev), torch.zeros((0, 1), device=dev))
        with torch.cuda.stream(self.ctx.torch_stream()):
            return (torch.as_tensor(_DevBuf(p.value, (b, 21, 5, 5), "<f4"), device=dev), torch.as_tensor(_DevBuf(q.value, (b, 2, 25), "<f4"), device=dev),
                    torch.as_tensor(_DevBuf(z.value, (b,), "<f4"), device=dev).unsqueeze(1))

    @staticmethod
    def indices(size, batch_size, seed=0):
        """the ring slots onb_replay_sample gathers for (seed, size): distinct, pseudo-random (host helper, no device)"""
        import ctypes as C
        b = min(int(batch_size), int(size))
        out = np.zeros(b, dtype=np.int64)
        rc = L.load().onb_replay_indices(int(size), int(batch_size), int(seed), L.ptr(out))
        if rc != 0:
            raise L.OnbError(rc, "onb_replay_indices: bad arguments")
        return out

    def close(self):
        if getattr(self, "_h", None):
            self.ctx._lib.onb_replay_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
