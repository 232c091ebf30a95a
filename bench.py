#!/usr/bin/env python3
"""bench.py -- env steps/s (and MCTS sims/s) of the B200-native Onitama self-play hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload env|mcts|playout] [--impl ours|reference] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1, NCCL only for the barrier / max-over-ranks of the timings: games shard
across GPUs with no data-path collective, scaling = weak). A "step" is one pass of the hot path over one batch:
  env     (BASELINE config 3, the default): one lockstep step of 1 048 576 games/GPU = legal moves -> random action
          (counter RNG) -> apply -> terminal detection -> auto-reset -> legal mask + 21x5x5 f32 planes of the new state.
  mcts    (BASELINE config 4): one full search = 16 384 trees/GPU x 400 simulations, uniform-prior evaluator.
  playout (BASELINE config 1): 4 096 random-vs-random games to terminal.
The default run measures env as the headline and appends the mcts numbers under "mcts" in the same JSON line.
--impl reference times the CPU restatement of the reference path (oracle/, all host threads) on the same workload.
--dump-outputs DIR writes what the last timed step computed (env, and the mcts section or workload) as DIR/<name>.npy, for a fixed
seeded sample of the games / trees, so that two builds can be compared output for output on identical inputs.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENV_GAMES = 1 << 20
MCTS_TREES = 1 << 14
MCTS_SIMS = 400
MCTS_C = 2.0
PLAYOUT_GAMES = 4096
SELFPLAY_GAMES = 16384
SELFPLAY_SIMS = 800
GAMES_SLOTS = 2048     # `games` workload: slots per GPU (a step plays 2 x slots whole games)
SEED = 20240607
DUMP_SAMPLE = 4096     # --dump-outputs: games / trees per dumped array (env planes: 8.6 MB)
NET_PRECISION = {"fused-f32": "f32", "fused": "f16", "fused-tf32": "tf32", "torch": "torch"}
NET_KERNEL = {"fused-f32": "k_net_forward_x3p<true> (CTA pairs, tcgen05 cta_group::2)", "fused": "k_net_forward_f16q<true> (CTA pairs, tcgen05 cta_group::2, four accumulators)", "fused-tf32": "k_net_forward<2,tf32>",
              "torch": "library kernels"}
NET_DTYPE = {"fused-f32": "f32-faithful network: split f16 operands (x = x1 + 2^-11 x2), 3 products per multiply-add, f32 accumulate",
             "fused": "f16 x f16 -> f32 network (FAST MODE: operands rounded to 11 bits, not the reference's f32 arithmetic)",
             "fused-tf32": "tf32 x tf32 -> f32 network (operands rounded to 11 bits)", "torch": "f32/tf32 (network, cuDNN)"}
# algorithmic bytes per unit of work (DESIGN.md section 5)
ENV_BYTES_PER_STEP = 16 + 16 + 8 + 2100  # state read, state write, legal mask, planes


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def read_tensor_peak():
    """dense bf16/f16 tensor peak in TFLOP/s: the sustained figure (the network runs inside a long step)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d.get("bf16_tflops_sustained") or d["bf16_tflops"]), "measured (MEASURED_PEAKS.json, sustained cuBLAS bf16)"
        except Exception:
            pass
    return 1590.0, "fallback (B200_PROFILING.md)"


def read_traffic(kernel):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


class ClockSampler:
    """SM clock and throttle reasons read IN PROCESS through NVML: one sample immediately before the timed region, one immediately
    after, and as many as fit while the host waits for the region to drain (sample() is called from the wait loop), so even a
    6 ms region is covered. Falls back to one `nvidia-smi` query per sample() if pynvml is missing."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
               ("hw_power_brake_slowdown", 0x80))

    def __init__(self, index, uuid=None):
        self.rows, self.h, self.nv, self.index = [], None, None, index
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)) if uuid and not str(uuid).startswith("GPU-") else str(uuid))
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                phys = index
                if vis:
                    try:
                        phys = int(vis.split(",")[index])
                    except Exception:
                        phys = index
                self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def sample(self, tag="during"):
        try:
            if self.h is not None:
                nv = self.nv
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((tag, mhz, self.max_mhz, mask))
            else:
                q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.rows.append((tag, float(out[0]), float(out[1]), int(out[2].strip(), 16)))
        except Exception:
            pass

    def result(self, window):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0, "window": window}
        sm = sorted(r[1] for r in self.rows)
        reasons = set()
        for r in self.rows:
            for name, bit in self.REASONS:
                if r[3] & bit:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[2] for r in self.rows), "reasons": sorted(reasons), "samples": len(sm),
                "sm_mhz_min": sm[0], "sm_mhz_first_last": [self.rows[0][1], self.rows[-1][1]], "source": "nvml (in process)" if self.h is not None else "nvidia-smi",
                "window": window}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def oracle():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    return oracle_lib


class CpuEnv:
    """The CPU arm of config 3 on a game array that lives across timed steps (like the GPU context's): `n` games, every call
    steps all of them `steps` times (random action, apply, auto-reset, legal mask, 21x5x5 planes), all host threads."""

    def __init__(self, n_games, threads):
        self.O = oracle()
        self.n, self.threads, self.step = n_games, threads, 0
        self.g = self.O.new_games(n_games, seed=SEED)

    def run(self, steps):
        sink = ctypes.c_double()
        dt = self.O.lib().orc_bench_env_steps(self.g.ctypes.data, self.n, 0, self.step, steps, SEED, self.threads, 1, ctypes.byref(sink))
        self.step += steps
        return self.n * steps / dt, dt


def cpu_env(n_games, steps, threads):
    return CpuEnv(n_games, threads).run(steps)


def cfg4_roots(O, n, seed):
    import numpy as np
    base = O.new_games(n, seed=seed)
    g = base.copy()
    for step in range(16):
        live = (np.arange(n) % 16) > step
        h = g.copy()
        O.env_step_random(h, seed, step)
        g[live] = h[live]
    dead = g["result"] != 0
    g[dead] = base[dead]
    return g


def cpu_mcts(n_trees, sims, threads):
    O = oracle()
    roots = cfg4_roots(O, n_trees, SEED)
    sink = ctypes.c_double()
    dt = O.lib().orc_bench_mcts(roots.ctypes.data, n_trees, MCTS_C, sims, threads, ctypes.byref(sink))
    return n_trees * sims / dt, dt


def cpu_selfplay(n_trees, sims):
    """Config 5 the way the reference runs it: the oracle's PUCT arena with the PyTorch module on the CPU as evaluator, one
    position per forward call (net.rs:217-219 unsqueezes to batch 1), playouts one after the other (mcts_arena.rs:75-102)."""
    import time
    import numpy as np
    import torch
    from onitama_alphazero_b200.net import ConvResNet
    O = oracle()
    torch.manual_seed(1234)
    model = ConvResNet(64, 21, 3).eval()

    @torch.no_grad()
    def eval_one(planes525):
        p, v = model(torch.from_numpy(np.asarray(planes525, dtype=np.float32)).reshape(1, 21, 5, 5))
        return p.reshape(50).numpy(), float(v.reshape(()))

    roots = cfg4_roots(O, n_trees, SEED)
    t0 = time.perf_counter()
    done = 0
    for t in range(n_trees):
        if roots["result"][t] == 0:
            O.mcts_search(roots[t:t + 1], MCTS_C, sims, callback=eval_one)
            done += sims
    dt = time.perf_counter() - t0
    return done / dt, dt, torch.get_num_threads()


def dump_sample(n):
    """--dump-outputs: the fixed, seeded subset of the n games / trees whose outputs are written (sorted indices)"""
    import numpy as np
    return np.sort(np.random.default_rng(SEED).choice(n, min(n, DUMP_SAMPLE), replace=False))


def write_dump(path, arrays):
    import numpy as np
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20, "dump larger than 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        np.save(os.path.join(path, name + ".npy"), a)


def all_deals():
    return [[a, b, c, d, e] for a in range(16) for b in range(a + 1, 16) for c in range(16) if c not in (a, b)
            for d in range(c + 1, 16) if d not in (a, b) for e in range(16) if e not in (a, b, c, d)]


def cpu_perft(n_decks, depth, threads):
    import numpy as np
    O = oracle()
    decks = np.array(all_deals(), dtype=np.uint8)
    sel = np.ascontiguousarray(decks[np.random.RandomState(0).choice(len(decks), n_decks, replace=False)])
    totals = np.zeros(depth, dtype=np.uint64)
    dt = O.lib().orc_bench_perft(sel.ctypes.data, n_decks, depth, threads, totals.ctypes.data)
    return float(totals.sum()) / dt, dt


def cpu_playout(n_games, threads):
    O = oracle()
    t0 = time.perf_counter()
    _, plies, _, total = O.playout_games(n_games, SEED)
    dt = time.perf_counter() - t0
    return total / dt, dt


def run_reference(args, rank):
    """The reference's own CPU implementation of the path (C++ restatement: the Rust workspace cannot be built here),
    all host threads, bounded sample of the same workload."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    wl = args.workload
    vals = []
    if wl == "env":
        # the config the line prints: the same 1 048 576 games, ONE lockstep step of all of them per timed step, game array kept
        # across steps (so the positions are the mid-game mix the GPU arm sees, not 1 M opening moves)
        env = CpuEnv(ENV_GAMES, cores)
        for i in range(args.warmup + args.steps):
            v, dt = env.run(1)
            if i >= args.warmup:
                vals.append((v, dt))
        sample = "%d games x 1 lockstep step per timed step, %d threads (same step contents: move gen, random action, apply, reset, mask, planes)" % (ENV_GAMES, cores)
        unit, metric = "env_steps/s", "env_steps_per_sec"
    elif wl == "mcts":
        n = 1024
        sample = "%d trees x %d sims per timed step, uniform evaluator" % (n, MCTS_SIMS)
        for i in range(args.warmup + args.steps):
            v, dt = cpu_mcts(n, MCTS_SIMS, cores)
            if i >= args.warmup:
                vals.append((v, dt))
        unit, metric = "sims/s", "mcts_sims_per_sec"
    elif wl == "perft":
        nd, dp = 16 * cores, 5
        sample = "%d deals x depth %d per timed step (same move generation / transition, recursive DFS)" % (nd, dp)
        for i in range(args.warmup + args.steps):
            v, dt = cpu_perft(nd, dp, cores)
            if i >= args.warmup:
                vals.append((v, dt))
        unit, metric = "nodes/s", "perft_nodes_per_sec"
    elif wl == "uct":
        import time as _t
        O = oracle()
        n = 512
        roots = cfg4_roots(O, n, SEED)
        sample = "%d trees x %d playouts per timed step, plain UCT with random rollouts" % (n, MCTS_SIMS)
        for i in range(args.warmup + args.steps):
            t0 = _t.perf_counter()
            O.uct_search_batch(roots, 2.0 ** 0.5, 5, MCTS_SIMS, seed=SEED, threads=cores)
            dt = _t.perf_counter() - t0
            if i >= args.warmup:
                vals.append((n * MCTS_SIMS / dt, dt))
        unit, metric = "playouts/s", "uct_playouts_per_sec"
    elif wl == "selfplay":
        sample = "2 trees x 100 sims per timed step, oracle arena + the PyTorch module on the CPU, one position per forward call as in the reference"
        for i in range(args.warmup + args.steps):
            v, dt, cores = cpu_selfplay(2, 100)
            if i >= args.warmup:
                vals.append((v, dt))
        unit, metric = "sims/s", "mcts_sims_per_sec"
    else:
        sample = "%d games to terminal, single thread" % PLAYOUT_GAMES
        cores = 1
        for i in range(args.warmup + args.steps):
            v, dt = cpu_playout(PLAYOUT_GAMES, 1)
            if i >= args.warmup:
                vals.append((v, dt))
        unit, metric = "env_steps/s", "env_steps_per_sec"
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(dt for _, dt in vals) / len(vals)
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32" if wl != "mcts" else "u32+f64",
            "data": "synthetic", "config": workload_config(wl),
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "note": "C++ restatement of the reference CPU path (oracle/onb_oracle.cpp); the Rust reference cannot be built in this image"}
    emit_line(line)


def workload_config(wl):
    if wl == "env":
        return {"workload": "BASELINE config 3: batched env stepping, %d concurrent games/GPU, legal-move masks + 21x5x5 f32 plane encoding, "
                            "random policy (counter RNG), auto-reset" % ENV_GAMES, "games_per_gpu": ENV_GAMES,
                "l2": "per-step output 2.2 GB/GPU >> 126 MB L2 (inputs larger than L2, no flush needed)"}
    if wl == "mcts":
        return {"workload": "BASELINE config 4: batched PUCT MCTS, %d sims/move, %d concurrent trees/GPU, uniform-prior evaluator, eval mode"
                            % (MCTS_SIMS, MCTS_TREES), "trees_per_gpu": MCTS_TREES, "sims": MCTS_SIMS, "c_puct": MCTS_C,
                "l2": "touched node pools ~2.4 GB/GPU >> 126 MB L2"}
    if wl == "selfplay":
        return {"workload": "BASELINE config 5: AlphaZero self-play, %d sims/move, 3-block ConvResNet (64 ch, random init, fixed seed) evaluating "
                            "the leaf buffer in place, %d concurrent games/GPU, one ply per step, replay samples gathered to GPU 0"
                            % (SELFPLAY_SIMS, SELFPLAY_GAMES), "games_per_gpu": SELFPLAY_GAMES, "sims": SELFPLAY_SIMS, "c_puct": MCTS_C,
                "l2": "node pools + leaf batches >> L2"}
    if wl == "games":
        return {"workload": "whole self-play games inside the library (onb_self_play): %d slots/GPU, %d games per step, %d sims/move, 3-block ConvResNet "
                            "on the tensor cores, every started game played to its end, train-mode root noise" % (GAMES_SLOTS, 2 * GAMES_SLOTS, SELFPLAY_SIMS),
                "slots_per_gpu": GAMES_SLOTS, "sims": SELFPLAY_SIMS, "l2": "node pools + sample buffers >> L2"}
    if wl == "uct":
        return {"workload": "plain UCT with random rollouts (the reference's Mcts agent, evaluator.rs opponent): %d playouts/move, %d concurrent "
                            "trees/GPU, config-4 roots, c = sqrt(2), min_node_visits = 5" % (MCTS_SIMS, MCTS_TREES), "trees_per_gpu": MCTS_TREES,
                "playouts": MCTS_SIMS, "l2": "node pools >> L2"}
    if wl == "perft":
        return {"workload": "BASELINE config 2: perft-style legal-move enumeration depth 6 from the standard opening over all 131040 canonical "
                            "card deals, 1 GPU", "deals": 131040, "depth": 6, "l2": "DFS phase is register resident (~0 B/node); L2 flushed between iterations"}
    return {"workload": "BASELINE config 1: random-vs-random, %d games to terminal" % PLAYOUT_GAMES, "games": PLAYOUT_GAMES,
            "l2": "L2 flushed between timed iterations (256 MB write)"}


# ------------------------------------------------------------------------------------------------ GPU arm
_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: everything else that libraries print there (NCCL's version banner, ...) is sent to
    stderr by pointing fd 1 at fd 2 for the rest of the run; emit_line() writes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default per workload: env 1000, mcts 20, perft 5, selfplay 3, playout 50)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed warm-up steps (default per workload, >= 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="env", choices=["env", "mcts", "playout", "perft", "selfplay", "uct", "games"])
    ap.add_argument("--subbatches", type=int, default=4, help="env e2e: sub-batches in flight inside onb_actor (>= 4 hides the copies under three kernels)")
    ap.add_argument("--gather", default="abi", choices=["abi", "torch"],
                    help="selfplay workload, N > 1: gather the replay samples with onb_gather_samples (C ABI) or torch.distributed")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary mcts measurement of the default env run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfplay", action="store_true", help="skip the config-5 section of the default env run (12 000 launches: too many for an ncu launch list)")
    ap.add_argument("--eval-mode", action="store_true",
                    help="selfplay workload: search without the root exploration noise (self_play of train.rs searches in train mode)")
    ap.add_argument("--net", default="fused-f32", choices=["fused-f32", "fused", "fused-tf32", "torch"],
                    help="selfplay workload: the tensor-core network kernel -- fused-f32 = f32-faithful split-operand arithmetic (the headline: "
                         "the reference computes in f32), fused = the f16 fast mode, fused-tf32 = tf32 operands -- or the PyTorch module as a black box")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="env and mcts workloads: after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32 or "
                         "float64, a fixed seeded sample of %d games / trees; the default env run adds its mcts section as mcts_*)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("env", "mcts")):
        ap.error("--dump-outputs covers the env and mcts workloads of --impl ours")
    claim_stdout()
    dflt = {"env": (1000, 50), "mcts": (20, 5), "perft": (5, 3), "selfplay": (3, 3), "playout": (50, 5), "uct": (5, 3), "games": (1, 3)}[args.workload]
    if args.impl == "reference":
        dflt = (3, 1)
    args.steps_given = args.steps is not None
    args.steps = dflt[0] if args.steps is None else args.steps
    args.warmup = dflt[1] if args.warmup is None else args.warmup
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device. The product path has no CPU fallback (use --impl reference for the CPU arm).")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner goes to stdout otherwise: stdout carries ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    import onitama_alphazero_b200 as onb

    # a real (non-default) torch stream: the context launches on it, torch's events/copies are ordered with the kernels
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    peak, peak_src = read_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    try:
        dev_uuid = torch.cuda.get_device_properties(local_rank).uuid
    except Exception:
        dev_uuid = None
    sampler_box = {}

    def new_sampler():
        # NVML handle is created once (nvmlInit + lookup take milliseconds); every timed region gets its own row list
        if "s" not in sampler_box:
            sampler_box["s"] = ClockSampler(local_rank, dev_uuid)
        sampler_box["s"].rows = []
        return sampler_box["s"]

    def timed(fn, warmup, steps, between=None):
        """W untimed warm-up steps, then exactly K steps between two CUDA events on the launch stream, barrier + synchronize on both
        sides, max over ranks. Clocks: NVML is read immediately before the first event, while the host waits for the second one
        (every rank samples its own GPU; rank 0's samples are reported), and immediately after."""
        sampler = new_sampler()
        for i in range(warmup):
            fn(i)
            if between:
                between()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if between is None:
            sampler.sample("before")
            e0.record(stream)
            for i in range(steps):
                fn(warmup + i)
            e1.record(stream)
            while not e1.query():
                sampler.sample("during")
            sampler.sample("after")
            barrier()
            ms = e0.elapsed_time(e1)
        else:  # L2 flush between iterations: time each iteration on its own
            ms = 0.0
            for i in range(steps):
                between()
                sampler.sample("before")
                e0.record(stream)
                fn(warmup + i)
                e1.record(stream)
                while not e1.query():
                    sampler.sample("during")
                ms += e0.elapsed_time(e1)
            sampler.sample("after")
            barrier()
        clocks = sampler.result("immediately before / during / immediately after the timed region") if rank == 0 else None
        return max_over_ranks(ms), clocks

    out = {}
    wl = args.workload

    # ---------------------------------------------------------------- env (config 3)
    def bench_env(steps, warmup):
        n = ENV_GAMES
        flags = onb.OUT_MASKS | onb.OUT_PLANES
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream)
        ctx.reset()
        ms, clocks = timed(lambda i: ctx.step_random(i, auto_reset=True, out_flags=flags), warmup, steps)
        st = ctx.stats()
        assert int(st[onb.STAT_STEPS]) == n * (steps + warmup), "kernel did not step every game"
        dump = {}
        if args.dump_outputs and rank == 0:   # the last timed step's states, masks and planes, before the e2e runs below reset the games
            idx = dump_sample(n)
            sel = torch.from_numpy(idx).cuda()
            dump = {"env_games": idx.astype(np.float64),
                    "env_states": ctx.get_states()[idx].view("<u4").reshape(len(idx), 6).astype(np.float64),
                    "env_masks": ctx.tensor(onb.BUF_MASKS)[sel].cpu().numpy().view(np.uint32).astype(np.float64),
                    "env_planes": ctx.tensor(onb.BUF_PLANES)[sel].cpu().numpy(),
                    "env_stats": st.astype(np.float64)}
        value = world * n * steps / (ms * 1e-3)
        kernel_ms = ms / steps  # one k_env_step launch per step
        achieved = ENV_BYTES_PER_STEP * n / (kernel_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": read_traffic("k_env_step"),
                "kernel": "k_env_step<uniform,planes>", "algorithmic_bytes_per_launch": ENV_BYTES_PER_STEP * n, "peak_source": peak_src}
        # e2e: the reference-facing call with HOST buffers. A host actor feeds every game's action from pinned host memory and gets
        # back what a self-play driver consumes per step -- which games were decided and by whom (2 bits/game) plus the counters --
        # through onb_actor_submit / onb_actor_wait: the context's games as N_SUB sub-batches, each on its own stream inside the
        # library (H2D actions -> step kernel incl. masks + planes in HBM -> D2H results -> event), the host blocking on ONE event per
        # sub-batch. Actions are a recorded trajectory (so every step is a legal, mid-game step exactly like the device-timed run).
        from onitama_alphazero_b200.engine import Actor
        HL = onb._lib
        n_sub = args.subbatches
        e_steps = min(steps, 300)
        k_all = warmup + e_steps
        host_actions = torch.empty((k_all, n), dtype=torch.int16).pin_memory()
        ctx.reset()
        acts_dev = ctx.tensor(onb.BUF_ACTIONS)
        for i in range(k_all):
            ctx.step_random(i, auto_reset=True, out_flags=onb.OUT_ACTIONS)
            host_actions[i].copy_(acts_dev, non_blocking=True)
        want_tail = ctx.get_states(n - 4096, 4096).tobytes()   # the replayed games must end where the recorded ones did
        trace_ptr = host_actions.data_ptr()

        def e2e_run(host_flags, native):
            ctx.reset()
            ctx.stats(clear=True)
            with Actor(ctx, n_sub=n_sub, out_flags=flags, host_flags=host_flags) as act:
                firsts = [v["first"] for v in act.views]

                def run(i0, k):
                    if native:   # the same ring driven inside the library (no host think time, no Python in the loop)
                        act.replay((trace_ptr + 2 * n * i0, n, k), step0=i0, auto_reset=True)
                        return
                    for i in range(i0, i0 + k):
                        row = trace_ptr + 2 * n * i
                        for j in range(n_sub):
                            act.wait(j)   # the host now holds the results of step i-1 of this sub-batch and decides its next actions
                            act.submit(j, row + 2 * firsts[j], step=i, auto_reset=True)
                    for j in range(n_sub):
                        act.wait(j)

                run(0, warmup)
                act.join()
                barrier()
                sampler = new_sampler()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                sampler.sample("before")
                e0.record(stream)
                run(warmup, e_steps)
                act.join()
                e1.record(stream)
                sampler.sample("after")
                barrier()
                ems = max_over_ranks(e0.elapsed_time(e1))
                st2 = ctx.stats()
                assert int(st2[onb.STAT_STEPS]) == n * k_all and int(st2[HL.STAT_BAD_ACTIONS]) == 0
                if host_flags & HL.HOST_STATS:
                    assert int(act.views[-1]["stats"][onb.STAT_STEPS]) <= n * k_all
                assert ctx.get_states(n - 4096, 4096).tobytes() == want_tail, "replayed trajectory diverged"
            d2h = (8 * n if host_flags & HL.HOST_MASKS else 0) + (n // 4 if host_flags & HL.HOST_DONE else 0) + (64 * n_sub if host_flags & HL.HOST_STATS else 0)
            return world * n * e_steps / (ems * 1e-3), ems / e_steps, d2h, sampler.result("before / after the e2e region") if rank == 0 else None

        v_done, ms_done, d2h_done, e_clocks = e2e_run(HL.HOST_DONE | HL.HOST_STATS, False)
        v_native, ms_native, _, _ = e2e_run(HL.HOST_DONE | HL.HOST_STATS, True)
        v_masks, ms_masks, d2h_masks, _ = e2e_run(HL.HOST_MASKS | HL.HOST_DONE | HL.HOST_STATS, False)
        e2e = {"value": v_done, "unit": "env_steps/s", "h2d_bytes_per_step": 2 * n, "d2h_bytes_per_step": d2h_done, "ms_per_step": ms_done,
               "steps": e_steps, "sub_batches": n_sub, "clocks": e_clocks,
               "path": "onb_actor_submit/onb_actor_wait from the host loop: actions of every game from pinned host memory (H2D), step kernel "
                       "incl. legal masks + planes written to HBM for the network, D2H of the per-game decided/winner bits (2 bits/game) and "
                       "the counters every step; %d sub-batches in flight on the library's own streams" % n_sub,
               "variants": {"native_ring": {"value": v_native, "ms_per_step": ms_native,
                                            "path": "onb_actor_replay: the same ring driven inside the library, no host think time"},
                            "masks_to_host": {"value": v_masks, "ms_per_step": ms_masks, "d2h_bytes_per_step": d2h_masks,
                                              "path": "as the headline plus the 8 B/game legal masks copied to the host every step (round 1's e2e bytes)"}}}
        ctx.close()
        del host_actions
        return dict(metric="env_steps_per_sec", value=value, unit="env_steps/s", ms_per_step=ms / steps, dtype="u32", roofline=roof, e2e=e2e,
                    gpu_launches=steps, clocks=clocks, dump=dump)

    # ---------------------------------------------------------------- mcts (config 4)
    def bench_mcts(steps, warmup):
        n, sims = MCTS_TREES, MCTS_SIMS
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream, mcts_max_sims=sims, planes=False)
        # roots = positions after p = (id mod 16) random plies of config-1 games (built with the env kernels);
        # a game that ended before its p-th ply is searched from its start position instead
        ctx.reset()
        base = ctx.get_states()
        cur = base.copy()
        for step in range(16):
            ctx.step_random(step)
            nxt = ctx.get_states()
            live = (np.arange(n) % 16) > step
            cur[live] = nxt[live]
            ctx.set_states(cur)
        dead = cur["result"] != 0
        cur[dead] = base[dead]
        ctx.set_states(cur)
        roots_np = cur

        def one(i):
            ctx.mcts_begin(MCTS_C, sims)
            ctx.mcts_run(onb.EVAL_UNIFORM, sims)
            ctx.mcts_finish(to_host=False)

        ms, clocks = timed(one, warmup, steps)
        nn, fl = ctx.mcts_tree_info()
        assert int((fl & 2).sum()) == 0, "node pool overflow"
        dump = {}
        if args.dump_outputs and rank == 0:   # the last timed search's results as onb_mcts_finish hands them to a caller
            idx = dump_sample(n)
            r = ctx.mcts_finish(to_host=True)
            dump = {"mcts_trees": idx.astype(np.float64), "mcts_best": r["best"][idx].astype(np.float64),
                    "mcts_pi": r["pi"][idx].reshape(len(idx), 50), "mcts_root_visits": r["root_visits"][idx].astype(np.float64),
                    "mcts_root_q": r["root_q"][idx], "mcts_child_visits": r["child_visits"][idx].astype(np.float64)}
        value = world * n * sims * steps / (ms * 1e-3)
        # measured tree shape -> algorithmic bytes per simulation (DESIGN.md section 5), from the GPU's own trees:
        # mean select depth d = sum of visits of non-root nodes / sims, mean children k = (nodes - 1) / expanded nodes
        mean_nodes = float(nn.mean())
        ds, ks = [], []
        for t in range(0, n, n // 32):
            tr = ctx.mcts_dump_tree(int(t))
            ds.append(float(tr["visits"][1:].sum()) / sims)
            ks.append((len(tr["visits"]) - 1) / max(1, int((tr["flags"] & 1).sum())))
        d_mean, kk = float(np.mean(ds)), float(np.mean(ks))
        bytes_per_sim = d_mean * (16 + kk * 20) + kk * 30 + (d_mean + 1) * 24 + 16
        run_ms = ms / steps
        achieved = bytes_per_sim * n * sims / (run_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": read_traffic("k_mcts_run"),
                "kernel": "k_mcts_run<uniform>", "algorithmic_bytes_per_sim": bytes_per_sim, "mean_depth": d_mean, "mean_children": kk,
                "mean_nodes_per_tree": mean_nodes, "peak_source": peak_src,
                "note": "latency/occupancy-bound pointer chasing; launch time includes k_mcts_begin and k_mcts_finish (<1%)"}
        # e2e: roots from pinned host memory -> search -> best/pi/visits back on the host
        roots_host = torch.from_numpy(roots_np.view(np.uint8).reshape(n, 24).copy()).pin_memory()
        host_view = roots_host.numpy().view(onb.STATE_DTYPE).reshape(n)

        def pinned(shape, tdtype, ndtype):
            t = torch.empty(shape, dtype=tdtype).pin_memory()
            return t, t.numpy().view(ndtype)
        keep = []
        outs = {}
        for key, shape, td, nd in (("best", (n,), torch.int16, np.uint16), ("pi", (n, 2, 25), torch.float32, np.float32),
                                   ("root_visits", (n,), torch.int32, np.uint32), ("root_q", (n,), torch.float64, np.float64),
                                   ("child_visits", (n, 40), torch.int32, np.uint32)):
            t, a = pinned(shape, td, nd)
            keep.append(t)
            outs[key] = a

        def e2e_one(i):
            ctx.set_states(host_view)
            ctx.mcts_begin(MCTS_C, sims)
            ctx.mcts_run(onb.EVAL_UNIFORM, sims)
            ctx.mcts_finish(to_host=True, out=outs)

        ems, _ = timed(e2e_one, 1, max(1, steps))
        e2e = {"value": world * n * sims * max(1, steps) / (ems * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": 24 * n,
               "d2h_bytes_per_step": n * (2 + 200 + 4 + 8 + 160), "ms_per_step": ems / max(1, steps),
               "path": "onb_env_set_states(host roots) + onb_mcts_begin/run/finish(host best, pi, visits, q)"}
        # train mode (root exploration noise, AlphaZeroMctsConfig::train) for reference: same search with onb_mcts_set_noise
        ctx.mcts_set_noise(True, 0.25, 0.03, SEED)
        tms, _ = timed(one, 2, 3)
        ctx.mcts_set_noise(False)
        roof["train_mode_noise"] = {"value": world * n * sims * 3 / (tms * 1e-3), "unit": "sims/s", "ms_per_step": tms / 3}
        ctx.close()
        return dict(metric="mcts_sims_per_sec", value=value, unit="sims/s", ms_per_step=run_ms, dtype="u32+f64", roofline=roof, e2e=e2e,
                    gpu_launches=3 * steps, clocks=clocks, dump=dump)

    # ---------------------------------------------------------------- playout (config 1)
    def bench_playout(steps, warmup):
        n = PLAYOUT_GAMES
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream, planes=False)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        total = {"steps": 0}

        def one(i):
            ctx.reset()
            ctx.playout(want_plies=False, want_trace=False)

        ms, clocks = timed(one, warmup, steps, between=lambda: flush.fill_(1))
        st = ctx.stats()
        per_iter = int(st[onb.STAT_STEPS]) // (steps + warmup)
        value = world * per_iter * steps / (ms * 1e-3)
        ctx.close()
        roof = {"bound": "hbm", "achieved": 44.0 * per_iter / (ms / steps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": 44.0 * per_iter / (ms / steps * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "k_env_playout",
                "note": "4096 games cannot fill 148 SMs; launch/latency-bound by construction", "peak_source": peak_src}
        e2e = {"value": value, "unit": "env_steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "path": "same call (reset + playout); timing includes the reset's host sync"}
        return dict(metric="env_steps_per_sec", value=value, unit="env_steps/s", ms_per_step=ms / steps, dtype="u32", roofline=roof, e2e=e2e,
                    gpu_launches=2 * steps, clocks=clocks)

    # ---------------------------------------------------------------- perft (config 2)
    def bench_perft(steps, warmup):
        decks = np.array(all_deals(), dtype=np.uint8)
        lo, cnt = rank * len(decks) // world, (rank + 1) * len(decks) // world - rank * len(decks) // world
        roots = onb.start_states(decks[lo:lo + cnt])  # if sharded (N > 1): deals are partitioned, "strong" scaling
        ctx = onb.Context(8, device=local_rank, stream=stream.cuda_stream, planes=False)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        res = {}

        def one(i):
            res["nodes"], res["wins"], res["zero"] = ctx.perft(roots, 6)

        ms, clocks = timed(one, warmup, steps, between=lambda: flush.fill_(1))
        # the same enumeration with EVERY leaf visited (k_perft_flat: register DFS below the frontier, no bulk counting of quiet replies):
        # the like-for-like figure against the CPU arm, which enumerates every leaf too (VERDICT r01 weak #8)
        os.environ["ONB_PERFT_DFS"] = "1"
        counted = res["nodes"].copy()
        ms_leaf, _ = timed(one, 1, max(1, min(steps, 3)), between=lambda: flush.fill_(1))
        os.environ.pop("ONB_PERFT_DFS", None)
        assert np.array_equal(counted, res["nodes"]), "bulk-counted and per-leaf enumeration disagree"
        total = int(res["nodes"].sum())
        tot_t = torch.tensor([total], device="cuda", dtype=torch.int64)
        if world > 1:
            dist.all_reduce(tot_t)
        total_all = int(tot_t.item())
        if world == 1:
            assert int(res["nodes"][:, 0].sum()) == 1375920 and int(res["nodes"][:, 1].sum()) == 14375088 and int(res["zero"].sum()) == 0
        value = total_all * steps / (ms * 1e-3)
        ctx.close()
        # breadth-first levels 1..4 go through HBM: a frontier node is written once (16 B state + 4 B root id) and read once
        bfs_nodes = int(res["nodes"][:, :4].sum())
        roof = {"bound": "hbm", "achieved": 40.0 * bfs_nodes / (ms / steps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": 40.0 * bfs_nodes / (ms / steps * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "k_perft_leaf2 (+ k_perft_expand)",
                "note": "frontier of plies 1-4 in HBM (40 B/node written + read, chunked to < 7 GB); plies 5 and 6 are counted per frontier node in "
                        "registers by k_perft_leaf2 (issue-bound: quiet replies are counted in bulk), so the HBM fraction stays small by design",
                "peak_source": peak_src, "nodes_per_call": total, "frontier_nodes_per_call": bfs_nodes,
                "algorithms": {"bulk_counted": {"value": value, "unit": "nodes/s", "ms_per_step": ms / steps,
                                                "what": "value of this line: the last two plies are COUNTED per frontier node (quiet replies in bulk), "
                                                        "not visited one by one"},
                               "per_leaf": {"value": total_all * max(1, min(steps, 3)) / (ms_leaf * 1e-3), "unit": "nodes/s",
                                            "ms_per_step": ms_leaf / max(1, min(steps, 3)),
                                            "what": "k_perft_flat: every leaf is generated and visited, as the CPU arm does -- the like-for-like "
                                                    "comparison with cpu_baseline"}}}
        e2e = {"value": value, "unit": "nodes/s", "h2d_bytes_per_step": 24 * cnt, "d2h_bytes_per_step": 3 * 8 * 6 * cnt,
               "path": "onb_perft(host roots) -> host counters (the timed call itself copies both ways)"}
        return dict(metric="perft_nodes_per_sec", value=value, unit="nodes/s", ms_per_step=ms / steps, dtype="u32", roofline=roof, e2e=e2e,
                    gpu_launches=80 * steps, clocks=clocks)

    # ---------------------------------------------------------------- plain UCT with random rollouts (the reference's Mcts agent)
    def bench_uct(steps, warmup):
        n, sims = MCTS_TREES, MCTS_SIMS
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream, mcts_max_sims=sims, planes=False)
        ctx.reset()
        base = ctx.get_states()
        cur = base.copy()
        for step in range(16):   # the config-4 roots: positions after (id mod 16) random plies
            ctx.step_random(step)
            nxt = ctx.get_states()
            live = (np.arange(n) % 16) > step
            cur[live] = nxt[live]
            ctx.set_states(cur)
        dead = cur["result"] != 0
        cur[dead] = base[dead]
        ctx.set_states(cur)

        def one(i):
            ctx.uct_search(2.0 ** 0.5, 5, sims, to_host=False)

        ms, clocks = timed(one, warmup, steps)
        nn, fl = ctx.mcts_tree_info()
        assert int((fl & 2).sum()) == 0, "node pool overflow"
        value = world * n * sims * steps / (ms * 1e-3)
        ctx.close()
        roof = {"bound": "hbm", "achieved": 0.0, "peak": peak, "unit": "GB/s", "frac": 0.0, "traffic": None, "kernel": "k_uct_run",
                "note": "a playout is a short tree descent plus a random game of ~35 plies played in registers by the 8 lanes of the tree's "
                        "group: issue-bound, ~0 algorithmic bytes per ply", "mean_nodes_per_tree": float(nn.mean()), "peak_source": peak_src}
        e2e = {"value": value, "unit": "playouts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "path": "device-resident"}
        return dict(metric="uct_playouts_per_sec", value=value, unit="playouts/s", ms_per_step=ms / steps, dtype="u32+f32", roofline=roof, e2e=e2e,
                    gpu_launches=3 * steps, clocks=clocks)

    # ---------------------------------------------------------------- whole self-play games, natively (onb_self_play)
    def bench_games(steps, warmup):
        from onitama_alphazero_b200.net import ConvResNet
        n, sims = GAMES_SLOTS, SELFPLAY_SIMS
        torch.manual_seed(1234)
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream, mcts_max_sims=sims)
        ctx.net_load(ConvResNet(64, 21, 3), precision=NET_PRECISION[args.net])
        quota = 2 * n           # a step = 2 games per slot, every one of them played to its end (onb_self_play never drops a started game)
        cap = n * 400           # plies of sample buffer: two games of at most 152 plies per slot and slack
        tot = {"games": 0, "samples": 0, "plies": 0}

        def one(i):
            r = ctx.self_play_native(MCTS_C, sims, quota, evaluator=onb.EVAL_NET, train=not args.eval_mode, noise_seed=SEED + i, sample_cap=cap)
            if i >= warmup:
                tot["games"] += r["games"]; tot["samples"] += int(r["planes"].shape[0]); tot["plies"] += r["plies_run"]

        ms, clocks = timed(one, warmup, steps)
        ctx.close()
        g = torch.tensor([tot["games"], tot["samples"], tot["plies"]], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(g)
        games, samples, plies = [float(x) for x in g.tolist()]
        value = games / (ms * 1e-3)
        flop = 2.0 * 25 * 64 * 9 * (21 + 6 * 64) + 2.0 * (25 * 64 * 3 + 2500 + 1600 + 64)
        tpeak, tsrc = read_tensor_peak()
        ach = flop * sims * (samples / world) / (ms * 1e-3) / 1e12   # one search of `sims` evaluations per recorded sample (= per live slot and ply)
        roof = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": read_traffic("k_net_forward"),
                "kernel": NET_KERNEL[args.net], "peak_source": tsrc,
                "samples_per_sec": samples / (ms * 1e-3), "plies_per_step": plies / world / max(1, steps),
                "note": "a step = 2 x slots complete games; every ply searches the slots with a game in progress (x 800 network evaluations); finished "
                        "slots start their next game at once while games remain, idle slots are not searched",
                "flop_basis": "recorded samples x sims network evaluations (idle slots are not searched)"}
        e2e = {"value": value, "unit": "games/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8 * plies / world / max(1, steps),
               "path": "onb_self_play: one 8-byte counter per ply crosses PCIe; samples stay in device buffers for the trainer"}
        return dict(metric="selfplay_games_per_sec", value=value, unit="games/s", ms_per_step=ms / steps,
                    dtype="u32+f64 (search), " + NET_DTYPE[args.net], roofline=roof, e2e=e2e, gpu_launches=int(plies / world) * (3 * sims + 12),
                    clocks=clocks)

    # ---------------------------------------------------------------- self-play with the network (config 5)
    def bench_selfplay(steps, warmup, net_mode=None):
        from onitama_alphazero_b200.net import ConvResNet, make_evaluator
        net_mode = net_mode or args.net
        n, sims = SELFPLAY_GAMES, SELFPLAY_SIMS
        torch.manual_seed(1234)
        model = ConvResNet(64, 21, 3)
        ctx = onb.Context(n, seed=SEED, device=local_rank, game_id_base=rank * n, stream=stream.cuda_stream, mcts_max_sims=sims)
        fused = net_mode != "torch"
        if fused:
            ctx.net_load(model, precision=NET_PRECISION[net_mode])   # onb_net_load: the network becomes part of the library's search
            net = None
        else:
            net = make_evaluator(model.cuda(local_rank))
        ctx.reset()
        if not args.eval_mode:   # TrainingAlphaZeroMcts of self_play: Dirichlet-style noise at the root (mcts_arena.rs:186-202)
            ctx.mcts_set_noise(True, 0.25, 0.03, SEED)
        planes_t, pi_t = ctx.tensor(onb.BUF_PLANES), ctx.tensor(onb.BUF_PI)
        got = {"samples": 0}
        # the replay gather of section 8e through the C ABI (onb_comm_* / onb_gather_samples: the library's own NCCL communicator, created
        # from an id that rank 0 hands out); --gather torch keeps the torch.distributed twin (sharding.gather_replay)
        comm = None
        if world > 1 and args.gather == "abi":
            from onitama_alphazero_b200.sharding import Comm
            idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                idt.copy_(torch.frombuffer(bytearray(Comm.unique_id()), dtype=torch.uint8))
            dist.broadcast(idt, src=0)
            torch.cuda.synchronize()
            comm = Comm(ctx, world, rank, bytes(idt.cpu().numpy().tobytes()))

        def one_ply(i):
            ctx.encode(to_host=False)                      # sample planes of the searched position (train.rs:58)
            if fused:   # onb_mcts_run(ONB_EVAL_NET): select -> tensor-core ConvResNet -> expand/backup, x sims, no host in the loop
                ctx.search_device(MCTS_C, sims, evaluator=onb.EVAL_NET)
            else:       # select -> torch module (zero-copy leaf batch, CUDA graph) -> expand/backup, x sims
                ctx.search_device(MCTS_C, sims, net=net, use_graph=True)
            z = torch.zeros(n, device=planes_t.device)
            if comm is not None:
                out_s = comm.gather_samples(planes_t, pi_t, z, dst=0)   # onb_gather_samples: the ply's samples to the trainer GPU over NVLink
            else:
                out_s = onb.gather_replay(planes_t, pi_t, z, dst=0)
            if out_s is not None:
                got["samples"] = int(out_s[0].shape[0])
            ctx.mcts_play_best()

        ms, clocks = timed(one_ply, warmup, steps)
        value = world * n * sims * steps / (ms * 1e-3)
        if comm is not None:
            comm.close()
        ctx.close()
        per_sim = 1217.0 + 2100 + 204
        if fused:
            # the dominant kernel is the network: 7 3x3 convolutions (21->64, 6 x 64->64) on 25 squares + heads = 11.68 MFLOP per evaluation
            flop = 2.0 * 25 * 64 * 9 * (21 + 6 * 64) + 2.0 * (25 * 64 * 3 + 2500 + 1600 + 64)
            tpeak, tsrc = read_tensor_peak()
            ach = flop * n * sims * steps / (ms * 1e-3) / 1e12
            roof = {"bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": read_traffic("k_net_forward"),
                    "kernel": NET_KERNEL[net_mode], "flop_per_evaluation": flop,
                    "note": "achieved = USEFUL network FLOPs (one f32 multiply-add per weight and square, as the reference computes) of the whole "
                            "ply / ply time, search kernels included in the time; the f32-faithful mode spends three f16 tensor-core products per "
                            "useful multiply-add (split operands), so its tensor pipe does 3x this figure; the MMAs also compute the zero-padding "
                            "cells (25 of 36.6 rows are real squares) and are bound by shared-memory operand reads at N = 64; peak = dense bf16/f16",
                    "peak_source": tsrc}
            if net_mode == "fused-f32":   # what the tensor pipe executes for those useful FLOPs: 3 f16 products per multiply-add
                roof["split_products_per_multiply_add"] = 3
                roof["tensor_pipe_tflops"] = 3 * ach
                roof["tensor_pipe_frac"] = 3 * ach / tpeak
        else:
            roof = {"bound": "hbm", "achieved": per_sim * n * sims * steps / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": per_sim * n * sims * steps / (ms * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "k_mcts_select + k_mcts_expand_backup",
                    "note": "the step is dominated by the black-box network (library kernels, ~11.7 MFLOP per evaluation), not by these kernels",
                    "peak_source": peak_src}
        e2e = {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 16 * world if comm is not None else 0,
               "path": "device-resident self-play ply (search + sample gather + play); nothing but the gather's sample counts crosses PCIe by design",
               "gather": "onb_gather_samples (C ABI, NCCL send/recv over NVLink)" if comm is not None else ("torch.distributed gather" if world > 1 else "single rank")}
        roof["search_mode"] = "eval (no root noise)" if args.eval_mode else "train (root exploration noise, epsilon 0.25, alpha 0.03)"
        return dict(metric="mcts_sims_per_sec", value=value, unit="sims/s", ms_per_step=ms / steps, dtype="u32+f64 (search), " + NET_DTYPE[net_mode],
                    network=net_mode, roofline=roof, e2e=e2e, gpu_launches=((3 if fused else 2) * sims + 4) * steps, clocks=clocks,
                    samples_per_ply=got["samples"])

    if wl == "env":
        out = bench_env(args.steps, args.warmup)
    elif wl == "selfplay":
        out = bench_selfplay(args.steps, args.warmup)
    elif wl == "uct":
        out = bench_uct(args.steps, args.warmup)
    elif wl == "games":
        out = bench_games(args.steps, args.warmup)
    elif wl == "perft":
        out = bench_perft(args.steps, args.warmup)
    elif wl == "mcts":
        out = bench_mcts(args.steps, args.warmup)
    else:
        out = bench_playout(args.steps, args.warmup)

    secondary = None
    third = None
    dumps = dict(out.get("dump", {}))
    if wl == "env" and not args.no_secondary:
        # the config-4 and config-5 sections obey --steps/--warmup too (their own defaults when the flags are absent; config 5 is
        # capped at 30 plies of 0.3 s so that an env-sized --steps cannot turn the run into minutes) and carry their own clocks
        m_steps, m_warm = (args.steps, args.warmup) if args.steps_given else (20, 5)
        m_steps = min(m_steps, 200)
        m = bench_mcts(m_steps, max(3, m_warm))
        dumps.update(m["dump"])
        secondary = {k: m[k] for k in ("metric", "value", "unit", "ms_per_step", "roofline", "e2e", "gpu_launches", "clocks")}
        secondary["config"] = workload_config("mcts")
        secondary["steps"], secondary["warmup"] = m_steps, max(3, m_warm)
        try:  # config 5 with the network on the tensor cores (one ply of 16 384 games x 800 simulations per step)
            if args.no_selfplay:
                raise RuntimeError("skipped (--no-selfplay)")
            s_steps, s_warm = (min(args.steps, 10), min(max(3, args.warmup), 5)) if args.steps_given else (3, 3)
            sp = bench_selfplay(s_steps, s_warm, "fused-f32")   # headline: the reference's f32 arithmetic
            third = {k: sp[k] for k in ("metric", "value", "unit", "ms_per_step", "dtype", "network", "roofline", "e2e", "gpu_launches", "clocks")}
            third["config"] = workload_config("selfplay")
            third["steps"], third["warmup"] = s_steps, s_warm
            fast = bench_selfplay(s_steps, s_warm, "fused")     # explicitly labelled fast mode (f16 operands)
            third["fast_mode_f16"] = {k: fast[k] for k in ("value", "unit", "ms_per_step", "dtype", "network", "gpu_launches")}
            third["fast_mode_f16"]["roofline_frac"] = fast["roofline"]["frac"]
        except Exception as exc:  # never lose the headline over the extra measurement
            third = {"error": repr(exc)}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        if wl == "env":
            env = CpuEnv(ENV_GAMES, cores)
            env.run(8)   # leave the opening positions behind (untimed)
            v, dt = env.run(24)
            cpu_baseline = {"value": v, "unit": "env_steps/s", "cores": cores, "kind": "port",
                            "sample": "the same %d games x 24 lockstep steps incl. mask + plane encode, after 8 untimed steps (%.1f s wall, %d threads)"
                                      % (ENV_GAMES, dt, cores)}
            v1, dt1 = cpu_env(1 << 15, 32, 1)
            cpu_baseline["single_core_value"] = v1
            if secondary is not None:
                vm, dtm = cpu_mcts(8192, MCTS_SIMS, cores)
                vm1, _ = cpu_mcts(512, MCTS_SIMS, 1)
                secondary["cpu_baseline"] = {"value": vm, "unit": "sims/s", "cores": cores, "kind": "port", "single_core_value": vm1,
                                             "sample": "8192 trees x 400 sims, uniform evaluator (%.1f s wall, %d threads)" % (dtm, cores)}
        elif wl == "mcts":
            v, dt = cpu_mcts(8192, MCTS_SIMS, cores)
            v1, _ = cpu_mcts(512, MCTS_SIMS, 1)
            cpu_baseline = {"value": v, "unit": "sims/s", "cores": cores, "kind": "port", "single_core_value": v1,
                            "sample": "8192 trees x 400 sims, uniform evaluator (%.1f s wall, %d threads)" % (dt, cores)}
        elif wl == "selfplay":
            v, dt, th = cpu_selfplay(4, 100)
            cpu_baseline = {"value": v, "unit": "sims/s", "cores": th, "kind": "port",
                            "sample": "4 trees x 100 sims, oracle arena + the PyTorch module on the CPU, one position per forward call as in the "
                                      "reference (%.1f s wall, %d torch threads)" % (dt, th)}
        elif wl == "games":
            v, dt, th = cpu_selfplay(2, 100)
            cpu_baseline = {"value": v / (SELFPLAY_SIMS * 27.5), "unit": "games/s", "cores": th, "kind": "port",
                            "sample": "derived: %.1f sims/s of the oracle arena + PyTorch module on the CPU (2 trees x 100 sims, %.1f s) / (%d sims x 27.5 "
                                      "plies per game)" % (v, dt, SELFPLAY_SIMS)}
        elif wl == "uct":
            O = oracle()
            import time as _t
            roots = cfg4_roots(O, 1024, SEED)
            t0 = _t.perf_counter()
            r = O.uct_search_batch(roots, 2.0 ** 0.5, 5, MCTS_SIMS, seed=SEED, threads=cores)
            dt = _t.perf_counter() - t0
            cpu_baseline = {"value": 1024 * MCTS_SIMS / dt, "unit": "playouts/s", "cores": cores, "kind": "port",
                            "sample": "1024 trees x 400 playouts (%.1f s wall, %d threads, %.1f rollout plies per playout)"
                                      % (dt, cores, r["rollout_plies"] / (1024.0 * MCTS_SIMS))}
        elif wl == "perft":
            v, dt = cpu_perft(16 * cores, 5, cores)
            cpu_baseline = {"value": v, "unit": "nodes/s", "cores": cores, "kind": "port", "algorithm": "per-leaf (recursive DFS visits every node; "
                            "compare with roofline.algorithms.per_leaf)",
                            "sample": "%d random deals x depth 5, recursive DFS (%.1f s wall, %d threads)" % (16 * cores, dt, cores)}
        else:
            v, dt = cpu_playout(PLAYOUT_GAMES, 1)
            cpu_baseline = {"value": v, "unit": "env_steps/s", "cores": 1, "kind": "port", "sample": "the same 4096 games, one thread (%.2f s)" % dt}

    if rank == 0:
        line = {"metric": out["metric"], "value": out["value"], "unit": out["unit"], "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": out["ms_per_step"], "higher_is_better": True, "scaling": "strong" if wl == "perft" else "weak", "vs_baseline": None, "dtype": out["dtype"],
                "data": "synthetic", "config": workload_config(wl), "roofline": out["roofline"], "cpu_baseline": cpu_baseline, "e2e": out["e2e"],
                "gpu_launches": out["gpu_launches"], "clocks": out["clocks"], "impl": "ours"}
        if secondary is not None:
            line["mcts"] = secondary
        if third is not None:
            line["selfplay"] = third
        if args.dump_outputs:
            write_dump(args.dump_outputs, dumps)
        emit_line(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
