"""Speed of the on-device policy/value network at 64 and 128 hidden channels (onb_net_forward), with cuDNN as the baseline.

For widths 64 / 128, modes f16 / tf32 / f32 (ONB_NET_*) and 3 / 5 residual blocks: time per call on 16 384 positions (CUDA events on
the context's stream, after warm-up), positions/s, useful TFLOP/s computed from the shapes (2 x 25 squares x 9 taps x C_in x C_out per
convolution and position; heads not counted) and, for the 128-wide kernel, the L2 -> SM weight bytes per call computed from its
layout (every pass of NB boards streams the whole weight blob once). The 64-wide rows run the default kernels; one more row runs the
round-1 f16 kernel (ONB_NET_F16_QUAD=0), whose weight stream is 7 boards per pass of 8 KB taps. Inputs and weights stay in L2 across
calls, as they do inside a search. Then cuDNN (channels-last, torch defaults: TF32 convolutions) on the same 128-wide nets, and one
config-5-shaped search: 16 384 trees x 800 simulations, ONB_EVAL_NET, 3-block 128-wide net (f16) next to the 64-wide one.
Usage: python tools/net_wide_speed.py [--json PATH] [--reps 50]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

B = 16384
KB = 1024


def macs(width, blocks):
    return 25 * 9 * (21 * width + 2 * blocks * width * width)


def wide_weight_bytes(mode, blocks):
    """bytes of weights one pass of k_net_wide streams, and boards per pass (GeoW in onb_net.cu)"""
    nmat = 2 if mode == "f32" else 1
    kb = 2 if mode != "tf32" else 4
    blk = 128 * 128
    per_pass = 9 * nmat * blk + 2 * blocks * 9 * nmat * kb * blk
    return per_pass, (7 if mode == "f16" else 3)


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the name from torch is still reported
        q = "nvidia-smi unavailable: %s" % e
    return name, q


def time_calls(fn, stream, reps, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        fn()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("net_wide_speed: needs a CUDA device")
    import __graft_entry__ as ge
    ge.build()
    import onitama_alphazero_b200 as onb
    from onitama_alphazero_b200.net import ConvResNet

    name, smi = gpu_info()
    print("GPU: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (name, smi), flush=True)
    out = {"gpu": name, "nvidia_smi": smi, "positions": B, "rows": []}
    g = torch.Generator().manual_seed(0)
    planes = (torch.rand(B, 21, 5, 5, generator=g) > 0.7).float().numpy()

    def row(d):
        out["rows"].append(d)
        wb = "%8.2f GB" % (d["weight_bytes"] / 1e9) if d.get("weight_bytes") else "       n/a"
        print("%-34s %8.3f ms  %7.2f M pos/s  %7.1f TFLOP/s useful  weights L2->SM %s" % (d["case"], d["ms"], d["pos_per_s"] / 1e6, d["tflops"], wb),
              flush=True)

    with onb.Context(B, mcts_max_sims=2, planes=False) as ctx:
        ctx.write(onb.BUF_LEAF_PLANES, planes)
        stream = ctx.torch_stream()
        cases = [(w, m, b, None) for w in (64, 128) for b in (3, 5) for m in ("f16", "tf32", "f32")] + [(64, "f16", 3, "0"), (64, "f16", 5, "0")]
        for width, mode, blocks, quad in cases:
            torch.manual_seed(1234)
            ctx.net_load(ConvResNet(width, 21, blocks), precision=mode)
            if quad is not None:
                os.environ["ONB_NET_F16_QUAD"] = quad
            try:
                ms = time_calls(lambda: ctx.net_forward(onb.BUF_LEAF_PLANES), stream, args.reps)
            finally:
                os.environ.pop("ONB_NET_F16_QUAD", None)
            if width == 128:
                per_pass, nb = wide_weight_bytes(mode, blocks)
                wbytes = per_pass * -(-B // nb)
            elif quad is not None:  # round-1 k_net_forward<true>: 7 boards per pass, 8 KB per tap
                wbytes = 9 * (1 + 2 * blocks) * 8 * KB * -(-B // 7)
            else:
                wbytes = None
            label = "%3d ch %s %d blocks%s" % (width, mode, blocks, " (round-1 kernel)" if quad is not None else "")
            row(dict(case=label, width=width, mode=mode, blocks=blocks, ms=ms, pos_per_s=B / ms * 1e3,
                     tflops=2 * macs(width, blocks) * B / (ms * 1e-3) / 1e12, weight_bytes=wbytes))

    x = torch.from_numpy(planes).cuda().contiguous(memory_format=torch.channels_last)
    for blocks in (3, 5):
        torch.manual_seed(1234)
        m = ConvResNet(128, 21, blocks).cuda().eval().to(memory_format=torch.channels_last)
        with torch.no_grad():
            ms = time_calls(lambda: m(x), torch.cuda.current_stream(), args.reps)
        row(dict(case="128 ch cuDNN channels-last %d blocks" % blocks, width=128, mode="cudnn", blocks=blocks, ms=ms, pos_per_s=B / ms * 1e3,
                 tflops=2 * macs(128, blocks) * B / (ms * 1e-3) / 1e12, weight_bytes=None))

    sims = 800
    for width in (64, 128):
        with onb.Context(B, seed=1, mcts_max_sims=sims) as ctx:
            torch.manual_seed(1234)
            ctx.net_load(ConvResNet(width, 21, 3), precision="f16")
            ctx.reset()
            ctx.search_device(2.0, 16, evaluator=onb.EVAL_NET)   # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.search_device(2.0, sims, evaluator=onb.EVAL_NET)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        rate = B * sims / dt
        out["rows"].append(dict(case="search %d ch f16" % width, width=width, trees=B, sims=sims, seconds=dt, sims_per_s=rate))
        print("search: %d trees x %d sims, ONB_EVAL_NET, 3-block %d-wide net (f16): %.3f s -> %.3g sims/s" % (B, sims, width, dt, rate), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
