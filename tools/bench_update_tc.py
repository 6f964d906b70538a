"""Time the gradient phase of the headline update (`kernels.Updater.grad`: ppo_grad_tc_kernel + the partial reduction) on
one GPU, at the benchmark's minibatch: m = 2,097,152 samples gathered from B = 8,388,608 CartPole-shaped records
(65,536 envs x 128 steps).  The advantage moments are prepared once, as bench.py does per iteration, so the timed calls
are the grad kernel and its reduction only.  The records (2 x 268 MB) do not fit in L2.

  python tools/bench_update_tc.py [--iters 100] [--warmup 10] [--dump DIR]
  python tools/bench_update_tc.py --lib old.so --lib new.so --rounds 5     # A/B: alternating subprocesses, one JSON line each

AUR_UPDATE_IMPL=tc4 selects the four-threads-per-sample kernel.  --dump DIR writes the reduced gradients with the statistic
sums (grads.npy) and the per-CTA partials of the last call (partials.npy)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().split(",")])) if r.returncode == 0 else {}


def run(args):
    import numpy as np
    import torch
    from aur_ppo_b200 import _lib, kernels
    from tools.microbench import _policy
    desc, flat = _policy(False)
    B, m = args.B, args.m
    g = torch.Generator(device="cuda").manual_seed(3)
    dbuf = [torch.randn(B, 4, generator=g, device="cuda") * 0.5, torch.randint(0, 2, (B,), generator=g, device="cuda").float(),
            -0.7 + 0.1 * torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda"),
            torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda")]
    idx = torch.randperm(B, generator=g, device="cuda")[:m].to(torch.int32)
    up = kernels.Updater(desc, flat.clone())
    rec = kernels.pack_records(*dbuf)
    up.prepare_moments(dbuf[3], idx.view(1, m))

    def call():
        up.grad(*dbuf, idx, records=rec, moments_index=0)

    for _ in range(args.warmup):
        call()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.iters)]
    for a, b in ev:
        a.record()
        call()
        b.record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in ev)
    res = {"bench": "update_grad", "lib": _lib.LIB_PATH, "impl": os.environ.get("AUR_UPDATE_IMPL", "tc"), "B": B, "m": m,
           "iters": args.iters, "ms_median": ts[len(ts) // 2], "ms_min": ts[0], "ms_max": ts[-1],
           "samples_per_s": m / (ts[len(ts) // 2] * 1e-3), "gpu": gpu_info()}
    if args.dump:
        os.makedirs(args.dump, exist_ok=True)
        np.save(os.path.join(args.dump, "grads.npy"), up.grads.cpu().numpy())
        # [2][CTAs per net][UPD_PSTRIDE] partial rows at the start of the workspace (the tail: moments and a ticket)
        np.save(os.path.join(args.dump, "partials.npy"), up.workspace.cpu().numpy())
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100, help="timed calls (CUDA events around each)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--B", type=int, default=65536 * 128)
    ap.add_argument("--m", type=int, default=65536 * 128 // 4)
    ap.add_argument("--dump", metavar="DIR", default=None)
    ap.add_argument("--lib", action="append", default=[], help="library to time in a subprocess (repeat to alternate builds)")
    ap.add_argument("--rounds", type=int, default=1, help="with --lib: alternations of the libraries")
    args = ap.parse_args()
    if args.iters < 1:
        ap.error("--iters must be >= 1")
    if not args.lib:
        run(args)
        return
    if args.dump:
        ap.error("--dump times one library: run without --lib, with AUR_LIB_PATH set")
    rest = ["--iters", str(args.iters), "--warmup", str(args.warmup), "--B", str(args.B), "--m", str(args.m)]
    for _ in range(args.rounds):
        for lib in args.lib:
            env = dict(os.environ, AUR_LIB_PATH=os.path.abspath(lib))
            subprocess.run([sys.executable, os.path.abspath(__file__)] + rest, env=env, check=True)


if __name__ == "__main__":
    main()
