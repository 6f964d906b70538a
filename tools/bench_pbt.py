#!/usr/bin/env python
"""Population-based training rounds on one GPU: one JSON line per measurement, written to --out and printed.

  * round: one PBT round (aur_pop_episode_fitness + aur_pop_pbt_step, three launches) at K x n_member = 64 x 1,024,
    1,024 x 64 and 4,096 x 16 (CartPole-v1, hidden 64 x 2), CUDA events over --rounds rounds after --warmup rounds.  The
    fitness fed to the rank / exploit kernels is a fixed random vector (every member ranked), so every round copies the state
    of floor(0.25 K) members; the default episode fitness is computed in the same round and discarded.  The [K][P] rows
    and moments are 64 x 37 KB x 3 = 7 MB at K = 64 (L2-resident after the first round) and 450 MB at K = 4,096.
  * iteration: the README's 64 x 1,024 population (T = 128, 4 epochs x 4 minibatches), ms per iteration without PBT and with a
    round after every iteration (pbt interval 1: the round plus the host read of its donors / fitness / hyper-parameters that
    train() does), host clock around synchronised iterations.
  * learning: CartPole, K = 16 members with learning rates log-spaced over 1e-5 .. 1e-2, the same budget with and without PBT
    (interval 2, fraction 0.25, learning_rate and entropy_coeff perturbed by 0.8 / 1.2): the mean return of the episodes each
    member finished in the last iteration, and the population's mean and best.  Reported, not asserted.

The card's name and power limit are read in the same process and put on every line.
Usage: python tools/bench_pbt.py [--rounds 200] [--warmup 20] [--iters 10] [--learn-iters 40] [--out profiles/bench/pbt_bench.jsonl]"""
import argparse
import ctypes
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from aur_ppo_b200 import _lib, kernels  # noqa: E402
from aur_ppo_b200.population import ppo_population  # noqa: E402
from tools.bench_population import card, params_for  # noqa: E402


def bench_round(K, n, warmup, rounds):
    L = _lib.lib()
    dev = torch.device("cuda:0")
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    P = kernels.policy_param_count(desc)
    seeds = torch.arange(K, dtype=torch.int64, device=dev)
    pop = _lib.PopDesc(K, 0, n, seeds.data_ptr())
    rows = [torch.randn(K, P, device=dev) for _ in range(3)]
    steps = torch.ones(K, dtype=torch.int64, device=dev)
    hp = torch.tensor([[2.5e-4, 0.01, 0.2, 0.5, 0.5, float("inf")]] * K, dtype=torch.float64, device=dev)
    totals = torch.rand(K, 3, dtype=torch.float64, device=dev) * 100 + 1
    snapshot, episode_fitness = torch.zeros(K, 3, dtype=torch.float64, device=dev), torch.empty(K, dtype=torch.float64, device=dev)
    fitness = torch.randn(K, dtype=torch.float64, device=dev)
    rank, donor, order = (torch.empty(m, dtype=torch.int32, device=dev) for m in (K, K, K + 1))
    a = _lib.PopPbtArgs()
    a.fitness, a.q, a.down, a.up, a.mask, a.seed = fitness.data_ptr(), 0.25, 0.8, 1.2, 0b11, 1
    a.params, a.adam_m, a.adam_v = (r.data_ptr() for r in rows)
    a.steps, a.hparams, a.norm, a.norm_ld = steps.data_ptr(), hp.data_ptr(), None, 0
    a.rank_out, a.donor_out, a.order = rank.data_ptr(), donor.data_ptr(), order.data_ptr()
    st = kernels._stream()

    def one(r):
        _lib.check(L.aur_pop_episode_fitness(ctypes.byref(pop), totals.data_ptr(), snapshot.data_ptr(), episode_fitness.data_ptr(), st),
                   "aur_pop_episode_fitness")
        a.round = r
        _lib.check(L.aur_pop_pbt_step(ctypes.byref(pop), ctypes.byref(desc), ctypes.byref(a), st), "aur_pop_pbt_step")

    for r in range(1, warmup + 1):
        one(r)
    torch.cuda.synchronize()
    L.aur_launch_count_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(rounds):
        one(warmup + 1 + r)
    e1.record()
    torch.cuda.synchronize()
    launches = L.aur_launch_count() / rounds
    ms = e0.elapsed_time(e1) / rounds
    moved = int((donor >= 0).sum())
    return dict(kind="round", K=K, n_member=n, P=P, recipients_per_round=moved, round_us=round(ms * 1e3, 2), launches_per_round=launches)


def _members_lr(K, lo=1e-5, hi=1e-2):
    return [dict(seed=float(k + 1), learning_rate=float(v)) for k, v in enumerate(np.geomspace(lo, hi, K))]


def bench_iteration(warmup, iters):
    K, n = 64, 1024
    out = dict(kind="iteration", K=K, n_member=n, T=128)
    for label, pbt in (("no_pbt", None), ("pbt_interval_1", dict(interval=1))):
        pop = ppo_population(params_for(n, warmup + iters), [dict(seed=float(k + 1)) for k in range(K)], pbt=pbt)
        pop.reset_envs()

        def step(u):
            pop.run_update(u)
            if pbt is not None:
                pop._record_round(u, pop.pbt_step())

        for u in range(1, warmup + 1):
            step(u)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for u in range(warmup + 1, warmup + iters + 1):
            step(u)
        torch.cuda.synchronize()
        out[f"{label}_ms_per_iter"] = round((time.perf_counter() - t0) * 1e3 / iters, 3)
        del pop
        torch.cuda.empty_cache()
    out["pbt_overhead_pct"] = round(100 * (out["pbt_interval_1_ms_per_iter"] / out["no_pbt_ms_per_iter"] - 1), 2)
    return out


def bench_learning(iters, n=256):
    K = 16
    out = dict(kind="learning", env="CartPole-v1", K=K, n_member=n, T=128, iterations=iters, lr_range=[1e-5, 1e-2])
    for label, pbt in (("no_pbt", None), ("pbt", dict(interval=2))):
        params = params_for(n, 0)
        params["total_timesteps"] = n * 128 * iters
        pop = ppo_population(params, _members_lr(K), pbt=pbt)
        pop.reset_envs()
        for u in range(1, iters + 1):
            if u == iters:
                before = pop.totals.cpu().numpy().copy()
            pop.run_update(u)
            if pbt is not None and u % pbt["interval"] == 0 and u < iters:
                pop._record_round(u, pop.pbt_step())
        d = pop.totals.cpu().numpy() - before
        final = np.where(d[:, 0] > 0, d[:, 1] / np.maximum(d[:, 0], 1), np.nan)
        out[f"{label}_final_return_per_member"] = [round(float(v), 1) for v in final]
        out[f"{label}_final_return_mean"] = round(float(np.nanmean(final)), 2)
        out[f"{label}_final_return_best"] = round(float(np.nanmax(final)), 2)
        if pbt is not None:
            out["pbt_final_learning_rates"] = [float(f"{mp['learning_rate']:.3g}") for mp in pop.member_params]
        del pop
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--learn-iters", type=int, default=40)
    ap.add_argument("--shapes", default="64x1024,1024x64,4096x16")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench", "pbt_bench.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pbt needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    lines = [bench_round(*(int(x) for x in spec.lower().split("x")), args.warmup, args.rounds) for spec in args.shapes.split(",")]
    lines.append(bench_iteration(2, args.iters))
    if args.learn_iters > 0:
        lines.append(bench_learning(args.learn_iters))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            line.update(gpu=name, power_limit=power)
            f.write(json.dumps(line) + "\n")
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
