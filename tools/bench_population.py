#!/usr/bin/env python
"""Populations vs one run at a time on one GPU: for each (K, n_member) shape, one JSON line with

  * ms per population iteration (all K members) and the aggregate env-steps/s, split into rollout / GAE / update by CUDA events;
  * library launches per iteration (aur_launch_count);
  * the same K members as K sequential standalone `ppo` objects (ms per round of K iterations, env-steps/s);
  * for reference, one standalone run of K * n_member envs.

T = 128, 4 epochs x 4 minibatches, CartPole-v1, hidden 64 x 2 (the README's headline shape).  The card's name and power limit
are read in the same process and printed on every line.  Usage: python tools/bench_population.py [--iters 5] [--warmup 2]
[--shapes 64x1024,16x4096,256x256,1x65536] [--no-sequential]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from aur_ppo_b200 import _lib, kernels, run_ppo  # noqa: E402
from aur_ppo_b200.population import member_params, ppo_population  # noqa: E402
from aur_ppo_b200.ppo import ppo  # noqa: E402

T, EPOCHS, NMB = 128, 4, 4


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def params_for(n_envs, iters):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False, num_envs=n_envs, num_steps=T, num_minibatches=NMB, num_update_epochs=EPOCHS,
             total_timesteps=n_envs * T * (iters + 10))
    return p


def time_iters(step, warmup, iters, events=True):
    """step(u, ev) runs iteration u; returns (ms per iteration, [rollout, gae, update] ms per iteration)."""
    for u in range(1, warmup + 1):
        step(u, None)
    torch.cuda.synchronize()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(iters)]
    t0 = time.perf_counter()
    for i in range(iters):
        step(warmup + 1 + i, evs[i] if events else None)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / iters
    split = [0.0, 0.0, 0.0]
    if events:
        for e in evs:
            for j in range(3):
                split[j] += e[j].elapsed_time(e[j + 1]) / iters
    return wall, split


def bench_shape(K, n, warmup, iters, sequential):
    L = _lib.lib()
    params = params_for(n, warmup + iters)
    members = [dict(seed=float(k + 1)) for k in range(K)]
    pop = ppo_population(params, members)
    pop.reset_envs()
    launches = []

    def pop_step(u, ev):
        L.aur_launch_count_reset()
        pop.run_update(u, events=ev)
        launches.append(L.aur_launch_count())

    ms, split = time_iters(pop_step, warmup, iters)
    steps = K * n * T
    out = dict(K=K, n_member=n, T=T, epochs=EPOCHS, minibatches=NMB, population_ms_per_iter=round(ms, 3),
               population_env_steps_per_s=round(steps / ms * 1e3),
               population_split_ms=dict(rollout=round(split[0], 3), gae=round(split[1], 3), update=round(split[2], 3)),
               launches_per_iter=launches[-1])
    del pop
    torch.cuda.empty_cache()
    if sequential:
        runs = []
        for k in range(K):
            s = ppo(member_params(params, members[k]))
            s.envs.reset(seed=list(s.plan.env_ids))
            s._env_step = 0
            s._stats_rows = torch.zeros(EPOCHS * NMB, kernels.NUM_STATS, device=s.device)
            runs.append(s)

        def seq_step(u, ev):
            for s in runs:
                s.run_update(u)

        ms_seq, _ = time_iters(seq_step, warmup, iters, events=False)
        out.update(sequential_ms_per_round=round(ms_seq, 3), sequential_env_steps_per_s=round(steps / ms_seq * 1e3),
                   speedup_vs_sequential=round(ms_seq / ms, 2))
        del runs
        torch.cuda.empty_cache()
    big = ppo(params_for(K * n, warmup + iters))
    big.envs.reset(seed=list(big.plan.env_ids))
    big._env_step = 0
    big._stats_rows = torch.zeros(EPOCHS * NMB, kernels.NUM_STATS, device=big.device)
    ms_big, split_big = time_iters(lambda u, ev: big.run_update(u, events=ev), warmup, iters)
    out.update(single_run_envs=K * n, single_run_ms_per_iter=round(ms_big, 3), single_run_env_steps_per_s=round(steps / ms_big * 1e3),
               single_run_split_ms=dict(rollout=round(split_big[0], 3), gae=round(split_big[1], 3), update=round(split_big[2], 3)),
               population_vs_single_run=round(ms_big / ms, 3))
    del big
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shapes", default="64x1024,16x4096,256x256,1x65536")
    ap.add_argument("--no-sequential", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_population needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    for spec in args.shapes.split(","):
        K, n = (int(x) for x in spec.lower().split("x"))
        line = bench_shape(K, n, args.warmup, args.iters, not args.no_sequential)
        line.update(gpu=name, power_limit=power)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
