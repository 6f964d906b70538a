#!/usr/bin/env python
"""What saving the training state costs: one JSON line per workload, written to --out and printed.

Workloads: the bench-sized single run (CartPole-v1, 65,536 envs x 128 steps, 4 epochs x 4 minibatches, hidden 64 x 2) and the
README's 64 x 1,024 population (same T, epochs and minibatches).  For each:
  * state_bytes: the size of the state file;
  * save_ms: save_state() alone, host clock around a call followed by a device synchronise, --repeats calls (median, min, max),
    first with an empty episode history, then with the history of --history-iters iterations (T episodes per member and
    iteration: at these sizes CartPole logs one finished episode at every step); with that history also its parts: the
    device-to-host copies, the history lists turned into tensors, torch.save into memory, and the write + fsync of the bytes;
  * iteration ms without and with a save after every iteration, in alternating blocks of --iters iterations (host clock
    around synchronised iterations, as train() synchronises once per iteration to log), and the overhead of a save every
    iteration and every 10 iterations derived from the medians, all with that history.
The state files go to a temporary directory under --dir (default: the working directory, where train() writes them).  The
card's name and power limit are read in the same process and put on every line.
Usage: python tools/bench_training_state.py [--iters 5] [--blocks 4] [--repeats 7] [--history-iters 1000]
                                           [--out profiles/bench/training_state.jsonl]"""
import argparse
import io
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from aur_ppo_b200 import kernels, state  # noqa: E402
from aur_ppo_b200.population import ppo_population  # noqa: E402
from aur_ppo_b200.ppo import ppo  # noqa: E402
from tools.bench_population import card, params_for  # noqa: E402


def _single(n_iters):
    torch.manual_seed(1)
    p = ppo(params_for(65536, n_iters))
    p.envs.reset(seed=list(p.plan.env_ids))
    p._stats_rows = torch.zeros(p.num_update_epochs * p.num_minibatches, kernels.NUM_STATS, device=p.device)
    return p


def _population(n_iters):
    pop = ppo_population(params_for(1024, n_iters), [dict(seed=float(k + 1)) for k in range(64)])
    pop.reset_envs()
    return pop


def _fill_history(obj, n):
    """n episodes per member, as train() would have logged them: fp32 returns, lengths, increasing global steps."""
    rng = np.random.default_rng(0)
    lists = lambda: (rng.uniform(8, 500, n).astype(np.float32).tolist(), rng.integers(8, 500, n).tolist(),
                     (np.arange(n, dtype=np.int64) * 65536).tolist())
    if isinstance(obj, ppo):
        obj.total_returns, obj.total_episode_lengths, obj.x_indices = lists()
    else:
        per = [lists() for _ in range(obj.K)]
        obj.total_returns, obj.total_episode_lengths, obj.x_indices = ([p[j] for p in per] for j in range(3))


def _histories(obj):
    """(list, dtype) of every episode-history list save_state() stores."""
    groups = [(obj.total_returns, np.float64), (obj.total_episode_lengths, np.int64), (obj.x_indices, np.int64)]
    if isinstance(obj, ppo):
        return groups
    return [(h, dt) for lists, dt in groups for h in lists]


def _save_ms(obj, path, repeats):
    out = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        obj.save_state(path)
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return out


def bench(label, make, iters, blocks, repeats, history_iters, directory):
    obj = make(2 + 2 * blocks * iters + repeats)
    path = os.path.join(directory, f"{label}.pt")
    u = 0

    def iteration(save):
        nonlocal u
        u += 1
        out = obj.run_update(u)
        out["stats"].cpu()                    # the per-iteration host read of train()
        obj._iteration = u
        if save:
            obj.save_state(path)

    for _ in range(2):
        iteration(True)
    torch.cuda.synchronize()
    empty_ms = _save_ms(obj, path, repeats)
    empty_bytes = os.path.getsize(path)
    n_hist = history_iters * obj.buffer.rewards.shape[0]
    _fill_history(obj, n_hist)
    save_ms = _save_ms(obj, path, repeats)
    # where a save's time goes: device-to-host copies, history lists to tensors, torch.save into memory, write + fsync
    parts = {"d2h": [], "history": [], "serialise": [], "write_fsync": []}
    for _ in range(repeats):
        t0 = time.perf_counter()
        host = dict(tensors=state.to_host(obj._state_tensors()), env=state.to_host(state.env_tensors(obj.envs)))
        t1 = time.perf_counter()
        host["history"] = [state.history(h, dt) for h, dt in _histories(obj)]
        t2 = time.perf_counter()
        buf = io.BytesIO()
        torch.save(host, buf)
        t3 = time.perf_counter()
        with open(path + ".parts", "wb") as f:
            f.write(buf.getbuffer())
            f.flush()
            os.fsync(f.fileno())
        t4 = time.perf_counter()
        for key, dt in zip(parts, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            parts[key].append(dt * 1e3)
    os.remove(path + ".parts")
    times = {False: [], True: []}
    for b in range(2 * blocks):
        save = bool(b % 2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            iteration(save)
        torch.cuda.synchronize()
        times[save].append((time.perf_counter() - t0) * 1e3 / iters)
    off, on = statistics.median(times[False]), statistics.median(times[True])
    save_med = statistics.median(save_ms)
    line = dict(workload=label, state_bytes_no_history=empty_bytes, save_ms_no_history_median=round(statistics.median(empty_ms), 3),
                history_iters=history_iters, history_episodes_per_member=n_hist,
                state_bytes=os.path.getsize(path), save_ms_median=round(save_med, 3),
                save_ms_min=round(min(save_ms), 3), save_ms_max=round(max(save_ms), 3),
                **{f"{key}_ms_median": round(statistics.median(v), 3) for key, v in parts.items()},
                iter_ms_no_save=[round(t, 3) for t in times[False]], iter_ms_save_every_iter=[round(t, 3) for t in times[True]],
                iter_ms_no_save_median=round(off, 3), iter_ms_save_every_iter_median=round(on, 3),
                overhead_pct_save_every_iter=round(100 * (on / off - 1), 2),
                overhead_pct_save_every_10_iters=round(100 * save_med / (10 * off), 3))
    del obj
    torch.cuda.empty_cache()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5, help="iterations per timed block")
    ap.add_argument("--blocks", type=int, default=4, help="blocks per mode (without / with saving, alternating)")
    ap.add_argument("--repeats", type=int, default=7, help="timed save_state() calls")
    ap.add_argument("--history-iters", type=int, default=1000, help="iterations of episode history in the measured state")
    ap.add_argument("--dir", default=".", help="directory under which the state files go (a temporary subdirectory)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench", "training_state.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_training_state needs a CUDA device")
    torch.cuda.set_device(0)
    name, power = card()
    lines = []
    with tempfile.TemporaryDirectory(dir=args.dir) as d:
        for label, make in (("single_cartpole_65536x128", _single), ("population_64x1024x128", _population)):
            lines.append(bench(label, make, args.iters, args.blocks, args.repeats, args.history_iters, d))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for line in lines:
            line.update(gpu=name, power_limit=power)
            f.write(json.dumps(line) + "\n")
            print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
