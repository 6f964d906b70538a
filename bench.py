#!/usr/bin/env python
"""Benchmarks of the PPO hot path, one JSON line per run.

  python bench.py --gpus N --steps K --warmup W                  # headline: BASELINE configs[1]
  python bench.py --workload pendulum|scale1m|equiv|cnn ...      # configs[2], configs[4], configs[3], its plain-CNN sibling
  python bench.py --impl reference [--workload ...] ...          # the reference's CPU path (oracle port), bounded sample
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs as DIR/<name>.npy

Workloads (SURVEY.md section 8, sizes per BASELINE.json):
  ppo       CartPole-v1, 65536 envs PER GPU (weak scaling), T = 128, 4 minibatches x 4 epochs           configs[1]
  pendulum  Pendulum-v1 + the 5 wrappers, 65536 envs PER GPU, T = 256, the reference's continuous
            override (run_ppo.py:44-51): 32 minibatches x 10 epochs, lr 3e-4, entropy 0                  configs[2]
  scale1m   CartPole-v1, 1,048,576 envs IN TOTAL sharded over the GPUs (strong scaling), T = 128,
            plus a GAE sweep T = 128..2048 on 131072 columns per GPU                                      configs[4]
  equiv     equivariant actor-critic update, minibatch 4096 (--precision fp32|split|bf16)                      configs[3]
A step = one PPO iteration: T * num_envs env steps (fused rollout), one GAE pass and
epochs * num_minibatches fused updates.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env_steps_per_s"
UNIT = "env-steps/s"
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # nominal: 148 SMs x 128 FMA lanes x 2 flop x max SM clock (context, not a measured roofline)
CPU_SAMPLE_ENVS = {"ppo": 1024, "pendulum": 256, "scale1m": 1024}   # the CPU arm steps a bounded sample of the workload (see reference_arm_note)
if os.environ.get("AUR_BENCH_CPU_ENVS"):                              # tests shrink the sample (tests/test_bench_contract.py)
    CPU_SAMPLE_ENVS = {k: int(os.environ["AUR_BENCH_CPU_ENVS"]) for k in CPU_SAMPLE_ENVS}

WORKLOADS = {
    "ppo": dict(gym_id="CartPole-v1", continuous=False, T=128, nm=4, epochs=4, envs_per_gpu=65536, total_envs=None,
                lr=2.5e-4, ent=0.01, obs=4, act=2, baseline="BASELINE configs[1]", scaling="weak"),
    "pendulum": dict(gym_id="Pendulum-v1", continuous=True, T=256, nm=32, epochs=10, envs_per_gpu=65536, total_envs=None,
                     lr=3e-4, ent=0.0, obs=3, act=1, baseline="BASELINE configs[2]", scaling="weak"),
    "scale1m": dict(gym_id="CartPole-v1", continuous=False, T=128, nm=4, epochs=4, envs_per_gpu=None, total_envs=1048576,
                    lr=2.5e-4, ent=0.01, obs=4, act=2, baseline="BASELINE configs[4]", scaling="strong"),
}
GAE_SWEEP_T = (128, 256, 512, 1024, 2048)
GAE_SWEEP_COLS = 131072                              # config E at 8 GPUs: 1M / 8 columns per GPU


def num_envs_for(w, n_gpus):
    return w["total_envs"] if w["total_envs"] else w["envs_per_gpu"] * n_gpus


# --dump-outputs: a larger output is written as a fixed sample, so that the whole dump stays small (well under 64 MB)
DUMP_COLUMNS = 2048            # env columns of the [T, N, ...] rollout / GAE arrays
DUMP_ELEMENTS = 1 << 20        # elements of any other array


def seeded_sample(n, k):
    """k of range(n), sorted; the same for every run and build (seed 0)."""
    import torch
    if n <= k:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy: float64 stays float64, every other dtype becomes float32."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_ELEMENTS:
            t = t.reshape(-1)[seeded_sample(t.numel(), DUMP_ELEMENTS).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy())


HIDDEN = 64        # --hidden_dim (src/run_ppo.py:36): 64 is the reference default and every BASELINE config; 128 / 256 run the wide kernels


def mlp_flops_fwd(w, hidden=None):
    """fp32 FLOPs of one actor + critic forward per sample (2 x multiply-adds)."""
    hidden = hidden or HIDDEN
    o, a = w["obs"], w["act"]
    return 2 * (o * hidden + hidden * hidden + hidden * a) + 2 * (o * hidden + hidden * hidden + hidden)


def workload_config(name, n_gpus):
    w = WORKLOADS[name]
    n_envs = num_envs_for(w, n_gpus)
    return {"workload": f"{w['gym_id']} PPO iteration: fused rollout + GAE + update ({w['baseline']})",
            "name": name, "num_envs_per_gpu": n_envs // n_gpus, "num_envs": n_envs, "num_steps": w["T"],
            "num_minibatches": w["nm"], "update_epochs": w["epochs"], "hidden_dim": HIDDEN, "num_layers": 2,
            "continuous": w["continuous"], "wrappers": w["continuous"],
            "parallelism": f"dp{n_gpus} (env columns sharded; per minibatch one packed [grads|stats] exchange done by the "
                           f"update kernels over NVLink peer memory, AUR_DP_EXCHANGE=nccl selects a library all-reduce)",
            "l2": "working set per iteration >> 126 MB L2 (no explicit flush needed); the GAE sweep flushes L2 between launches",
            "reference_arm_note": f"the CPU arm (--impl reference and cpu_baseline) steps a BOUNDED SAMPLE of this workload: "
                                  f"num_envs={CPU_SAMPLE_ENVS[name]} x T={w['T']}, same minibatch count and epochs (a serial Python env "
                                  f"loop is ~flat in env-steps/s over num_envs; see cpu_points for num_envs 4 and 1024)"}


def params(name, n_gpus, total_iters):
    w = WORKLOADS[name]
    n = num_envs_for(w, n_gpus)
    return {'gym_id': w["gym_id"], 'seed': 1.0, 'num_steps': w["T"], 'gae': True,
            'total_timesteps': n * w["T"] * max(total_iters, 1), 'anneal_lr': True, 'gae_lambda': 0.95,
            'num_update_epochs': w["epochs"], 'num_envs': n, 'num_minibatches': w["nm"], 'entropy_coeff': w["ent"],
            'value_coeff': 0.5, 'clip_coeff': 0.2, 'clip_vloss': True, 'max_grad_norm': 0.5, 'target_kl': None,
            'norm_adv': True, 'capture_video': False, 'hidden_dim': HIDDEN, 'continuous': w["continuous"],
            'learning_rate': w["lr"], 'exp_name': 'bench', 'num_layers': 2, 'dropout': 0.0, 'gamma': 0.99, 'track': False,
            'tensorboard': False, 'save': False}


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons during the timed region (NVML)."""

    def __init__(self, index=0, period=0.1):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz = index, period, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# --------------------------------------------------------------------- reference arm (CPU)
def host_threads():
    """All the host threads torch may use, set explicitly (torchrun exports OMP_NUM_THREADS=1)."""
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    torch.set_num_threads(max(n, 1))
    return torch.get_num_threads()


def cpu_reference_iteration(name, num_envs, iters, warmup, seed=1):
    """The reference's CPU path restated (oracle/): gym-style SyncVectorEnv of per-env Python objects
    stepped serially (with the continuous wrapper stack of ppo.py:92-97 when the workload has it), reference
    actor_critic math on torch CPU, run_gae loop, update loop with Adam.
    Returns (seconds per iteration, env steps per iteration)."""
    import numpy as np
    import torch
    from oracle import gym_restated as G
    from oracle import ppo_ref as R
    from tests.helpers import random_policy
    w = WORKLOADS[name]
    T, cont, O = w["T"], w["continuous"], w["obs"]
    torch.manual_seed(seed)
    np.random.seed(seed)
    pol, _ = random_policy(O, w["act"], HIDDEN, 2, cont, seed=seed)
    opt = R.RefAdam(pol.tensors(), lr=w["lr"], eps=1e-5)
    envs = G.SyncVectorEnv([G.make_env(w["gym_id"], cont) for _ in range(num_envs)], O)
    next_obs = torch.from_numpy(envs.reset(seed=list(range(num_envs)))[0])
    next_done = torch.zeros(num_envs)
    N = num_envs
    obs = torch.zeros(T, N, O); actions = torch.zeros(T, N, w["act"]) if cont else torch.zeros(T, N)
    logps = torch.zeros(T, N); rewards = torch.zeros(T, N); dones = torch.zeros(T, N); values = torch.zeros(T, N)
    batch = N * T
    mb = max(batch // w["nm"], 1)
    times, phases = [], []
    for it in range(warmup + iters):
        t0 = time.perf_counter()
        for t in range(T):                                   # ppo.py:201-205
            obs[t], dones[t] = next_obs, next_done
            with torch.no_grad():
                a, lp, _, v = pol.evaluate(next_obs)
            values[t], actions[t], logps[t] = v.flatten(), a, lp
            o, r, term, trunc, info = envs.step(a.numpy())
            rewards[t] = torch.tensor(r).view(-1)
            next_obs, next_done = torch.from_numpy(o), torch.from_numpy(term.astype(np.float32))
        t_r = time.perf_counter()
        with torch.no_grad():                                # ppo.py:159-166
            ret, adv = R.gae(rewards, values, dones, pol.value(next_obs), next_done, 0.99, 0.95)
        t_g = time.perf_counter()
        b = (obs.reshape(-1, O), actions.reshape(-1, w["act"]) if cont else actions.reshape(-1), logps.reshape(-1),
             adv.reshape(-1), ret.reshape(-1), values.reshape(-1))
        inds = np.arange(batch)
        for ep in range(w["epochs"]):                        # ppo.py:215-269
            np.random.shuffle(inds)
            for s in range(0, batch, mb):
                mi = torch.from_numpy(inds[s:s + mb])
                R.ppo_update_step(pol, opt, b[0][mi], b[1][mi], b[2][mi], b[3][mi], b[4][mi], b[5][mi], ent_c=w["ent"])
        t_u = time.perf_counter()
        times.append(t_u - t0)
        phases.append((t_r - t0, t_g - t_r, t_u - t_g))
    times, phases = times[warmup:], phases[warmup:]
    med = lambda i: sorted(p[i] for p in phases)[len(phases) // 2]
    CPU_PHASES[(name, num_envs)] = {"rollout_env_steps_per_s": N * T / med(0), "gae_GBps": (20 * T * N + 8 * N) / med(1) / 1e9,
                                    "update_samples_per_s": w["epochs"] * batch / med(2),
                                    "phase_ms_median": {"rollout": med(0) * 1e3, "gae": med(1) * 1e3, "update": med(2) * 1e3}}
    return sum(times) / len(times), N * T


CPU_PHASES = {}


def host_info():
    """BASELINE.md section 3: what is always printed with the CPU numbers."""
    import numpy as np
    import torch
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"cpu_model": model, "os_cpu_count": os.cpu_count(), "torch_num_threads": torch.get_num_threads(),
            "torch": torch.__version__, "numpy": np.__version__,
            "path": "2 (BASELINE.md section 3 fallback): oracle restatement of gym 0.26.2 + reference model math on torch CPU; gym "
                    "itself is not installed and not installable (profiles/r2_pip_gym_attempt.log)",
            "note": "env stepping is one Python loop on one core by construction (SyncVectorEnv); torch CPU ops use all threads"}


def cpu_sample_text(name, n, iters):
    w = WORKLOADS[name]
    return (f"oracle port of the reference CPU path (gym-style SyncVectorEnv of Python env objects"
            f"{' + ClipAction/NormalizeObservation/NormalizeReward wrappers' if w['continuous'] else ''} + torch CPU), "
            f"{w['gym_id']} num_envs={n} x T={w['T']}, {w['epochs']} epochs x {w['nm']} minibatches per step, {iters} timed "
            f"iterations; gym itself is not installed, so this is oracle/gym_restated.py + oracle/ppo_ref.py")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload in ("equiv", "cnn"):
        return run_reference_cnn(args)
    name = args.workload
    w = WORKLOADS[name]
    cores = host_threads()
    n = CPU_SAMPLE_ENVS[name]
    sec, steps = cpu_reference_iteration(name, n, args.steps, args.warmup)
    v = steps / sec
    # BASELINE.md section 3: the reference's own CPU-runnable case (configs[0], num_envs = 4) and one scaled point
    points = []
    if name == "ppo":
        for pn, it in ((4, 8), (n, 0)):
            if it:
                ps, pst = cpu_reference_iteration(name, pn, it, 2)
                points.append(dict({"num_envs": pn, "value": pst / ps, "unit": UNIT, "ms_per_iteration": ps * 1e3}, **CPU_PHASES[(name, pn)]))
            else:
                points.append(dict({"num_envs": pn, "value": v, "unit": UNIT, "ms_per_iteration": sec * 1e3}, **CPU_PHASES[(name, pn)]))
    sample = cpu_sample_text(name, n, args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": w["scaling"],
            "vs_baseline": None, "dtype": "f32 (MLP) / f64 (env state)", "data": "synthetic",
            "config": workload_config(name, args.gpus),
            "sampled": {"num_envs": n, "num_steps": w["T"], "env_steps_per_step": steps,
                        "note": "value = env-steps of the SAMPLE / its time; one CPU process whatever --gpus says"},
            "cpu_points": points, "cpu_phases": CPU_PHASES.get((name, n)), "host": host_info(),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_reference_cnn(args):
    """--impl reference for configs[3] / its sibling: the torch-CPU port of the update on a bounded minibatch."""
    plain = args.workload == "cnn"
    cores = host_threads()
    cb = cnn_cpu_baseline(plain, min_seconds=5.0 * max(args.steps, 1) / 10.0 + 5.0)
    line = {"impl": "reference", "metric": "update_samples_per_s", "value": cb["value"], "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 4096 / cb["value"] * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": equiv_config(plain),
            "cpu_baseline": dict(cb, cores=cores),
            "e2e": {"value": cb["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------ own arm
def gae_sweep(torch, kernels, dev, cols, hbm_peak):
    """GAE-only launches on synthetic [T, cols] inputs (SURVEY.md section 8d), L2 flushed before every launch,
    CUDA events around each launch -> one rooflines[] entry per T."""
    out = []
    g = torch.Generator(device=dev).manual_seed(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for T in GAE_SWEEP_T:
        rew = torch.rand(T, cols, generator=g, device=dev)
        val = torch.randn(T, cols, generator=g, device=dev)
        term = (torch.rand(T, cols, generator=g, device=dev) < 1.0 / 200).float()
        nv = torch.randn(cols, generator=g, device=dev)
        nd = torch.zeros(cols, device=dev)
        ret, adv = torch.empty_like(rew), torch.empty_like(rew)
        ts = []
        for i in range(3 + 10):
            flush.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            kernels.gae(rew, val, term, nv, nd, 0.99, 0.95, True, out=(ret, adv))
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        ms = ts[len(ts) // 2]
        nbytes = 20 * T * cols + 8 * cols
        gbps = nbytes / (ms * 1e-3) / 1e9
        out.append({"kernel": f"gae_bulk_kernel [T={T}, N={cols}] (cold L2)", "bound": "hbm", "achieved": gbps, "peak": hbm_peak,
                    "unit": "GB/s", "frac": gbps / hbm_peak, "traffic": None, "algorithmic_bytes": nbytes, "ms": ms})
        del rew, val, term, ret, adv
    return out


def run_ours(args):
    import math
    import torch
    import torch.distributed as dist
    from aur_ppo_b200 import _lib, kernels
    name = args.workload
    w = WORKLOADS[name]
    T, EPOCHS, NM = w["T"], w["epochs"], w["nm"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    from aur_ppo_b200.ppo import ppo
    n_gpus = world
    torch.manual_seed(1)            # the initial policy comes from torch's generator: every run starts from the same weights
    agent = ppo(params(name, n_gpus, args.steps + args.warmup))
    n_mb_iter = EPOCHS * math.ceil(agent.local_batch / agent.local_minibatch)
    agent._stats_rows = torch.zeros(n_mb_iter, 16, device=agent.device)
    id0 = agent.rank * agent.local_envs
    agent.envs.reset(seed=list(range(id0, id0 + agent.local_envs)))
    L = _lib.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value) with per-phase events
    upd = 0
    for _ in range(args.warmup):
        upd += 1
        agent.run_update(upd)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    L.aur_launch_count_reset()
    if agent.exchange is not None:
        agent.exchange.wait_stats(reset=True)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for k in range(args.steps):
        upd += 1
        agent.run_update(upd, events=ev[k])
    end.record()
    barrier()
    launches = int(L.aur_launch_count())
    wait_stats = None
    if agent.exchange is not None:                      # device-measured spin time on peers' flags inside the timed region
        ws_ = agent.exchange.wait_stats()
        wt = torch.tensor([ws_["adam_wall_wait_us"] / max(ws_["adam_launches"], 1),
                           ws_["moment_spin_us_sum"] / max(ws_["moment_spins"], 1)], device=agent.device, dtype=torch.float64)
        wmax, wmin = wt.clone(), wt.clone()
        dist.all_reduce(wmax, op=dist.ReduceOp.MAX); dist.all_reduce(wmin, op=dist.ReduceOp.MIN)
        wait_stats = {"rank0": ws_, "grad_wall_wait_us_per_minibatch_max_rank": float(wmax[0]),
                      "grad_wall_wait_us_per_minibatch_min_rank": float(wmin[0]),
                      "moment_spin_us_per_spinning_cta_max_rank": float(wmax[1]),
                      "what": "measured on the device (globaltimer, accumulated in the exchange area): wall time the clip + Adam kernel "
                              "of a minibatch stood still until every peer's gradient sums had arrived (the rank that arrives last "
                              "waits ~0, the others wait for it), and the spin time of the gradient kernels' CTAs on the moment flags "
                              "(only the first minibatch of an iteration can spin: the moments travel once per iteration)"}
    clocks = sampler.finish()
    if args.dump_outputs and rank == 0:             # the last timed iteration, before the e2e loop below moves the agent on
        b, cols = agent.buffer, seeded_sample(agent.local_envs, DUMP_COLUMNS).to(agent.device)
        dump_outputs(args.dump_outputs, {
            "params": agent.flat, "stats": agent._stats_rows, "obs": b.states[:, cols], "actions": b.actions[:, cols],
            "log_probs": b.log_probs[:, cols], "values": b.values[:, cols], "rewards": b.rewards[:, cols],
            "dones": b.terminals[:, cols], "next_value": b.next_value[cols], "returns": agent._returns[:, cols],
            "advantages": agent._advantages[:, cols]})
    ms_total = start.elapsed_time(end)
    t_roll = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
    t_gae = sum(e[1].elapsed_time(e[2]) for e in ev) / args.steps
    t_upd = sum(e[2].elapsed_time(e[3]) for e in ev) / args.steps
    tt = torch.tensor([ms_total, t_roll, t_gae, t_upd], device=agent.device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, t_roll, t_gae, t_upd = [float(x) for x in tt.cpu()]
    ms_per_step = ms_total / args.steps
    local_envs = agent.local_envs
    steps_per_iter = local_envs * n_gpus * T
    value = steps_per_iter / (ms_per_step * 1e-3)

    # ---- e2e through the public API with host buffers: every step uploads the policy parameters and
    # the learning rate from pinned host memory, runs ppo.run_update(), and reads back the updated
    # parameters, the per-minibatch statistics and the finished-episode log.
    P = agent.flat.numel()
    h_params = torch.empty(P, dtype=torch.float32).pin_memory()
    h_params.copy_(agent.flat.cpu())
    h_stats = torch.empty(agent._stats_rows.shape, dtype=torch.float32).pin_memory()
    barrier()
    d2h = 0
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for k in range(args.steps):
        upd += 1
        agent.flat.copy_(h_params, non_blocking=True)                 # H2D: parameters
        out = agent.run_update(min(upd, agent.num_updates))
        h_params.copy_(agent.flat, non_blocking=True)                 # D2H: updated parameters
        h_stats[:out["stats"].shape[0]].copy_(out["stats"], non_blocking=True)
        agent.envs.first_finished_episodes()                          # D2H: per-step first finished episode (syncs)
        d2h += 8 * T
    t1.record()
    barrier()
    e2e_ms = t0.elapsed_time(t1) / args.steps
    te = torch.tensor([e2e_ms], device=agent.device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.cpu()[0])
    e2e_value = steps_per_iter / (e2e_ms * 1e-3)
    h2d_bytes = P * 4
    d2h_bytes = P * 4 + h_stats.numel() * 4 + d2h // args.steps

    exchange_kind = "in-kernel all-reduce over NVLink peer memory" if agent.exchange is not None else ("nccl all_reduce" if world > 1 else "none")
    if agent.exchange is not None and agent.exchange.status() != 0:
        raise SystemExit("data-parallel exchange: a kernel timed out waiting for a peer rank")
    m = agent.local_minibatch
    dev = agent.device
    agent.close()
    del agent
    torch.cuda.empty_cache()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")
    sweep = []
    if name == "scale1m":                                             # every rank runs it (same work), rank 0 reports
        sweep = gae_sweep(torch, kernels, dev, GAE_SWEEP_COLS, hbm_peak)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    tensor_peak = next((float(peaks[k]) for k in ("bf16_tflops_sustained", "bf16_dense_tflops_sustained", "bf16_tflops")
                        if k in peaks), 1414.7)
    n_mb = n_mb_iter
    fwd = float(mlp_flops_fwd(w))
    upd_flops = 3.0 * fwd
    upd_samples_per_s = n_mb * m * n_gpus / (t_upd * 1e-3)
    roll_steps_per_s = steps_per_iter / (t_roll * 1e-3)
    gae_bytes = 20 * T * local_envs + 8 * local_envs
    gae_gbps = gae_bytes / (t_gae * 1e-3) / 1e9
    upd_gbps = 40.0 * m / (t_upd / n_mb * 1e-3) / 1e9
    upd_tflops = upd_flops * m / (t_upd / n_mb * 1e-3) / 1e12
    # DRAM bytes per launch from the committed `ncu --set full` capture of THIS round's binary (profiles/r2_traffic.json,
    # config-B shapes); null when the workload's shapes differ from the captured ones
    traffic, traffic_src = {}, None
    if name == "ppo" and HIDDEN == 64:
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            traffic, traffic_src = tj.get("dram_bytes_per_launch", {}), tj.get("source")
        except Exception:
            traffic = {}
    roll_bytes = 36.0 * local_envs * T
    rooflines = [
        {"kernel": "gae_bulk_kernel", "bound": "hbm", "achieved": gae_gbps, "peak": hbm_peak, "unit": "GB/s",
         "frac": gae_gbps / hbm_peak, "traffic": traffic.get("gae_bulk_kernel"), "algorithmic_bytes": gae_bytes,
         "ms": t_gae, "note": "inside the iteration: inputs were just written by the rollout (partly L2-resident)"},
        {"kernel": "rollout_tc_kernel + critic_values_tc_kernel", "bound": "hbm", "achieved": roll_bytes / (t_roll * 1e-3) / 1e9,
         "peak": hbm_peak, "unit": "GB/s", "frac": roll_bytes / (t_roll * 1e-3) / 1e9 / hbm_peak,
         "traffic": (traffic.get("rollout_tc_kernel", 0) + traffic.get("critic_values_tc_kernel", 0)) or None, "ms": t_roll,
         "fp32_tflops": fwd * local_envs * T / (t_roll * 1e-3) / 1e12,
         "fp32_frac_of_nominal": fwd * local_envs * T / (t_roll * 1e-3) / 1e12 / FP32_PEAK_TFLOPS},
        {"kernel": "ppo_grad_tc_kernel (+shuffle, moments, reduce, adam)", "bound": "tensor", "achieved": upd_tflops,
         "peak": tensor_peak, "unit": "TFLOP/s", "frac": upd_tflops / tensor_peak, "traffic": traffic.get("ppo_grad_tc_kernel"),
         "ms": t_upd / n_mb, "algorithmic_flops": upd_flops * m, "algorithmic_bytes": 40.0 * m,
         "hbm_GBps": upd_gbps, "hbm_frac": upd_gbps / hbm_peak,
         "fp32_equiv_frac_of_nominal_fp32": upd_tflops / FP32_PEAK_TFLOPS,
         "note": "compute side of the roofline (>1000 FLOP per gathered byte).  The 64x64 contractions run on tcgen05 as "
                 "bf16 two-term splits; achieved = ALGORITHMIC fwd+bwd FLOP per sample / time against the measured dense "
                 "bf16 peak.  ncu: the kernel is issue-bound on the per-sample SIMT work, see profiles/"},
    ] + sweep
    if HIDDEN != 64:      # the wide kernels (update_wide.cu; rollout_tc_kernel<ENV, 128> or, at 256, the layer-wise rollout of rollout_wide.cu)
        rooflines[2]["kernel"] = "layer-wise tensor-core update (update_wide.cu: wide_gemm128 / tc_gemm / tc_gemm_tn + SIMT layers)"
        rooflines[2]["note"] = ("hidden %d: every H x H contraction is a tcgen05 GEMM over two-plane bf16 operands, activations staged in "
                                "HBM per 262,144-sample sub-batch; achieved = ALGORITHMIC fwd+bwd FLOP per sample / time" % HIDDEN)
        rooflines[2].pop("algorithmic_bytes", None)
        if HIDDEN > 128:
            rooflines[1]["kernel"] = "layer-wise actor per step (rollout_wide.cu: rows_first / skinny_gemm / rows_head) + rollout_tc_kernel<ENV, 0> + value pass"
    dominant = max(rooflines[:3], key=lambda r: r["ms"] * (n_mb if "update" in r["kernel"] or r["kernel"].startswith("ppo_grad") else 1))
    roofline = {k: dominant[k] for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
    roofline["kernel"] = dominant["kernel"]
    roofline["peak_source"] = peak_src
    roofline["traffic_source"] = traffic_src
    for k in ("fp32_tflops", "fp32_frac_of_nominal", "hbm_GBps", "hbm_frac", "note"):
        if k in dominant:
            roofline[k] = dominant[k]

    cpu_baseline = None
    if n_gpus == 1 and not args.no_cpu_baseline:
        cores = host_threads()
        iters = 4 if name != "pendulum" else 2
        sec, steps = cpu_reference_iteration(name, CPU_SAMPLE_ENVS[name], iters, 1)
        cpu_baseline = {"value": steps / sec, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": cpu_sample_text(name, CPU_SAMPLE_ENVS[name], iters),
                        "phases": CPU_PHASES.get((name, CPU_SAMPLE_ENVS[name])), "host": host_info()}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "f32 (MLP, GAE, Adam) / f64 (env state)", "data": "synthetic", "config": workload_config(name, n_gpus),
            "rollout_env_steps_per_s": roll_steps_per_s, "update_samples_per_s": upd_samples_per_s,
            "gae_GBps": gae_gbps, "gae_frac_of_hbm_peak": gae_gbps / hbm_peak,
            "phase_ms": {"rollout": t_roll, "gae": t_gae, "update": t_upd},
            "roofline": roofline, "rooflines": rooflines, "cpu_baseline": cpu_baseline, "dp_exchange": exchange_kind,
            "dp_wait": wait_stats,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms,
                    "what": "per step: H2D policy parameters from pinned memory -> ppo.run_update() -> D2H updated "
                            "parameters, per-minibatch statistics, finished-episode log; env state stays in HBM"},
            "gpu_launches": launches, "clocks": clocks}
    if n_gpus == 1 and name == "ppo" and not args.no_extras:
        line["other_workloads"] = other_workloads(args)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_workloads(args):
    """The other BASELINE configs, measured in the SAME default run (N = 1 only) so that they are driver-run numbers too: each
    is this script in a child process (own CUDA context, the parent has released its memory) with a short step count; its
    JSON line is condensed into one entry.  The headline `value` is computed before any of this starts."""
    import subprocess
    runs = [("pendulum", ["--workload", "pendulum", "--steps", "3"]),
            ("scale1m", ["--workload", "scale1m", "--steps", "3"]),
            ("equiv_fp32", ["--workload", "equiv", "--precision", "fp32", "--steps", "3"]),
            ("equiv_bf16", ["--workload", "equiv", "--precision", "bf16", "--steps", "5"]),
            ("cnn_fp32", ["--workload", "cnn", "--precision", "fp32", "--steps", "3"]),
            ("ppo_hidden128", ["--workload", "ppo", "--hidden_dim", "128", "--steps", "3"])]
    out = {}
    for tag, extra in runs:
        t0 = time.perf_counter()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--gpus", "1", "--warmup", "3", "--no-cpu-baseline", "--no-extras"] + extra,
                               capture_output=True, text=True, timeout=420)
            d = json.loads(r.stdout.strip().splitlines()[-1])
            e = {k: d.get(k) for k in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "dtype", "precision", "scaling", "phase_ms",
                                       "rollout_env_steps_per_s", "update_samples_per_s", "gae_frac_of_hbm_peak", "gpu_launches", "clocks")
                 if d.get(k) is not None}
            e["workload"] = d["config"]["workload"]
            e["e2e"] = {k: d["e2e"].get(k) for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")}
            e["roofline"] = {k: d["roofline"].get(k) for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "issued_tflops") if k in d["roofline"]}
            if tag == "scale1m":
                e["gae_sweep"] = [{"kernel": x["kernel"], "GBps": x["achieved"], "frac": x["frac"], "ms": x["ms"]} for x in d.get("rooflines", [])[3:]]
            e["wall_s"] = round(time.perf_counter() - t0, 1)
            out[tag] = e
        except Exception as ex:      # never let a side measurement take the headline line down
            out[tag] = {"error": repr(ex)[:300]}
    return out


def equiv_config(plain):
    return {"workload": ("plain CNN actor-critic update (robot_actor_critic equivariant=False), minibatch 4096, obs "
                         "1x128x128 + gripper state (sibling of BASELINE configs[3])") if plain else
                        ("equivariant actor-critic update, minibatch 4096, obs 1x128x128 + gripper state "
                         "(BASELINE configs[3])"),
            "l2": "activations >> L2 per step",
            "reference_arm_note": "the CPU arm (--impl reference and cpu_baseline) runs the torch-CPU port of the same update "
                                  "on a BOUNDED minibatch (32 for the plain CNN, 8 for the equivariant model)"}


def run_equiv(args, plain: bool = False):
    """BASELINE configs[3]: equivariant actor-critic update on synthetic close_loop_block_picking-shaped
    observations (1x128x128 heightmap + gripper state), minibatch 4096.  One step = one full update
    (two encoders forward + loss + backward + clip + Adam).  plain=True: the sibling non-equivariant CNN
    (robot_actor_critic equivariant=False, SURVEY.md section 8(f) rank 3) on the same inputs."""
    import torch
    from aur_ppo_b200 import _lib, equiv, plain_cnn
    B = 4096
    torch.cuda.set_device(0)
    split = args.precision != "bf16"
    if plain:
        params = plain_cnn.init_params(seed=0)
    else:
        params = equiv.init_params(seed=0)
        for k in ("actor.head.psi_triv", "actor.head.psi_irrep", "critic.head2.w"):
            params[k].mul_(0.1)
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.rand(B, 1, 128, 128, generator=g, device="cuda") * 0.32
    state = (torch.rand(B, generator=g, device="cuda") > 0.5).float()
    action = torch.randn(B, 5, generator=g, device="cuda")
    adv, ret, vold = (torch.randn(B, generator=g, device="cuda") for _ in range(3))
    oldlp = torch.full((B,), -7.0, device="cuda")
    model = (plain_cnn.PlainActorCritic if plain else equiv.EquivActorCritic)(params, B, precision=args.precision)
    for _ in range(args.warmup):
        model.update(state, obs, action, oldlp, adv, ret, vold)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    L = _lib.lib()
    L.aur_launch_count_reset()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        st = model.update(state, obs, action, oldlp, adv, ret, vold)
    t1.record()
    torch.cuda.synchronize()
    launches = int(L.aur_launch_count())
    clocks = sampler.finish()
    if args.dump_outputs:                           # the last timed update, before the e2e loop below runs more of them
        dump_outputs(args.dump_outputs, {"params": model._flat["p"], "stats": st, "values": model.value, "log_probs": model.logp})
    ms = t0.elapsed_time(t1) / args.steps
    # e2e: observations, states, actions and targets uploaded from pinned host memory every step, stats read back
    # Two device buffer sets and a copy stream: the upload of step i+1 (269 MB of observations) runs while step i computes;
    # every step's inputs still cross PCIe inside the timed region and every step's statistics are read back.
    host = [t.cpu().pin_memory() for t in (obs, state, action, oldlp, adv, ret, vold)]
    dev = [[torch.empty_like(t) for t in (obs, state, action, oldlp, adv, ret, vold)] for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    free = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream()

    def upload(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(free[i & 1])
            for d, h in zip(dev[i & 1], host):
                d.copy_(h, non_blocking=True)
            ready[i & 1].record(copy_stream)
    for ev in free:
        ev.record(main)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    upload(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            upload(i + 1)
        main.wait_event(ready[i & 1])
        dv = dev[i & 1]
        st = model.update(dv[1], dv[0], dv[2], dv[3], dv[4], dv[5], dv[6])
        free[i & 1].record(main)
        st_host = st.cpu()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / args.steps
    h2d = sum(t.numel() * t.element_size() for t in host)
    # forward FLOPs per encoder and sample: equivariant 2.80e9 (SURVEY.md section 8a row X); plain CNN 2 * 9 * sum(cin * cout * H * W)
    # = 9.4 + 4 x 37.7 + 42.5 + 0.6 MFLOP = 2.034e8 (real channels; the padded contractions issue ~2.2x that in layers 0-2)
    flops = 3 * 2 * (2.034e8 if plain else 2.80e9) * B
    cpu_baseline = None
    if not args.no_cpu_baseline:
        cores = host_threads()
        cpu_baseline = dict(cnn_cpu_baseline(plain), cores=cores)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    tf = flops / (ms * 1e-3) / 1e12
    line = {"metric": "update_samples_per_s", "value": B / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "fp32-equivalent (the reference's precision): bf16x3 operand planes (hi + mid + lo = 24 mantissa bits), "
                              "six products on tcgen05, TMEM accumulation promoted into fp32 registers every 32 MMA steps; measured "
                              "~7e-7 per layer, gradients within 3e-5 of float64 on identical routing; fp32 parameters and Adam",
                      "split": "bf16x2 operand planes (hi + mid = 16 mantissa bits), three products, the same promotion: ~5e-6 per "
                               "layer, gradients within 1e-4 at well-conditioned points (the reference's fp32 convolutions run as "
                               "TF32, ~5e-4, under cuDNN's default); fp32 parameters and Adam",
                      "bf16": "bf16 operands / fp32 accumulate (tcgen05), fp32 parameters and Adam: BELOW the reference's fp32 "
                              "precision (fast mode)"}[args.precision],
            "data": "synthetic", "precision": args.precision,
            "config": dict(equiv_config(plain), precision=args.precision),
            "roofline": {"bound": "tensor", "achieved": tf, "peak": peak, "unit": "TFLOP/s", "frac": tf / peak, "traffic": None,
                         "issued_tflops": tf * {"fp32": 6.0, "split": 3.0, "bf16": 1.0}[args.precision],
                         "kernel": "conv_igemm_kernel + wgrad3x3_kernel (whole update, %.1f TFLOP algorithmic)" % (flops / 1e12),
                         "peak_source": "measured sustained bf16 (MEASURED_PEAKS.json)" if peaks else "fallback",
                         "note": ("channels 16 / 32 are padded to the 64-wide K chunk and layer 0 runs 4 rotated copies: the "
                                  "narrow layers are HBM / epilogue bound, see DESIGN.md section 4.8") if plain else None},
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": B / (e2e_ms * 1e-3), "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                    "ms_per_step": e2e_ms},
            "gpu_launches": launches, "clocks": clocks}
    print(json.dumps(line))


def cnn_cpu_baseline(plain=True, min_seconds=10.0):
    """The reference's CPU path for the CNN update restated (oracle/cnn_ref.py = base_actor / base_critic forward,
    oracle/equiv_ref.py = the restated equivariant model; robot_ppo.update loss, autograd backward, actor-only clip,
    torch Adam) on the host cores, bounded sample."""
    import torch
    if plain:
        from oracle import cnn_ref as C
        B = 32
        p = {k: v.clone().requires_grad_(True) for k, v in C.formula_params(C.param_shapes(), seed=0).items()}
    else:
        from oracle import equiv_ref as C
        B = 8
        p = {k: v.clone().requires_grad_(True) for k, v in C.init_params(seed=0).items()}
    opt = torch.optim.Adam(list(p.values()), lr=3e-4, eps=1e-5)
    g = torch.Generator().manual_seed(0)
    obs = torch.rand(B, 1, 128, 128, generator=g) * 0.32
    state = (torch.rand(B, generator=g) > 0.5).float()
    action = torch.randn(B, 5, generator=g)
    adv, ret, vold = (torch.randn(B, generator=g) for _ in range(3))
    oldlp = torch.full((B,), -7.0)

    def step():
        opt.zero_grad()
        loss, _ = C.update_loss(p, state, obs, action, oldlp, adv, ret, vold)
        loss.backward()
        torch.nn.utils.clip_grad_norm_([v for k, v in p.items() if k.startswith("actor.")], 0.5)
        opt.step()
    step()
    n, t0 = 0, time.perf_counter()
    while n < 3 or time.perf_counter() - t0 < min_seconds:
        step()
        n += 1
    dt = time.perf_counter() - t0
    return {"value": n * B / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"oracle port (torch CPU conv2d + autograd + Adam, fp32), minibatch {B} x {n} updates"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-extras", dest="no_extras", action="store_true",
                    help="default N = 1 run only: skip the short side measurements of the other BASELINE configs (other_workloads)")
    ap.add_argument("--workload", type=str, default="ppo", choices=["ppo", "pendulum", "scale1m", "equiv", "cnn"],
                    help="ppo = BASELINE configs[1] (default, the headline line); pendulum = configs[2]; scale1m = configs[4] "
                         "(1M envs over the GPUs + GAE sweep); equiv = configs[3]; cnn = its plain-CNN sibling")
    ap.add_argument("--precision", type=str, default="fp32", choices=["fp32", "split", "bf16"],
                    help="equiv / cnn: fp32 = three bf16 operand planes, fp32-equivalent like the reference (default); split = two "
                         "planes (~5e-6 per layer); bf16 = single-plane fast mode, below the reference's precision")
    ap.add_argument("--hidden_dim", type=int, default=64, choices=[64, 128, 256],
                    help="policy width of the MLP workloads (src/run_ppo.py:36); 64 is every BASELINE config, 128 / 256 exercise the wide kernels")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64; "
                         "large arrays as a fixed sample) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    global HIDDEN
    HIDDEN = args.hidden_dim
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload in ("equiv", "cnn"):
        run_equiv(args, plain=args.workload == "cnn")
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
