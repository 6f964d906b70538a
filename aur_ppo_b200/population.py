"""A population of K independent PPO runs trained in shared launches on one GPU.

The reference's results are seed and hyper-parameter sweeps (src/grid_search.sh, src/robot.sh; `--trials` is parsed and
ignored, src/run_ppo.py:41), each run a separate process.  `ppo_population(params, members)` trains K such runs at once:
every member has its own seed (initial weights, Philox sampling key, shuffle key) and its own learning rate, entropy / clip /
value coefficients, max_grad_norm and target_kl; everything else is shared.  Member k computes exactly -- bit for bit -- what
`ppo(params_k)` computes from the same initial weights with `philox_seed = shuffle_seed = seed_k` (include/aur_ppo.h,
"populations"), in the same number of kernel launches per iteration whatever K is:

  per iteration            one aur_pop_rollout, one aur_gae_f32, one aur_ppo_pack_records, one aur_pop_shuffle_indices,
                           one aur_pop_adv_moments_multi (all members, all minibatches)
  per minibatch            one aur_pop_update_grad (all members), one aur_pop_update_apply (all members)
  per PBT round (opt-in)   one aur_pop_episode_fitness, one aur_pop_pbt_step (two launches), between iterations

Population-based training (`pbt=dict(interval=...)`): every `interval` iterations the bottom `fraction` of the members (by the
mean return of the episodes they finished since the last round) copy the weights, Adam state and wrapper statistics of
members drawn from the top `fraction`, then multiply the copied hyper-parameters named in `keys` by one of `factors`
(include/aur_ppo.h, "population-based training").  With `pbt=None` nothing changes.

Layout: the rollout buffers are those of a single run of K * n_member envs; member k owns columns k * n_member ...
"""
from __future__ import annotations

import ctypes
import json
import math
import time
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib, compat, kernels, parallel
from .envs import DeviceVecEnv, pcg64_seed_states
from .models.actor_critic import actor_critic
from .ppo import _SPACES, torch_buffer
from .run_ppo import SWEEP_KEYS

# the keys a member may set; every other key of `params` is shared by the whole population
MEMBER_KEYS = ("seed", "learning_rate", "entropy_coeff", "clip_coeff", "value_coeff", "max_grad_norm", "target_kl")
POP_ENVS = ("CartPole-v1", "Pendulum-v1", "MountainCar-v0")
PBT_DEFAULTS = dict(fraction=0.25, keys=("learning_rate", "entropy_coeff"), factors=(0.8, 1.2))
ADAM_BETAS, ADAM_EPS = (0.9, 0.999), 1e-5


def member_params(params: Dict, member: Dict) -> Dict:
    """The standalone `ppo` params of one member: `params` with the member's overrides, sampling and shuffle keyed by its seed."""
    p = dict(params)
    p.update(member)
    p["philox_seed"] = p["shuffle_seed"] = int(p["seed"])
    return p


def check_members(params: Dict, members: Sequence[Dict]) -> List[Dict]:
    """Validate the member overrides (AurError on an empty population, a non-dict, or a shared key that differs)."""
    if not members:
        raise _lib.AurError("a population needs at least one member")
    out = []
    for k, m in enumerate(members):
        if not isinstance(m, dict):
            raise _lib.AurError(f"member {k}: expected a dict of overrides, got {type(m).__name__}")
        for key, v in m.items():
            if key not in MEMBER_KEYS and (key not in params or params[key] != v):
                raise _lib.AurError(f"member {k}: {key!r} is shared by the population (per-member keys: {', '.join(MEMBER_KEYS)})")
        out.append({key: v for key, v in m.items() if key in MEMBER_KEYS})
    return out


def check_pbt(pbt: Optional[Dict], K: int) -> Optional[Dict]:
    """Validate a PBT config (AurError) -> dict(interval, fraction, keys, factors, mask) with the defaults filled in."""
    if pbt is None:
        return None
    if not isinstance(pbt, dict):
        raise _lib.AurError(f"pbt: expected a dict, got {type(pbt).__name__}")
    unknown = set(pbt) - {"interval", *PBT_DEFAULTS}
    if unknown:
        raise _lib.AurError(f"pbt: unknown settings {sorted(unknown)} (interval, fraction, keys, factors)")
    cfg = dict(PBT_DEFAULTS, **pbt)
    if K < 2:
        raise _lib.AurError(f"pbt needs a population of at least two members (got {K})")
    interval = cfg.get("interval")
    if isinstance(interval, bool) or not isinstance(interval, int) or interval < 1:
        raise _lib.AurError(f"pbt interval must be an integer >= 1 (got {interval!r})")
    q = cfg["fraction"]
    if isinstance(q, bool) or not isinstance(q, (int, float)) or not 0.0 < q <= 0.5:
        raise _lib.AurError(f"pbt fraction must be in (0, 0.5] (got {q!r})")
    keys = (cfg["keys"],) if isinstance(cfg["keys"], str) else tuple(cfg["keys"])
    bad = [k for k in keys if k not in SWEEP_KEYS]
    if bad:
        raise _lib.AurError(f"pbt keys {bad} are not hyper-parameters a member has (one of {', '.join(SWEEP_KEYS)})")
    try:
        down, up = (float(v) for v in cfg["factors"])
    except (TypeError, ValueError):
        raise _lib.AurError(f"pbt factors must be two numbers (got {cfg['factors']!r})")
    if not all(math.isfinite(v) and v > 0 for v in (down, up)):
        raise _lib.AurError(f"pbt factors must be finite and > 0 (got {down}, {up})")
    return dict(interval=interval, fraction=float(q), keys=keys, factors=(down, up),
                mask=sum(1 << SWEEP_KEYS.index(k) for k in set(keys)))


def _bind_flat(policy: actor_critic, row: torch.Tensor) -> None:
    """Make every parameter of `policy` a view of `row` (the flat_parameters() order) after copying its values there."""
    flat = policy.flat_parameters()
    row.copy_(flat)
    offs = policy._flat_offsets
    for p, o in zip(policy._ordered_parameters(), offs):
        p.data = row[o:o + p.numel()].view_as(p)
    object.__setattr__(policy, "_flat", row)


class ppo_population:
    def __init__(self, params: Dict, members: Sequence[Dict], pbt: Optional[Dict] = None):
        self.params_dict = params
        self.members = check_members(params, members)
        self.member_params = [member_params(params, m) for m in self.members]
        self.K = K = len(self.members)
        self.pbt = check_pbt(pbt, K)
        for key in ("gym_id", "num_envs", "num_steps", "num_minibatches", "num_update_epochs", "gamma", "gae_lambda", "gae",
                    "norm_adv", "clip_vloss", "anneal_lr", "total_timesteps", "hidden_dim", "num_layers", "continuous", "exp_name"):
            setattr(self, key, params[key])
        if torch.distributed.is_available() and torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
            raise _lib.AurError("populations run on one GPU (world_size > 1 is not supported)")
        try:
            plan = parallel.current_plan(self.num_envs, self.num_steps, self.num_minibatches)
        except ValueError as e:
            raise _lib.AurError(str(e))
        if plan.world_size > 1:
            raise _lib.AurError("populations run on one GPU (world_size > 1 is not supported)")
        if self.gym_id not in POP_ENVS:
            raise _lib.AurError(f"gym_id {self.gym_id!r} has no population kernel (supported: {', '.join(POP_ENVS)}); no fallback")
        sp = _SPACES[self.gym_id]
        if bool(self.continuous) != (sp["n"] is None):
            raise _lib.AurError(f"{self.gym_id} is {'continuous' if sp['n'] is None else 'discrete'}; got continuous={self.continuous}")
        if int(self.hidden_dim) != 64 or int(self.num_layers) != 2:
            raise _lib.AurError(f"populations run the 64 x 2 tensor-core kernels; got hidden_dim {self.hidden_dim}, "
                                f"num_layers {self.num_layers} (no fallback)")
        self.n_member = int(self.num_envs)
        self.batch_size = self.n_member * int(self.num_steps)
        self.minibatch_size = self.batch_size // int(self.num_minibatches)
        self.num_updates = int(self.total_timesteps) // self.batch_size
        self.per_epoch = self.batch_size // max(self.minibatch_size, 1)
        self.n_mb = int(self.num_update_epochs) * self.per_epoch
        if self.minibatch_size < 1 or self.batch_size % self.minibatch_size or not 1 <= self.n_mb <= kernels.Updater.MAX_MINIBATCHES:
            raise _lib.AurError(f"populations need num_envs * num_steps divisible into whole minibatches and at most "
                                f"{kernels.Updater.MAX_MINIBATCHES} minibatches per iteration (got batch {self.batch_size}, "
                                f"minibatch {self.minibatch_size}, {self.n_mb} minibatches)")
        if K * self.batch_size >= 2 ** 31:
            raise _lib.AurError(f"K * num_envs * num_steps must be < 2^31 (got {K * self.batch_size})")
        if not torch.cuda.is_available():
            raise _lib.AurError("aur_ppo_b200.population needs a CUDA device: the hot path has no CPU fallback")
        _lib.lib()
        self.device = torch.device(params.get("device", f"cuda:{torch.cuda.current_device()}"))
        dev = self.device
        self.run_name = f"{self.gym_id}__{self.exp_name}__{params['seed']}__{int(time.time())}"

        # ---- members' policies: torch.manual_seed(seed_k) before each actor_critic is built; parameters are rows of [K][P]
        self.state_dim = sp["obs"]
        self.action_dim = sp["act_shape"] if self.continuous else sp["n"]
        self.policies: List[actor_critic] = []
        for mp in self.member_params:
            torch.manual_seed(int(mp["seed"]))
            with torch.cuda.device(dev):
                self.policies.append(actor_critic(self.state_dim[0], self.action_dim, 64, 2, params.get("dropout", 0.0),
                                                  self.continuous).to(dev))
        self.desc = kernels.policy_desc(*self.policies[0].kernel_shape())
        self.P = kernels.policy_param_count(self.desc)
        self.params = torch.empty(K, self.P, dtype=torch.float32, device=dev)
        for k, pol in enumerate(self.policies):
            _bind_flat(pol, self.params[k])
        self.exp_avg = torch.zeros(K, self.P, device=dev)
        self.exp_avg_sq = torch.zeros(K, self.P, device=dev)
        self.grads = torch.zeros(K, self.P + kernels.NUM_STATS, device=dev)
        self.steps = torch.zeros(K, dtype=torch.int64, device=dev)
        self.active = torch.ones(K, dtype=torch.int32, device=dev)
        # hyper-parameter table, written once; target_kl None = +inf (never stops early)
        hp = np.zeros((K, 6), dtype=np.float64)
        for k, mp in enumerate(self.member_params):
            tkl = mp.get("target_kl")
            hp[k] = (mp["learning_rate"], mp["entropy_coeff"], mp["clip_coeff"], mp["value_coeff"], mp["max_grad_norm"],
                     math.inf if tkl is None else float(tkl))
        self.hparams = torch.from_numpy(hp).to(dev)
        self.any_target_kl = any(mp.get("target_kl") is not None for mp in self.member_params)
        seeds = np.array([int(mp["seed"]) & 0xFFFFFFFFFFFFFFFF for mp in self.member_params], dtype=np.uint64)
        self.seeds = torch.from_numpy(seeds.view(np.int64)).to(dev)          # uint64 keys, stored as their int64 bit patterns
        self.pop = _lib.PopDesc(K, 0, self.n_member, self.seeds.data_ptr())
        self.bias_corr = None
        self._iterations = 0
        self._ensure_bias_corr(self.num_updates * self.n_mb + 1)

        # ---- envs, buffers, workspace
        self.envs = DeviceVecEnv(self.gym_id, K * self.n_member, wrappers=bool(self.continuous), device=dev)
        self.buffer = torch_buffer(self.state_dim, sp["act_shape"], self.num_steps, K * self.n_member, dev)
        self._returns = torch.empty_like(self.buffer.rewards)
        self._advantages = torch.empty_like(self.buffer.rewards)
        self._records = None
        self._b_inds = torch.empty(K, self.n_mb, self.minibatch_size, dtype=torch.int32, device=dev)
        self.moments = torch.zeros(K, self.n_mb, 3, dtype=torch.float64, device=dev)
        ws = int(_lib.lib().aur_pop_update_workspace_bytes(ctypes.byref(self.pop), ctypes.byref(self.desc), self.n_mb,
                                                           self.minibatch_size))
        if ws < 0:
            _lib.check(ws, "aur_pop_update_workspace_bytes")
        self.workspace = torch.empty((ws + 3) // 4, dtype=torch.float32, device=dev)
        self.first_finished = torch.empty(K, int(self.num_steps), dtype=torch.int64, device=dev)
        self.totals = torch.zeros(K, 3, dtype=torch.float64, device=dev)
        self._stats_rows = torch.zeros(K, self.n_mb, kernels.NUM_STATS, device=dev)
        self.rows_done = [0] * K
        self._shuffle_count = 0
        self._env_step = 0
        self.total_returns: List[List[float]] = [[] for _ in range(K)]
        self.total_episode_lengths: List[List[int]] = [[] for _ in range(K)]
        self.x_indices: List[List[int]] = [[] for _ in range(K)]
        # PBT: the fitness snapshot of the episode totals, the round's outputs and the history of rounds
        self.pbt_round = 0
        self.lineage: List[Dict] = []
        if self.pbt is not None:
            self.pbt_snapshot = torch.zeros(K, 3, dtype=torch.float64, device=dev)
            self.pbt_fitness = torch.empty(K, dtype=torch.float64, device=dev)
            self.pbt_rank = torch.empty(K, dtype=torch.int32, device=dev)
            self.pbt_donor = torch.empty(K, dtype=torch.int32, device=dev)
            self.pbt_order = torch.empty(K + 1, dtype=torch.int32, device=dev)

    def _ensure_bias_corr(self, max_step: int) -> None:
        """Adam bias corrections 1 - beta^s for s = 0 .. max_step (aur_pop_update_apply reads entry steps[k] + 1, which must exist),
        computed with the host pow the single-run aur_ppo_update_apply uses (math.pow is the C library's pow).  Grows the table
        when a caller runs more iterations than num_updates."""
        have = 0 if self.bias_corr is None else self.bias_corr.shape[0]
        if max_step < have:
            return
        n = max(max_step + 1, 2 * have)
        bc = np.empty((n, 2), dtype=np.float64)
        for s in range(n):
            bc[s, 0] = 1.0 - math.pow(ADAM_BETAS[0], float(s))
            bc[s, 1] = 1.0 - math.pow(ADAM_BETAS[1], float(s))
        self.bias_corr = torch.from_numpy(bc).to(self.device)

    # ------------------------------------------------------------------ hot path pieces
    def reset_envs(self) -> None:
        """envs.reset(seed=[...]) of every member (src/ppo.py:188): member k's env n is seeded n, as a single run seeds it."""
        n, K = self.n_member, self.K
        st = pcg64_seed_states(range(n))
        self.envs.pcg.copy_(torch.from_numpy(np.tile(st, (1, K)).view(np.int64)))
        with torch.cuda.device(self.device):
            es = self.envs.state_struct()
            rc = _lib.lib().aur_env_reset(self.envs.kind, K * n, int(self.envs.wrappers), ctypes.byref(es),
                                          self.envs.next_obs.data_ptr(), self.envs.next_done.data_ptr(), kernels._stream())
        _lib.check(rc, "aur_env_reset")
        self._env_step = 0

    def rollout(self) -> None:
        T, N = self.buffer.rewards.shape
        b, env = self.buffer, self.envs
        a = _lib.RolloutArgs()
        a.env_kind, a.wrappers, a.N, a.T = env.kind, int(env.wrappers), N, T
        a.policy = self.desc
        a.params = self.params.data_ptr()
        a.env = env.state_struct()
        a.obs_buf, a.act_buf, a.logp_buf = b.states.data_ptr(), b.actions.data_ptr(), b.log_probs.data_ptr()
        a.val_buf, a.rew_buf, a.done_buf = b.values.data_ptr(), b.rewards.data_ptr(), b.terminals.data_ptr()
        a.next_obs, a.next_done, a.next_value = env.next_obs.data_ptr(), env.next_done.data_ptr(), b.next_value.data_ptr()
        a.seed, a.step0, a.env_id0 = 0, self._env_step, 0
        self.first_finished.fill_(-1)
        a.log = _lib.EpisodeLog(None, None, 0, 0, self.first_finished.data_ptr(), self.totals.data_ptr())
        a.gamma = env.gamma
        with torch.cuda.device(self.device):
            rc = _lib.lib().aur_pop_rollout(ctypes.byref(self.pop), ctypes.byref(a), kernels._stream())
        _lib.check(rc, "aur_pop_rollout")
        self._env_step += T

    def run_update(self, update: int, events=None) -> Dict[str, torch.Tensor]:
        """One iteration of every member (ppo.run_update); returns device tensors: stats [K][n_mb][16] (member k's first
        rows_done[k] rows are its minibatches), b_values / b_returns [T * K * n_member].
        events: optional 4 CUDA events recorded at the phase boundaries (start, rollout done, GAE done, update done)."""
        L = _lib.lib()
        st = kernels._stream()
        rec = (lambda i: events[i].record()) if events is not None else (lambda i: None)
        frac = 1.0 - (update - 1.0) / self.num_updates if self.anneal_lr else 1.0
        self.lr_frac = frac
        self._iterations += 1
        self._ensure_bias_corr(self._iterations * self.n_mb)     # no member can step more often than every minibatch
        rec(0)
        self.rollout()
        rec(1)
        ret, adv = kernels.gae(self.buffer.rewards, self.buffer.values, self.buffer.terminals, self.buffer.next_value,
                               self.envs.next_done, self.gamma, self.gae_lambda, bool(self.gae), out=(self._returns, self._advantages))
        rec(2)
        flat = self.buffer.flatten(ret, adv)
        self._records = kernels.pack_records(*[flat[i] for i in (0, 2, 1, 3, 4, 5)], out=self._records)
        E, m = int(self.num_update_epochs), self.minibatch_size
        with torch.cuda.device(self.device):
            _lib.check(L.aur_pop_shuffle_indices(ctypes.byref(self.pop), int(self.num_steps), E, self._shuffle_count,
                                                 self._b_inds.data_ptr(), st), "aur_pop_shuffle_indices")
            self._shuffle_count += E
            if self.norm_adv:
                _lib.check(L.aur_pop_adv_moments_multi(ctypes.byref(self.pop), self.n_mb, m, self._b_inds.data_ptr(),
                                                       flat[3].data_ptr(), self.moments.data_ptr(), self.workspace.data_ptr(), st),
                           "aur_pop_adv_moments_multi")
            self.active.fill_(1)
            u = _lib.PopUpdateArgs()
            u.policy, u.norm_adv, u.clip_vloss, u.n_mb, u.m = self.desc, int(bool(self.norm_adv)), int(bool(self.clip_vloss)), self.n_mb, m
            u.idx, u.rec_actor, u.rec_critic = self._b_inds.data_ptr(), self._records[0].data_ptr(), self._records[1].data_ptr()
            u.params, u.hparams, u.active = self.params.data_ptr(), self.hparams.data_ptr(), self.active.data_ptr()
            u.adv_moments = self.moments.data_ptr() if self.norm_adv else None
            u.workspace, u.grads_out = self.workspace.data_ptr(), self.grads.data_ptr()
            rows = [0] * self.K
            live = np.ones(self.K, dtype=bool)
            j = 0
            for ep in range(E):
                for i in range(self.per_epoch):
                    u.mb_index = j
                    _lib.check(L.aur_pop_update_grad(ctypes.byref(self.pop), ctypes.byref(u), st), "aur_pop_update_grad")
                    _lib.check(L.aur_pop_update_apply(ctypes.byref(self.pop), ctypes.byref(self.desc), self.hparams.data_ptr(),
                                                      self.params.data_ptr(), self.grads.data_ptr(), self.exp_avg.data_ptr(),
                                                      self.exp_avg_sq.data_ptr(), self.steps.data_ptr(), self.active.data_ptr(),
                                                      self.bias_corr.data_ptr(), self.bias_corr.shape[0], frac, ADAM_BETAS[0],
                                                      ADAM_BETAS[1], ADAM_EPS, m, self._stats_rows.data_ptr(), self.n_mb, j,
                                                      int(self.any_target_kl and i == self.per_epoch - 1), st),
                               "aur_pop_update_apply")
                    j += 1
                for k in np.nonzero(live)[0]:
                    rows[k] += self.per_epoch
                if self.any_target_kl:
                    live = self.active.cpu().numpy() != 0       # one read per epoch: the single run's `.item()` (ppo.py:271)
                    if not live.any():
                        break
        self.rows_done = rows
        rec(3)
        return dict(stats=self._stats_rows, b_values=flat[5], b_returns=flat[4])

    def pbt_step(self, fitness: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """One PBT round between iterations (three launches): fitness (aur_pop_episode_fitness, the mean return of each member's
        episodes since the previous round) unless a [K] fp64 device tensor is given, then rank + exploit / explore
        (aur_pop_pbt_step) keyed by the population's seed and the round number.  Returns device tensors donor [K] int32 (-1:
        kept its own state), fitness [K] fp64 and rank [K] int32."""
        if self.pbt is None:
            raise _lib.AurError("pbt_step: this population was built without a pbt config")
        cfg = self.pbt
        L = _lib.lib()
        st = kernels._stream()
        with torch.cuda.device(self.device):
            if fitness is None:
                _lib.check(L.aur_pop_episode_fitness(ctypes.byref(self.pop), self.totals.data_ptr(), self.pbt_snapshot.data_ptr(),
                                                     self.pbt_fitness.data_ptr(), st), "aur_pop_episode_fitness")
                fitness = self.pbt_fitness
            elif fitness.dtype != torch.float64 or fitness.shape != (self.K,) or fitness.device != self.device:
                raise _lib.AurError(f"pbt_step: fitness must be a [{self.K}] float64 tensor on {self.device}")
            fitness = fitness.contiguous()
            self.pbt_round += 1
            a = _lib.PopPbtArgs()
            a.fitness = fitness.data_ptr()
            a.q, (a.down, a.up), a.mask = cfg["fraction"], cfg["factors"], cfg["mask"]
            a.seed, a.round = int(self.params_dict["seed"]) & 0xFFFFFFFFFFFFFFFF, self.pbt_round
            a.params, a.adam_m, a.adam_v = self.params.data_ptr(), self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr()
            a.steps, a.hparams = self.steps.data_ptr(), self.hparams.data_ptr()
            a.norm = self.envs.norm.data_ptr() if self.envs.norm is not None else None
            a.norm_ld = self.K * self.n_member
            a.rank_out, a.donor_out, a.order = self.pbt_rank.data_ptr(), self.pbt_donor.data_ptr(), self.pbt_order.data_ptr()
            _lib.check(L.aur_pop_pbt_step(ctypes.byref(self.pop), ctypes.byref(self.desc), ctypes.byref(a), st), "aur_pop_pbt_step")
        return dict(donor=self.pbt_donor, fitness=fitness, rank=self.pbt_rank)

    def _record_round(self, iteration: int, out: Dict[str, torch.Tensor]) -> Dict:
        """Read a round's donors, fitness and hyper-parameter table back once; update member_params and the lineage."""
        donor = out["donor"].cpu().numpy()
        fitness = out["fitness"].cpu().numpy()
        hp = self.hparams.cpu().numpy()
        for k, mp in enumerate(self.member_params):
            mp.update({key: float(hp[k, j]) for j, key in enumerate(SWEEP_KEYS)})
            if math.isinf(mp["target_kl"]):
                mp["target_kl"] = None
        self.any_target_kl = any(mp["target_kl"] is not None for mp in self.member_params)
        entry = dict(iteration=int(iteration), fitness=[None if math.isnan(f) else float(f) for f in fitness],
                     donor=[int(d) for d in donor], hparams=[{key: mp[key] for key in SWEEP_KEYS} for mp in self.member_params])
        self.lineage.append(entry)
        return entry

    # --------------------------------------------------------------------------- train
    def member_slice(self, t: torch.Tensor, k: int) -> torch.Tensor:
        """Member k's [T, n_member, ...] part of a [T, K * n_member, ...] population buffer."""
        return t[:, k * self.n_member:(k + 1) * self.n_member]

    def train(self):
        """ppo.train for every member -> one (total_returns, total_episode_lengths, x_indices) per member."""
        K, n, T = self.K, self.n_member, int(self.num_steps)
        writers = [None] * K
        if self.params_dict.get("tensorboard", True):
            from torch.utils.tensorboard import SummaryWriter
            for k, mp in enumerate(self.member_params):
                writers[k] = SummaryWriter(f"runs/{self.run_name}__m{k}")
                writers[k].add_text("parameters/what", "what")
                writers[k].add_text("hyperparameters", "|param|value|\n|-|-|\n%s" % (
                    "\n".join([f"|{key}|{str(mp[key])}|" for key in mp])))
        start_time = time.time()
        self.reset_envs()
        for update in range(1, self.num_updates + 1):
            step_base = self._env_step
            out = self.run_update(update)
            keys = self.first_finished.cpu().numpy().view(np.uint64)
            b_ret = out["b_returns"].view(T, K, n)
            b_val = out["b_values"].view(T, K, n)
            var_y = torch.var(b_ret, dim=(0, 2), unbiased=False)
            ev = 1 - torch.var(b_ret - b_val, dim=(0, 2), unbiased=False) / var_y
            stats = out["stats"]
            host_stats = stats.cpu().numpy()
            host_ev = torch.stack([var_y, ev]).cpu().numpy()
            global_step = (step_base + T) * n
            for k in range(K):
                kk = keys[k]
                ts = np.nonzero(kk != np.uint64(0xFFFFFFFFFFFFFFFF))[0]
                v = kk[ts]
                lens = ((v >> np.uint64(32)) & np.uint64(1023)).astype(np.int64)
                rets = (v & np.uint64(0xFFFFFFFF)).astype(np.uint32).view(np.float32)
                gss = (step_base + ts + 1) * n
                w = writers[k]
                if w is not None:
                    for gs, r, ln in zip(gss.tolist(), rets.tolist(), lens.tolist()):
                        w.add_scalar("charts/episodic_return", r, gs)
                        w.add_scalar("charts/episodic_length", ln, gs)
                self.total_returns[k].extend(rets.tolist())
                self.total_episode_lengths[k].extend(lens.tolist())
                self.x_indices[k].extend(gss.tolist())
                r = self.rows_done[k]
                last = host_stats[k, r - 1]
                explained_var = float("nan") if host_ev[0, k] == 0 else float(host_ev[1, k])
                if w is not None:
                    w.add_scalar("charts/learning_rate", self.lr_frac * self.member_params[k]["learning_rate"], global_step)
                    w.add_scalar("losses/value_loss", last[1], global_step)
                    w.add_scalar("losses/policy_loss", last[0], global_step)
                    w.add_scalar("losses/entropy", last[2], global_step)
                    w.add_scalar("losses/old_approx_kl", last[3], global_step)
                    w.add_scalar("losses/approx_kl", last[4], global_step)
                    w.add_scalar("losses/clipfrac", host_stats[k, :r, 5].mean(), global_step)
                    w.add_scalar("losses/explained_variance", explained_var, global_step)
                    w.add_scalar("charts/SPS", int(global_step / (time.time() - start_time)), global_step)
            if self.pbt is not None and update % self.pbt["interval"] == 0 and update < self.num_updates:
                entry = self._record_round(update, self.pbt_step())
                for k, w in enumerate(writers):
                    if w is not None:
                        f = entry["fitness"][k]
                        w.add_scalar("pbt/fitness", float("nan") if f is None else f, global_step)
                        w.add_scalar("pbt/donor", entry["donor"][k], global_step)
        for w in writers:
            if w is not None:
                w.close()
        if self.params_dict.get("save", True):
            for k in range(K):
                compat.save_policy(self.standalone_policy(k), f"actor_critic_{self.num_layers}_m{k}.pt")
            if self.pbt is not None:
                with open("pbt_lineage.json", "w") as f:
                    json.dump(self.lineage, f, indent=1)
        return [(self.total_returns[k], self.total_episode_lengths[k], self.x_indices[k]) for k in range(K)]

    def standalone_policy(self, k: int) -> actor_critic:
        """A copy of member k's actor_critic that owns its parameters (what a checkpoint should hold, not the [K][P] buffer)."""
        pol = self.policies[k]
        with torch.cuda.device(self.device):
            out = actor_critic(pol.state_dim, pol.action_dim, pol.hidden_dim, pol.num_layers, pol.dropout, pol.continuous).to(self.device)
        out.load_state_dict({name: t.detach().clone() for name, t in pol.state_dict().items()})
        return out
