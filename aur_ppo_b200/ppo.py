"""Drop-in for the reference's `ppo` class (src/ppo.py:42-321) on the B200 hot path.

Same constructor (`ppo(params)` with the run_ppo.py:53-81 dict), same attributes (`policy`,
`optimizer`, `buffer`, `envs`, `batch_size`, `minibatch_size`, `num_updates`), same `train()`
return value, same TensorBoard tags and checkpoint file.  What differs is where the work runs:

  reference                                   here
  ------------------------------------------  -----------------------------------------------
  gym.vector.SyncVectorEnv on the host        DeviceVecEnv: env state lives in HBM
  T x (evaluate, D2H, N env.step, H2D)        one aur_rollout launch per update   (ppo.py:201-205)
  T x 9 elementwise kernels                   one aur_gae_f32 launch              (ppo.py:125-157)
  ~100 kernels + 2 syncs per minibatch        moments, grad, reduce, adam         (ppo.py:220-269)
  np.random.shuffle + index H2D per epoch     keyed bijection written by shuffle_kernel (no sort)

There is no CPU path: without a CUDA device or without libaurppo.so the constructor raises.
Under torch.distributed each rank owns num_envs / world_size env columns; the only exchange is
the packed [grads | stats] buffer (and three fp64 advantage moments) per minibatch, summed by the
update kernels themselves over NVLink peer memory (parallel.PeerExchange; AUR_DP_EXCHANGE=nccl
selects two library all_reduce calls instead).
"""
from __future__ import annotations

import math
import os
import random
import time
from typing import Dict, List, Optional

import numpy as np
import torch

from . import _lib, compat, kernels, parallel, state
from .envs import DeviceVecEnv
from .models.actor_critic import actor_critic


class torch_buffer:
    """src/ppo.py:20-39: [T,N,...] fp32 rollout storage (actions are fp32 even when discrete)."""

    def __init__(self, observation_shape, action_shape, num_steps, num_envs, device="cuda"):
        self.observation_shape = tuple(observation_shape)
        self.action_shape = tuple(action_shape)
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=device)
        self.states = z(num_steps, num_envs, *self.observation_shape)
        self.actions = z(num_steps, num_envs, *self.action_shape)
        self.log_probs = z(num_steps, num_envs)
        self.rewards = z(num_steps, num_envs)
        self.terminals = z(num_steps, num_envs)
        self.values = z(num_steps, num_envs)
        self.next_value = z(num_envs)

    def flatten(self, returns, advantages):
        b_obs = self.states.reshape((-1,) + self.observation_shape)
        b_logprobs = self.log_probs.reshape(-1)
        b_actions = self.actions.reshape((-1,) + self.action_shape)
        b_advantages = advantages.reshape(-1)
        b_returns = returns.reshape(-1)
        b_values = self.values.reshape(-1)
        return b_obs, b_logprobs, b_actions, b_advantages, b_returns, b_values


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(lr, eps=1e-5) facade (src/ppo.py:80) over the fused clip+Adam kernel:
    `param_groups[0]["lr"]` is what the kernel reads each step, the moments live in flat buffers."""

    def __init__(self, params, updater: kernels.Updater, lr: float, eps: float = 1e-5, betas=(0.9, 0.999)):
        super().__init__(list(params), dict(lr=lr, eps=eps, betas=betas, weight_decay=0, amsgrad=False))
        self.updater = updater

    def step(self, closure=None, max_grad_norm: float = 0.5, stats_out=None):
        return self.updater.apply(self.param_groups[0]["lr"], max_grad_norm, stats_out=stats_out)

    def zero_grad(self, set_to_none: bool = True):
        pass   # the gradient buffer is overwritten by every aur_ppo_update_grad call


_SPACES = {"CartPole-v1": dict(obs=(4,), act_shape=(), n=2), "Pendulum-v1": dict(obs=(3,), act_shape=(1,), n=None),
           "MountainCar-v0": dict(obs=(2,), act_shape=(), n=3), "Acrobot-v1": dict(obs=(6,), act_shape=(), n=3),
           "MountainCarContinuous-v0": dict(obs=(2,), act_shape=(1,), n=None)}


class ppo:
    def __init__(self, params: Dict):
        self.params_dict = params
        self.all_steps = None
        self.minibatch_size = None
        for key, value in params.items():
            if key not in ("batch_size", "minibatch_size"):
                setattr(self, key, value)
        if not torch.cuda.is_available():
            raise _lib.AurError("aur_ppo_b200.ppo needs a CUDA device: the hot path has no CPU fallback")
        _lib.lib()
        # ---- data-parallel layout: env columns sharded over ranks
        try:
            self.plan = parallel.current_plan(self.num_envs, self.num_steps, self.num_minibatches)
        except ValueError as e:
            raise _lib.AurError(str(e))
        self.world_size, self.rank = self.plan.world_size, self.plan.rank
        self.device = torch.device(params.get("device", f"cuda:{torch.cuda.current_device()}"))
        self.local_envs = self.plan.local_envs
        if self.gym_id not in _SPACES:
            raise _lib.AurError(f"gym_id {self.gym_id!r} has no device kernel (compiled: {sorted(_SPACES)})")
        sp = _SPACES[self.gym_id]
        if bool(self.continuous) != (sp["n"] is None):
            raise _lib.AurError(f"{self.gym_id} is {'continuous' if sp['n'] is None else 'discrete'}; got continuous={self.continuous}")

        self.all_steps = self.num_steps * self.num_envs
        self.batch_size = int(self.num_envs * self.num_steps)
        self.minibatch_size = int(self.all_steps // self.num_minibatches)
        self.num_updates = self.total_timesteps // self.batch_size
        self.local_batch = self.plan.local_batch
        self.local_minibatch = self.plan.local_minibatch
        self.run_name = f"{self.gym_id}__{self.exp_name}__{self.seed}__{int(time.time())}"

        self.envs = DeviceVecEnv(self.gym_id, self.local_envs, wrappers=bool(self.continuous), device=self.device,
                                 env_id0=self.plan.env_id0)
        self.state_dim = sp["obs"]
        self.action_dim = sp["act_shape"] if self.continuous else sp["n"]
        with torch.cuda.device(self.device):
            self.policy = actor_critic(self.state_dim[0], self.action_dim, self.hidden_dim, self.num_layers, self.dropout,
                                       self.continuous).to(self.device)
        parallel.broadcast_parameters(self.policy, self.plan)      # identical initial weights on every rank
        self.flat = self.policy.flat_parameters()
        self.desc = kernels.policy_desc(*self.policy.kernel_shape())
        self.buffer = torch_buffer(self.state_dim, sp["act_shape"], self.num_steps, self.local_envs, self.device)
        # data-parallel exchange: "peer" = in-kernel all-reduce over NVLink peer memory (default), "nccl" = library all-reduce
        self.exchange_kind = str(params.get("exchange", os.environ.get("AUR_DP_EXCHANGE", "peer")))
        self.exchange = None
        if self.plan.world_size > 1 and self.exchange_kind == "peer":
            self.exchange = parallel.PeerExchange(self.plan, self.desc)
            self.updater = kernels.Updater(self.desc, self.flat, eps=1e-5, exchange=self.exchange)
        else:
            self.updater = kernels.Updater(self.desc, self.flat, eps=1e-5, allreduce=parallel.make_allreduce(self.plan))
        self.optimizer = FusedAdam(self.policy.parameters(), self.updater, lr=self.learning_rate, eps=1e-5)
        self.philox_seed = int(params.get("philox_seed", 1))
        # minibatch shuffles: one stream per (rank, epoch) so that ranks draw independent permutations
        self.shuffle_seed = int(params.get("shuffle_seed", self.philox_seed))
        self._shuffle_count = self.rank << 40
        # the permutations of ALL epochs of an iteration (they do not depend on the parameters): [epochs, local_batch]
        self._b_inds = torch.empty(max(int(self.num_update_epochs), 1), self.local_batch, dtype=torch.int32, device=self.device)
        self._records = None
        self.total_returns: List[float] = []
        self.total_episode_lengths: List[int] = []
        self.x_indices: List[int] = []
        self._returns = torch.empty_like(self.buffer.rewards)
        self._advantages = torch.empty_like(self.buffer.rewards)
        self._env_step = 0
        self._iteration = 0              # iterations of train() completed
        self._train_seconds = 0.0        # wall-clock seconds train() has run them in
        self._resumed = False            # load_state() restored a state: the next train() continues it

    def close(self) -> None:
        """Unmap the peer exchange areas (data-parallel runs); collective: every rank calls it."""
        if getattr(self, "exchange", None) is not None:
            self.exchange.close()
            self.exchange = None

    def _check_exchange(self) -> None:
        """Data-parallel health check, once per update: if any rank's kernels gave up waiting for a peer (the Adam kernel then
        skips its step), EVERY rank learns it here (one tiny all-reduce on the control plane) and raises after the collective
        close, so no rank is left hanging at a barrier."""
        if self.exchange is None:
            return
        bad = torch.tensor([float(self.exchange.status() != 0)])
        if torch.distributed.get_backend() == "nccl":
            bad = bad.to(self.device)
        torch.distributed.all_reduce(bad, op=torch.distributed.ReduceOp.MAX)
        if float(bad.item()) != 0.0:
            self.close()
            raise _lib.AurError("data-parallel exchange: a kernel timed out waiting for a peer rank (update skipped on every rank)")

    # ------------------------------------------------------------------ hot path pieces
    def make_env(self, gym_id, idx, capture_video):
        raise _lib.AurError("envs are device-resident here; there are no per-env gym thunks (src/ppo.py:85-99)")

    def rollout(self, actions_in: Optional[torch.Tensor] = None) -> None:
        """ppo.py:201-205 for all T steps: fills self.buffer, leaves critic(next_obs) in buffer.next_value."""
        kernels.rollout(self.envs, self.desc, self.flat, self.buffer, seed=self.philox_seed, step0=self._env_step,
                        actions_in=actions_in)
        self._env_step += self.num_steps

    def advantages(self, next_obs=None, next_done=None):
        """ppo.py:159-166 -> (returns, advantages) [T,N]."""
        return kernels.gae(self.buffer.rewards, self.buffer.values, self.buffer.terminals, self.buffer.next_value,
                           self.envs.next_done, self.gamma, self.gae_lambda, bool(self.gae),
                           out=(self._returns, self._advantages))

    def pack(self, flat_bufs) -> None:
        """Gather-friendly per-sample records of this iteration's batch (one 32-byte sector per sample and net)."""
        b_obs, b_logprobs, b_actions, b_advantages, b_returns, b_values = flat_bufs
        self._records = kernels.pack_records(b_obs, b_actions, b_logprobs, b_advantages, b_returns, b_values,
                                             out=self._records)

    def update_minibatch(self, flat_bufs, mb_inds: torch.Tensor, stats_out: Optional[torch.Tensor] = None,
                         moments_index: Optional[int] = None) -> torch.Tensor:
        """ppo.py:220-269 for one minibatch of local row indices -> device stats tensor (written to stats_out if given).
        moments_index: entry of the iteration's pre-computed advantage moments (run_update), else computed here."""
        b_obs, b_logprobs, b_actions, b_advantages, b_returns, b_values = flat_bufs
        self.updater.grad(b_obs, b_actions, b_logprobs, b_advantages, b_returns, b_values, mb_inds,
                          m_total=mb_inds.numel() * self.world_size, clip_coeff=self.clip_coeff,
                          entropy_coeff=self.entropy_coeff, value_coeff=self.value_coeff, norm_adv=bool(self.norm_adv),
                          clip_vloss=bool(self.clip_vloss), records=self._records, moments_index=moments_index)
        return self.optimizer.step(max_grad_norm=self.max_grad_norm, stats_out=stats_out)

    def run_update(self, update: int, events=None) -> Dict[str, torch.Tensor]:
        """One full iteration of the outer loop (ppo.py:192-273) without logging; returns device tensors.
        events: optional 4 CUDA events recorded at the phase boundaries (start, rollout done, GAE done, update done)."""
        rec = (lambda i: events[i].record()) if events is not None else (lambda i: None)
        if self.anneal_lr:
            frac = 1.0 - (update - 1.0) / self.num_updates
            self.optimizer.param_groups[0]["lr"] = frac * self.learning_rate
        rec(0)
        self.rollout()
        rec(1)
        returns, advantages = self.advantages()
        rec(2)
        flat_bufs = self.buffer.flatten(returns, advantages)
        self.pack(flat_bufs)
        n_mb = 0
        stats_rows = self._stats_rows
        # np.random.shuffle(b_inds) of every epoch (ppo.py:214-215) up front, then the advantage moments of every minibatch in
        # ONE launch (data-parallel: one exchange per iteration instead of one per minibatch)
        for ep in range(self.num_update_epochs):
            kernels.shuffle_indices(self.local_batch, seed=self.shuffle_seed, stream_id=self._shuffle_count, out=self._b_inds[ep])
            self._shuffle_count += 1
        per_epoch = self.local_batch // self.local_minibatch
        ahead = (bool(self.norm_adv) and self.local_batch % self.local_minibatch == 0 and
                 self.num_update_epochs * per_epoch <= kernels.Updater.MAX_MINIBATCHES)
        if ahead:
            self.updater.prepare_moments(flat_bufs[3], self._b_inds.view(-1, self.local_minibatch))
        for ep in range(self.num_update_epochs):
            b_inds = self._b_inds[ep]
            for j, start in enumerate(range(0, self.local_batch, self.local_minibatch)):
                mb = b_inds[start:start + self.local_minibatch]
                self.update_minibatch(flat_bufs, mb, stats_out=stats_rows[n_mb], moments_index=ep * per_epoch + j if ahead else None)
                n_mb += 1
            if self.target_kl is not None:
                if stats_rows[n_mb - 1, 4].item() > self.target_kl:
                    break
        rec(3)
        return dict(stats=stats_rows[:n_mb], b_values=flat_bufs[5], b_returns=flat_bufs[4])

    # --------------------------------------------------------------------------- training state
    def _state_tensors(self) -> Dict[str, torch.Tensor]:
        return dict(flat=self.flat, exp_avg=self.updater.exp_avg, exp_avg_sq=self.updater.exp_avg_sq,
                    totals=self.envs.totals)

    def _refuse_data_parallel(self) -> None:
        if self.world_size > 1:
            raise _lib.AurError("training state: data-parallel runs (world_size > 1) cannot be saved or resumed")

    def save_state(self, path: str) -> None:
        """Write what train() needs to continue after iteration `self._iteration` to `path` (state.py, DESIGN.md section 13)."""
        self._refuse_data_parallel()
        if self._iteration < 1:
            raise _lib.AurError("save_state: no iteration of train() has completed yet; there is nothing to resume")
        body = dict(tensors=state.to_host(self._state_tensors()), env=state.to_host(state.env_tensors(self.envs)),
                    step_count=int(self.updater.step_count), env_step=int(self._env_step),
                    shuffle_count=int(self._shuffle_count), iteration=int(self._iteration),
                    train_seconds=float(self._train_seconds), run_name=self.run_name,
                    total_returns=state.history(self.total_returns, np.float64),
                    total_episode_lengths=state.history(self.total_episode_lengths, np.int64),
                    x_indices=state.history(self.x_indices, np.int64), last_stats=getattr(self, "last_stats", None))
        state.write(path, "ppo", state.fingerprint(self.params_dict), body)

    def load_state(self, path: str) -> None:
        """Restore a state written by save_state into this freshly built run (same configuration); the next train() then
        continues with the following iteration, without an env reset.  Everything is checked before anything is changed.
        Tensors are copied in place: `flat` stays the buffer the policy's parameters view."""
        self._refuse_data_parallel()
        st = state.read(path, "ppo", state.fingerprint(self.params_dict))
        f = state.fields(st, ("tensors", "env", "step_count", "env_step", "shuffle_count", "iteration", "train_seconds",
                              "run_name", "total_returns", "total_episode_lengths", "x_indices", "last_stats"))
        try:
            scalars = dict(step_count=int(f["step_count"]), env_step=int(f["env_step"]), shuffle_count=int(f["shuffle_count"]),
                           iteration=int(f["iteration"]), train_seconds=float(f["train_seconds"]), run_name=str(f["run_name"]),
                           total_returns=f["total_returns"].tolist(), total_episode_lengths=f["total_episode_lengths"].tolist(),
                           x_indices=f["x_indices"].tolist(), last_stats=None if f["last_stats"] is None else dict(f["last_stats"]))
        except (AttributeError, TypeError, ValueError) as e:
            raise _lib.AurError(f"training state {path!r}: malformed entry ({e})")
        mine = self._state_tensors()
        state.restore([(k, t, f["tensors"].get(k)) for k, t in mine.items()] + state.restore_env(self.envs, f["env"]))
        self.updater.step_count = scalars["step_count"]
        self._env_step, self._shuffle_count = scalars["env_step"], scalars["shuffle_count"]
        self._iteration, self._train_seconds = scalars["iteration"], scalars["train_seconds"]
        self.run_name = scalars["run_name"]
        self.total_returns = scalars["total_returns"]
        self.total_episode_lengths = scalars["total_episode_lengths"]
        self.x_indices = scalars["x_indices"]
        if scalars["last_stats"] is not None:
            self.last_stats = scalars["last_stats"]
        self._resumed = True

    # --------------------------------------------------------------------------- train
    def train(self, save_state_every: int = 0, state_path: str = "training_state.pt", resume: Optional[str] = None):
        """ppo.py:175-309.  save_state_every N > 0: write the training state to `state_path` after every N-th iteration and
        after the last one.  resume: continue the run whose state that file holds (no env reset, same schedule); the same as
        load_state(resume) followed by train()."""
        if int(save_state_every) < 0:
            raise _lib.AurError(f"save_state_every must be >= 0 (got {save_state_every})")
        if save_state_every or resume is not None:
            self._refuse_data_parallel()
        if resume is not None:
            self.load_state(resume)
        writer = None
        if self.rank == 0 and self.params_dict.get("tensorboard", True):
            if self.track:
                import wandb
                wandb.init(project="ppo", entity="Aurelian", sync_tensorboard=True, config=None, name=self.run_name,
                           monitor_gym=True, save_code=True)
            from torch.utils.tensorboard import SummaryWriter
            writer = SummaryWriter(f"runs/{self.run_name}")
            writer.add_text("parameters/what", "what")
            writer.add_text("hyperparameters", "|param|value|\n|-|-|\n%s" % (
                "\n".join([f"|{key}|{str(self.params_dict[key])}|" for key in self.params_dict])))
        seed = 1                                    # hard-coded in the reference (ppo.py:180-184)
        random.seed(seed)
        np.random.seed(seed)
        torch.manual_seed(seed)

        global_step = 0
        resuming, self._resumed = self._resumed, False
        if not resuming:
            self.envs.reset(seed=list(self.plan.env_ids))
            self._env_step = 0
            self._iteration, self._train_seconds = 0, 0.0
        start_time = time.time() - self._train_seconds
        n_rows = self.num_update_epochs * math.ceil(self.local_batch / max(self.local_minibatch, 1))
        self._stats_rows = torch.zeros(n_rows, kernels.NUM_STATS, device=self.device)

        for update in range(self._iteration + 1, self.num_updates + 1):
            step_base = self._env_step
            out = self.run_update(update)
            self._check_exchange()
            # ---- episodic statistics (ppo.py:114-122): the first finished env of each step
            ts, _, rets, lens = self.envs.first_finished_episodes()
            gss = (step_base + ts + 1) * self.num_envs
            if writer is not None:
                for gs, ret, length in zip(gss.tolist(), rets.tolist(), lens.tolist()):
                    writer.add_scalar("charts/episodic_return", ret, gs)
                    writer.add_scalar("charts/episodic_length", length, gs)
            self.total_returns.extend(rets.tolist())
            self.total_episode_lengths.extend(lens.tolist())
            self.x_indices.extend(gss.tolist())
            global_step = (step_base + self.num_steps) * self.num_envs
            # ---- per-update scalars (ppo.py:277-292); explained variance computed on device
            stats = out["stats"]
            b_values, b_returns = out["b_values"], out["b_returns"]
            var_y = torch.var(b_returns, unbiased=False)
            ev = 1 - torch.var(b_returns - b_values, unbiased=False) / var_y
            host = torch.cat([stats[-1, :8], stats[:, 5].mean().reshape(1), var_y.reshape(1), ev.reshape(1)]).cpu().numpy()
            explained_var = float("nan") if host[9] == 0 else float(host[10])
            self.last_stats = dict(value_loss=float(host[1]), policy_loss=float(host[0]), entropy=float(host[2]),
                                   old_approx_kl=float(host[3]), approx_kl=float(host[4]), clipfrac=float(host[8]),
                                   explained_variance=explained_var, grad_norm=float(host[6]))
            if writer is not None:
                writer.add_scalar("charts/learning_rate", self.optimizer.param_groups[0]["lr"], global_step)
                writer.add_scalar("losses/value_loss", host[1], global_step)
                writer.add_scalar("losses/policy_loss", host[0], global_step)
                writer.add_scalar("losses/entropy", host[2], global_step)
                writer.add_scalar("losses/old_approx_kl", host[3], global_step)
                writer.add_scalar("losses/approx_kl", host[4], global_step)
                writer.add_scalar("losses/clipfrac", host[8], global_step)
                writer.add_scalar("losses/explained_variance", explained_var, global_step)
                writer.add_scalar("charts/SPS", int(global_step / (time.time() - start_time)), global_step)
            self._iteration, self._train_seconds = update, time.time() - start_time
            if save_state_every and (update % save_state_every == 0 or update == self.num_updates):
                self.save_state(state_path)

        self.envs.close()
        self.close()
        if writer is not None:
            writer.close()
        if self.rank == 0 and self.params_dict.get("save", True):
            compat.save_policy(self.policy, "actor_critic_" + str(self.num_layers) + ".pt")
            self.plot_episodic_returns(np.array(self.total_returns), np.array(self.x_indices), "episodic returns")
            self.plot_episodic_returns(np.array(self.total_episode_lengths), np.array(self.x_indices), "episodic lengths")
        return self.total_returns, self.total_episode_lengths, self.x_indices

    # ---------------------------------------------------------------------------- plots
    def moving_average(self, data, window_size):
        return np.convolve(data, np.ones(window_size) / window_size, mode="valid")

    def plot_episodic_returns(self, episodic_returns, x_indices, title, window_size=10):
        """ppo.py:313-321; skipped (with a note) when matplotlib is not installed."""
        try:
            import matplotlib
            matplotlib.use("Agg")
            import matplotlib.pyplot as plt
        except Exception:
            print(f"[aur_ppo_b200] matplotlib not available: skipping plot {title!r}")
            return
        if len(episodic_returns) < window_size:
            return
        plt.figure()
        plt.plot(x_indices, episodic_returns, label="Episodic Returns")
        plt.plot(x_indices[window_size - 1:], self.moving_average(episodic_returns, window_size),
                 label=f"Moving Average (Window Size = {window_size})", color="red")
        plt.title("Episodic Returns with Moving Average for " + self.gym_id)
        plt.xlabel("Timestep")
        plt.ylabel("Return")
        plt.legend()
        os.makedirs("../plots", exist_ok=True)
        plt.savefig("../plots/" + title + "_num_layers_" + str(self.num_layers) + "_dropout_" + str(self.dropout) +
                    "_num_envs_" + str(self.num_envs) + "_num_mb_" + str(self.num_minibatches) + ".png")
        plt.close()
