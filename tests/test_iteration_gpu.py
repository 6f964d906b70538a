"""Whole iterations of the outer loop (src/ppo.py:192-273) on the device against the restatement, on the same inputs:
rollout -> GAE -> `num_update_epochs` x `num_minibatches` updates with the learning-rate anneal, twice in a row.

* the env trajectory of both iterations replays bit for bit on the checker (oracle/envs.c in its own trig mode) from the actions
  the device sampled;
* the stored log-probs / values are the restated model's at the parameters the iteration started from (2e-5);
* returns / advantages equal `run_gae` on the device's own rewards / values bit for bit;
* the parameter change of each iteration equals the restated update loop's (same keyed shuffles, same minibatch order, Adam with
  the annealed learning rate) within 1e-4 relative L2 of the CHANGE (parameters within 1e-6 absolute).

Covers the host orchestration (ppo.run_update: shuffle stream ids, moments of all minibatches ahead or per minibatch, minibatch
slicing with a ragged tail, the target_kl stop, GAE or plain returns, anneal) for the 64-wide fused kernels and for the wide
tensor-core paths (128 / 256 units), on CartPole, Pendulum, MountainCar and Acrobot."""
import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, kernels, run_ppo
from oracle import envs as E
from oracle import ppo_ref as R
from tests.helpers import flat_from_named

pytestmark = pytest.mark.gpu


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False)
    p.update(kw)
    return p


def _named_from_module(policy):
    return {k: v.detach().cpu().numpy().copy() for k, v in policy.state_dict().items()}


_KIND = {"CartPole-v1": E.CARTPOLE, "Pendulum-v1": E.PENDULUM, "MountainCar-v0": E.MOUNTAINCAR, "Acrobot-v1": E.ACROBOT}


def _row(gym_id, hidden=64, layers=2, **kw):
    """One case: the env, the policy width and whatever it sets besides the defaults of the loop below (N, T, NM, EP and any
    run_ppo parameter)."""
    return dict(gym_id=gym_id, hidden=hidden, layers=layers, **kw)


ITERATION_ROWS = {
    "CartPole-v1-False-64-2": _row("CartPole-v1"),
    "CartPole-v1-False-128-2": _row("CartPole-v1", 128),
    "Pendulum-v1-True-64-2": _row("Pendulum-v1"),
    "Pendulum-v1-True-128-2": _row("Pendulum-v1", 128),
    "CartPole-v1-False-256-2": _row("CartPole-v1", 256),
    "CartPole-v1-False-128-3": _row("CartPole-v1", 128, 3),
    # the first whole-iteration parity of MountainCar-v0: the 64-wide kernels, the 128 x 2 tensor-core rollout, and at 256 the
    # layer-wise rollout with the external-actor env step; the wide rows feed the update a 3-output head from 2 inputs.  At
    # 1e-3 the wide nets move 2-3 times as far as the CartPole rows do, so they learn at half the rate to keep the absolute
    # parameter bar as strict
    "mountaincar-64x2": _row("MountainCar-v0"),
    "mountaincar-128x2": _row("MountainCar-v0", 128, learning_rate=5e-4),
    "mountaincar-256x2": _row("MountainCar-v0", 256, learning_rate=5e-4),
    # the runtime-width SIMT rollout at 128 units (Acrobot has no tensor-core rollout) feeding wide_first_kernel<8>
    "acrobot-128x2": _row("Acrobot-v1", 128),
    # the wide update's clip_vloss == 0 branch inside the loop.  Its value loss is (v - vold)^2 and vold is the rollout's own
    # value, so the critic's gradient is only the rounding difference between two forward passes, which Adam scales up to
    # full-size steps on both sides: the critic's change and the stats that hold it are not comparable, only the actor's
    # are; the value loss must stay small, which a wrong target would not
    "cartpole-128x2-novclip": _row("CartPole-v1", 128, clip_vloss=False, actor_only=True),
    # norm_adv off: run_update skips prepare_moments, and the wide continuous head takes raw advantages
    "pendulum-128x2-nonorm": _row("Pendulum-v1", 128, norm_adv=False),
    # 288 minibatches x 2 epochs = 576 > Updater.MAX_MINIBATCHES: moments per minibatch instead of prepare_moments.  72 times
    # as many Adam steps as the other rows, so a 20 times smaller learning rate keeps the absolute parameter bar as strict
    "cartpole-576-minibatches": _row("CartPole-v1", num_minibatches=288, learning_rate=5e-5),
    # returns by normal_advantage (ppo.py:145-157) through the host loop
    "cartpole-no-gae": _row("CartPole-v1", gae=False),
    # approx_kl passes target_kl after the first of three epochs: the loop stops there, as the restated loop does
    "cartpole-target-kl": _row("CartPole-v1", num_update_epochs=3, target_kl=1e-7),
}


@pytest.mark.parametrize("row", list(ITERATION_ROWS))
def test_two_iterations_vs_oracle(row):
    from aur_ppo_b200.ppo import ppo
    kw = dict(ITERATION_ROWS[row])
    gym_id, hidden, layers = kw.pop("gym_id"), kw.pop("hidden"), kw.pop("layers")
    kind = _KIND[gym_id]
    cont = gym_id == "Pendulum-v1"
    obs_dim = E.OBS_DIM[kind]
    N, T, U = 24, 48, 2
    NM, EP = kw.pop("num_minibatches", 4), kw.pop("num_update_epochs", 2)
    lr, actor_only = kw.pop("learning_rate", 1e-3), kw.pop("actor_only", False)
    torch.manual_seed(3)
    p = _params(gym_id=gym_id, continuous=cont, hidden_dim=hidden, num_layers=layers, num_envs=N, num_steps=T, num_minibatches=NM,
                num_update_epochs=EP, total_timesteps=N * T * U, learning_rate=lr, entropy_coeff=0.01 if not cont else 0.0, **kw)
    agent = ppo(p)
    batch, mb = N * T, N * T // NM
    per_epoch = -(-batch // mb)
    # the prelude of train() (ppo.py:180-190)
    agent.envs.reset(seed=list(agent.plan.env_ids))
    agent._env_step = 0
    agent._stats_rows = torch.zeros(EP * per_epoch, kernels.NUM_STATS, device=agent.device)
    # which way run_update computes the advantage moments: all minibatches ahead in one launch, or each minibatch itself
    ahead = p["norm_adv"] and batch % mb == 0 and EP * per_epoch <= kernels.Updater.MAX_MINIBATCHES

    names = list(agent.policy.state_dict().keys())
    pol = R.RefPolicy(_named_from_module(agent.policy), cont)
    pol.requires_grad_(False)
    opt = R.RefAdam(pol.tensors(), lr=lr, eps=1e-5)
    shuffle_count = agent._shuffle_count
    compared = ~flat_from_named({n: np.full(t.shape, actor_only and n.startswith("critic."))
                                 for n, t in agent.policy.state_dict().items()}).astype(bool)
    acts_all, per_iter = [], []
    loss_kw = dict(max_grad_norm=p["max_grad_norm"], clip_coeff=p["clip_coeff"], ent_c=p["entropy_coeff"], vf_c=p["value_coeff"],
                   norm_adv=bool(p["norm_adv"]), clip_vloss=bool(p["clip_vloss"]))
    for u in range(1, U + 1):
        before = agent.flat.detach().cpu().numpy().copy()
        out = agent.run_update(u)
        torch.cuda.synchronize()
        b = agent.buffer
        dev = {k: getattr(b, k).cpu().numpy().copy() for k in ("states", "actions", "log_probs", "rewards", "terminals", "values")}
        dev["next_value"] = b.next_value.cpu().numpy().copy()
        dev["next_done"] = agent.envs.next_done.cpu().numpy().copy()
        dev["returns"], dev["advantages"] = agent._returns.cpu().numpy().copy(), agent._advantages.cpu().numpy().copy()
        acts_all.append(dev["actions"])
        # ---- the restated model at the parameters this iteration started from
        ot = torch.from_numpy(dev["states"].reshape(-1, obs_dim))
        at = torch.from_numpy(dev["actions"].reshape(-1, 1) if cont else dev["actions"].reshape(-1))
        with torch.no_grad():
            _, lp, _, v = pol.evaluate(ot, at)
        np.testing.assert_allclose(dev["log_probs"].reshape(-1), lp.numpy(), rtol=2e-5, atol=5e-6)
        np.testing.assert_allclose(dev["values"].reshape(-1), v.numpy().reshape(-1), rtol=2e-5, atol=5e-6)
        # ---- run_gae on the device's own rewards / values: bit for bit
        rollout = [torch.from_numpy(dev[k]) for k in ("rewards", "values", "terminals", "next_value", "next_done")]
        with torch.no_grad():
            if p["gae"]:
                ret, adv = R.gae(*rollout, p["gamma"], p["gae_lambda"])
            else:
                ret, adv = R.normal_advantage(*rollout, p["gamma"])
        assert np.array_equal(ret.numpy(), dev["returns"]) and np.array_equal(adv.numpy(), dev["advantages"])
        # ---- the update loop (ppo.py:208-269) with the device's keyed shuffles
        opt.lr = R.lr_anneal(lr, u, U)
        assert abs(agent.optimizer.param_groups[0]["lr"] - opt.lr) < 1e-15
        flat_b = (ot, at if not cont else at.reshape(-1, 1), torch.from_numpy(dev["log_probs"].reshape(-1)), adv.reshape(-1),
                  ret.reshape(-1), torch.from_numpy(dev["values"].reshape(-1)))
        ref_stats, n_ref = None, 0
        for ep in range(EP):
            inds = R.feistel_shuffle(batch, agent.shuffle_seed, shuffle_count + ep)    # drawn for every epoch up front
            for s in range(0, batch, mb):
                mi = torch.from_numpy(inds[s:s + mb].astype(np.int64))
                ref_stats = R.ppo_update_step(pol, opt, *[t[mi] for t in flat_b], **loss_kw)[0]
                n_ref += 1
            if p["target_kl"] is not None and ref_stats["approx_kl"] > p["target_kl"]:
                break
        shuffle_count += EP
        # ---- the branch run_update took
        assert out["stats"].shape[0] == n_ref
        if p["target_kl"] is not None:
            assert n_ref == per_epoch                      # stopped after the first epoch
        else:
            assert n_ref == EP * per_epoch
        if ahead:
            assert agent.updater.moments_all is not None and agent.updater.moments_all.shape[0] == EP * per_epoch
        else:
            assert agent.updater.moments_all is None       # prepare_moments never ran
        after = agent.flat.detach().cpu().numpy()
        want = flat_from_named({n: pol.p[n].detach().numpy() for n in names})
        d_dev, d_ref = (after - before)[compared], (want - before)[compared]
        rel = float(np.linalg.norm(d_dev - d_ref) / np.linalg.norm(d_ref))
        print(f"{row} ({gym_id} hidden {hidden} x {layers}), iteration {u}: {n_ref} minibatches, |param change| "
              f"{np.linalg.norm(d_ref):.3e}, relative L2 error of the change {rel:.2e}")
        assert rel < 1e-4                      # measured 8e-6 .. 1.9e-5 (profiles/r2_whole_iteration_parity.txt)
        np.testing.assert_allclose(after[compared], want[compared], rtol=0, atol=1e-6)
        last = out["stats"][-1].cpu().numpy()
        for i, k in enumerate(kernels.STAT_NAMES):
            if actor_only and k in ("value_loss", "loss", "grad_norm"):
                continue                       # these hold the critic, whose change is not comparable (see the row)
            np.testing.assert_allclose(last[i], ref_stats[k], rtol=2e-3, atol=2e-5, err_msg=k)
        if actor_only:                         # v - vold stays at the critic's drift; v - returns would be of order 1
            assert last[kernels.STAT_NAMES.index("value_loss")] < 1e-2
        # keep the restated parameters ON the device's (the comparison above is per iteration, not cumulative)
        with torch.no_grad():
            for n, t in zip(names, pol.tensors()):
                t.copy_(agent.policy.state_dict()[n].detach().cpu())
        per_iter.append(dev)
    assert agent._shuffle_count == shuffle_count
    # ---- both iterations' trajectory on the checker, from the sampled actions
    acts = np.concatenate(acts_all).reshape(U * T, N, -1)
    acts = acts if cont else acts[..., 0].astype(np.int64)
    cv = E.CVecEnv(kind, N, wrappers=cont, trig=E.TRIG_CR)
    cur, _ = cv.reset(list(range(N)))
    cur_done = np.zeros(N, np.float32)
    for t in range(U * T):
        dev = per_iter[t // T]
        assert np.array_equal(dev["states"][t % T], cur) and np.array_equal(dev["terminals"][t % T], cur_done), t
        cur, r, term, trunc, info = cv.step(acts[t])
        assert np.array_equal(dev["rewards"][t % T], r.astype(np.float32)), t
        cur_done = term.astype(np.float32)
    assert np.array_equal(agent.envs.next_obs.cpu().numpy(), cur)


def test_a_batch_that_does_not_divide_into_minibatches_is_refused():
    """1,152 samples in 5 minibatches would leave a short last minibatch (the reference slices one); the run refuses it when it
    is built, so run_update never sees a ragged batch."""
    from aur_ppo_b200.ppo import ppo
    with pytest.raises(_lib.AurError, match="local batch must divide into num_minibatches"):
        ppo(_params(num_envs=24, num_steps=48, num_minibatches=5))
