"""Populations on the device: member k of a ppo_population computes exactly -- np.array_equal -- what a standalone `ppo` of
its params computes from the same initial weights: rollout buffers, next_obs / next_done / next_value, returns / advantages,
parameters, Adam moments and step count, per-minibatch statistics and the episode log, iteration after iteration.  Also:
placement independence, target_kl per member, launches per iteration independent of K, the single-run kernel switches having no
effect on a population, and the CLI end to end."""
import glob
import os

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, compat, kernels, run_ppo
from aur_ppo_b200.population import member_params, ppo_population
from aur_ppo_b200.ppo import ppo

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def default_impls():
    """The standalone reference runs the default (tensor-core) kernels; a test elsewhere may have left a switch set."""
    L = _lib.lib()
    prev = (L.aur_rollout_get_impl(), L.aur_ppo_update_get_impl())
    L.aur_rollout_set_impl(1)
    L.aur_ppo_update_set_impl(1)
    yield
    L.aur_rollout_set_impl(prev[0])
    L.aur_ppo_update_set_impl(prev[1])


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False)
    p.update(kw)
    return p


def _np(t):
    return t.detach().cpu().numpy().copy()


def _member_state(pop, k):
    n = pop.n_member
    cols = slice(k * n, (k + 1) * n)
    b = pop.buffer
    out = {f: _np(getattr(b, f)[:, cols]) for f in ("states", "actions", "log_probs", "rewards", "terminals", "values")}
    out.update(next_value=_np(b.next_value[cols]), next_obs=_np(pop.envs.next_obs[cols]), next_done=_np(pop.envs.next_done[cols]),
               returns=_np(pop._returns[:, cols]), advantages=_np(pop._advantages[:, cols]), params=_np(pop.params[k]),
               exp_avg=_np(pop.exp_avg[k]), exp_avg_sq=_np(pop.exp_avg_sq[k]), steps=int(pop.steps[k]),
               stats=_np(pop._stats_rows[k, :pop.rows_done[k]]), first_finished=_np(pop.first_finished[k]))
    return out


def _standalone_state(s, out):
    b = s.buffer
    st = {f: _np(getattr(b, f)) for f in ("states", "actions", "log_probs", "rewards", "terminals", "values")}
    st.update(next_value=_np(b.next_value), next_obs=_np(s.envs.next_obs), next_done=_np(s.envs.next_done), returns=_np(s._returns),
              advantages=_np(s._advantages), params=_np(s.flat), exp_avg=_np(s.updater.exp_avg),
              exp_avg_sq=_np(s.updater.exp_avg_sq), steps=s.updater.step_count, stats=_np(out["stats"]),
              first_finished=_np(s.envs.first_finished))
    return st


def _standalone(pop, params, members, k):
    s = ppo(member_params(params, members[k]))
    s.flat.copy_(pop.params[k])                       # the member's initial weights
    s.envs.reset(seed=list(s.plan.env_ids))
    s._env_step = 0
    s._stats_rows = torch.zeros(pop.n_mb, kernels.NUM_STATS, device=s.device)
    return s


def _assert_equal(got, want, what):
    assert got.keys() == want.keys()
    for key in want:
        if key == "steps":
            assert got[key] == want[key], (what, key)
        else:
            assert got[key].shape == want[key].shape, (what, key, got[key].shape, want[key].shape)
            assert np.array_equal(got[key], want[key]), f"{what}: {key} differs (max |d| {np.abs(got[key] - want[key]).max()})"


def _check_vs_standalone(params, members, iters, check=None):
    pop = ppo_population(params, members)
    pop.reset_envs()
    ks = range(len(members)) if check is None else check
    alone = {k: _standalone(pop, params, members, k) for k in ks}
    for u in range(1, iters + 1):
        pop.run_update(u)
        got = {k: _member_state(pop, k) for k in ks}
        for k in ks:
            out = alone[k].run_update(u)
            _assert_equal(got[k], _standalone_state(alone[k], out), f"iteration {u}, member {k}")
    return pop


CARTPOLE_MEMBERS = [dict(seed=1.0), dict(seed=2.0, learning_rate=1e-3), dict(seed=3.0, entropy_coeff=0.0, clip_coeff=0.1),
                    dict(seed=4.0, learning_rate=5e-4, entropy_coeff=0.05, clip_coeff=0.3, value_coeff=0.25, max_grad_norm=1.0)]


def test_cartpole_members_equal_standalone_runs():
    # n_member = 200 is not a multiple of 128: the last CTA of every member has idle lanes
    params = _params(num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2, total_timesteps=200 * 32 * 2)
    pop = _check_vs_standalone(params, CARTPOLE_MEMBERS, iters=2)
    assert all(r == 8 for r in pop.rows_done)


def test_pendulum_with_wrappers_members_equal_standalone_runs():
    params = _params(gym_id="Pendulum-v1", continuous=True, num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2,
                     total_timesteps=200 * 32 * 2, learning_rate=3e-4, entropy_coeff=0.0)
    members = [dict(seed=1.0), dict(seed=2.0, learning_rate=1e-3, clip_coeff=0.1), dict(seed=3.0, entropy_coeff=0.01)]
    _check_vs_standalone(params, members, iters=2)


def test_large_members_use_the_full_single_run_partition():
    # one minibatch of 16,384 * 8 / 4 = 32,768 samples per member: 256 tiles, so every net gets the single run's #SM CTAs
    params = _params(num_envs=16384, num_steps=8, num_minibatches=4, num_update_epochs=1, total_timesteps=16384 * 8)
    assert params["num_envs"] * params["num_steps"] // params["num_minibatches"] >= 128 * torch.cuda.get_device_properties(0).multi_processor_count
    _check_vs_standalone(params, [dict(seed=1.0), dict(seed=2.0, learning_rate=1e-3)], iters=1)


def test_a_member_gives_the_same_bits_wherever_it_sits():
    params = _params(num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2, total_timesteps=200 * 32 * 2)
    me = dict(seed=11.0, learning_rate=7e-4, entropy_coeff=0.02)
    others = [dict(seed=20.0 + i, learning_rate=1e-4 * (i + 1)) for i in range(7)]
    alone = ppo_population(params, [me])
    crowd = ppo_population(params, others[:5] + [me] + others[5:])
    for p in (alone, crowd):
        p.reset_envs()
    for u in (1, 2):
        alone.run_update(u)
        crowd.run_update(u)
        _assert_equal(_member_state(crowd, 5), _member_state(alone, 0), f"iteration {u}, slot 5 of 8 vs K = 1")


def test_target_kl_stops_one_member_after_its_first_epoch():
    params = _params(num_envs=256, num_steps=32, num_minibatches=4, num_update_epochs=3, total_timesteps=256 * 32 * 2,
                     learning_rate=1e-3)
    members = [dict(seed=1.0), dict(seed=2.0, target_kl=1e-12), dict(seed=3.0, target_kl=10.0)]
    pop = _check_vs_standalone(params, members, iters=2)
    assert pop.rows_done == [12, 4, 12]


def test_launches_per_iteration_do_not_depend_on_K():
    params = _params(num_envs=128, num_steps=16, num_minibatches=4, num_update_epochs=2, total_timesteps=128 * 16 * 4)
    L = _lib.lib()
    counts = []
    for K in (1, 64):
        pop = ppo_population(params, [dict(seed=float(k + 1)) for k in range(K)])
        pop.reset_envs()
        pop.run_update(1)                       # first call: attributes, library-owned allocations
        torch.cuda.synchronize()
        L.aur_launch_count_reset()
        pop.run_update(2)
        torch.cuda.synchronize()
        counts.append(L.aur_launch_count())
    assert counts[0] == counts[1], counts
    # rollout + 2 value passes, GAE, records, shuffle, 2 moments launches; then grad + reduce + Adam per minibatch
    assert counts[0] == 8 + 3 * 8


def test_cli_population_end_to_end(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    out = run_ppo.main(["--population", "3", "--num_envs", "256", "--num_steps", "32", "--total_timesteps", str(256 * 32 * 3),
                        "--no_tensorboard"])
    assert len(out) == 3 and all(len(r[0]) == len(r[2]) for r in out)
    files = sorted(glob.glob(str(tmp_path / "actor_critic_2_m*.pt")))
    assert [os.path.basename(f) for f in files] == ["actor_critic_2_m0.pt", "actor_critic_2_m1.pt", "actor_critic_2_m2.pt"]
    weights = []
    for f in files:
        pol = compat.load_policy(f)
        assert os.path.getsize(f) < 200_000                        # the member's parameters, not the whole [K][P] buffer
        action, logp, ent, value = pol.evaluate(torch.randn(5, 4))
        assert action.shape == (5,) and value.shape == (5, 1) and torch.isfinite(logp).all()
        weights.append(torch.cat([p.detach().reshape(-1) for p in pol.parameters()]))
    assert not torch.equal(weights[0], weights[1])                 # different seeds, different members


def test_mountaincar_members_equal_standalone_runs_beyond_num_updates():
    # total_timesteps allows ONE update; the second iteration (annealed learning rate 0) needs Adam steps beyond the bias-correction
    # table sized at construction, which the population grows
    params = _params(gym_id="MountainCar-v0", num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2,
                     total_timesteps=200 * 32)
    members = [dict(seed=1.0), dict(seed=2.0, learning_rate=1e-3, entropy_coeff=0.0), dict(seed=3.0, clip_coeff=0.3)]
    pop = _check_vs_standalone(params, members, iters=2)
    assert pop.num_updates == 1 and all(int(s) == 16 for s in pop.steps.cpu())


@pytest.mark.parametrize("rollout_impl,update_impl", [(0, 0), (0, 3), (1, 2)])
def test_populations_ignore_the_single_run_kernel_switches(rollout_impl, update_impl):
    params = _params(num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2, total_timesteps=200 * 32 * 2)
    members = CARTPOLE_MEMBERS[:2]
    L = _lib.lib()
    states = []
    for switches in ((rollout_impl, update_impl), (1, 1)):
        L.aur_rollout_set_impl(switches[0])
        L.aur_ppo_update_set_impl(switches[1])
        pop = ppo_population(params, members)
        pop.reset_envs()
        for u in (1, 2):
            pop.run_update(u)
        states.append([_member_state(pop, k) for k in range(len(members))])
    for k in range(len(members)):
        _assert_equal(states[0][k], states[1][k], f"member {k} with rollout impl {rollout_impl}, update impl {update_impl} left set")
