"""Population-based training on the device, np.array_equal throughout: the rank / exploit kernels against oracle/pbt_ref.py on
crafted fitness vectors; a round on a live population copying exactly the donor's state and nothing else; a population with
PBT equal, iteration after iteration, to one without PBT to which each round's donors are transplanted by plain indexing; the
default episode fitness; launch counts; the CLI end to end."""
import ctypes
import glob
import json
import os

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, compat, kernels, population, run_ppo
from aur_ppo_b200.population import ppo_population
from oracle import pbt_ref
from tests.test_population_gpu import _assert_equal, _member_state, _np, _params, default_impls  # noqa: F401 (autouse fixture)

pytestmark = pytest.mark.gpu

NAN, INF = float("nan"), float("inf")


# ------------------------------------------------------------------------------------------------ 1. decision kernels
def _fitness(kind, K, rng):
    if kind == "random":
        return rng.standard_normal(K)
    if kind == "ties":
        return rng.integers(-2, 3, K).astype(np.float64)
    f = rng.integers(-1, 2, K).astype(np.float64)                   # -1, 0, 1 with specials mixed in
    special = np.array([NAN, INF, -INF, 0.0, -0.0])
    pick = rng.random(K) < 0.5
    f[pick] = special[rng.integers(0, 5, int(pick.sum()))]
    return f


@pytest.mark.parametrize("K", [2, 3, 64, 1000, 5000])
def test_decision_kernels_equal_the_oracle(K):
    L = _lib.lib()
    dev = torch.device("cuda:0")
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    P = kernels.policy_param_count(desc)
    seeds = torch.arange(K, dtype=torch.int64, device=dev)
    pop = _lib.PopDesc(K, 0, 4, seeds.data_ptr())
    rng = np.random.default_rng(K)
    rows0 = [torch.randn(K, P, device=dev) for _ in range(3)]
    steps0 = torch.from_numpy(rng.integers(1, 1000, K)).to(dev)
    hp0 = np.exp(rng.uniform(-8, 0, (K, 6)))
    hp0[rng.random(K) < 0.3, 5] = INF
    rank, donor, order = (torch.empty(n, dtype=torch.int32, device=dev) for n in (K, K, K + 1))
    cases = [("random", 0.25, 0b000011, 1, 1), ("ties", 0.5, 0b111111, 2 ** 40 + 3, 7), ("special", 0.1, 0b100001, 5, 2 ** 33 + 5),
             ("special", 0.5, 0b010100, 2 ** 63 + 9, 3), ("ties", 0.3, 0, 77, 1)]
    for kind, q, mask, seed, rnd in cases:
        f = _fitness(kind, K, rng)
        rows = [r.clone() for r in rows0]
        steps = steps0.clone()
        hp = torch.from_numpy(hp0).to(dev)
        fit = torch.from_numpy(f).to(dev)
        a = _lib.PopPbtArgs()
        a.fitness, a.q, a.down, a.up, a.mask, a.seed, a.round = fit.data_ptr(), q, 0.8, 1.25, mask, seed, rnd
        a.params, a.adam_m, a.adam_v = (r.data_ptr() for r in rows)
        a.steps, a.hparams, a.norm, a.norm_ld = steps.data_ptr(), hp.data_ptr(), None, 0
        a.rank_out, a.donor_out, a.order = rank.data_ptr(), donor.data_ptr(), order.data_ptr()
        _lib.check(L.aur_pop_pbt_step(ctypes.byref(pop), ctypes.byref(desc), ctypes.byref(a), None), "aur_pop_pbt_step")
        want_rank, want_donor, want_hp = pbt_ref.decide(f, q, 0.8, 1.25, mask, seed, rnd, hp0)
        what = f"K {K}, {kind}, q {q}, seed {seed}, round {rnd}"
        assert np.array_equal(_np(rank), want_rank), what
        assert np.array_equal(_np(donor), want_donor), what
        assert np.array_equal(_np(hp), want_hp), what
        assert int(order[K]) == int((~np.isnan(f)).sum()), what
        src = torch.arange(K, device=dev)
        rec = torch.from_numpy(want_donor >= 0).to(dev)
        src[rec] = torch.from_numpy(want_donor.astype(np.int64)).to(dev)[rec]
        for r, r0 in zip(rows, rows0):
            assert torch.equal(r, r0[src]), what
        assert torch.equal(steps, steps0[src]), what


# ------------------------------------------------------------------------------------------------ 2. exploit on a live population
ENVS = {
    "cartpole": dict(),
    "pendulum": dict(gym_id="Pendulum-v1", continuous=True, learning_rate=3e-4, entropy_coeff=0.0),
}


def _pop_params(env, iters):
    return _params(num_envs=200, num_steps=32, num_minibatches=4, num_update_epochs=2, total_timesteps=200 * 32 * iters, **ENVS[env])


def _members(K):
    return [dict(seed=float(k + 1), learning_rate=1e-4 * (k + 1), entropy_coeff=0.001 * k) for k in range(K)]


def _env_state(pop):
    e = pop.envs
    out = dict(phys=_np(e.phys), pcg=_np(e.pcg), elapsed=_np(e.elapsed), ep_return=_np(e.ep_return), ep_length=_np(e.ep_length),
               seeds=_np(pop.seeds), states=_np(pop.buffer.states), next_obs=_np(e.next_obs))
    if e.norm is not None:
        out["norm"] = _np(e.norm)
    return out


@pytest.mark.parametrize("env", ["cartpole", "pendulum"])
def test_a_round_copies_exactly_the_donor_state(env):
    K = 8
    pop = ppo_population(_pop_params(env, 2), _members(K), pbt=dict(interval=1, fraction=0.5))
    pop.reset_envs()
    pop.run_update(1)
    rows0 = [_np(t) for t in (pop.params, pop.exp_avg, pop.exp_avg_sq)]
    steps0, hp0, env0 = _np(pop.steps), _np(pop.hparams), _env_state(pop)
    f = np.array([0.5, 3.0, NAN, -1.0, 2.0, 7.0, -4.0, 1.0])
    out = pop.pbt_step(torch.from_numpy(f).to(pop.device))
    donor = _np(out["donor"])
    _, want_donor, want_hp = pbt_ref.decide(f, 0.5, 0.8, 1.2, 0b11, int(pop.params_dict["seed"]), 1, hp0)
    # order 5, 1, 4, 7, 0, 3, 6 (2 is not ranked); n_sel = floor(0.5 * 7) = 3: members 0, 3, 6 receive from 5, 1 or 4
    assert np.array_equal(donor, want_donor) and np.nonzero(donor >= 0)[0].tolist() == [0, 3, 6]
    assert set(donor[[0, 3, 6]].tolist()) <= {5, 1, 4}
    assert np.array_equal(_np(pop.hparams), want_hp)
    rows = [_np(t) for t in (pop.params, pop.exp_avg, pop.exp_avg_sq)]
    steps, env1 = _np(pop.steps), _env_state(pop)
    for k in range(K):
        src = donor[k] if donor[k] >= 0 else k
        for r, r0 in zip(rows, rows0):
            assert np.array_equal(r[k], r0[src]), (k, src)
        assert steps[k] == steps0[src]
    # env physics, PCG, TimeLimit counters, episode accumulators, seeds and buffers: untouched for every member
    for key in env0:
        if key != "norm":
            assert np.array_equal(env1[key], env0[key]), key
    if "norm" in env0:
        n, D = pop.n_member, pop.state_dim[0]
        for k in range(K):
            src = donor[k] if donor[k] >= 0 else k
            cols, dcols = slice(k * n, (k + 1) * n), slice(src * n, (src + 1) * n)
            assert np.array_equal(env1["norm"][:2 * D + 4, cols], env0["norm"][:2 * D + 4, dcols]), (k, "wrapper statistics")
            assert np.array_equal(env1["norm"][2 * D + 4, cols], env0["norm"][2 * D + 4, cols]), (k, "return accumulator")


# ------------------------------------------------------------------------------------------------ 3. transplant equivalence
def _full_state(pop, k):
    st = _member_state(pop, k)
    n = pop.n_member
    e = pop.envs
    st.update(hparams=_np(pop.hparams[k]), phys=_np(e.phys[:, k * n:(k + 1) * n]), pcg=_np(e.pcg[:, k * n:(k + 1) * n]),
              elapsed=_np(e.elapsed[k * n:(k + 1) * n]), ep_return=_np(e.ep_return[k * n:(k + 1) * n]))
    if e.norm is not None:
        st["norm"] = _np(e.norm[:, k * n:(k + 1) * n])
    return st


def _transplant(b, donor, hp):
    rec = np.nonzero(donor >= 0)[0]
    if len(rec) == 0:
        return
    d = torch.from_numpy(donor[rec].astype(np.int64)).to(b.device)
    r = torch.from_numpy(rec.astype(np.int64)).to(b.device)
    for t in (b.params, b.exp_avg, b.exp_avg_sq, b.steps):
        t[r] = t[d]
    b.hparams.copy_(torch.from_numpy(hp))
    if b.envs.norm is not None:
        n, D = b.n_member, b.state_dim[0]
        for k, dk in zip(rec.tolist(), donor[rec].tolist()):
            b.envs.norm[:2 * D + 4, k * n:(k + 1) * n] = b.envs.norm[:2 * D + 4, dk * n:(dk + 1) * n]


@pytest.mark.parametrize("env", ["cartpole", "pendulum"])
def test_a_round_is_exactly_a_state_transplant(env):
    K, iters = 8, 3
    params = _pop_params(env, iters)
    pbt = dict(interval=1, fraction=0.5, keys=("learning_rate", "entropy_coeff", "clip_coeff"), factors=(0.5, 2.0))
    a = ppo_population(params, _members(K), pbt=pbt)
    b = ppo_population(params, _members(K))
    for p in (a, b):
        p.reset_envs()
    rng = np.random.default_rng(3)
    moved = 0
    for u in range(1, iters + 1):
        a.run_update(u)
        b.run_update(u)
        for k in range(K):
            _assert_equal(_full_state(a, k), _full_state(b, k), f"{env}, iteration {u}, member {k}")
        if u == iters:
            break
        # CartPole: the default fitness (episodes finish within an iteration); Pendulum's 200-step episodes do not, so a
        # crafted vector with a NaN stands in
        fit = None if env == "cartpole" else torch.from_numpy(np.where(rng.random(K) < 0.2, NAN, rng.standard_normal(K))).to(a.device)
        hp_before = _np(b.hparams)
        out = a.pbt_step(fit)
        f, donor = _np(out["fitness"]), _np(out["donor"])
        _, want_donor, want_hp = pbt_ref.decide(f, 0.5, 0.5, 2.0, 0b111, int(params["seed"]), u, hp_before)
        assert np.array_equal(donor, want_donor) and np.array_equal(_np(a.hparams), want_hp)
        moved += int((donor >= 0).sum())
        _transplant(b, donor, want_hp)
    assert moved > 0


# ------------------------------------------------------------------------------------------------ 4. default fitness
def test_episode_fitness_is_the_mean_return_since_the_last_round():
    K = 4
    pop = ppo_population(_pop_params("cartpole", 2), _members(K), pbt=dict(interval=1))
    L = _lib.lib()
    pop.reset_envs()
    snap = np.zeros((K, 3))
    for u in (1, 2):
        pop.run_update(u)
        tot = _np(pop.totals)
        _lib.check(L.aur_pop_episode_fitness(ctypes.byref(pop.pop), pop.totals.data_ptr(), pop.pbt_snapshot.data_ptr(),
                                             pop.pbt_fitness.data_ptr(), None), "aur_pop_episode_fitness")
        d = tot - snap
        assert (d[:, 0] > 0).all()
        assert np.array_equal(_np(pop.pbt_fitness), d[:, 1] / d[:, 0]), u
        assert np.array_equal(_np(pop.pbt_snapshot), tot)
        snap = tot
    # no episode finished since the snapshot: NaN for every member
    _lib.check(L.aur_pop_episode_fitness(ctypes.byref(pop.pop), pop.totals.data_ptr(), pop.pbt_snapshot.data_ptr(),
                                         pop.pbt_fitness.data_ptr(), None), "aur_pop_episode_fitness")
    assert np.isnan(_np(pop.pbt_fitness)).all()
    # Pendulum: 200-step episodes, none finishes in 32 steps
    pend = ppo_population(_pop_params("pendulum", 1), _members(3), pbt=dict(interval=1))
    pend.reset_envs()
    pend.run_update(1)
    out = pend.pbt_step()
    assert np.isnan(_np(out["fitness"])).all() and (_np(out["donor"]) == -1).all()


# ------------------------------------------------------------------------------------------------ 5. launch counts
def test_a_round_is_three_launches_and_iterations_are_unchanged():
    params = _params(num_envs=128, num_steps=16, num_minibatches=4, num_update_epochs=2, total_timesteps=128 * 16 * 4)
    L = _lib.lib()
    for K in (2, 256):
        members = [dict(seed=float(k + 1)) for k in range(K)]
        counts = []
        for pbt in (None, dict(interval=1)):
            pop = ppo_population(params, members, pbt=pbt)
            pop.reset_envs()
            pop.run_update(1)
            torch.cuda.synchronize()
            L.aur_launch_count_reset()
            pop.run_update(2)
            torch.cuda.synchronize()
            counts.append(L.aur_launch_count())
        assert counts[0] == counts[1] == 8 + 3 * 8, (K, counts)
        L.aur_launch_count_reset()
        pop.pbt_step()
        torch.cuda.synchronize()
        assert L.aur_launch_count() == 3, K


# ------------------------------------------------------------------------------------------------ 6. CLI
def test_cli_pbt_end_to_end(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    made = []

    class Recording(ppo_population):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            made.append(self)

    monkeypatch.setattr(population, "ppo_population", Recording)
    out = run_ppo.main(["--population", "4", "--pbt_interval", "1", "--num_envs", "256", "--num_steps", "32",
                        "--total_timesteps", str(256 * 32 * 3), "--no_tensorboard"])
    assert len(out) == 4 and len(made) == 1
    pop = made[0]
    lineage = json.load(open(tmp_path / "pbt_lineage.json"))
    assert [e["iteration"] for e in lineage] == [1, 2] and len(pop.lineage) == 2
    for e, want in zip(lineage, pop.lineage):
        assert e["donor"] == want["donor"] and e["hparams"] == want["hparams"] and e["fitness"] == want["fitness"]
        assert len(e["donor"]) == 4 and len(e["hparams"]) == 4
    assert sum(d >= 0 for e in lineage for d in e["donor"]) == 2             # n_sel = floor(0.25 * 4) = 1 per round
    assert [pop.member_params[k]["learning_rate"] for k in range(4)] == [h["learning_rate"] for h in lineage[-1]["hparams"]]
    files = sorted(glob.glob(str(tmp_path / "actor_critic_2_m*.pt")))
    assert [os.path.basename(f) for f in files] == [f"actor_critic_2_m{k}.pt" for k in range(4)]
    for f in files:
        pol = compat.load_policy(f)
        action, logp, ent, value = pol.evaluate(torch.randn(5, 4))
        assert action.shape == (5,) and torch.isfinite(logp).all()
