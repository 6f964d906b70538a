"""Saving and resuming training, np.array_equal throughout: a run (A) trains U iterations without stopping; the same run (B) is
killed right after it wrote its state at iteration k, and a fresh object resumes from that file, through train(resume=...) and
through load_state() + train().  A and B must end with the same
parameters, Adam state, env state, rollout buffers, returns / advantages, episode lists, statistics and checkpoint files -- for
single runs on every kind of kernel path and for populations with and without PBT.  Also: resuming a finished run trains
nothing, saving adds no launch, a state from another configuration is refused before any kernel runs, and an incomplete state
is refused before anything changes."""
import json
import math
import os
import shutil

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, compat, kernels, run_ppo, state
from aur_ppo_b200.population import ppo_population
from aur_ppo_b200.ppo import ppo
from tests.test_population_gpu import default_impls  # noqa: F401 (autouse fixture)

pytestmark = pytest.mark.gpu


class _Killed(Exception):
    pass


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=True, num_envs=256, num_steps=32)
    p.update(kw)
    return p


def _np(t):
    return t.detach().cpu().numpy().copy()


def _same(a, b, what):
    if isinstance(a, float) and isinstance(b, float) and math.isnan(a) and math.isnan(b):
        return
    if isinstance(a, np.ndarray):
        assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b, equal_nan=a.dtype.kind == "f"), what
    elif isinstance(a, dict):
        assert a.keys() == b.keys(), what
        for k in a:
            _same(a[k], b[k], f"{what}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            _same(x, y, f"{what}[{i}]")
    else:
        assert a == b, (what, a, b)


def _buffers(obj):
    b = obj.buffer
    out = {f: _np(getattr(b, f)) for f in ("states", "actions", "log_probs", "rewards", "terminals", "values", "next_value")}
    out.update(returns=_np(obj._returns), advantages=_np(obj._advantages))
    out.update({f"env.{k}": _np(t) for k, t in state.env_tensors(obj.envs).items()})
    return out


def _ppo_snapshot(p, out):
    snap = dict(flat=_np(p.flat), exp_avg=_np(p.updater.exp_avg), exp_avg_sq=_np(p.updater.exp_avg_sq),
                step_count=p.updater.step_count, totals=_np(p.envs.totals), env_step=p._env_step, shuffle=p._shuffle_count,
                lists=out, last_stats=p.last_stats, lr=p.optimizer.param_groups[0]["lr"])
    snap.update(_buffers(p))
    return snap


def _pop_snapshot(p, out):
    snap = {k: _np(t) for k, t in p._state_tensors().items()}
    snap.update(_buffers(p))
    snap.update(lists=out, env_step=p._env_step, shuffle=p._shuffle_count, iterations=p._iterations,
                member_params=p.member_params, any_target_kl=p.any_target_kl, pbt_round=p.pbt_round, lineage=p.lineage)
    return snap


def _checkpoints(d):
    out = {}
    for f in sorted(os.listdir(d)):
        if f.startswith("actor_critic_"):
            out[f] = {n: _np(t) for n, t in compat.load_policy(os.path.join(d, f)).state_dict().items()}
        elif f == "pbt_lineage.json":
            out[f] = json.load(open(os.path.join(d, f)))
    return out


def _a_and_resumed_b(make, k, tmp_path, monkeypatch, snapshot):
    """(A's snapshot and files, B's snapshot and files, the final state path) for an uninterrupted run A and a run B killed
    after its state write at iteration k and resumed with train(resume=...).  A third object resumed with load_state() and a
    plain train() must end exactly as B."""
    for d in ("a", "b", "d"):
        os.makedirs(tmp_path / d)
    path, path_k = str(tmp_path / "state.pt"), str(tmp_path / "state_k.pt")
    monkeypatch.chdir(tmp_path / "a")
    a = make()
    sa = snapshot(a, a.train())
    monkeypatch.chdir(tmp_path / "b")
    real = state.write

    def write_then_die(*args, **kw):
        real(*args, **kw)
        raise _Killed()

    monkeypatch.setattr(state, "write", write_then_die)
    with pytest.raises(_Killed):
        make().train(save_state_every=k, state_path=path)
    monkeypatch.setattr(state, "write", real)
    assert torch.load(path, weights_only=True)["iteration"] == k
    shutil.copy(path, path_k)
    b = make()
    sb = snapshot(b, b.train(save_state_every=k, state_path=path, resume=path))
    assert b._iteration == a.num_updates
    monkeypatch.chdir(tmp_path / "d")
    d = make()
    d.load_state(path_k)
    sd = snapshot(d, d.train())
    _same(sd, sb, "load_state() + train() vs train(resume=...)")
    _same(_checkpoints(tmp_path / "d"), _checkpoints(tmp_path / "b"), "load_state() + train() checkpoints")
    return (sa, _checkpoints(tmp_path / "a")), (sb, _checkpoints(tmp_path / "b")), path


def _make_ppo(params):
    def make():
        torch.manual_seed(1)
        return ppo(dict(params))
    return make


PPO_CASES = {
    # fused 64 x 2 tensor-core kernels; lr annealing; target_kl low enough that epochs stop early
    "cartpole_target_kl": (dict(target_kl=1e-6), 4, 2),
    # 128-step rollouts so that 200-step episodes finish
    "pendulum_wrappers": (dict(gym_id="Pendulum-v1", continuous=True, learning_rate=3e-4, entropy_coeff=0.0, num_steps=128), 3, 1),
    "cartpole_hidden128": (dict(hidden_dim=128), 3, 2),
    "acrobot_generic": (dict(gym_id="Acrobot-v1"), 3, 1),
}


@pytest.mark.parametrize("case", list(PPO_CASES))
def test_a_resumed_run_equals_an_uninterrupted_one(case, tmp_path, monkeypatch):
    kw, U, k = PPO_CASES[case]
    params = _params(**kw)
    params["total_timesteps"] = params["num_envs"] * params["num_steps"] * U
    (sa, fa), (sb, fb), path = _a_and_resumed_b(_make_ppo(params), k, tmp_path, monkeypatch, _ppo_snapshot)
    _same(sb, sa, case)
    _same(fb, fa, f"{case} checkpoints")
    assert list(fa) == ["actor_critic_2.pt"]
    if case == "cartpole_target_kl":
        assert sa["step_count"] < U * 4 * 4, "no epoch stopped early: target_kl does not bite"
    # the final state: resuming it runs no iteration, returns the same lists and writes the same checkpoint
    os.makedirs(tmp_path / "c")
    monkeypatch.chdir(tmp_path / "c")
    c = _make_ppo(params)()
    L = _lib.lib()
    torch.cuda.synchronize()
    L.aur_launch_count_reset()
    out = c.train(resume=path)
    torch.cuda.synchronize()
    assert L.aur_launch_count() == 0
    _same(out, sa["lists"], f"{case} final resume")
    _same(c.last_stats, sa["last_stats"], f"{case} final resume")
    _same(_checkpoints(tmp_path / "c"), fa, f"{case} final resume checkpoint")


def _members(K):
    return run_ppo.expand_members(1.0, K // 2, ["learning_rate=1e-4,1e-3"])


POP_CASES = {
    "cartpole_pbt": (dict(), 6, dict(interval=1, fraction=0.5), 4, 2),
    "pendulum_wrappers": (dict(gym_id="Pendulum-v1", continuous=True, learning_rate=3e-4, entropy_coeff=0.0, num_steps=128), 4,
                          None, 3, 1),
}


@pytest.mark.parametrize("case", list(POP_CASES))
def test_a_resumed_population_equals_an_uninterrupted_one(case, tmp_path, monkeypatch):
    kw, K, pbt, U, k = POP_CASES[case]
    params = _params(num_envs=200, **kw)
    params["total_timesteps"] = params["num_envs"] * params["num_steps"] * U
    members = _members(K)
    make = lambda: ppo_population(dict(params), members, pbt=pbt)
    (sa, fa), (sb, fb), path = _a_and_resumed_b(make, k, tmp_path, monkeypatch, _pop_snapshot)
    _same(sb, sa, case)
    _same(fb, fa, f"{case} checkpoints")
    assert sorted(f for f in fa if f.startswith("actor_critic")) == [f"actor_critic_2_m{m}.pt" for m in range(K)]
    if pbt is not None:
        assert sa["pbt_round"] == U - 1 and "pbt_lineage.json" in fa
        assert any(d >= 0 for e in sa["lineage"] for d in e["donor"]), "no PBT round copied anything"
        assert len({mp["learning_rate"] for mp in sa["member_params"]}) > 2   # PBT moved the learning rates
    # the final state: no iteration, same lists
    os.makedirs(tmp_path / "c")
    monkeypatch.chdir(tmp_path / "c")
    c = make()
    L = _lib.lib()
    torch.cuda.synchronize()
    L.aur_launch_count_reset()
    out = c.train(resume=path)
    torch.cuda.synchronize()
    assert L.aur_launch_count() == 0
    _same(out, sa["lists"], f"{case} final resume")
    _same(_checkpoints(tmp_path / "c"), fa, f"{case} final resume checkpoints")


def test_saving_adds_no_launch(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    U = 3
    params = _params(total_timesteps=256 * 32 * U, save=False)
    L = _lib.lib()
    counts = []
    for how in ("by hand", 0, 1):
        p = _make_ppo(params)()
        torch.cuda.synchronize()
        L.aur_launch_count_reset()
        if how == "by hand":           # what train() launched before it could save: env reset + U iterations
            p.envs.reset(seed=list(p.plan.env_ids))
            p._stats_rows = torch.zeros(p.num_update_epochs * p.num_minibatches, kernels.NUM_STATS, device=p.device)
            for u in range(1, U + 1):
                p.run_update(u)
        else:
            p.train(save_state_every=how, state_path=str(tmp_path / "s.pt"))
        torch.cuda.synchronize()
        counts.append(L.aur_launch_count())
    assert counts[0] == counts[1] == counts[2] > 0, counts


def test_another_configuration_is_refused_before_any_kernel(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    path = str(tmp_path / "s.pt")
    params = _params(total_timesteps=256 * 32 * 2, save=False)
    _make_ppo(params)().train(save_state_every=1, state_path=path)
    pop_path = str(tmp_path / "pop.pt")
    members = _members(2)
    ppo_population(dict(params), members).train(save_state_every=2, state_path=pop_path)
    L = _lib.lib()
    bad = [(lambda: _make_ppo(dict(params, learning_rate=1e-3))(), path, "learning_rate"),
           (lambda: _make_ppo(dict(params, num_envs=128))(), path, "num_envs"),
           (lambda: _make_ppo(params)(), pop_path, "'population' run"),
           (lambda: ppo_population(dict(params), members), path, "'ppo' run"),
           (lambda: ppo_population(dict(params), members, pbt=dict(interval=1)), pop_path, r"pbt"),
           (lambda: ppo_population(dict(params), _members(4)), pop_path, "members")]
    for make, p, what in bad:
        obj = make()
        torch.cuda.synchronize()
        L.aur_launch_count_reset()
        with pytest.raises(_lib.AurError, match=what):
            obj.train(resume=p)
        torch.cuda.synchronize()
        assert L.aur_launch_count() == 0, what


def test_incomplete_states_are_refused_and_change_nothing(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    params = _params(total_timesteps=256 * 32 * 2, save=False)
    p = _make_ppo(params)()
    with pytest.raises(_lib.AurError, match="no iteration"):
        p.save_state(str(tmp_path / "early.pt"))          # before train(): nothing to resume from
    assert not os.path.exists(tmp_path / "early.pt")
    path = str(tmp_path / "s.pt")
    p.train(save_state_every=1, state_path=path)
    full = torch.load(path, weights_only=True)
    fresh = _make_ppo(params)()
    before = {k: _np(t) for k, t in dict(fresh._state_tensors(), **state.env_tensors(fresh.envs)).items()}
    for drop in ("env_step", "x_indices", "last_stats", "iteration"):
        torch.save({k: v for k, v in full.items() if k != drop}, path)
        with pytest.raises(_lib.AurError, match="lacks|no completed iteration"):
            fresh.load_state(path)
    torch.save(dict(full, iteration=0), path)
    with pytest.raises(_lib.AurError, match="no completed iteration"):
        fresh.load_state(path)
    torch.save(dict(full, x_indices=[1, 2]), path)
    with pytest.raises(_lib.AurError, match="malformed"):
        fresh.load_state(path)
    after = {k: _np(t) for k, t in dict(fresh._state_tensors(), **state.env_tensors(fresh.envs)).items()}
    _same(after, before, "a refused state changed the run")
    assert fresh._iteration == 0 and fresh._env_step == 0 and not fresh._resumed
