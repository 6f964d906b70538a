"""The training-state file (aur_ppo_b200/state.py) and the CLI flags that write and resume it.  CPU only: a round trip through
torch.load(weights_only=True), every refusal of a state that does not fit the run, atomic writes, and argument parsing."""
import os

import pytest
import torch

from aur_ppo_b200 import _lib, population, ppo as ppo_mod, run_ppo, state
from tests.test_host_api import REF_KEYS


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(kw)
    return p


def _body():
    return dict(tensors=dict(flat=torch.arange(10, dtype=torch.float32), steps=torch.tensor([3, 4], dtype=torch.int64)),
                env=dict(phys=torch.randn(4, 6, dtype=torch.float64)), iteration=3, run_name="CartPole-v1__x__1.0__7",
                total_returns=[1.0, 2.5], last_stats=dict(value_loss=0.25, explained_variance=float("nan")),
                lineage=[dict(iteration=1, fitness=[None, 1.5], donor=[-1, 0])])


def test_round_trip_loads_with_weights_only(tmp_path):
    path = str(tmp_path / "s.pt")
    fp = state.fingerprint(_params())
    body = _body()
    state.write(path, "ppo", fp, body)
    raw = torch.load(path, weights_only=True)
    assert (raw["format"], raw["version"], raw["kind"]) == ("aur_ppo_training_state", 1, "ppo")
    got = state.read(path, "ppo", fp)
    assert got["fingerprint"] == fp
    assert torch.equal(got["tensors"]["flat"], body["tensors"]["flat"]) and got["tensors"]["steps"].dtype == torch.int64
    assert torch.equal(got["env"]["phys"], body["env"]["phys"])
    assert got["iteration"] == 3 and got["run_name"] == body["run_name"] and got["total_returns"] == [1.0, 2.5]
    assert got["lineage"] == body["lineage"] and got["last_stats"]["value_loss"] == 0.25
    assert not os.path.exists(path + ".tmp")


def test_non_computing_keys_may_differ(tmp_path):
    path = str(tmp_path / "s.pt")
    state.write(path, "ppo", state.fingerprint(_params()), _body())
    other = _params(track=True, capture_video=True, exp_name="renamed", tensorboard=False, save=False, device="cuda:3")
    state.read(path, "ppo", state.fingerprint(other))


def test_each_differing_key_is_named(tmp_path):
    path = str(tmp_path / "s.pt")
    state.write(path, "ppo", state.fingerprint(_params(philox_seed=5)), _body())
    changed = dict(learning_rate=1e-3, num_envs=8, total_timesteps=1000, gym_id="Pendulum-v1", target_kl=0.01)
    with pytest.raises(_lib.AurError) as e:
        state.read(path, "ppo", state.fingerprint(_params(philox_seed=6, **changed)))
    for key in ["philox_seed", *changed]:
        assert key in str(e.value), key
    # a key present on one side only
    with pytest.raises(_lib.AurError, match="shuffle_seed"):
        state.read(path, "ppo", state.fingerprint(_params(philox_seed=5, shuffle_seed=5)))


def _pop_fp(members=None, pbt=dict(interval=2), **kw):
    members = members or [dict(seed=1.0, learning_rate=1e-4), dict(seed=2.0, learning_rate=1e-3)]
    return state.fingerprint(_params(**kw), population.check_members(_params(**kw), members),
                             population.check_pbt(pbt, len(members)) if pbt is not None else None)


def test_population_members_and_pbt_config_are_compared(tmp_path):
    path = str(tmp_path / "s.pt")
    state.write(path, "population", _pop_fp(), _body())
    state.read(path, "population", _pop_fp(exp_name="other"))
    with pytest.raises(_lib.AurError, match="members"):
        state.read(path, "population", _pop_fp(members=[dict(seed=1.0, learning_rate=1e-4), dict(seed=2.0, learning_rate=2e-3)]))
    with pytest.raises(_lib.AurError, match="members"):
        state.read(path, "population", _pop_fp(members=[dict(seed=1.0, learning_rate=1e-4)] * 3))
    for pbt, what in ((dict(interval=3), "pbt.interval"), (dict(interval=2, fraction=0.5), "pbt.fraction"),
                      (dict(interval=2, keys=("clip_coeff",)), "pbt.keys"), (dict(interval=2, factors=(0.5, 2.0)), "pbt.factors"),
                      (None, "pbt")):
        with pytest.raises(_lib.AurError, match=what.replace(".", r"\.")):
            state.read(path, "population", _pop_fp(pbt=pbt))
    with pytest.raises(_lib.AurError, match="params.gamma"):
        state.read(path, "population", _pop_fp(gamma=0.9))


def test_kind_format_and_version_are_checked(tmp_path):
    path = str(tmp_path / "s.pt")
    fp = state.fingerprint(_params())
    state.write(path, "ppo", fp, _body())
    with pytest.raises(_lib.AurError, match="'ppo' run and cannot be loaded into a 'population'"):
        state.read(path, "population", fp)
    state.write(path, "population", _pop_fp(), _body())
    with pytest.raises(_lib.AurError, match="'population' run and cannot be loaded into a 'ppo'"):
        state.read(path, "ppo", fp)
    obj = torch.load(path, weights_only=True)
    for key, value, what in (("version", 2, "version 2"), ("format", "something_else", "not an aur_ppo training state")):
        torch.save(dict(obj, **{key: value}), path)
        with pytest.raises(_lib.AurError, match=what):
            state.read(path, "population", _pop_fp())
    with pytest.raises(_lib.AurError, match="does not exist"):
        state.read(str(tmp_path / "missing.pt"), "ppo", fp)
    with open(path, "wb") as f:
        f.write(b"not a torch file")
    with pytest.raises(_lib.AurError, match="not a readable state file"):
        state.read(path, "ppo", fp)


def test_loading_refuses_pickled_code(tmp_path):
    path = str(tmp_path / "s.pt")
    torch.save(dict(format=state.FORMAT, version=1, kind="ppo", fingerprint={}, hook=_Opaque()), path)
    with pytest.raises(_lib.AurError, match="not a readable state file"):
        state.read(path, "ppo", {})


class _Opaque:
    pass


def test_tensor_shape_and_dtype_are_checked_before_any_copy():
    a, b = torch.zeros(4), torch.zeros(2, 3, dtype=torch.int64)
    with pytest.raises(_lib.AurError, match=r"b is torch.int64 \(2, 4\)"):
        state.restore([("a", a, torch.ones(4)), ("b", b, torch.ones(2, 4, dtype=torch.int64))])
    with pytest.raises(_lib.AurError, match=r"a is torch.float64"):
        state.restore([("a", a, torch.ones(4, dtype=torch.float64))])
    with pytest.raises(_lib.AurError, match="a is missing"):
        state.restore([("a", a, None)])
    assert not a.any() and not b.any()                    # nothing was copied
    state.restore([("a", a, torch.ones(4)), ("b", b, torch.full((2, 3), 7))])
    assert (a == 1).all() and (b == 7).all()


def test_a_failed_write_leaves_the_previous_state(tmp_path, monkeypatch):
    path = str(tmp_path / "s.pt")
    fp = state.fingerprint(_params())
    state.write(path, "ppo", fp, _body())
    before = open(path, "rb").read()
    real_save = torch.save

    def dies_midway(obj, f, *a, **kw):
        f.write(b"PK\x03\x04 half a zip")
        raise RuntimeError("disk full")

    monkeypatch.setattr(torch, "save", dies_midway)
    body = _body()
    body["iteration"] = 4
    with pytest.raises(RuntimeError, match="disk full"):
        state.write(path, "ppo", fp, body)
    monkeypatch.setattr(torch, "save", real_save)
    assert open(path, "rb").read() == before
    assert state.read(path, "ppo", fp)["iteration"] == 3
    assert not os.path.exists(path + ".tmp")


def test_cli_defaults_keep_the_reference_keys():
    args = run_ppo.build_parser().parse_args([])
    assert list(run_ppo.params_from_args(args).keys()) == REF_KEYS
    assert args.save_state_every == 0 and args.resume is None
    args = run_ppo.build_parser().parse_args(["--save_state_every", "2", "--resume", "run.pt"])
    assert list(run_ppo.params_from_args(args).keys()) == REF_KEYS
    assert (args.save_state_every, args.resume) == (2, "run.pt")


class _Recorder:
    made = []

    def __init__(self, *a, **kw):
        self.args = a
        _Recorder.made.append(self)

    def train(self, **kw):
        self.train_kw = kw
        return []


def test_cli_passes_the_state_options_to_train(monkeypatch):
    monkeypatch.setattr(ppo_mod, "ppo", _Recorder)
    monkeypatch.setattr(population, "ppo_population", _Recorder)
    _Recorder.made.clear()
    run_ppo.main(["--save_state_every", "3"])
    run_ppo.main(["--resume", "x.pt", "--population", "2", "--pbt_interval", "1"])
    run_ppo.main([])
    kws = [r.train_kw for r in _Recorder.made]
    assert kws == [dict(save_state_every=3, resume=None), dict(save_state_every=0, resume="x.pt"),
                   dict(save_state_every=0, resume=None)]
    assert len(_Recorder.made[1].args[1]) == 2                 # the population got its members
    with pytest.raises(SystemExit):
        run_ppo.main(["--save_state_every", "-1"])


def test_numpy_scalars_are_stored_as_python_values(tmp_path):
    import numpy as np
    path = str(tmp_path / "s.pt")
    params = _params(total_timesteps=np.int64(4096), learning_rate=np.float32(1e-3), seed=np.float64(2.0))
    state.write(path, "ppo", state.fingerprint(params), dict(_body(), iteration=np.int64(3)))
    got = state.read(path, "ppo", state.fingerprint(params))
    assert type(got["fingerprint"]["total_timesteps"]) is int and got["iteration"] == 3
    state.read(path, "ppo", state.fingerprint(_params(total_timesteps=4096, learning_rate=float(np.float32(1e-3)), seed=2.0)))


def test_a_value_that_cannot_be_loaded_is_refused_at_write(tmp_path):
    path = str(tmp_path / "s.pt")
    fp = state.fingerprint(_params())
    state.write(path, "ppo", fp, _body())
    before = open(path, "rb").read()
    with pytest.raises(_lib.AurError, match="_Opaque cannot be stored"):
        state.write(path, "ppo", fp, dict(_body(), extra=[_Opaque()]))
    with pytest.raises(_lib.AurError, match="cannot be stored"):
        state.fingerprint(_params(device=object(), gym_id=_Opaque()))
    assert open(path, "rb").read() == before and not os.path.exists(path + ".tmp")


def test_a_state_without_a_completed_iteration_is_refused(tmp_path):
    path = str(tmp_path / "s.pt")
    fp = state.fingerprint(_params())
    for it in (0, None, "3"):
        state.write(path, "ppo", fp, dict(_body(), iteration=it))
        with pytest.raises(_lib.AurError, match="no completed iteration"):
            state.read(path, "ppo", fp)


def test_histories_round_trip_exactly():
    import numpy as np
    rets = [float(v) for v in np.random.default_rng(0).standard_normal(1000).astype(np.float32)] + [500.0]
    xs = [3 * 2 ** 40, 0, 7]
    assert state.history(rets, np.float64).tolist() == rets and state.history(xs, np.int64).tolist() == xs
    assert state.history([], np.int64).tolist() == []
    assert state.fields(dict(a=1, b=2), ("a",)) == dict(a=1)
    with pytest.raises(_lib.AurError, match=r"lacks \['c'\]"):
        state.fields(dict(a=1), ("a", "c"))
