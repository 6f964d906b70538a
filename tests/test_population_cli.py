"""Populations without a GPU: the --population / --sweep expansion into member dicts, and the requests ppo_population refuses
(AurError before any kernel runs) - a shared key that differs between members, shapes / envs outside the population kernels,
data-parallel runs.  Also the population entry points' argument checks through the C ABI."""
import ctypes

import pytest

from aur_ppo_b200 import _lib, run_ppo
from aur_ppo_b200.population import check_members, member_params, ppo_population


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False)
    p.update(kw)
    return p


def test_no_flag_is_a_single_run():
    assert run_ppo.expand_members(1.0, 0, []) == []


def test_population_gives_consecutive_seeds():
    args = run_ppo.build_parser().parse_args(["--population", "3", "--seed", "7"])
    assert run_ppo.expand_members(args.seed, args.population, args.sweep) == [{"seed": 7.0}, {"seed": 8.0}, {"seed": 9.0}]


def test_sweep_is_the_cartesian_product_with_the_seeds():
    args = run_ppo.build_parser().parse_args(["--population", "2", "--sweep", "learning_rate=1e-3,3e-4",
                                              "--sweep", "target_kl=none,0.02"])
    got = run_ppo.expand_members(args.seed, args.population, args.sweep)
    assert len(got) == 8
    assert got[0] == {"seed": 1.0, "learning_rate": 1e-3, "target_kl": None}
    assert got[1] == {"seed": 2.0, "learning_rate": 1e-3, "target_kl": None}
    assert got[2] == {"seed": 1.0, "learning_rate": 1e-3, "target_kl": 0.02}
    assert got[-1] == {"seed": 2.0, "learning_rate": 3e-4, "target_kl": 0.02}


def test_sweep_alone_runs_one_seed_per_combination():
    assert run_ppo.expand_members(1.0, 0, ["clip_coeff=0.1,0.2"]) == [{"seed": 1.0, "clip_coeff": 0.1}, {"seed": 1.0, "clip_coeff": 0.2}]


@pytest.mark.parametrize("spec", ["num_envs=4,8", "seed=1,2", "learning_rate", "learning_rate=", "entropy_coeff=0.1,,0.2"])
def test_bad_sweeps_are_refused(spec):
    with pytest.raises(ValueError):
        run_ppo.expand_members(1.0, 2, [spec])
    with pytest.raises(SystemExit):
        run_ppo.main(["--sweep", spec])


def test_trials_is_still_parsed_and_ignored():
    args = run_ppo.build_parser().parse_args(["--trials", "5"])
    assert args.trials == 5 and "trials" not in run_ppo.params_from_args(args)
    assert run_ppo.expand_members(args.seed, args.population, args.sweep) == []


def test_member_params_key_sampling_and_shuffles_by_seed():
    p = member_params(_params(), {"seed": 5.0, "learning_rate": 1e-3})
    assert p["philox_seed"] == p["shuffle_seed"] == 5 and p["learning_rate"] == 1e-3 and p["num_envs"] == 4


def test_a_shared_key_equal_to_params_is_accepted():
    assert check_members(_params(), [{"seed": 2.0, "num_envs": 4}]) == [{"seed": 2.0}]


@pytest.mark.parametrize("member", [{"num_envs": 8}, {"gamma": 0.9}, {"gym_id": "Pendulum-v1"}, {"hidden_dim": 128},
                                    {"not_a_key": 1}])
def test_a_shared_key_that_differs_raises(member):
    with pytest.raises(_lib.AurError, match="shared"):
        ppo_population(_params(), [{"seed": 1.0}, dict(member, seed=2.0)])


def test_empty_population_raises():
    with pytest.raises(_lib.AurError):
        ppo_population(_params(), [])


@pytest.mark.parametrize("kw", [dict(hidden_dim=128), dict(num_layers=3), dict(gym_id="Acrobot-v1"),
                                dict(gym_id="MountainCarContinuous-v0", continuous=True), dict(num_envs=6, num_minibatches=4,
                                                                                              num_steps=3)])
def test_unsupported_requests_raise(kw):
    with pytest.raises(_lib.AurError):
        ppo_population(_params(**kw), [{"seed": 1.0}, {"seed": 2.0}])


def test_data_parallel_raises(monkeypatch):
    from aur_ppo_b200 import parallel, population
    monkeypatch.setattr(population.parallel, "current_plan", lambda *a: parallel.ShardPlan(2, 0, 4, 128, 4))
    with pytest.raises(_lib.AurError, match="one GPU"):
        ppo_population(_params(), [{"seed": 1.0}])


def test_c_abi_refuses_outside_the_population_scope():
    L = _lib.lib()
    pop = _lib.PopDesc(2, 0, 128, 8)              # the seed pointer is never dereferenced by these checks
    wide = _lib.PolicyDesc(4, 2, 128, 2, 0)
    assert L.aur_pop_update_workspace_bytes(ctypes.byref(pop), ctypes.byref(wide), 4, 1024) == -2     # AUR_ERR_UNSUPPORTED
    assert b"64 x 2" in L.aur_last_error()
    ok = _lib.PolicyDesc(4, 2, 64, 2, 0)
    assert L.aur_pop_update_workspace_bytes(ctypes.byref(pop), ctypes.byref(ok), 4, 1024) > 0
    bad = _lib.PopDesc(0, 0, 128, 8)
    assert L.aur_pop_update_workspace_bytes(ctypes.byref(bad), ctypes.byref(ok), 4, 1024) == -1
    assert L.aur_pop_shuffle_indices(ctypes.byref(pop), 16, 2, 0, None, None) == -1
    assert L.aur_pop_update_grad(ctypes.byref(pop), None, None) == -1
