"""Population-based training without a GPU: the --pbt_* flags and every request they, ppo_population and the C ABI refuse;
the oracle's decision rule (oracle/pbt_ref.py) on hand-worked cases; the ctypes layout of aur_pop_pbt_args against the C
header."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from aur_ppo_b200 import _lib, run_ppo
from aur_ppo_b200.population import check_pbt, ppo_population
from oracle import pbt_ref
from oracle.ppo_ref import philox4x32_10

NAN, INF = float("nan"), float("inf")


def _params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False)
    p.update(kw)
    return p


def _pbt_of(argv):
    args = run_ppo.build_parser().parse_args(argv)
    return run_ppo.pbt_from_args(args, len(run_ppo.expand_members(args.seed, args.population, args.sweep)))


# ------------------------------------------------------------------------------------------------ flags
def test_pbt_is_off_by_default():
    args = run_ppo.build_parser().parse_args(["--population", "4"])
    assert args.pbt_interval == 0 and _pbt_of(["--population", "4"]) is None


def test_pbt_flags_give_the_config():
    got = _pbt_of(["--population", "4", "--pbt_interval", "3", "--pbt_fraction", "0.5", "--pbt_keys", "clip_coeff, target_kl"])
    assert got == dict(interval=3, fraction=0.5, keys=("clip_coeff", "target_kl"))
    assert _pbt_of(["--sweep", "learning_rate=1e-4,1e-3", "--pbt_interval", "1"]) == dict(
        interval=1, fraction=0.25, keys=("learning_rate", "entropy_coeff"))


def test_pbt_config_defaults_and_mask():
    cfg = check_pbt(dict(interval=2), 4)
    assert cfg == dict(interval=2, fraction=0.25, keys=("learning_rate", "entropy_coeff"), factors=(0.8, 1.2), mask=0b11)
    assert check_pbt(dict(interval=1, keys=("target_kl", "clip_coeff")), 2)["mask"] == 0b100100
    assert check_pbt(None, 1) is None


@pytest.mark.parametrize("argv", [
    ["--pbt_interval", "1"],                                          # a single run
    ["--population", "1", "--pbt_interval", "1"],                     # one member
    ["--sweep", "learning_rate=1e-3", "--pbt_interval", "2"],         # one member
    ["--population", "4", "--pbt_interval", "-1"],
    ["--population", "4", "--pbt_interval", "1", "--pbt_fraction", "0"],
    ["--population", "4", "--pbt_interval", "1", "--pbt_fraction", "0.6"],
    ["--population", "4", "--pbt_interval", "1", "--pbt_fraction", "nan"],
    ["--population", "4", "--pbt_interval", "1", "--pbt_keys", "seed"],
    ["--population", "4", "--pbt_interval", "1", "--pbt_keys", "learning_rate,gamma"],
])
def test_bad_pbt_flags_are_parser_errors(argv):
    with pytest.raises(SystemExit):
        run_ppo.main(argv + ["--no_tensorboard", "--no_save"])


@pytest.mark.parametrize("pbt", [
    dict(interval=0), dict(interval=1.5), dict(interval=True), dict(), dict(interval=1, fraction=0.0),
    dict(interval=1, fraction=0.51), dict(interval=1, keys=("num_envs",)), dict(interval=1, keys=("seed",)),
    dict(interval=1, factors=(0.0, 1.2)), dict(interval=1, factors=(0.8, INF)), dict(interval=1, factors=(0.8,)),
    dict(interval=1, period=3), [1],
])
def test_bad_pbt_configs_raise(pbt):
    with pytest.raises(_lib.AurError):
        ppo_population(_params(), [{"seed": 1.0}, {"seed": 2.0}], pbt=pbt)


def test_pbt_needs_two_members():
    with pytest.raises(_lib.AurError, match="two members"):
        ppo_population(_params(), [{"seed": 1.0}], pbt=dict(interval=1))


# ------------------------------------------------------------------------------------------------ the oracle
def _hp(K):
    return np.array([[1e-3 * (k + 1), 0.01, 0.2, 0.5, 0.5, INF] for k in range(K)])


def test_oracle_worked_example():
    # fitness [3, NaN, 1, 2], q = 0.5: order [0, 3, 2], n_sel = floor(1.5) = 1, recipient 2 (rank 2 >= 3 - 1), donor 0
    rank, donor, hp = pbt_ref.decide([3.0, NAN, 1.0, 2.0], 0.5, 0.8, 1.2, 0b1, 7, 1, _hp(4))
    assert rank.tolist() == [0, -1, 2, 1]
    assert donor.tolist() == [-1, -1, 0, -1]
    w1 = philox4x32_10((2, 1, 0, pbt_ref.PHILOX_C3), (7, 0))[1]
    assert hp[2, 0] == 1e-3 * (1.2 if w1 & 1 else 0.8)
    assert hp[2, 1:].tolist() == _hp(4)[0, 1:].tolist()                 # unmasked fields copied, target_kl inf kept
    assert np.array_equal(np.delete(hp, 2, 0), np.delete(_hp(4), 2, 0))


def test_oracle_ties_go_to_the_lower_index():
    rank, order = pbt_ref.rank_members([1.0, 2.0, 1.0, 2.0, -0.0, 0.0, INF, -INF])
    assert order.tolist() == [6, 1, 3, 0, 2, 4, 5, 7]
    assert rank.tolist() == [3, 1, 4, 2, 5, 6, 0, 7]


def test_oracle_two_members_at_half():
    rank, donor, hp = pbt_ref.decide([0.5, 1.5], 0.5, 0.8, 1.2, 0, 3, 9, _hp(2))
    assert rank.tolist() == [1, 0] and donor.tolist() == [1, -1]
    assert np.array_equal(hp, _hp(2)[[1, 1]])                         # mask 0: a plain copy


@pytest.mark.parametrize("fitness,q", [([1.0], 0.5), ([1.0, 2.0, 3.0], 0.25), ([NAN, NAN, 4.0], 0.5), ([NAN] * 4, 0.5)])
def test_oracle_rounds_that_change_nothing(fitness, q):
    K = len(fitness)
    rank, donor, hp = pbt_ref.decide(fitness, q, 0.8, 1.2, 0b111111, 1, 1, _hp(K))
    assert (donor == -1).all() and np.array_equal(hp, _hp(K))


def test_oracle_target_kl_inf_stays_inf_and_donors_are_the_top():
    K = 40
    f = np.arange(K, dtype=np.float64)[::-1].copy()                  # member 0 best
    rank, donor, hp = pbt_ref.decide(f, 0.25, 0.5, 2.0, 0b111111, 11, 5, _hp(K))
    rec = np.nonzero(donor >= 0)[0]
    assert rec.tolist() == list(range(30, 40)) and set(donor[rec].tolist()) <= set(range(10))
    assert np.isinf(hp[rec, 5]).all()


def test_oracle_exploit_copies_rows_and_statistics_but_not_the_return_accumulator():
    K, P, n, D = 3, 5, 2, 3
    rows = [np.arange(K * P, dtype=np.float32).reshape(K, P) + 100 * i for i in range(3)]
    steps = np.array([4, 8, 12])
    norm = np.arange((2 * D + 5) * K * n, dtype=np.float64).reshape(2 * D + 5, K * n)
    want = norm.copy()
    pbt_ref.exploit(np.array([-1, -1, 0]), rows, steps, norm, n, D)
    assert rows[0][2].tolist() == rows[0][0].tolist() and steps.tolist() == [4, 8, 4]
    want[:2 * D + 4, 4:6] = want[:2 * D + 4, 0:2]
    assert np.array_equal(norm, want)


# ------------------------------------------------------------------------------------------------ C ABI
def _args(**kw):
    a = _lib.PopPbtArgs()
    a.fitness = a.params = a.adam_m = a.adam_v = a.steps = a.hparams = a.rank_out = a.donor_out = a.order = 8
    a.q, a.down, a.up, a.mask, a.seed, a.round = 0.25, 0.8, 1.2, 3, 1, 1
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("kw", [dict(q=0.0), dict(q=0.5000001), dict(q=NAN), dict(down=0.0), dict(up=-1.0), dict(up=INF),
                                dict(down=NAN), dict(mask=64), dict(fitness=None), dict(params=None), dict(adam_v=None),
                                dict(steps=None), dict(hparams=None), dict(order=None), dict(donor_out=None),
                                dict(norm=8, norm_ld=100)])
def test_c_abi_pbt_argument_errors(kw):
    L = _lib.lib()
    pop = _lib.PopDesc(2, 0, 128, 8)              # no pointer is dereferenced before the checks pass
    ok = _lib.PolicyDesc(4, 2, 64, 2, 0)
    assert L.aur_pop_pbt_step(ctypes.byref(pop), ctypes.byref(ok), ctypes.byref(_args(**kw)), None) == -1
    assert b"aur_pop_pbt_step" in L.aur_last_error()


def test_c_abi_pbt_refuses_outside_the_population_scope():
    L = _lib.lib()
    pop = _lib.PopDesc(2, 0, 128, 8)
    wide = _lib.PolicyDesc(4, 2, 128, 2, 0)
    assert L.aur_pop_pbt_step(ctypes.byref(pop), ctypes.byref(wide), ctypes.byref(_args()), None) == -2
    assert b"64 x 2" in L.aur_last_error()
    bad = _lib.PopDesc(0, 0, 128, 8)
    ok = _lib.PolicyDesc(4, 2, 64, 2, 0)
    assert L.aur_pop_pbt_step(ctypes.byref(bad), ctypes.byref(ok), ctypes.byref(_args()), None) == -1
    assert L.aur_pop_pbt_step(ctypes.byref(pop), ctypes.byref(ok), None, None) == -1
    assert L.aur_pop_episode_fitness(ctypes.byref(pop), None, 8, 8, None) == -1
    assert L.aur_pop_episode_fitness(ctypes.byref(bad), 8, 8, 8, None) == -1


def test_pbt_args_layout_matches_the_header(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    fields = [f for f, _ in _lib.PopPbtArgs._fields_ if not f.startswith("_")]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "include/aur_ppo.h"\nint main(void) {\n'
                   '  printf("%zu", sizeof(aur_pop_pbt_args));\n'
                   + "".join(f'  printf(" %zu", offsetof(aur_pop_pbt_args, {f}));\n' for f in fields)
                   + '  printf("\\n");\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-std=c99", "-I", root, str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(_lib.PopPbtArgs)] + [getattr(_lib.PopPbtArgs, f).offset for f in fields]
