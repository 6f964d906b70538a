"""Rollout kernel vs the CPU checker (GPU).  Env transitions, rewards and done flags are
compared BIT FOR BIT (north_star); log-probs and values within 2e-5 (fp32 MLP, fast tanh)."""
import os

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, envs as denv, kernels
from oracle import envs as E
from oracle import ppo_ref as R
from tests.helpers import flat_from_named, golden_policy, random_policy

pytestmark = pytest.mark.gpu
TOL = dict(rtol=2e-5, atol=2e-6)


@pytest.fixture(autouse=True, params=["tc", "simt"])
def rollout_impl(request):
    """Every test runs against both rollout kernels: actor hidden layer on tcgen05 (default) and the SIMT kernel."""
    L = _lib.lib()
    prev = L.aur_rollout_get_impl()
    assert L.aur_rollout_set_impl(1 if request.param == "tc" else 0) == 0
    yield request.param
    L.aur_rollout_set_impl(prev)



def test_device_sincos_equals_host_copy_bitwise():
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(-0.3, 0.3, 200_000), rng.uniform(-100, 100, 200_000),
                        rng.uniform(-1.6e6, 1.6e6, 100_000), [0.0, -0.0, np.pi / 4, -np.pi / 4, 1e-300, 0.7853981633974484]])
    s, c = kernels.sincos_f64(torch.from_numpy(x).cuda())
    hs, hc = E.det_sincos(x)
    assert np.array_equal(s.cpu().numpy(), hs) and np.array_equal(c.cpu().numpy(), hc)


@pytest.mark.parametrize("tag", ["disc", "cont", "disc3", "cont2"])
def test_policy_evaluate_matches_reference_golden(golden_dir, tag):
    pol, named, g = golden_policy(golden_dir, tag)
    nl = len([k for k in named if k.startswith("critic.net.") and k.endswith(".weight")]) - 1
    obs, act = g[f"{tag}_obs"], g[f"{tag}_act"].astype(np.float32)
    cont = pol.continuous
    A = named["actor_logstd"].size if cont else int(named[[k for k in named if k.startswith("actor.net.")][-1]].shape[0])
    desc = kernels.policy_desc(obs.shape[1], A, 64, nl, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    assert flat.numel() == kernels.policy_param_count(desc)
    a, lp, ent, v = kernels.policy_evaluate(desc, flat, torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda())
    np.testing.assert_allclose(lp.cpu().numpy(), g[f"{tag}_logp"], **TOL)
    np.testing.assert_allclose(ent.cpu().numpy(), g[f"{tag}_ent"], **TOL)
    np.testing.assert_allclose(v.cpu().numpy(), g[f"{tag}_value_flat"], **TOL)
    np.testing.assert_array_equal(a.cpu().numpy().reshape(act.shape), act)


def test_unsupported_shapes_fail_loudly():
    for desc in (kernels.policy_desc(4, 2, 66, 2, False), kernels.policy_desc(4, 2, 512, 2, False)):
        with pytest.raises(_lib.AurError, match="hidden_dim"):
            kernels.policy_evaluate(desc, torch.zeros(1000000, device="cuda"), torch.zeros(4, 4, device="cuda"))
    with pytest.raises(_lib.AurError, match="obs_dim"):
        kernels.policy_evaluate(kernels.policy_desc(9, 2, 64, 2, False), torch.zeros(100000, device="cuda"), torch.zeros(4, 9, device="cuda"))
    with pytest.raises(_lib.AurError, match="no device kernel"):
        denv.DeviceVecEnv("LunarLander-v2", 4)


def _oracle_replay(kind, N, wrappers, seeds, actions, T):
    cv = E.CVecEnv(kind, N, wrappers=wrappers, trig=E.TRIG_CR)
    obs0, _ = cv.reset(seeds)
    D = cv.obs_dim
    obs = np.zeros((T, N, D), np.float32); rew = np.zeros((T, N), np.float32); done = np.zeros((T, N), np.float32)
    cur, cur_done = obs0, np.zeros(N, np.float32)
    episodes = []
    for t in range(T):
        obs[t], done[t] = cur, cur_done
        cur, r, term, trunc, info = cv.step(actions[t])
        rew[t] = r.astype(np.float32)
        cur_done = term.astype(np.float32)
        if "final_info" in info:
            for i, it in enumerate(info["final_info"]):
                if it is not None:
                    episodes.append((t, i, float(it["episode"]["r"]), int(it["episode"]["l"])))
    return cv, obs0, obs, rew, done, cur, cur_done, episodes


@pytest.mark.parametrize("N,T", [(5, 700), (300, 256), (16384, 96)])   # E=1 ragged, E=1, E=2 (>= 9472 envs)
def test_cartpole_replay_is_bit_exact(N, T):
    pol, named = random_policy(4, 2, 64, 2, False, seed=3)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(N))
    rng = np.random.default_rng(N)
    actions = rng.integers(0, 2, (T, N))
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.CARTPOLE, N, False, seeds, actions, T)

    env = denv.DeviceVecEnv("CartPole-v1", N, log_capacity=N * 64)
    o, _ = env.reset(seeds)
    assert np.array_equal(o.cpu().numpy(), obs0)
    buf = kernels.RolloutBuffers(T, N, 4, (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions.astype(np.float32)).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.terminals.cpu().numpy(), done)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(buf.actions.cpu().numpy(), actions.astype(np.float32))
    assert np.array_equal(env.next_obs.cpu().numpy(), last_obs)
    assert np.array_equal(env.next_done.cpu().numpy(), last_done)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())          # fp64 state, bit for bit
    # what the training loop reads: per step, the first finished env in env order (ppo.py:114-122)
    ft, fenv, fret, flen = env.first_finished_episodes()
    want_first = {}
    for (t, i, r, l) in sorted(episodes, key=lambda r: (r[0], r[1])):
        want_first.setdefault(t, (i, r, l))
    assert list(ft) == sorted(want_first)
    assert [(int(e), float(r), int(l)) for e, r, l in zip(fenv, fret, flen)] == [want_first[t] for t in sorted(want_first)]
    tot = env.totals.cpu().numpy()
    assert tot[0] == len(episodes) and tot[2] == sum(e[3] for e in episodes)
    got = env.drain_episodes()
    assert got == sorted(episodes, key=lambda r: (r[0], r[1]))
    assert len(got) > 0
    # log-probs / values against the oracle model on the same observations
    sub = slice(0, min(N, 64))
    ot = torch.from_numpy(obs[:, sub].reshape(-1, 4)); at = torch.from_numpy(actions[:, sub].reshape(-1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
    np.testing.assert_allclose(buf.log_probs[:, sub].cpu().numpy().reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values[:, sub].cpu().numpy().reshape(-1), v.numpy().reshape(-1), **TOL)
    with torch.no_grad():
        nv = pol.value(torch.from_numpy(last_obs[sub]))
    np.testing.assert_allclose(buf.next_value[sub].cpu().numpy(), nv.numpy(), **TOL)


# N, T, hidden, layers.  Past 64 x 2 each width is the first MountainCar-v0 run of its kernels: 128 x 2 takes
# rollout_tc_kernel<MountainCar, 128> + critic_values_tc_kernel<128> with 2 observations; 256 x 2 and 128 x 3 take the
# layer-wise actor (rollout_wide.cu) and rollout_tc_kernel<MountainCar, 0>, the external-actor mode with 3 logits; simt takes
# the runtime-width kernel at 128 / 256 units
MOUNTAINCAR_REPLAYS = {"7-450": (7, 450, 64, 2), "300-256": (300, 256, 64, 2), "128x2": (300, 256, 128, 2),
                       "256x2": (130, 256, 256, 2), "128x3": (130, 256, 128, 3)}


@pytest.mark.parametrize("case", list(MOUNTAINCAR_REPLAYS))
def test_mountaincar_replay_is_bit_exact(case, rollout_impl):
    """MountainCar-v0 ((f) rank 4: more classic-control envs behind --gym_id): obs 2, 3 discrete actions, TimeLimit 200."""
    N, T, hidden, layers = MOUNTAINCAR_REPLAYS[case]
    L = _lib.lib()
    pol, named = random_policy(2, 3, hidden, layers, False, seed=8)
    desc = kernels.policy_desc(2, 3, hidden, layers, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(N))
    rng = np.random.default_rng(N)
    # energy pumping on half of the envs so that some episodes terminate before the TimeLimit truncation
    actions = rng.integers(0, 3, (T, N))
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay_adaptive(E.MOUNTAINCAR, N, seeds, actions, T)
    env = denv.DeviceVecEnv("MountainCar-v0", N, log_capacity=N * 16)
    o, _ = env.reset(seeds)
    assert np.array_equal(o.cpu().numpy(), obs0)
    buf = kernels.RolloutBuffers(T, N, 2, (), "cuda")
    L.aur_launch_count_reset()
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions.astype(np.float32)).cuda())
    torch.cuda.synchronize()
    layerwise = rollout_impl == "tc" and (hidden, layers) not in ((64, 2), (128, 2))
    assert (L.aur_launch_count() >= T) == layerwise          # the layer-wise actor launches per step, a fused rollout does not
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.terminals.cpu().numpy(), done)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(env.next_obs.cpu().numpy(), last_obs)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())
    got = env.drain_episodes()
    assert got == sorted(episodes, key=lambda r: (r[0], r[1])) and len(got) > 0
    assert any(l < 200 for (_, _, _, l) in got) and done.sum() > 0           # real terminations, not only truncations
    sub = slice(0, min(N, 64))
    ot = torch.from_numpy(obs[:, sub].reshape(-1, 2)); at = torch.from_numpy(actions[:, sub].reshape(-1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
        nv = pol.value(torch.from_numpy(last_obs[sub]))
    np.testing.assert_allclose(buf.log_probs[:, sub].cpu().numpy().reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values[:, sub].cpu().numpy().reshape(-1), v.numpy().reshape(-1), **TOL)
    np.testing.assert_allclose(buf.next_value[sub].cpu().numpy(), nv.numpy(), **TOL)


def _oracle_replay_adaptive(kind, N, seeds, actions, T):
    """Like _oracle_replay, but even-numbered envs follow the energy-pumping policy (push in the direction of motion):
    `actions` is overwritten in place with what was actually played."""
    cv = E.CVecEnv(kind, N, wrappers=False, trig=E.TRIG_CR)
    obs0, _ = cv.reset(seeds)
    D = cv.obs_dim
    obs = np.zeros((T, N, D), np.float32); rew = np.zeros((T, N), np.float32); done = np.zeros((T, N), np.float32)
    cur, cur_done = obs0, np.zeros(N, np.float32)
    episodes = []
    for t in range(T):
        obs[t], done[t] = cur, cur_done
        actions[t, ::2] = np.where(cur[::2, 1] >= 0, 2, 0)
        cur, r, term, trunc, info = cv.step(actions[t])
        rew[t] = r.astype(np.float32)
        cur_done = term.astype(np.float32)
        if "final_info" in info:
            for i, it in enumerate(info["final_info"]):
                if it is not None:
                    episodes.append((t, i, float(it["episode"]["r"]), int(it["episode"]["l"])))
    return cv, obs0, obs, rew, done, cur, cur_done, episodes


@pytest.mark.parametrize("wrappers", [True, False])
def test_pendulum_replay_is_bit_exact(wrappers):
    N, T = 200, 450           # crosses two TimeLimit truncations
    pol, named = random_policy(3, 1, 64, 2, True, seed=4)
    desc = kernels.policy_desc(3, 1, 64, 2, True)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(100, 100 + N))
    rng = np.random.default_rng(9)
    actions = rng.normal(0, 1.6, (T, N, 1)).astype(np.float32)
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.PENDULUM, N, wrappers, seeds, actions, T)
    env = denv.DeviceVecEnv("Pendulum-v1", N, wrappers=wrappers, log_capacity=N * 8)
    o, _ = env.reset(seeds)
    assert np.array_equal(o.cpu().numpy(), obs0)
    buf = kernels.RolloutBuffers(T, N, 3, (1,), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(buf.terminals.cpu().numpy(), done) and not done.any()
    assert np.array_equal(env.next_obs.cpu().numpy(), last_obs)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())
    if wrappers:
        assert np.array_equal(env.norm.cpu().numpy().T, cv.norm_stats())
    got = env.drain_episodes()
    assert [(g[0], g[1], g[3]) for g in got] == [(e[0], e[1], e[3]) for e in sorted(episodes, key=lambda r: (r[0], r[1]))]
    np.testing.assert_array_equal([g[2] for g in got], [e[2] for e in sorted(episodes, key=lambda r: (r[0], r[1]))])
    ot = torch.from_numpy(obs[:, :32].reshape(-1, 3)); at = torch.from_numpy(actions[:, :32].reshape(-1, 1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
    np.testing.assert_allclose(buf.log_probs[:, :32].cpu().numpy().reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values[:, :32].cpu().numpy().reshape(-1), v.numpy().reshape(-1), **TOL)


def test_sampled_rollout_then_replay_on_the_checker():
    """Sampled mode: the actions the kernel drew, replayed on the CPU checker, reproduce every
    transition; and the draw follows the Philox stream restated in the oracle."""
    N, T = 512, 200
    pol, named = random_policy(4, 2, 64, 2, False, seed=5)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    env = denv.DeviceVecEnv("CartPole-v1", N, env_id0=1000)
    env.reset(list(range(N)))
    buf = kernels.RolloutBuffers(T, N, 4, (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=77, step0=5, actions_in=None)
    actions = buf.actions.cpu().numpy().astype(np.int64)
    cv, obs0, obs, rew, done, last_obs, last_done, _ = _oracle_replay(E.CARTPOLE, N, False, list(range(N)), actions, T)
    assert np.array_equal(buf.states.cpu().numpy(), obs) and np.array_equal(buf.terminals.cpu().numpy(), done)
    # inverse-CDF rule on the oracle's probabilities with the restated Philox uniform, every draw not within 1e-5 of the
    # CDF boundary
    with torch.no_grad():
        p = torch.softmax(pol._mlp("actor", torch.from_numpy(obs.reshape(-1, 4))), -1).double().numpy()
    gid = np.tile(1000 + np.arange(N, dtype=np.uint64), T)
    step = np.repeat(5 + np.arange(T, dtype=np.uint64), N)
    u = (R.sampler_words_np(77, gid, step)[0] >> 8) * 2.0 ** -24
    want, margin = R.categorical_icdf(p, u)
    keep = margin > 1e-5
    assert keep.mean() > 0.99 and np.array_equal(want[keep], actions.reshape(-1)[keep])
    # action frequencies follow the policy (chi-square style bound on the mean)
    with torch.no_grad():
        lg = pol._mlp("actor", torch.from_numpy(obs.reshape(-1, 4)))
        pm = torch.softmax(lg, -1)[:, 1].mean().item()
    assert abs(actions.mean() - pm) < 4 * np.sqrt(0.25 / actions.size)


def test_sharding_and_chunking_invariance():
    """Two half-size launches with env_id0 offsets == one launch; two T/2 calls == one T call."""
    N, T = 256, 64
    _, named = random_policy(4, 2, 64, 2, False, seed=6)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()

    def run(n, id0, seeds, chunks):
        env = denv.DeviceVecEnv("CartPole-v1", n, env_id0=id0)
        env.reset(seeds)
        outs, step = [], 0
        for tc in chunks:
            buf = kernels.RolloutBuffers(tc, n, 4, (), "cuda")
            kernels.rollout(env, desc, flat, buf, seed=9, step0=step)
            step += tc
            outs.append(buf)
        cat = lambda f: torch.cat([getattr(b, f) for b in outs], 0)
        return cat("states"), cat("actions"), cat("rewards"), cat("terminals"), cat("log_probs"), env.phys.clone()

    full = run(N, 0, list(range(N)), [T])
    a = run(N // 2, 0, list(range(N // 2)), [T])
    b = run(N // 2, N // 2, list(range(N // 2, N)), [T])
    for i in range(5):
        assert torch.equal(full[i], torch.cat([a[i], b[i]], 1))
    assert torch.equal(full[5], torch.cat([a[5], b[5]], 1))
    two = run(N, 0, list(range(N)), [T // 2, T // 2])
    for i in range(6):
        assert torch.equal(full[i], two[i])


def test_pendulum_sampling_moments():
    N, T = 4096, 8
    pol, named = random_policy(3, 1, 64, 2, True, seed=8)
    desc = kernels.policy_desc(3, 1, 64, 2, True)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    env = denv.DeviceVecEnv("Pendulum-v1", N, wrappers=True)
    env.reset(list(range(N)))
    buf = kernels.RolloutBuffers(T, N, 3, (1,), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=3, step0=0)
    obs = buf.states.cpu().reshape(-1, 3)
    with torch.no_grad():
        mean = pol._mlp("actor", obs).reshape(-1)
    std = float(np.exp(named["actor_logstd"].ravel()[0]))
    z = (buf.actions.cpu().reshape(-1) - mean) / std
    n = z.numel()
    assert abs(z.mean().item()) < 5 / np.sqrt(n) and abs(z.var().item() - 1) < 5 * np.sqrt(2 / n)
    assert abs((z ** 3).mean().item()) < 0.1 and abs((z ** 4).mean().item() - 3) < 0.2
    with torch.no_grad():
        _, lp, _, _ = pol.evaluate(obs, buf.actions.cpu().reshape(-1, 1))
    np.testing.assert_allclose(buf.log_probs.cpu().reshape(-1).numpy(), lp.numpy(), rtol=2e-5, atol=5e-6)


def test_full_size_rollout_properties():
    """BASELINE config B rollout (65536 envs x 128 steps, sampled actions), through size-independent properties: a
    random subset of env columns replays bit-exactly on the CPU checker with the actions the device drew, every reward
    is 1, and the episode totals merged on the device equal what the done / truncation pattern implies."""
    N, T = 65536, 128
    pol, named = random_policy(4, 2, 64, 2, False, seed=4)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    env = denv.DeviceVecEnv("CartPole-v1", N)
    env.reset(list(range(N)))
    buf = kernels.RolloutBuffers(T, N, 4, (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=7, step0=0)
    torch.cuda.synchronize()
    assert torch.all(buf.rewards == 1.0)
    acts = buf.actions.cpu().numpy()
    assert set(np.unique(acts)) <= {0.0, 1.0} and 0.3 < acts.mean() < 0.7
    cols = np.sort(np.random.default_rng(0).choice(N, 96, replace=False))
    cv = E.CVecEnv(E.CARTPOLE, len(cols), wrappers=False, trig=E.TRIG_CR)
    cur, _ = cv.reset([int(c) for c in cols])            # env i is seeded with its global id
    cur_done = np.zeros(len(cols), np.float32)
    states, terminals = buf.states.cpu().numpy(), buf.terminals.cpu().numpy()
    finished = 0
    for t in range(T):
        assert np.array_equal(states[t, cols], cur) and np.array_equal(terminals[t, cols], cur_done), t
        cur, r, term, trunc, info = cv.step(acts[t, cols].astype(np.int32))
        cur_done = term.astype(np.float32)
        finished += int((term | trunc).sum())
    assert np.array_equal(env.next_obs.cpu().numpy()[cols], cur)
    assert np.array_equal(env.phys.cpu().numpy().T[cols], cv.phys())
    tot = env.totals.cpu().numpy()
    # every terminated step is followed by a `done` flag in the next row (or in next_done after the last row)
    n_term = int(buf.terminals[1:].sum().item() + env.next_done.sum().item())
    assert tot[0] == n_term and finished > 0              # no TimeLimit truncation can occur in 128 steps
    # log-probs / values of the subset against the oracle model
    ot = torch.from_numpy(states[:, cols[:16]].reshape(-1, 4)); at = torch.from_numpy(acts[:, cols[:16]].reshape(-1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
    np.testing.assert_allclose(buf.log_probs.cpu().numpy()[:, cols[:16]].reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values.cpu().numpy()[:, cols[:16]].reshape(-1), v.numpy().reshape(-1), **TOL)


# ---- runtime-width policies (hidden_dim != 64, widths up to 8): csrc/policy.cuh::mlp_forward_dyn ---------------------
@pytest.mark.parametrize("obs_dim,act_dim,hidden,layers,cont", [(4, 2, 32, 2, False), (4, 2, 128, 3, False), (8, 4, 64, 2, False),
                                                                (6, 3, 256, 2, False), (3, 1, 100, 1, True), (8, 8, 64, 2, True),
                                                                (5, 6, 20, 4, True), (4, 3, 256, 4, False)])
def test_policy_evaluate_runtime_widths_vs_oracle(obs_dim, act_dim, hidden, layers, cont, rollout_impl):
    """actor_critic.evaluate / value (models/actor_critic.py:31-51) for the shapes `-d` / `-nl` and the shipped checkpoints
    (state 8 / 4 actions) produce, against the restated torch model."""
    if rollout_impl != "tc":
        pytest.skip("one kernel behind this path")
    pol, named = random_policy(obs_dim, act_dim, hidden, layers, cont, seed=hidden)
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    g = torch.Generator().manual_seed(1)
    B = 3000
    obs = torch.randn(B, obs_dim, generator=g)
    act = torch.randn(B, act_dim, generator=g) if cont else torch.randint(0, act_dim, (B,), generator=g).float()
    with torch.no_grad():
        _, lp, ent, v = pol.evaluate(obs, act)
    a, glp, gent, gv = kernels.policy_evaluate(desc, flat, obs.cuda(), act.cuda())
    np.testing.assert_allclose(glp.cpu().numpy(), lp.numpy(), rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(gent.cpu().numpy(), ent.numpy(), rtol=2e-5, atol=5e-6)
    np.testing.assert_allclose(gv.cpu().numpy().reshape(-1), v.numpy().reshape(-1), rtol=2e-5, atol=5e-6)
    # sampling: replaying the drawn actions reproduces the log-probs bit for bit; discrete frequencies follow the softmax
    a1, lp1, _, _ = kernels.policy_evaluate(desc, flat, obs.cuda(), None, seed=7, step=3)
    a2, lp2, _, _ = kernels.policy_evaluate(desc, flat, obs.cuda(), a1, seed=7, step=3)
    assert torch.equal(lp1, lp2) and torch.equal(a1, a2)
    if cont:
        z = a1.cpu().reshape(B, act_dim)
        assert torch.isfinite(z).all()
        if act_dim > 4:   # the second Philox block feeds dims 4..7: they must not repeat dims 0..3
            assert not torch.equal(z[:, 0], z[:, 4])
    else:
        assert set(np.unique(a1.cpu().numpy())) <= set(range(act_dim))


@pytest.mark.parametrize("hidden,layers,N,T", [(32, 2, 300, 200), (128, 2, 70, 300), (256, 2, 40, 120), (96, 3, 64, 150), (128, 3, 200, 90),
                                               (256, 4, 130, 60)])
def test_cartpole_replay_runtime_width(hidden, layers, N, T, rollout_impl):
    """`--hidden_dim` other than 64: transitions stay bit-exact (same env code), log-probs / values follow the wider MLP.
    128 / 256 units have two paths: tcgen05 (128 x 2: rollout_tc_kernel<ENV, 128> + critic_values_tc_kernel<128>; otherwise the
    layer-wise actor of rollout_wide.cu with the env step in rollout_tc_kernel<ENV, 0>) and the runtime-width SIMT kernel."""
    if rollout_impl != "tc" and hidden not in (128, 256):
        pytest.skip("one kernel behind this path")
    pol, named = random_policy(4, 2, hidden, layers, False, seed=hidden)
    desc = kernels.policy_desc(4, 2, hidden, layers, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(N))
    actions = np.random.default_rng(N).integers(0, 2, (T, N))
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.CARTPOLE, N, False, seeds, actions, T)
    env = denv.DeviceVecEnv("CartPole-v1", N, log_capacity=N * 64)
    env.reset(seeds)
    buf = kernels.RolloutBuffers(T, N, 4, (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions.astype(np.float32)).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.terminals.cpu().numpy(), done)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())
    assert env.drain_episodes() == sorted(episodes, key=lambda r: (r[0], r[1]))
    ot = torch.from_numpy(obs.reshape(-1, 4)); at = torch.from_numpy(actions.reshape(-1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
        nv = pol.value(torch.from_numpy(last_obs))
    np.testing.assert_allclose(buf.log_probs.cpu().numpy().reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values.cpu().numpy().reshape(-1), v.numpy().reshape(-1), **TOL)
    np.testing.assert_allclose(buf.next_value.cpu().numpy(), nv.numpy(), **TOL)
    # sampled actions: same Philox stream as the 64-wide kernels -> a sampled rollout replays on the checker
    env.reset(seeds)
    buf2 = kernels.RolloutBuffers(T, N, 4, (), "cuda")
    kernels.rollout(env, desc, flat, buf2, seed=5, step0=0)
    acts = buf2.actions.cpu().numpy().astype(np.int64)
    _, _, obs_s, rew_s, done_s, _, _, _ = _oracle_replay(E.CARTPOLE, N, False, seeds, acts, T)
    assert np.array_equal(buf2.states.cpu().numpy(), obs_s) and np.array_equal(buf2.rewards.cpu().numpy(), rew_s)
    assert np.array_equal(buf2.terminals.cpu().numpy(), done_s)


@pytest.mark.parametrize("hidden", [128, 256])
def test_pendulum_replay_runtime_width(hidden, rollout_impl):
    """Pendulum + wrappers at hidden 128 / 256: tensor-core kernels (tc) and the runtime-width SIMT kernel (simt)."""
    N, T = 50, 260
    pol, named = random_policy(3, 1, hidden, 2, True, seed=9)
    desc = kernels.policy_desc(3, 1, hidden, 2, True)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(N))
    env = denv.DeviceVecEnv("Pendulum-v1", N, wrappers=True, log_capacity=N * 8)
    env.reset(seeds)
    buf = kernels.RolloutBuffers(T, N, 3, (1,), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=2, step0=0)
    torch.cuda.synchronize()
    acts = buf.actions.cpu().numpy()
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.PENDULUM, N, True, seeds, acts, T)
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(torch.from_numpy(obs.reshape(-1, 3)), torch.from_numpy(acts.reshape(-1, 1)))
    np.testing.assert_allclose(buf.log_probs.cpu().numpy().reshape(-1), lp.numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(buf.values.cpu().numpy().reshape(-1), v.numpy().reshape(-1), rtol=2e-5, atol=5e-6)


@pytest.mark.parametrize("N,T,hidden", [(9, 600, 64), (300, 256, 64), (64, 200, 32)])
def test_acrobot_replay_is_bit_exact(N, T, hidden, rollout_impl):
    """Acrobot-v1 ((f) rank 4; obs 6 -> the runtime-width policy path): RK4 transitions, wrap / bound, termination and
    TimeLimit bit for bit against the C checker; log-probs / values against the restated model."""
    if rollout_impl != "tc":
        pytest.skip("one kernel behind this path")
    pol, named = random_policy(6, 3, hidden, 2, False, seed=21)
    desc = kernels.policy_desc(6, 3, hidden, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(N))
    rng = np.random.default_rng(N)
    # torque along the second joint's velocity most of the time, so that episodes actually terminate inside T
    actions = rng.integers(0, 3, (T, N))
    cv = E.CVecEnv(E.ACROBOT, N, trig=E.TRIG_CR)
    cv.reset(seeds)
    for t in range(T):
        greedy = np.where(cv.phys()[:, 3] > 0, 2, 0)
        actions[t] = np.where(rng.random(N) < 0.8, greedy, actions[t])
        cv.step(actions[t])
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.ACROBOT, N, False, seeds, actions, T)
    assert done.any() and (rew == 0).any()
    env = denv.DeviceVecEnv("Acrobot-v1", N, log_capacity=N * 64)
    o, _ = env.reset(seeds)
    assert np.array_equal(o.cpu().numpy(), obs0)
    buf = kernels.RolloutBuffers(T, N, 6, (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions.astype(np.float32)).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.terminals.cpu().numpy(), done)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(env.next_obs.cpu().numpy(), last_obs)
    assert np.array_equal(env.next_done.cpu().numpy(), last_done)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())
    assert env.drain_episodes() == sorted(episodes, key=lambda r: (r[0], r[1]))
    ot = torch.from_numpy(obs.reshape(-1, 6)); at = torch.from_numpy(actions.reshape(-1))
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(ot, at)
        nv = pol.value(torch.from_numpy(last_obs))
    np.testing.assert_allclose(buf.log_probs.cpu().numpy().reshape(-1), lp.numpy(), **TOL)
    np.testing.assert_allclose(buf.values.cpu().numpy().reshape(-1), v.numpy().reshape(-1), **TOL)
    np.testing.assert_allclose(buf.next_value.cpu().numpy(), nv.numpy(), **TOL)


@pytest.mark.parametrize("wrappers,hidden", [(True, 64), (False, 64), (True, 32)])
def test_mountaincar_continuous_replay_is_bit_exact(wrappers, hidden, rollout_impl):
    """MountainCarContinuous-v0 ((f) rank 4): float32 state / float64 arithmetic, ClipAction(-1, 1), the continuous wrapper
    stack with two observation dims and the 999-step TimeLimit (10-bit episode lengths in the log), bit for bit."""
    N, T = 40, 1100
    pol, named = random_policy(2, 1, hidden, 2, True, seed=14)
    desc = kernels.policy_desc(2, 1, hidden, 2, True)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seeds = list(range(50, 50 + N))
    rng = np.random.default_rng(3)
    # rock with the velocity (plus noise, some of it outside [-1, 1]) so that some episodes reach the flag
    actions = np.zeros((T, N, 1), np.float32)
    cv = E.CVecEnv(E.MOUNTAINCAR_CONT, N, wrappers=wrappers, trig=E.TRIG_CR)
    cv.reset(seeds)
    for t in range(T):
        vel = cv.phys()[:, 1]
        a = np.where(vel >= 0, 1.0, -1.0) * (np.arange(N) % 2) + rng.normal(0, 0.8, N)
        actions[t, :, 0] = a.astype(np.float32)
        cv.step(actions[t])
    cv, obs0, obs, rew, done, last_obs, last_done, episodes = _oracle_replay(E.MOUNTAINCAR_CONT, N, wrappers, seeds, actions, T)
    assert done.any() and any(e[3] == 999 for e in episodes)
    env = denv.DeviceVecEnv("MountainCarContinuous-v0", N, wrappers=wrappers, log_capacity=N * 64)
    o, _ = env.reset(seeds)
    assert np.array_equal(o.cpu().numpy(), obs0)
    buf = kernels.RolloutBuffers(T, N, 2, (1,), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(actions).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), obs)
    assert np.array_equal(buf.rewards.cpu().numpy(), rew)
    assert np.array_equal(buf.terminals.cpu().numpy(), done)
    assert np.array_equal(env.next_obs.cpu().numpy(), last_obs)
    assert np.array_equal(env.phys.cpu().numpy().T, cv.phys())
    if wrappers:
        assert np.array_equal(env.norm.cpu().numpy().T, cv.norm_stats())
    got = env.drain_episodes()
    want = sorted(episodes, key=lambda r: (r[0], r[1]))
    assert [(g[0], g[1], g[3]) for g in got] == [(e[0], e[1], e[3]) for e in want]
    np.testing.assert_array_equal([g[2] for g in got], [e[2] for e in want])
    ft, fenv, fret, flen = env.first_finished_episodes()
    first = {}
    for (t, i, r, l) in want:
        first.setdefault(t, (i, r, l))
    assert [(int(e), float(r), int(l)) for e, r, l in zip(fenv, fret, flen)] == [first[t] for t in sorted(first)]
    with torch.no_grad():
        _, lp, _, v = pol.evaluate(torch.from_numpy(obs.reshape(-1, 2)), torch.from_numpy(actions.reshape(-1, 1)))
    np.testing.assert_allclose(buf.log_probs.cpu().numpy().reshape(-1), lp.numpy(), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(buf.values.cpu().numpy().reshape(-1), v.numpy().reshape(-1), rtol=2e-5, atol=5e-6)


@pytest.mark.parametrize("tag,gym_id", [("cart128", "CartPole-v1"), ("pend128", "Pendulum-v1"), ("cart256", "CartPole-v1")])
def test_wide_rollout_matches_reference_golden(golden_dir, tag, gym_id, rollout_impl):
    """tests/golden/rollout_wide.npz (oracle/gen_golden_wide.py): log-probs / values of the REFERENCE'S OWN actor_critic.evaluate
    at 128 / 256 hidden units on the observations a seeded rollout visits under a fixed action tape.  The device rollout must
    visit the same observations bit for bit and store the reference's numbers (both kernel families)."""
    g = np.load(os.path.join(golden_dir, "rollout_wide.npz"))
    obs_dim, act_dim, hidden, layers, cont, N, T = [int(v) for v in g[f"{tag}_shape"]]
    named0 = {}
    for i, n in enumerate(str(x) for x in g[f"{tag}_names"]):
        shape = tuple(int(v) for v in g[f"{tag}_pshape_{n}"])
        k = np.arange(int(np.prod(shape)), dtype=np.float64)
        named0[n] = torch.from_numpy(0.1 * np.sin(0.37 * k + i)).to(torch.float32).numpy().reshape(shape)   # gen_golden.fill_params
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, bool(cont))
    flat = torch.from_numpy(flat_from_named(named0)).cuda()
    env = denv.DeviceVecEnv(gym_id, N, wrappers=bool(cont))
    env.reset(list(range(N)))
    buf = kernels.RolloutBuffers(T, N, obs_dim, (act_dim,) if cont else (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=torch.from_numpy(g[f"{tag}_actions"]).cuda())
    torch.cuda.synchronize()
    assert np.array_equal(buf.states.cpu().numpy(), g[f"{tag}_obs"])
    np.testing.assert_allclose(buf.log_probs.cpu().numpy(), g[f"{tag}_logp"], **TOL)
    np.testing.assert_allclose(buf.values.cpu().numpy(), g[f"{tag}_value"], **TOL)
    np.testing.assert_allclose(buf.next_value.cpu().numpy(), g[f"{tag}_next_value"], **TOL)


def test_layerwise_rollout_more_envs_than_one_sub_batch(rollout_impl):
    """rollout_wide.cu chunks every per-step actor pass (and the value pass) at 262,144 rows: with more envs than that, the
    second chunk must see its own rows.  The layer-wise path against the runtime-width SIMT kernel on the same seeds and action
    tape: identical trajectory, log-probs / values within 2e-5."""
    if rollout_impl != "tc":
        pytest.skip("compares the two paths itself")
    L = _lib.lib()
    N, T, hidden = 262144 + 4321, 2, 256
    _, named = random_policy(4, 2, hidden, 2, False, seed=8)
    desc = kernels.policy_desc(4, 2, hidden, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    actions = torch.randint(0, 2, (T, N), generator=torch.Generator().manual_seed(1)).float().cuda()
    res = {}
    for impl in (1, 0):
        assert L.aur_rollout_set_impl(impl) == 0
        env = denv.DeviceVecEnv("CartPole-v1", N)
        env.reset(list(range(N)))
        buf = kernels.RolloutBuffers(T, N, 4, (), "cuda")
        kernels.rollout(env, desc, flat, buf, seed=1, step0=0, actions_in=actions)
        torch.cuda.synchronize()
        res[impl] = (buf.states.clone(), buf.log_probs.clone(), buf.values.clone(), buf.next_value.clone(), env.next_obs.clone())
    L.aur_rollout_set_impl(1)
    assert torch.equal(res[1][0], res[0][0]) and torch.equal(res[1][4], res[0][4])
    for i in (1, 2, 3):
        torch.testing.assert_close(res[1][i], res[0][i], **TOL)
