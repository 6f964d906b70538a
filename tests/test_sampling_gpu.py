"""Every sampled action of the device samplers against the float64 restatement of oracle/ppo_ref.py, draw for draw: the
rollout kernels (SIMT, tensor-core, layer-wise, runtime width, population), policy_evaluate (64-wide and runtime-width
kernels, both Philox blocks), aur_squashed_gaussian_sample and the facades' head_eval_kernel, with ids and steps above
2^32.  Then the edge counters of tests/test_sampling_oracle.py on the device, and the draws against the specification
itself: chi-square of class counts, Kolmogorov-Smirnov per dimension, correlations.

Discrete draws: the class of the first CDF boundary above u, except draws closer to a boundary than the kernels'
probability error (from the log-prob bar they meet, rtol 2e-5: |dCDF| <= sum_j p_j |d log p_j| <= 2e-5 (1 + H)).
Continuous draws: |a - (mean + std z)| within the head's error plus the fp32 Box-Muller's (logf, sincosf, and u rounded
to fp32, which moves r = sqrt(-2 ln u) by at most min(2^-11.5, 2^-23 / r))."""
import ctypes

import numpy as np
import pytest
import torch
from scipy import special, stats

from aur_ppo_b200 import _lib, envs as denv, kernels, run_ppo
from aur_ppo_b200.population import ppo_population
from oracle import ppo_ref as R
from tests.helpers import flat_from_named, random_policy
from tests.test_sampling_oracle import EXTREME_COUNTERS

pytestmark = pytest.mark.gpu

LOGP_RTOL = 2e-5
HEAD_TOL = 1e-4       # |mean error| / (1 + |mean|) of a policy head computed by a kernel
ROUND_TOL = 1e-6      # the same for a mean given to the kernel: fp32 rounding of mean + std * z alone
Z_RTOL = 1e-5         # |z error| / (1 + r): logf, sincosf, the fp32 angle
R2_ERR = 2.0 ** -23   # |error of r^2| from u rounded to fp32
# Measured on one B200 (1000 W power limit), largest |a - a64| and its share of the tolerance:
#   rollouts 9.3e-6 (Pendulum, tensor-core kernel), 0.07;  policy_evaluate 4.3e-6, 0.03;  population 3.4e-6, 0.03;
#   squashed_gaussian_sample 3.9e-6, 0.13;  facade heads 1.0e-5 (equivariant), 0.15;
#   edge counters at u1 = 1 - 2^-24, where the device's u rounds to 1 and r to 0: 1.9e-4, 0.50.
# Discrete draws left out at a CDF boundary: 3e-5 .. 7e-4 of each check, no mismatch outside.


@pytest.fixture(params=["tc", "simt"])
def rollout_impl(request):
    L = _lib.lib()
    prev = L.aur_rollout_get_impl()
    assert L.aur_rollout_set_impl(1 if request.param == "tc" else 0) == 0
    yield request.param
    L.aur_rollout_set_impl(prev)


def _mlp64(named, prefix, x):
    idx = sorted({int(k.split(".")[2]) for k in named if k.startswith(prefix + ".net.")})
    h = np.asarray(x, np.float64)
    for j, i in enumerate(idx):
        h = h @ np.asarray(named[f"{prefix}.net.{i}.weight"], np.float64).T + np.asarray(named[f"{prefix}.net.{i}.bias"], np.float64)
        if j != len(idx) - 1:
            h = np.tanh(h)
    return h


def _named_from_flat(flat, obs_dim, A, hidden, layers, cont):
    named, o = {}, 0
    for prefix, out in (("actor", A), ("critic", 1)):
        dims = [obs_dim] + [hidden] * layers + [out]
        for li in range(len(dims) - 1):
            for name, shape in (("weight", (dims[li + 1], dims[li])), ("bias", (dims[li + 1],))):
                n = int(np.prod(shape))
                named[f"{prefix}.net.{2 * li}.{name}"] = flat[o:o + n].reshape(shape)
                o += n
    if cont:
        named["actor_logstd"] = flat[o:o + A].reshape(1, A)
        o += A
    assert o == flat.size
    return named


def _u24(word0):
    return (np.asarray(word0) >> np.uint32(8)).astype(np.float64) * 2.0 ** -24


def _normals(seed, idx, stream, A):
    """z [.., A] of Philox blocks 0 .. (A - 1) / 4 and the Box-Muller radius r each dim came from."""
    z = np.concatenate([R.normal4_f64(R.sampler_words_np(seed, idx, stream, blk)) for blk in range((A + 3) // 4)], axis=-1)
    r = np.repeat(np.hypot(z[..., 0::2], z[..., 1::2]), 2, axis=-1)
    return z[..., :A], r[..., :A]


def _check_discrete(logits, u, act, what):
    p = special.softmax(np.asarray(logits, np.float64), axis=1)
    want, margin = R.categorical_icdf(p, u)
    keep = margin > LOGP_RTOL * (1.0 + special.entr(p).sum(axis=1))
    bad = np.nonzero(keep & (want != act))[0]
    excluded = 1.0 - keep.mean()
    print(f"{what}: {act.size} draws, {bad.size} mismatches, {excluded:.2e} left out at a CDF boundary")
    assert bad.size == 0, (what, bad[:8], want[bad[:8]], act[bad[:8]], u[bad[:8]])
    assert excluded < 0.01
    return want


def _check_continuous(mean, std, z, r, act, what, head_tol=HEAD_TOL):
    want = mean + std * z
    err = np.abs(act - want)
    bound = head_tol * (1.0 + np.abs(mean)) + std * (Z_RTOL * (1.0 + r) + np.minimum(np.sqrt(R2_ERR), R2_ERR / np.maximum(r, 1e-300)))
    ratio = err / bound
    print(f"{what}: {act.size} draws, max |a - a64| {err.max():.3e}, max error / tolerance {ratio.max():.3f}")
    assert np.isfinite(act).all() and (err <= bound).all(), (what, np.unravel_index(ratio.argmax(), ratio.shape), err.max())


def _head_policy(obs_dim, A, cont, head, logstd=None, seed=0):
    """random_policy with the actor's output layer replaced: W3 = 0 and b3 = head, so every row's logits / mean are `head`
    exactly (0 * h + b in fp32), whatever the observation."""
    _, named = random_policy(obs_dim, A, 64, 2, cont, seed=seed)
    named["actor.net.4.weight"] = np.zeros_like(named["actor.net.4.weight"])
    named["actor.net.4.bias"] = np.asarray(head, np.float32)
    if cont:
        named["actor_logstd"] = np.asarray(logstd, np.float32).reshape(1, A)
    return kernels.policy_desc(obs_dim, A, 64, 2, cont), named


# ---- rollouts --------------------------------------------------------------------------------------------------------
# gym_id, obs, act, hidden, layers, continuous, wrappers, N, T, two kernels (tc and simt differ)
ROLLOUTS = {
    "cartpole-64x2": ("CartPole-v1", 4, 2, 64, 2, False, False, 10240, 6, True),      # simt: 2 envs per thread from 9,472
    "cartpole-128x2": ("CartPole-v1", 4, 2, 128, 2, False, False, 2048, 12, True),
    "cartpole-256x2": ("CartPole-v1", 4, 2, 256, 2, False, False, 2048, 8, True),     # tc: layer-wise actor (rollout_wide.cu)
    "cartpole-32x3": ("CartPole-v1", 4, 2, 32, 3, False, False, 2048, 12, False),
    "mountaincar": ("MountainCar-v0", 2, 3, 64, 2, False, False, 2048, 12, True),
    "acrobot": ("Acrobot-v1", 6, 3, 64, 2, False, False, 2048, 12, False),
    "pendulum-wrappers": ("Pendulum-v1", 3, 1, 64, 2, True, True, 2048, 12, True),
    "pendulum": ("Pendulum-v1", 3, 1, 64, 2, True, False, 2048, 12, True),
    "mountaincar-cont": ("MountainCarContinuous-v0", 2, 1, 64, 2, True, True, 2048, 12, False),
}


@pytest.mark.parametrize("case", list(ROLLOUTS))
def test_sampled_rollout_draws_follow_the_restatement(case, rollout_impl):
    gym_id, obs_dim, A, hidden, layers, cont, wrappers, N, T, two = ROLLOUTS[case]
    if rollout_impl == "simt" and not two:
        pytest.skip("one kernel behind this shape")
    _, named = random_policy(obs_dim, A, hidden, layers, cont, seed=hidden + A, scale=2.0)
    desc = kernels.policy_desc(obs_dim, A, hidden, layers, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    seed, env_id0, step0 = 0x9E3779B97F4A7C15, 2 ** 32 - N // 2, 2 ** 32 + 3       # env ids and steps cross 2^32
    env = denv.DeviceVecEnv(gym_id, N, wrappers=wrappers, env_id0=env_id0)
    env.reset(list(range(N)))
    buf = kernels.RolloutBuffers(T, N, obs_dim, (A,) if cont else (), "cuda")
    kernels.rollout(env, desc, flat, buf, seed=seed, step0=step0)
    head = _mlp64(named, "actor", buf.states.cpu().numpy().reshape(-1, obs_dim))
    gid = (np.uint64(env_id0) + np.arange(N, dtype=np.uint64))[None, :].repeat(T, 0).reshape(-1)
    step = (np.uint64(step0) + np.arange(T, dtype=np.uint64)).repeat(N)
    what = f"{case} ({rollout_impl})"
    if cont:
        z, r = _normals(seed, gid, step, A)
        std = np.exp(named["actor_logstd"].astype(np.float64))
        _check_continuous(head, std, z, r, buf.actions.cpu().numpy().reshape(-1, A), what)
    else:
        u = _u24(R.sampler_words_np(seed, gid, step)[0])
        _check_discrete(head, u, buf.actions.cpu().numpy().reshape(-1).astype(np.int64), what)


def _pop_params(**kw):
    p = run_ppo.params_from_args(run_ppo.build_parser().parse_args([]))
    p.update(tensorboard=False, save=False)
    p.update(kw)
    return p


@pytest.mark.parametrize("gym_id", ["CartPole-v1", "Pendulum-v1"])
def test_population_members_draw_with_their_own_keys(gym_id):
    """K = 3 members in one launch: member k draws with its own seed and member-local env ids."""
    cont = gym_id == "Pendulum-v1"
    n, T = 1024, 16
    params = _pop_params(gym_id=gym_id, continuous=cont, num_envs=n, num_steps=T, num_minibatches=4, num_update_epochs=1,
                         total_timesteps=n * T)
    seeds = [11, 2 ** 33 + 5, 7]
    pop = ppo_population(params, [dict(seed=float(s)) for s in seeds])
    pop.reset_envs()
    pop._env_step = 2 ** 32 - 7                                         # steps cross 2^32
    pop.rollout()
    obs_dim, A = (3, 1) if cont else (4, 2)
    gid = np.arange(n, dtype=np.uint64)[None, :].repeat(T, 0).reshape(-1)
    step = (np.uint64(2 ** 32 - 7) + np.arange(T, dtype=np.uint64)).repeat(n)
    zs = []
    for k, seed in enumerate(seeds):
        cols = slice(k * n, (k + 1) * n)
        named = _named_from_flat(pop.params[k].cpu().numpy(), obs_dim, A, 64, 2, cont)
        head = _mlp64(named, "actor", pop.buffer.states[:, cols].cpu().numpy().reshape(-1, obs_dim))
        act = pop.buffer.actions[:, cols].cpu().numpy()
        if cont:
            z, r = _normals(seed, gid, step, A)
            std = np.exp(named["actor_logstd"].astype(np.float64))
            _check_continuous(head, std, z, r, act.reshape(-1, A), f"{gym_id} member {k}")
            zs.append((act.reshape(-1) - head.reshape(-1)) / std.reshape(-1))
        else:
            _check_discrete(head, _u24(R.sampler_words_np(seed, gid, step)[0]), act.reshape(-1).astype(np.int64), f"{gym_id} member {k}")
    if cont:                                                            # the members' noise is independent
        c = np.corrcoef(np.stack(zs))
        print(f"correlation of the members' z over {zs[0].size} draws: {c[0, 1]:.2e} {c[0, 2]:.2e} {c[1, 2]:.2e}")
        assert np.abs(c - np.eye(3)).max() < 5 / np.sqrt(zs[0].size)


# ---- policy_evaluate -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cont", [False, True])
@pytest.mark.parametrize("A", range(1, 9))
def test_policy_evaluate_draws_follow_the_restatement(A, cont):
    """act_dim 1..4: the 64-wide kernel; 5..8: the runtime-width kernel, dims 4..7 from the second Philox block.  Rows cross
    2^32 and the step is above 2^32; the high halves of both must change the draws."""
    B = 16384
    _, named = random_policy(4, A, 64, 2, cont, seed=40 + A, scale=2.0)
    desc = kernels.policy_desc(4, A, 64, 2, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    obs = torch.randn(B, 4, generator=torch.Generator().manual_seed(A)).cuda()
    seed, row0, step = 2 ** 63 + 77, 2 ** 32 - B // 2, 5 * 2 ** 32 + 9
    act = kernels.policy_evaluate(desc, flat, obs, seed=seed, row0=row0, step=step)[0].cpu().numpy()
    head = _mlp64(named, "actor", obs.cpu().numpy())
    rows = np.uint64(row0) + np.arange(B, dtype=np.uint64)
    what = f"policy_evaluate act_dim {A} {'continuous' if cont else 'discrete'}"
    if cont:
        z, r = _normals(seed, rows, step, A)
        _check_continuous(head, np.exp(named["actor_logstd"].astype(np.float64)), z, r, act.reshape(B, A), what)
    else:
        _check_discrete(head, _u24(R.sampler_words_np(seed, rows, step)[0]), act.astype(np.int64), what)
    # the same rows with the step's high half dropped, and the rows above 2^32 at their low 32 bits, draw differently
    lo_step = kernels.policy_evaluate(desc, flat, obs, seed=seed, row0=row0, step=step & 0xFFFFFFFF)[0].cpu().numpy()
    lo_rows = np.roll(kernels.policy_evaluate(desc, flat, obs.roll(B // 2, 0), seed=seed, row0=0, step=step)[0].cpu().numpy(), B // 2, 0)
    for other in (lo_step, lo_rows[B // 2:]):
        mine = act if other is lo_step else act[B // 2:]
        if cont:
            assert (other != mine).all()
        elif A > 1:
            assert (other != mine).mean() > 0.02


# ---- squashed Gaussian and the facades' heads ------------------------------------------------------------------------
@pytest.mark.parametrize("A", [1, 5, 16])
def test_squashed_gaussian_draws_follow_the_restatement(A):
    B = 8192
    g = torch.Generator().manual_seed(A)
    mean = torch.randn(B, A, generator=g)
    log_std = torch.rand(B, A, generator=g) * 1.5 - 1.0
    seed, stream = 2 ** 40 + 3, 3 * 2 ** 32 + 17
    y, lp, mo, ent, pre = kernels.squashed_gaussian_sample(mean.cuda(), log_std.cuda(), None, seed=seed, stream_id=stream,
                                                           return_pre_tanh=True)
    z, r = _normals(seed, np.arange(B, dtype=np.uint64), stream, A)
    std = np.exp(log_std.numpy().astype(np.float64))
    _check_continuous(mean.numpy().astype(np.float64), std, z, r, pre.cpu().numpy(), f"squashed_gaussian_sample A={A}", ROUND_TOL)
    assert torch.equal(y, torch.tanh(pre))


@pytest.mark.parametrize("equivariant", [False, True])
def test_facade_head_draws_follow_the_restatement(equivariant):
    """head_eval_kernel's 5-dim Normal draw (robot_actor_critic.evaluate) through aur_plain_head_eval / aur_equiv_head_eval,
    which take the seed and the stream id: counter (b, 0, stream lo, stream hi ^ blk << 24)."""
    B = 8192
    g = torch.Generator().manual_seed(5)
    a_out = torch.randn(B, 16, generator=g).cuda()
    a_bias = (torch.randn(10, generator=g) * 0.5).cuda()
    logstd = (torch.rand(5, generator=g) * 1.5 - 1.0).cuda()
    seed, stream = 2 ** 50 + 99, 2 ** 32 + 41
    f = lambda *s: torch.empty(*s, device="cuda")
    unscaled, scaled, lp, ent, mean, ls = f(B, 5), f(B, 5), f(B), f(B), f(B, 5), f(B, 5)
    ranges = (ctypes.c_float * 10)(0.0, 1.0, -0.02, 0.02, -0.02, 0.02, -0.02, 0.02, -0.4, 0.4)
    outs = (unscaled.data_ptr(), scaled.data_ptr(), lp.data_ptr(), ent.data_ptr(), None, mean.data_ptr(), ls.data_ptr())
    L = _lib.lib()
    if equivariant:
        rc = L.aur_equiv_head_eval(B, a_out.data_ptr(), a_bias.data_ptr(), None, None, None, None, None, seed, stream, ranges,
                                   *outs, kernels._stream())
    else:
        rc = L.aur_plain_head_eval(B, a_out.data_ptr(), a_bias.data_ptr(), logstd.data_ptr(), None, None, None, None, None, seed,
                                   stream, ranges, *outs, kernels._stream())
    _lib.check(rc, "head_eval")
    o10 = (a_out[:, :10] + torch.cat([a_bias[:5], a_bias[5:] * (1 if equivariant else 0)])).cpu().numpy()
    want_mean = o10[:, [2, 0, 1, 3, 4]] if equivariant else o10[:, :5]
    want_ls = np.clip(o10[:, 5:], -20, 2) if equivariant else np.broadcast_to(logstd.cpu().numpy(), (B, 5))
    assert np.array_equal(mean.cpu().numpy(), want_mean) and np.array_equal(ls.cpu().numpy(), want_ls)
    z, r = _normals(seed, np.arange(B, dtype=np.uint64), stream, 5)
    _check_continuous(want_mean.astype(np.float64), np.exp(want_ls.astype(np.float64)), z, r, unscaled.cpu().numpy(),
                      f"{'equivariant' if equivariant else 'plain CNN'} head", ROUND_TOL)


# ---- edge counters ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,gid,step,word,value", EXTREME_COUNTERS)
def test_extreme_counters_on_the_device(seed, gid, step, word, value):
    """B = 1 at row0 = gid: the categorical u at 0 and at the top, the smallest radii and an angle of ~0."""
    for A in (3, 6):                                                     # 64-wide and runtime-width kernels
        desc, named = _head_policy(4, A, False, np.linspace(0.4, -0.3, A))
        act = kernels.policy_evaluate(desc, torch.from_numpy(flat_from_named(named)).cuda(), torch.zeros(1, 4, device="cuda"),
                                      seed=seed, row0=gid, step=step)[0].cpu().numpy().astype(np.int64)
        _check_discrete(named["actor.net.4.bias"][None, :], _u24(R.sampler_words_np(seed, np.array([gid], np.uint64), step)[0]), act,
                        f"act_dim {A} at gid {gid} step {step}")
    for A in (4, 8):
        mean, logstd = np.linspace(0.5, -1.0, A), np.linspace(-0.5, 0.3, A)
        desc, named = _head_policy(4, A, True, mean, logstd)
        act = kernels.policy_evaluate(desc, torch.from_numpy(flat_from_named(named)).cuda(), torch.zeros(1, 4, device="cuda"),
                                      seed=seed, row0=gid, step=step)[0].cpu().numpy()
        z, r = _normals(seed, np.array([gid], np.uint64), step, A)
        _check_continuous(named["actor.net.4.bias"].astype(np.float64)[None, :], np.exp(logstd.astype(np.float32).astype(np.float64)),
                          z, r, act.reshape(1, A), f"continuous act_dim {A} at gid {gid} step {step}")


def _dead_class_draws(A, dead, counters, vectors):
    """One policy_evaluate per (logit vector, counter): the class `dead` has logit 150 below the others, so its fp32
    probability is exactly 0 (expf underflows below -103.9)."""
    rng = np.random.default_rng(A)
    desc, named = _head_policy(4, A, False, np.zeros(A))
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    b3 = flat.numel() - (64 * 4 + 64 + 64 * 64 + 64 + 64 + 1) - A            # actor output bias: before the critic
    obs = torch.zeros(1, 4, device="cuda")
    got = []
    for _ in range(vectors):
        lg = (rng.standard_normal(A) * 2).astype(np.float32)
        lg[dead] = lg.min() - 150
        flat[b3:b3 + A] = torch.from_numpy(lg)
        for (seed, gid, step) in counters:
            got.append(int(kernels.policy_evaluate(desc, flat, obs, seed=seed, row0=gid, step=step)[0].item()))
    return np.array(got)


@pytest.mark.parametrize("A", [3, 4, 8])
def test_a_dead_class_is_never_drawn(A):
    """u = 0 must not take a dead first class (`u < c`, not `<=`); u in the top 16 values must not take a dead last class
    when the fp32 CDF ends below u."""
    zero = [(s, g, t) for s, g, t, w, v in EXTREME_COUNTERS if w == 0 and v == 0]
    top = [(s, g, t) for s, g, t, w, v in EXTREME_COUNTERS if w == 0 and v >= 0xFFFFF0]
    first = _dead_class_draws(A, 0, zero, 20)
    assert (first == 1).all(), np.bincount(first)
    last = _dead_class_draws(A, A - 1, top, 300)
    print(f"act_dim {A}: {last.size} draws at u >= 1 - 2^-20 with a dead last class, classes drawn {np.bincount(last, minlength=A)}")
    assert (last != A - 1).all() and (last == A - 2).mean() > 0.9


# ---- against the specification ---------------------------------------------------------------------------------------
M = 1 << 22


@pytest.mark.parametrize("A", [3, 4, 8])
def test_class_counts_follow_the_softmax(A):
    logits = np.linspace(-1.5, 1.0, A)[np.random.default_rng(A).permutation(A)]
    desc, named = _head_policy(4, A, False, logits)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    act = kernels.policy_evaluate(desc, flat, torch.zeros(M, 4, device="cuda"), seed=123, row0=0, step=1)[0]
    counts = torch.bincount(act.long(), minlength=A).cpu().numpy()
    p = special.softmax(named["actor.net.4.bias"].astype(np.float64))
    chi = stats.chisquare(counts, p * M)
    print(f"act_dim {A}: chi-square {chi.statistic:.2f} on {A - 1} dof, p-value {chi.pvalue:.3f}")
    assert counts.sum() == M and chi.pvalue > 1e-3


def test_normal_draws_follow_the_standard_normal():
    """act_dim 8, mean 0, std 1 (the action is z itself): Kolmogorov-Smirnov per dim, the 8 x 8 correlation, and the
    correlation between adjacent env ids, adjacent steps and two seeds (two population members' keys)."""
    desc, named = _head_policy(4, 8, True, np.zeros(8), np.zeros(8))
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    obs = torch.zeros(M, 4, device="cuda")
    draw = lambda seed, step: kernels.policy_evaluate(desc, flat, obs, seed=seed, row0=2 ** 32 - M // 2, step=step)[0].cpu().numpy().astype(np.float64)
    z = draw(9, 4)
    lim = 5 / np.sqrt(M)
    for d in range(8):
        ks = stats.kstest(z[:, d], "norm")
        print(f"dim {d}: KS statistic {ks.statistic:.2e}, p-value {ks.pvalue:.3f}")
        assert ks.pvalue > 1e-3
    c = np.corrcoef(z.T)
    print(f"largest off-diagonal correlation of z over {M} draws: {np.abs(c - np.eye(8)).max():.2e} (bound {lim:.2e})")
    assert np.abs(c - np.eye(8)).max() < lim
    pairs = {"adjacent env ids": (z[:-1], z[1:]), "adjacent steps": (z, draw(9, 5)), "two seeds": (z, draw(10, 4))}
    for what, (x, y) in pairs.items():
        cc = [np.corrcoef(x[:, d], y[:, d])[0, 1] for d in range(8)]
        print(f"{what}: largest correlation {np.abs(cc).max():.2e}")
        assert np.abs(cc).max() < lim
