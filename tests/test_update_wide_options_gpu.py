"""The layer-wise tensor-core update (csrc/update_wide.cu, `--hidden_dim` 128 / 256) under the loss options, actor heads and
minibatch sizes that run_ppo.py can reach and test_update_wide_gpu.py does not run, against the float64 restatement
(oracle/ppo_ref.py, RefPolicy(dtype=float64)).

Every row names the branch, instantiation or tile edge it is the first to run.  Each row takes two minibatch steps
(grad + apply).  Before each step, any sample whose float64 ratio or value delta lies within 1e-3 of a clip edge has its
oldlp / vold moved away: fp32 and fp64 may round such a sample to different sides, which would change its gradient by a
whole term.  The bars are the ones the other update tests use: gradients within 1e-4 of max|g| elementwise and 1e-4 relative
L2, stats 1e-4, parameters after Adam 1e-5 / 1e-6, and clipfrac as an exact count.  Each step prints the kernel's distance
to float64 next to the fp32 restatement's own distance to float64."""
import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, kernels
from oracle import ppo_ref as R
from tests.helpers import flat_from_named, random_policy

pytestmark = pytest.mark.gpu

EDGE = 1e-3           # no sample's float64 clip decision may lie closer than this to its edge
NUDGE = 0.013         # how far a sample near an edge is moved (log-prob or value units)


def _rel_l2(got, want):
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def _inputs(obs_dim, act_dim, hidden, layers, cont, m, B, seed):
    _, named = random_policy(obs_dim, act_dim, hidden, layers, cont, seed=seed)
    g = torch.Generator().manual_seed(seed * 7 + m)
    obs = torch.randn(B, obs_dim, generator=g) * 0.7
    act = torch.randn(B, act_dim, generator=g) if cont else torch.randint(0, act_dim, (B,), generator=g).float()
    with torch.no_grad():
        _, lp0, _, v0 = R.RefPolicy(named, cont).evaluate(obs, act)
    oldlp = lp0 + 0.25 * torch.randn(B, generator=g)             # some ratios leave the clip range
    adv = torch.randn(B, generator=g) * 3 + 0.5
    ret = torch.randn(B, generator=g)
    vold = v0.flatten() + 0.4 * torch.randn(B, generator=g)      # some value deltas leave the clip range
    idx = torch.randperm(B, generator=g)[:m]
    return named, [obs, act, oldlp, adv, ret, vold], idx


def _keep_off_the_edges(pol64, bufs, idx, clip, clip_vloss):
    """Move oldlp (policy ratio) or vold (value clip, and the max of the two value losses) of every sample of `idx` whose
    float64 decision lies within EDGE of its edge, in place; returns how many moves it took."""
    obs, act, oldlp, _, ret, vold = bufs
    moved = 0
    for _ in range(50):
        with torch.no_grad():
            _, lp, _, v = pol64.evaluate(obs[idx].double(), act[idx] if not pol64.continuous else act[idx].double())
        v = v.view(-1)
        ratio = torch.exp(lp - oldlp[idx].double())
        near_p = ((ratio - (1 - clip)).abs() < EDGE) | ((ratio - (1 + clip)).abs() < EDGE)
        near_v = torch.zeros_like(near_p)
        if clip_vloss:
            d = v - vold[idx].double()
            near_v = ((d - clip).abs() < EDGE) | ((d + clip).abs() < EDGE)
            # outside the clip range the larger of the two value losses picks the gradient term (inside, both are the same)
            vc = vold[idx].double() + d.clamp(-clip, clip)
            tie = ((v - ret[idx].double()).abs() - (vc - ret[idx].double()).abs()).abs() < EDGE
            near_v |= (d.abs() > clip) & tie
        if not bool(near_p.any() or near_v.any()):
            return moved
        oldlp[idx[near_p]] += NUDGE
        vold[idx[near_v]] += NUDGE
        moved += int(near_p.sum() + near_v.sum())
    raise AssertionError("could not move the samples off the clip edges")


# obs_dim, act_dim, hidden, layers, continuous, m, B, norm_adv, clip_vloss, clip_coeff, entropy_coeff, value_coeff
ROWS = {
    # wide_head_kernel's critic `clip_vloss == 0` branch (the reference's b_values quirk): discrete 128 x 2, continuous 256 x 2
    "novclip-disc128": (4, 2, 128, 2, False, 3000, 4096, True, False, 0.2, 0.01, 0.5),
    "novclip-cont256": (3, 1, 256, 2, True, 2500, 4096, True, False, 0.2, 0.0, 0.5),
    # the actor's `norm_adv == 0` branch (raw advantages, no moments launch): continuous 128 x 2, discrete 256 x 3 (middle layer)
    "nonorm-cont128": (3, 1, 128, 2, True, 2000, 4096, False, True, 0.2, 0.0, 0.5),
    "nonorm-disc256x3": (6, 3, 256, 3, False, 1500, 4096, False, True, 0.2, 0.01, 0.5),
    # coefficients other than 0.2 / 0.01 / 0.5 in the clip range, the entropy gradient and the value scale
    "coef-0.1-0-1": (4, 2, 128, 2, False, 2048, 4096, True, True, 0.1, 0.0, 1.0),
    "coef-0.3-0.05-0.25": (3, 1, 256, 2, True, 1800, 4096, True, True, 0.3, 0.05, 0.25),
    # the four heads no other test instantiates; obs 1 / 2 pad wide_first_kernel<4>, obs 5 / 7 pad wide_first_kernel<8>
    "head-disc1-obs1": (1, 1, 128, 2, False, 1500, 4096, True, True, 0.2, 0.01, 0.5),      # wide_head_kernel<0, 1>
    "head-disc4-obs7": (7, 4, 256, 2, False, 1500, 4096, True, True, 0.2, 0.01, 0.5),      # wide_head_kernel<0, 4>
    "head-cont2-obs2": (2, 2, 128, 3, True, 1500, 4096, True, True, 0.2, 0.0, 0.5),        # wide_head_kernel<1, 2>
    "head-cont3-obs5": (5, 3, 256, 2, True, 1500, 4096, True, True, 0.2, 0.0, 0.5),        # wide_head_kernel<1, 3>
    # minibatch sizes at the tile edges: one sample (std of one sample is NaN in the reference too, so no normalisation),
    # one short / one full 64-sample TMA box, one full / one just over a 1,024-sample partial row
    "m1": (4, 2, 128, 2, False, 1, 64, False, True, 0.2, 0.01, 0.5),
    "m63": (3, 1, 128, 2, True, 63, 1000, True, True, 0.2, 0.0, 0.5),
    "m64": (4, 2, 256, 2, False, 64, 1000, True, True, 0.2, 0.01, 0.5),
    "m1024": (4, 2, 128, 2, False, 1024, 4096, True, True, 0.2, 0.01, 0.5),
    "m1025": (6, 3, 128, 2, False, 1025, 4096, True, True, 0.2, 0.01, 0.5),
}


@pytest.mark.parametrize("row", list(ROWS))
def test_wide_update_options_vs_float64(row):
    obs_dim, act_dim, hidden, layers, cont, m, B, norm_adv, clip_vloss, clip, ent_c, vf_c = ROWS[row]
    L = _lib.lib()
    assert L.aur_ppo_update_get_wide() == 1
    named, bufs, idx = _inputs(obs_dim, act_dim, hidden, layers, cont, m, B, seed=hidden + layers + act_dim + obs_dim)
    names = list(named.keys())
    pol64, pol32 = R.RefPolicy(named, cont, dtype=torch.float64), R.RefPolicy(named, cont)
    opt64, opt32 = R.RefAdam(pol64.tensors(), lr=3e-4, eps=1e-5), R.RefAdam(pol32.tensors(), lr=3e-4, eps=1e-5)
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, cont)
    params = torch.from_numpy(flat_from_named(named)).cuda()
    up = kernels.Updater(desc, params)
    didx = idx.to(torch.int32).cuda()
    kw = dict(norm_adv=norm_adv, clip_vloss=clip_vloss)
    for step in range(2):
        moved = _keep_off_the_edges(pol64, bufs, idx, clip, clip_vloss)
        mb = [b[idx] for b in bufs]
        mb64 = [b if i == 1 and not cont else b.double() for i, b in enumerate(mb)]
        st64, raw64, _, _ = R.ppo_update_step(pol64, opt64, *mb64, max_grad_norm=0.5, clip_coeff=clip, ent_c=ent_c, vf_c=vf_c, **kw)
        st32, raw32, _, _ = R.ppo_update_step(pol32, opt32, *mb, max_grad_norm=0.5, clip_coeff=clip, ent_c=ent_c, vf_c=vf_c, **kw)
        dbuf = [b.cuda().contiguous() for b in bufs]
        L.aur_launch_count_reset()
        grads = up.grad(*dbuf, didx, clip_coeff=clip, entropy_coeff=ent_c, value_coeff=vf_c, **kw).clone()
        assert L.aur_launch_count() >= 2 * (5 + 3 * (layers - 2)) + 1 - (0 if norm_adv else 1)   # the layer-wise path ran
        stats = up.apply(3e-4, 0.5).cpu().numpy()
        want = flat_from_named({n: r.numpy() for n, r in zip(names, raw64)}, np.float64)
        ref32 = flat_from_named({n: r.numpy() for n, r in zip(names, raw32)}, np.float64)
        got = grads[:up.P].cpu().numpy().astype(np.float64)
        p_want = flat_from_named({n: pol64.p[n].numpy() for n in names}, np.float64)
        p_got = params.cpu().numpy().astype(np.float64)
        p_ref32 = flat_from_named({n: pol32.p[n].numpy() for n in names}, np.float64)
        s_rel = lambda st: max(abs(st[k] - st64[k]) / max(abs(st64[k]), 1e-30) for k in kernels.STAT_NAMES if k != "clipfrac")
        kst = {k: float(stats[i]) for i, k in enumerate(kernels.STAT_NAMES)}
        print(f"{row} step {step} ({moved} samples moved off a clip edge): distance to float64 -- gradient rel L2 kernel "
              f"{_rel_l2(got, want):.2e} / fp32 restatement {_rel_l2(ref32, want):.2e}; stats max rel kernel {s_rel(kst):.2e} / "
              f"fp32 {s_rel(st32):.2e}; parameters max abs kernel {np.abs(p_got - p_want).max():.2e} / "
              f"fp32 {np.abs(p_ref32 - p_want).max():.2e}; clipfrac {kst['clipfrac'] * m:.0f} / {st64['clipfrac'] * m:.0f} of {m}")
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * float(np.abs(want).max()) + 1e-9)
        assert _rel_l2(got, want) < 1e-4
        for i, k in enumerate(kernels.STAT_NAMES):
            if k == "clipfrac":
                count = stats[i] * m
                assert abs(count - round(count)) < 1e-3 and round(count) == round(st64[k] * m), (count, st64[k] * m)
            else:
                np.testing.assert_allclose(stats[i], st64[k], rtol=1e-4, atol=2e-6, err_msg=k)
        np.testing.assert_allclose(p_got, p_want, rtol=1e-5, atol=1e-6)
