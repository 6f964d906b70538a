"""Pins oracle/ppo_ref.py to the golden vectors generated from the reference's own
code (oracle/gen_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import ppo_ref as R


def _t(a):
    return torch.from_numpy(np.asarray(a))


def test_gae_known_answer_and_random(golden_dir):
    g = np.load(os.path.join(golden_dir, "gae.npz"))
    for name in g["names"]:
        rew, val, term, nv, nd = (_t(g[f"{name}_{k}"]) for k in ("rew", "val", "term", "nv", "nd"))
        gamma, lam = float(g[f"{name}_gamma"]), float(g[f"{name}_lam"])
        ret, adv = R.gae(rew, val, term, nv, nd, gamma, lam)
        assert np.array_equal(ret.numpy(), g[f"{name}_gae_ret"]), name
        assert np.array_equal(adv.numpy(), g[f"{name}_gae_adv"]), name
        ret2, adv2 = R.normal_advantage(rew, val, term, nv, nd, gamma)
        assert np.array_equal(ret2.numpy(), g[f"{name}_mc_ret"]), name
        assert np.array_equal(adv2.numpy(), g[f"{name}_mc_adv"]), name
    # the numbers quoted in SURVEY.md section 8(c)
    np.testing.assert_allclose(g["ka_gae_adv"].flatten()[:3], [3.8616199493, 1.5232572556, 2.5640804768], rtol=1e-7)
    np.testing.assert_allclose(g["ka_mc_ret"].flatten()[:3], [4.1805477142, 1.9900000095, 3.2126746178], rtol=1e-7)


def _policy(g, tag, prefix):
    names = [str(n) for n in g[f"{tag}_names"]]
    return R.RefPolicy({n: g[f"{tag}_{prefix}_{n}"] for n in names}, continuous="actor_logstd" in names), names


@pytest.mark.parametrize("tag", ["disc", "cont", "disc3", "cont2"])
def test_model_forward(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "model.npz"))
    pol, _ = _policy(g, tag, "p")
    obs, act = _t(g[f"{tag}_obs"]), _t(g[f"{tag}_act"])
    a, lp, ent, v = pol.evaluate(obs, act)
    np.testing.assert_allclose(lp.numpy(), g[f"{tag}_logp"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(ent.numpy(), g[f"{tag}_ent"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(v.numpy(), g[f"{tag}_value"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(pol.value(obs).numpy(), g[f"{tag}_value_flat"], rtol=2e-6, atol=1e-7)


@pytest.mark.parametrize("tag", ["disc", "disc_big", "cont", "disc_nonorm", "disc_novclip"])
def test_update_step(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "update.npz"))
    pol, names = _policy(g, tag, "p0")
    clip, ent_c, vf_c, mgn, lr, norm_adv, clip_vloss = g[f"{tag}_hyper"]
    opt = R.RefAdam(pol.tensors(), lr=float(lr), eps=1e-5)
    obs, act, oldlp, adv, ret, vold = (_t(g[f"{tag}_{k}"]) for k in ("obs", "act", "oldlp", "adv", "ret", "vold"))
    for step in range(2):
        stats, raw, nlp, nv = R.ppo_update_step(pol, opt, obs, act, oldlp, adv, ret, vold, max_grad_norm=float(mgn),
                                                clip_coeff=float(clip), ent_c=float(ent_c), vf_c=float(vf_c),
                                                norm_adv=bool(norm_adv), clip_vloss=bool(clip_vloss))
        want = g[f"{tag}_s{step}_stats"]
        got = [stats[k] for k in ("policy_loss", "value_loss", "entropy", "loss", "old_approx_kl", "approx_kl",
                                  "clipfrac", "grad_norm")]
        np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-7)
        for n, gr in zip(names, raw):
            np.testing.assert_allclose(gr.numpy(), g[f"{tag}_s{step}_g_{n}"], rtol=2e-4, atol=2e-7, err_msg=n)
        for n in names:
            np.testing.assert_allclose(pol.p[n].numpy(), g[f"{tag}_s{step}_p_{n}"], rtol=1e-5, atol=1e-7, err_msg=n)
    if tag == "disc":   # SURVEY.md 8(c) quoted values
        np.testing.assert_allclose(g["disc_s0_stats"][[0, 1, 2, 3, 7]],
                                   [-0.0097216293, 0.4503803849, 0.6908517480, 0.2085600495, 1.0845984221], rtol=2e-5)


def test_squashed_sample(golden_dir):
    g = np.load(os.path.join(golden_dir, "squash.npz"))
    x, act = _t(g["x"]), _t(g["act"])
    y, lp, mean, ent = R.squashed_sample(x[:, :5], x[:, 5:], act)
    np.testing.assert_allclose(y.numpy(), g["a"], rtol=1e-6)
    np.testing.assert_allclose(lp.numpy(), g["logp"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(mean.numpy(), g["mean"], rtol=1e-6)
    np.testing.assert_allclose(ent.numpy(), g["ent"], rtol=1e-6)


def test_philox_known_answer():
    # Random123 kat_vectors: philox4x32-10, counter/key all zero and all ones
    assert R.philox4x32_10((0, 0, 0, 0), (0, 0)) == (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)
    assert R.philox4x32_10((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2) == (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)
    assert R.philox4x32_10((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0)) == (
        0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)


def test_explained_variance_and_anneal():
    v = np.array([0.0, 1.0, 2.0, 3.0], np.float32)
    r = np.array([0.5, 1.0, 2.5, 2.0], np.float32)
    assert abs(R.explained_variance(v, r) - (1 - np.var(r - v) / np.var(r))) < 1e-12
    assert np.isnan(R.explained_variance(v, np.ones(4, np.float32)))
    assert R.lr_anneal(2.5e-4, 1, 10) == 2.5e-4
    assert abs(R.lr_anneal(2.5e-4, 6, 10) - 1.25e-4) < 1e-18


def test_feistel_shuffle_restatement_is_a_permutation():
    for n in (1, 2, 5, 1000, 4097, 1 << 16):
        p = R.feistel_shuffle(n, seed=9, stream_id=n)
        assert p.dtype == np.int32 and np.array_equal(np.sort(p), np.arange(n))
    a, b = R.feistel_shuffle(4096, 1, 0), R.feistel_shuffle(4096, 1, 1)
    assert (a == b).mean() < 0.01 and np.array_equal(a, R.feistel_shuffle(4096, 1, 0))
    assert abs(np.corrcoef(a, np.arange(4096))[0, 1]) < 0.08


@pytest.mark.parametrize("tag", ["disc128", "cont128", "disc128x3"])
def test_update_step_wide_shapes(golden_dir, tag):
    """The restated update against the reference's own gradients at 128 hidden units (tests/golden/update_wide.npz, written by
    oracle/gen_golden_wide.py from the imported reference): pins the checker of the wide GPU paths, not only the 64-wide one."""
    from tests.helpers import flat_from_named, golden_flat
    g = np.load(os.path.join(golden_dir, "update_wide.npz"))
    names = [str(n) for n in g[f"{tag}_names"]]
    named0 = {}
    for i, n in enumerate(names):
        shape = tuple(int(v) for v in g[f"{tag}_pshape_{n}"])
        k = np.arange(int(np.prod(shape)), dtype=np.float64)
        named0[n] = torch.from_numpy(0.1 * np.sin(0.37 * k + i)).to(torch.float32).numpy().reshape(shape)
    pol = R.RefPolicy(named0, bool(g[f"{tag}_shape"][4]))
    opt = R.RefAdam(pol.tensors(), lr=float(g[f"{tag}_hyper"][4]), eps=1e-5)
    t = lambda k: torch.from_numpy(g[f"{tag}_{k}"])
    for step in range(2):
        stats, raw, _, _ = R.ppo_update_step(pol, opt, t("obs"), t("act"), t("oldlp"), t("adv"), t("ret"), t("vold"), max_grad_norm=0.5)
        want, sel = golden_flat(g, tag, f"s{step}_g", names)
        got = flat_from_named({n: r.numpy() for n, r in zip(pol.p.keys(), raw)})[sel]
        assert float(np.linalg.norm(got - want) / np.linalg.norm(want)) < 1e-6
        ref = g[f"{tag}_s{step}_stats"]
        np.testing.assert_allclose([stats[k] for k in ("policy_loss", "value_loss", "entropy", "loss", "old_approx_kl", "approx_kl", "clipfrac",
                                                       "grad_norm")], ref, rtol=2e-5, atol=1e-7)
    want, sel = golden_flat(g, tag, "final_p", names)
    np.testing.assert_allclose(flat_from_named({n: pol.p[n].detach().numpy() for n in names})[sel], want, rtol=1e-6, atol=1e-7)
