"""Fused minibatch update vs the reference-generated golden vectors and the torch-autograd
oracle (GPU).  Tolerance: north_star's 1e-4 relative for losses and gradients."""
import os

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, kernels
from oracle import ppo_ref as R
from tests.helpers import flat_from_named, random_policy

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tc", "tc4", "simt"])
def update_impl(request):
    """Every test runs against all CUDA implementations of aur_ppo_update_grad: the tcgen05 kernel with two or four
    threads per sample and the independent SIMT fp32 kernel."""
    from aur_ppo_b200 import _lib
    L = _lib.lib()
    prev = L.aur_ppo_update_get_impl()
    assert L.aur_ppo_update_set_impl({"simt": 0, "tc": 1, "tc4": 2}[request.param]) == 0
    yield request.param
    L.aur_ppo_update_set_impl(prev)


def _flat_grads(names, grads):
    return flat_from_named({n: g for n, g in zip(names, grads)})


def _grad_close(got, want, rtol=1e-4, what=""):
    """north_star's "gradients within 1e-4 relative", read as: every entry within rtol * (|entry| + max|g|) - small entries
    are held to 1e-4 of the gradient's SCALE, not of themselves (an entry 1e6 times smaller than its neighbours carries
    their rounding).  What that leaves open is measured and bounded too: over the entries that matter (above 1e-3 of the
    scale) the largest ELEMENTWISE relative error must stay below 5e-3 (measured up to 2e-3 on entries ~1e-3 of the scale), and the relative L2 error of the whole gradient
    below 1e-4."""
    np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * float(np.abs(want).max()) + 1e-9)
    big = np.abs(want) > 1e-3 * float(np.abs(want).max())
    worst = float((np.abs(got - want)[big] / np.abs(want)[big]).max())
    l2 = float(np.linalg.norm(got.astype(np.float64) - want) / np.linalg.norm(want))
    print(f"{what} gradient: relative L2 {l2:.1e}, max elementwise relative error over |g| > 1e-3 max|g|: {worst:.1e} ({int(big.sum())} entries)")
    assert l2 < 1e-4 and worst < 5e-3, (l2, worst)         # measured: L2 <= 1e-5, elementwise <= 2.0e-3


@pytest.mark.parametrize("tag", ["disc", "disc_big", "cont", "disc_nonorm", "disc_novclip"])
def test_update_matches_reference_golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, "update.npz"))
    names = [str(n) for n in g[f"{tag}_names"]]
    named0 = {n: g[f"{tag}_p0_{n}"] for n in names}
    cont = "actor_logstd" in names
    obs, act = g[f"{tag}_obs"], g[f"{tag}_act"].astype(np.float32)
    clip, ent_c, vf_c, mgn, lr, norm_adv, clip_vloss = [float(v) for v in g[f"{tag}_hyper"]]
    desc = kernels.policy_desc(obs.shape[1], 1 if cont else 2, 64, 2, cont)
    params = torch.from_numpy(flat_from_named(named0)).cuda()
    up = kernels.Updater(desc, params)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    bufs = [dev(obs), dev(act), dev(g[f"{tag}_oldlp"]), dev(g[f"{tag}_adv"]), dev(g[f"{tag}_ret"]), dev(g[f"{tag}_vold"])]
    B = obs.shape[0]
    idx = torch.arange(B, dtype=torch.int32, device="cuda")
    for step in range(2):
        grads = up.grad(*bufs, idx, clip_coeff=clip, entropy_coeff=ent_c, value_coeff=vf_c, norm_adv=bool(norm_adv),
                        clip_vloss=bool(clip_vloss)).clone()
        stats = up.apply(lr, mgn).cpu().numpy()
        want_g = flat_from_named({n: g[f"{tag}_s{step}_g_{n}"] for n in names})
        _grad_close(grads[:up.P].cpu().numpy(), want_g, what=f"{tag} step {step}")
        want = g[f"{tag}_s{step}_stats"]    # policy, value, entropy, loss, old_kl, kl, clipfrac, gnorm
        got = [stats[0], stats[1], stats[2], stats[7], stats[3], stats[4], stats[5], stats[6]]
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=2e-6)
        want_p = flat_from_named({n: g[f"{tag}_s{step}_p_{n}"] for n in names})
        # Adam divides by sqrt(v) + eps: where |g| ~ eps a 1e-5 relative gradient error moves the step by ~1e-3 of lr
        np.testing.assert_allclose(params.cpu().numpy(), want_p, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("cont,m,B", [(False, 1000, 5000), (True, 777, 4096), (False, 256, 256), (False, 1, 64)])
def test_update_with_shuffled_gather_vs_oracle(cont, m, B):
    obs_dim, act_dim = (3, 1) if cont else (4, 2)
    pol, named = random_policy(obs_dim, act_dim, 64, 2, cont, seed=11)
    names = list(named.keys())
    desc = kernels.policy_desc(obs_dim, act_dim, 64, 2, cont)
    g = torch.Generator().manual_seed(m)
    b_obs = torch.randn(B, obs_dim, generator=g) * 0.7
    b_act = torch.randn(B, 1, generator=g) if cont else torch.randint(0, 2, (B,), generator=g).float()
    with torch.no_grad():
        _, lp0, _, v0 = pol.evaluate(b_obs, b_act)
    b_lp = lp0 + 0.25 * torch.randn(B, generator=g)             # some ratios leave the clip range
    b_adv = torch.randn(B, generator=g) * 3 + 0.5
    b_ret = torch.randn(B, generator=g)
    b_val = v0.flatten() + 0.4 * torch.randn(B, generator=g)    # some value deltas leave the clip range
    idx = torch.randperm(B, generator=g)[:m]
    opt = R.RefAdam(pol.tensors(), lr=3e-4, eps=1e-5)
    params = torch.from_numpy(flat_from_named(named)).cuda()
    up = kernels.Updater(desc, params)
    dbuf = [t.cuda().contiguous() for t in (b_obs, b_act, b_lp, b_adv, b_ret, b_val)]
    for step in range(3):
        if m == 1:
            kw = dict(norm_adv=False)      # std of one sample is NaN in the reference too
        else:
            kw = {}
        stats_ref, raw, _, _ = R.ppo_update_step(pol, opt, b_obs[idx], b_act[idx], b_lp[idx], b_adv[idx], b_ret[idx],
                                                 b_val[idx], max_grad_norm=0.5, **kw)
        grads = up.grad(*dbuf, idx.to(torch.int32).cuda(), **kw).clone()
        stats = up.apply(3e-4, 0.5).cpu().numpy()
        _grad_close(grads[:up.P].cpu().numpy(), _flat_grads(names, [r.numpy() for r in raw]))
        for i, k in enumerate(kernels.STAT_NAMES):
            np.testing.assert_allclose(stats[i], stats_ref[k], rtol=1e-4, atol=2e-6, err_msg=k)
        np.testing.assert_allclose(params.cpu().numpy(), flat_from_named({n: pol.p[n].detach().numpy() for n in names}),
                                   rtol=1e-5, atol=1e-6)


def test_identity_index_range_and_split_minibatch(update_impl):
    """idx=NULL + offset equals an explicit arange; two half-minibatch gradient buffers summed
    equal the whole (the data-parallel contract: m_total scales, partial sums add).  Besides 64 x 2, the layer-wise wide
    update (update_wide.cu) at 128 x 2 and at 256 x 3 (a middle layer): the first runs of its idx = NULL + idx_offset gather
    and of an m_total other than m_local there; they do not depend on update_impl, so they run once."""
    shapes = [(4, 2, 64, 2)] + ([(4, 2, 128, 2), (6, 3, 256, 3)] if update_impl == "tc" else [])
    for obs_dim, act_dim, hidden, layers in shapes:
        _, named = random_policy(obs_dim, act_dim, hidden, layers, False, seed=12)
        desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, False)
        g = torch.Generator().manual_seed(2)
        B = 2048
        bufs = [torch.randn(B, obs_dim, generator=g), torch.randint(0, act_dim, (B,), generator=g).float(),
                -0.7 + 0.2 * torch.randn(B, generator=g), torch.randn(B, generator=g), torch.randn(B, generator=g),
                torch.randn(B, generator=g)]
        dbuf = [t.cuda() for t in bufs]
        params = torch.from_numpy(flat_from_named(named)).cuda()
        up = kernels.Updater(desc, params)
        full = up.grad(*dbuf, torch.arange(512, 1536, dtype=torch.int32, device="cuda")).clone()
        rng = up.grad(*dbuf, None, idx_offset=512, m_local=1024).clone()
        assert torch.equal(full, rng), hidden
        # halves: moments must be the whole minibatch's, so feed them through the allreduce hook
        whole_moments = up.moments.clone()
        up.allreduce = lambda t: t.copy_(whole_moments) if t.dtype == torch.float64 else None
        a = up.grad(*dbuf, None, idx_offset=512, m_local=512, m_total=1024).clone()
        b = up.grad(*dbuf, None, idx_offset=1024, m_local=512, m_total=1024).clone()
        np.testing.assert_allclose((a + b)[:up.P].cpu().numpy(), full[:up.P].cpu().numpy(), rtol=2e-5, atol=1e-8, err_msg=str(hidden))
        np.testing.assert_allclose((a + b)[up.P:up.P + 6].cpu().numpy(), full[up.P:up.P + 6].cpu().numpy(), rtol=1e-5, err_msg=str(hidden))


def test_large_minibatch_properties():
    """Config-B sized minibatch (2,097,152 of 8,388,608 rows): too big for the autograd oracle in
    seconds, so check it through linearity: the packed sums over two disjoint halves add up to the
    whole, and a sampled sub-minibatch matches the oracle."""
    pol, named = random_policy(4, 2, 64, 2, False, seed=13)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    B, m = 8_388_608, 2_097_152
    g = torch.Generator(device="cuda").manual_seed(3)
    dbuf = [torch.randn(B, 4, generator=g, device="cuda") * 0.5, torch.randint(0, 2, (B,), generator=g, device="cuda").float(),
            -0.7 + 0.1 * torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda"),
            torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda")]
    idx = torch.randperm(B, generator=g, device="cuda")[:m].to(torch.int32)
    params = torch.from_numpy(flat_from_named(named)).cuda()
    up = kernels.Updater(desc, params)
    whole = up.grad(*dbuf, idx).clone()
    mom = up.moments.clone()
    up.allreduce = lambda t: t.copy_(mom) if t.dtype == torch.float64 else None
    h1 = up.grad(*dbuf, idx[: m // 2].contiguous(), m_total=m).clone()
    h2 = up.grad(*dbuf, idx[m // 2:].contiguous(), m_total=m).clone()
    np.testing.assert_allclose((h1 + h2)[:up.P].cpu().numpy(), whole[:up.P].cpu().numpy(), rtol=1e-4, atol=1e-7)
    sub = idx[:4096].long().cpu()
    _, stats_ref, _, _ = R.ppo_loss(pol, *[t[sub.cuda()].cpu() for t in dbuf])
    up.allreduce = None
    up.grad(*dbuf, idx[:4096].contiguous())
    st = (up.grads[up.P:up.P + 6] / 4096).cpu().numpy()
    np.testing.assert_allclose(st[:3], [stats_ref["policy_loss"], stats_ref["value_loss"], stats_ref["entropy"]], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("cont", [False, True])
def test_packed_records_give_the_same_update(cont, update_impl):
    """aur_ppo_pack_records only changes WHERE the gathered values are read from: same gradients, bit for bit."""
    obs_dim, act_dim = (3, 1) if cont else (4, 2)
    _, named = random_policy(obs_dim, act_dim, 64, 2, cont, seed=5)
    desc = kernels.policy_desc(obs_dim, act_dim, 64, 2, cont)
    B, m = 20000, 8192
    g = torch.Generator().manual_seed(77)
    bufs = [(torch.randn(B, obs_dim, generator=g) * 0.6).cuda(),
            (torch.randn(B, 1, generator=g) if cont else torch.randint(0, 2, (B,), generator=g).float()).cuda(),
            (-0.7 + 0.2 * torch.randn(B, generator=g)).cuda(), (torch.randn(B, generator=g) * 2).cuda(),
            torch.randn(B, generator=g).cuda(), torch.randn(B, generator=g).cuda()]
    idx = torch.randperm(B, generator=g)[:m].to(torch.int32).cuda()
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    rec = kernels.pack_records(*bufs)
    assert rec is not None and rec[0].shape == (B, 8)
    np.testing.assert_array_equal(rec[0][:, :obs_dim].cpu().numpy(), bufs[0].cpu().numpy())
    np.testing.assert_array_equal(rec[1][:, 4].cpu().numpy(), bufs[4].cpu().numpy())
    a, b = kernels.Updater(desc, flat.clone()), kernels.Updater(desc, flat.clone())
    for _ in range(2):
        ga = a.grad(*bufs, idx).clone(); a.apply(3e-4, 0.5)
        gb = b.grad(*bufs, idx, records=rec).clone(); b.apply(3e-4, 0.5)
        assert torch.equal(ga, gb)
    assert torch.equal(a.params, b.params)
    assert kernels.pack_records(torch.zeros(8, 6, device="cuda"), *bufs[1:]) is None   # obs_dim > 4 does not fit a record


def test_full_size_minibatch_properties():
    """BASELINE config B minibatch (2,097,152 samples of an 8,388,608-sample batch), through size-independent properties:
    (1) the tensor-core and the independent SIMT kernel agree within the 1e-4 bar, (2) gradient sums are additive over a
    split of the minibatch (checksum of checksums), (3) packed records give bit-identical results."""
    from aur_ppo_b200 import _lib
    L = _lib.lib()
    B, m = 8388608, 2097152
    _, named = random_policy(4, 2, 64, 2, False, seed=2)
    desc = kernels.policy_desc(4, 2, 64, 2, False)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    g = torch.Generator(device="cuda").manual_seed(3)
    bufs = [torch.randn(B, 4, generator=g, device="cuda") * 0.5, torch.randint(0, 2, (B,), generator=g, device="cuda").float(),
            -0.7 + 0.1 * torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda"),
            torch.randn(B, generator=g, device="cuda"), torch.randn(B, generator=g, device="cuda")]
    idx = kernels.shuffle_indices(B, seed=5, stream_id=0)[:m].contiguous()
    prev = L.aur_ppo_update_get_impl()
    try:
        out = {}
        for name, impl in (("tc", 1), ("simt", 0)):
            L.aur_ppo_update_set_impl(impl)
            up = kernels.Updater(desc, flat.clone())
            out[name] = up.grad(*bufs, idx).clone()
            if name == "tc":
                rec = kernels.pack_records(*bufs)
                assert torch.equal(up.grad(*bufs, idx, records=rec), out["tc"])
                # additivity (advantage normalisation off so that the halves share nothing but the weights)
                whole = up.grad(*bufs, idx, norm_adv=False).clone()
                a = up.grad(*bufs, idx[: m // 2].contiguous(), m_total=m, norm_adv=False).clone()
                b = up.grad(*bufs, idx[m // 2:].contiguous(), m_total=m, norm_adv=False).clone()
                scale = whole[:up.P].abs().max().item()
                np.testing.assert_allclose((a + b).cpu().numpy(), whole.cpu().numpy(), rtol=2e-5, atol=2e-6 * scale + 1e-9)
        P = policy_p = kernels.policy_param_count(desc)
        gt, gs = out["tc"][:P].cpu().numpy(), out["simt"][:P].cpu().numpy()
        np.testing.assert_allclose(gt, gs, rtol=1e-4, atol=1e-4 * float(np.abs(gs).max()))
        l2 = float(np.linalg.norm(gt.astype(np.float64) - gs) / np.linalg.norm(gs))
        print(f"2.1 M-sample minibatch, tcgen05 vs SIMT fp32 kernel: relative L2 {l2:.1e}")
        assert l2 < 1e-4          # includes the tensor core's truncating accumulator over 110 tiles per CTA
        np.testing.assert_allclose(out["tc"][P:P + 6].cpu().numpy(), out["simt"][P:P + 6].cpu().numpy(), rtol=1e-4)
    finally:
        L.aur_ppo_update_set_impl(prev)


@pytest.mark.parametrize("cont", [False, True])
def test_moments_of_all_minibatches_in_one_launch(cont):
    """aur_ppo_adv_moments_multi (what ppo.run_update uses: the moments of every minibatch of an iteration right after the
    shuffles) against the per-minibatch kernel and against float64 torch; the update that reads entry j is the update that
    computed its own moments."""
    from tests.helpers import flat_from_named, random_policy
    obs_dim, act_dim = (3, 1) if cont else (4, 2)
    _, named = random_policy(obs_dim, act_dim, 64, 2, cont, seed=9)
    desc = kernels.policy_desc(obs_dim, act_dim, 64, 2, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    B, n_mb, m = 40000, 7, 5000
    g = torch.Generator().manual_seed(3)
    obs = (torch.randn(B, obs_dim, generator=g) * 0.5).cuda()
    act = (torch.randn(B, act_dim, generator=g) if cont else torch.randint(0, act_dim, (B,), generator=g).float()).cuda()
    oldlp = (-0.7 + 0.2 * torch.randn(B, generator=g)).cuda(); adv = (torch.randn(B, generator=g) * 3 + 2).cuda()
    ret = torch.randn(B, generator=g).cuda(); vold = torch.randn(B, generator=g).cuda()
    idx_all = torch.stack([torch.randperm(B, generator=g)[:m] for _ in range(n_mb)]).to(torch.int32).cuda().contiguous()
    bufs = (obs, act, oldlp, adv, ret, vold)
    up = kernels.Updater(desc, flat.clone())
    up.prepare_moments(adv, idx_all)
    got = up.moments_all.cpu()
    for j in range(n_mb):
        a = adv[idx_all[j].long()].double().cpu()
        np.testing.assert_allclose(got[j].numpy(), [float(a.sum()), float((a * a).sum()), m], rtol=1e-13)
    ref = kernels.Updater(desc, flat.clone())
    for j in (0, 3, 6):
        g1 = up.grad(*bufs, idx_all[j], moments_index=j).clone()
        g2 = ref.grad(*bufs, idx_all[j]).clone()
        assert torch.equal(g1, g2) or float((g1 - g2).abs().max()) <= 1e-7 * float(g2.abs().max())
    with pytest.raises(_lib.AurError):
        up.grad(*bufs, idx_all[0], moments_index=n_mb)
