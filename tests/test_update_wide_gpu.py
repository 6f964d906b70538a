"""The layer-wise tensor-core update for wide policies (csrc/update_wide.cu: `--hidden_dim` 128 / 256, src/run_ppo.py:36)
against the torch-autograd restatement of src/ppo.py:220-269 (oracle/ppo_ref.py) and against the shape-generic SIMT kernel.
Tolerance: north_star's 1e-4 relative for losses and gradients."""
import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, kernels
from oracle import ppo_ref as R
from tests.helpers import flat_from_named, golden_flat, random_policy

pytestmark = pytest.mark.gpu


def _rel_l2(got, want):
    return float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-30))


def _setup(obs_dim, act_dim, hidden, layers, cont, m, B, seed):
    pol, named = random_policy(obs_dim, act_dim, hidden, layers, cont, seed=seed)
    g = torch.Generator().manual_seed(m)
    b_obs = torch.randn(B, obs_dim, generator=g) * 0.7
    b_act = torch.randn(B, act_dim, generator=g) if cont else torch.randint(0, act_dim, (B,), generator=g).float()
    with torch.no_grad():
        _, lp0, _, v0 = pol.evaluate(b_obs, b_act)
    b_lp = lp0 + 0.25 * torch.randn(B, generator=g)
    b_adv = torch.randn(B, generator=g) * 3 + 0.5
    b_ret = torch.randn(B, generator=g)
    b_val = v0.flatten() + 0.4 * torch.randn(B, generator=g)
    idx = torch.randperm(B, generator=g)[:m]
    return pol, named, (b_obs, b_act, b_lp, b_adv, b_ret, b_val), idx


SHAPES = [  # obs_dim, act_dim, hidden, layers, continuous, m, B
    (4, 2, 128, 2, False, 1000, 5000),          # one partial row, ragged
    (4, 2, 128, 2, False, 5000, 8192),          # five rows, the last one ragged and not a multiple of the 64-sample K block
    (3, 1, 128, 2, True, 4096, 4096),           # Pendulum-sized, Normal head + log-std gradient
    (4, 2, 256, 2, False, 3001, 4096),
    (6, 3, 128, 3, False, 2500, 4096),          # a middle layer (wide_act_kernel, delta ping-pong), Acrobot widths
    (8, 4, 256, 4, True, 1500, 2048),
    (4, 2, 128, 2, False, 65, 64 * 3),           # one K block and one sample
]


@pytest.mark.parametrize("obs_dim,act_dim,hidden,layers,cont,m,B", SHAPES)
def test_wide_update_vs_oracle(obs_dim, act_dim, hidden, layers, cont, m, B):
    L = _lib.lib()
    assert L.aur_ppo_update_get_wide() == 1
    pol, named, bufs, idx = _setup(obs_dim, act_dim, hidden, layers, cont, m, B, seed=hidden + layers)
    names = list(named.keys())
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, cont)
    opt = R.RefAdam(pol.tensors(), lr=3e-4, eps=1e-5)
    params = torch.from_numpy(flat_from_named(named)).cuda()
    up = kernels.Updater(desc, params)
    dbuf = [t.cuda().contiguous() for t in bufs]
    didx = idx.to(torch.int32).cuda()
    for step in range(2):
        stats_ref, raw, _, _ = R.ppo_update_step(pol, opt, *[b[idx] for b in bufs], max_grad_norm=0.5)
        L.aur_launch_count_reset()
        grads = up.grad(*dbuf, didx).clone()
        assert L.aur_launch_count() >= 2 * (5 + 3 * (layers - 2)) + 1      # the layer-wise path ran, not the fused generic kernel
        again = up.grad(*dbuf, didx).clone()
        assert torch.equal(grads, again)                                   # fixed accumulation order: bit-reproducible
        assert L.aur_ppo_update_set_wide(0) == 0
        try:
            simt = up.grad(*dbuf, didx).clone()
        finally:
            L.aur_ppo_update_set_wide(1)
        up.grad(*dbuf, didx)
        stats = up.apply(3e-4, 0.5).cpu().numpy()
        want = flat_from_named({n: r.numpy() for n, r in zip(names, raw)})
        got = grads[:up.P].cpu().numpy()
        print(f"H={hidden} L={layers} m={m} step {step}: rel L2 vs oracle {_rel_l2(got, want):.2e}, "
              f"vs the SIMT kernel {_rel_l2(got, simt[:up.P].cpu().numpy()):.2e}")
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * float(np.abs(want).max()) + 1e-9)
        assert _rel_l2(got, want) < 1e-4
        for i, k in enumerate(kernels.STAT_NAMES):
            np.testing.assert_allclose(stats[i], stats_ref[k], rtol=1e-4, atol=2e-6, err_msg=k)
        np.testing.assert_allclose(params.cpu().numpy(), flat_from_named({n: pol.p[n].detach().numpy() for n in names}),
                                   rtol=1e-5, atol=1e-6)


def test_wide_update_sub_batches_accumulate():
    """A minibatch larger than one 262,144-sample sub-batch: the second sub-batch adds into the first one's partial rows."""
    obs_dim, act_dim, hidden, layers, cont = 4, 2, 128, 2, False
    m = 262144 + 70001
    pol, named, bufs, idx = _setup(obs_dim, act_dim, hidden, layers, cont, m, m, seed=5)
    names = list(named.keys())
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, cont)
    opt = R.RefAdam(pol.tensors(), lr=3e-4, eps=1e-5)
    params = torch.from_numpy(flat_from_named(named)).cuda()
    up = kernels.Updater(desc, params)
    dbuf = [t.cuda().contiguous() for t in bufs]
    didx = idx.to(torch.int32).cuda()
    stats_ref, raw, _, _ = R.ppo_update_step(pol, opt, *[b[idx] for b in bufs], max_grad_norm=0.5)
    grads = up.grad(*dbuf, didx).clone()
    stats = up.apply(3e-4, 0.5).cpu().numpy()
    want = flat_from_named({n: r.numpy() for n, r in zip(names, raw)})
    got = grads[:up.P].cpu().numpy()
    print(f"m={m}: rel L2 vs oracle {_rel_l2(got, want):.2e}")
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * float(np.abs(want).max()) + 1e-9)
    for i, k in enumerate(kernels.STAT_NAMES):
        np.testing.assert_allclose(stats[i], stats_ref[k], rtol=1e-4, atol=2e-6, err_msg=k)


@pytest.mark.parametrize("tag", ["disc128", "cont128", "disc128x3"])
def test_wide_update_matches_reference_golden(golden_dir, tag):
    """tests/golden/update_wide.npz: two minibatch steps of ppo.py:220-269 computed by the REFERENCE'S OWN actor_critic +
    torch.optim.Adam at 128 hidden units (oracle/gen_golden_wide.py, run where /root/reference exists).  The initial parameters
    are the generator's closed form, re-created here from the stored names and shapes."""
    import os
    g = np.load(os.path.join(golden_dir, "update_wide.npz"))
    names = [str(n) for n in g[f"{tag}_names"]]
    obs_dim, act_dim, hidden, layers, cont = [int(v) for v in g[f"{tag}_shape"]]
    named0 = {}
    for i, n in enumerate(names):
        shape = tuple(int(v) for v in g[f"{tag}_pshape_{n}"])
        k = np.arange(int(np.prod(shape)), dtype=np.float64)
        named0[n] = torch.from_numpy(0.1 * np.sin(0.37 * k + i)).to(torch.float32).numpy().reshape(shape)   # gen_golden.fill_params
    clip, ent_c, vf_c, mgn, lr = [float(v) for v in g[f"{tag}_hyper"]]
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, bool(cont))
    params = torch.from_numpy(flat_from_named(named0)).cuda()
    up = kernels.Updater(desc, params)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    bufs = [dev(g[f"{tag}_obs"]), dev(g[f"{tag}_act"].astype(np.float32)), dev(g[f"{tag}_oldlp"]), dev(g[f"{tag}_adv"]),
            dev(g[f"{tag}_ret"]), dev(g[f"{tag}_vold"])]
    idx = torch.arange(bufs[0].shape[0], dtype=torch.int32, device="cuda")
    L = _lib.lib()
    for step in range(2):
        L.aur_launch_count_reset()
        grads = up.grad(*bufs, idx, clip_coeff=clip, entropy_coeff=ent_c, value_coeff=vf_c, norm_adv=True, clip_vloss=True).clone()
        assert L.aur_launch_count() >= 12                               # the layer-wise path, not the fused generic kernel
        stats = up.apply(lr, mgn).cpu().numpy()
        want, sel = golden_flat(g, tag, f"s{step}_g", names)
        got = grads[:up.P].cpu().numpy()[sel]
        print(f"{tag} step {step}: rel L2 vs the reference's gradients {_rel_l2(got, want):.2e}")
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * float(np.abs(want).max()) + 1e-9)
        assert _rel_l2(got, want) < 1e-4
        ref = g[f"{tag}_s{step}_stats"]
        np.testing.assert_allclose([stats[0], stats[1], stats[2], stats[7], stats[3], stats[4], stats[5], stats[6]], ref, rtol=1e-4, atol=2e-6)
    want, sel = golden_flat(g, tag, "final_p", names)
    np.testing.assert_allclose(params.cpu().numpy()[sel], want, rtol=1e-5, atol=1e-6)
