"""Out-of-bounds WRITE detection without compute-sanitizer (the tool is closed on this GPU pool: profiles/r2_sanitizer.md).
Every output buffer of a kernel family is carved out of a larger allocation whose surroundings hold a sentinel pattern;
after the launch the sentinels must be intact and the payload fully written (no sentinel left inside where the kernel is
specified to write everything).  Small and ragged shapes on purpose: that is where tile tails go wrong."""
import ctypes

import numpy as np
import pytest
import torch

from aur_ppo_b200 import _lib, envs as denv, kernels
from tests.helpers import flat_from_named, random_policy

pytestmark = pytest.mark.gpu
GUARD = 4096          # bytes on each side
SENT = 0xA5


class Guarded:
    def __init__(self, shape, dtype, fill_sentinel=True):
        n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        pad = (-n) % 256
        self.raw = torch.full((GUARD + n + pad + GUARD,), SENT, dtype=torch.uint8, device="cuda")
        self.n = n
        self.t = self.raw[GUARD:GUARD + n].view(dtype).view(*shape)
        if not fill_sentinel:
            self.t.zero_()

    def check(self, name, fully_written=False):
        front, back = self.raw[:GUARD], self.raw[GUARD + self.n:]
        assert bool((front == SENT).all()), f"{name}: bytes written BEFORE the buffer"
        assert bool((back == SENT).all()), f"{name}: bytes written AFTER the buffer"
        if fully_written and self.t.element_size() == 4:
            left = (self.t.contiguous().view(torch.int32) == np.int32(np.uint32(0xA5A5A5A5).view(np.int32))).sum().item()
            assert left == 0, f"{name}: {left} elements never written"


@pytest.mark.parametrize("T,N", [(16, 256), (7, 250), (128, 1000), (33, 4099)])
def test_gae_writes_stay_inside(T, N):
    g = torch.Generator(device="cuda").manual_seed(T)
    rew, val = torch.rand(T, N, generator=g, device="cuda"), torch.randn(T, N, generator=g, device="cuda")
    term = (torch.rand(T, N, generator=g, device="cuda") < 0.05).float()
    nv, nd = torch.randn(N, generator=g, device="cuda"), torch.zeros(N, device="cuda")
    ret, adv = Guarded((T, N), torch.float32), Guarded((T, N), torch.float32)
    kernels.gae(rew, val, term, nv, nd, 0.99, 0.95, True, out=(ret.t, adv.t))
    torch.cuda.synchronize()
    ret.check("returns", True); adv.check("advantages", True)


# gym_id, continuous, act_dim, N, T, hidden.  The wide rows are the first guarded runs of the layer-wise actor with the
# external-actor env step (CartPole 256 x 2) and of rollout_tc_kernel<ENV, 128> + critic_values_tc_kernel<128> (Pendulum and
# MountainCar 128 x 2); under impl 0 they run the runtime-width SIMT kernel
ROLLOUT_GUARDS = {"CartPole-v1-False-2-130-9": ("CartPole-v1", False, 2, 130, 9, 64),
                  "CartPole-v1-False-2-9600-5": ("CartPole-v1", False, 2, 9600, 5, 64),
                  "Pendulum-v1-True-1-257-7": ("Pendulum-v1", True, 1, 257, 7, 64),
                  "Acrobot-v1-False-3-100-6": ("Acrobot-v1", False, 3, 100, 6, 64),
                  "cartpole-256x2": ("CartPole-v1", False, 2, 130, 5, 256),
                  "pendulum-128x2": ("Pendulum-v1", True, 1, 257, 7, 128),
                  "mountaincar-128x2": ("MountainCar-v0", False, 3, 300, 6, 128)}


@pytest.mark.parametrize("case", list(ROLLOUT_GUARDS))
def test_rollout_writes_stay_inside(case):
    gym_id, cont, act, N, T, hidden = ROLLOUT_GUARDS[case]
    env = denv.DeviceVecEnv(gym_id, N, wrappers=cont)
    env.reset(list(range(N)))
    desc = kernels.policy_desc(env.obs_dim, act, hidden, 2, cont)
    P = kernels.policy_param_count(desc)
    flat = (torch.rand(P, device="cuda") - 0.5) * 0.2
    buf = kernels.RolloutBuffers(T, N, env.obs_dim, (act,) if cont else (), "cuda")
    G = dict(states=Guarded((T, N, env.obs_dim), torch.float32), actions=Guarded((T, N, act) if cont else (T, N), torch.float32),
             log_probs=Guarded((T, N), torch.float32), rewards=Guarded((T, N), torch.float32),
             terminals=Guarded((T, N), torch.float32), values=Guarded((T, N), torch.float32), next_value=Guarded((N,), torch.float32))
    for k, gd in G.items():
        setattr(buf, k, gd.t)
    for impl in (0, 1):
        _lib.lib().aur_rollout_set_impl(impl)
        kernels.rollout(env, desc, flat, buf, seed=1, step0=0)
        torch.cuda.synchronize()
        for k, gd in G.items():
            gd.check(f"{gym_id} impl {impl} {k}", True)
    _lib.lib().aur_rollout_set_impl(1)


# continuous, m, hidden, layers.  The wide rows are the first guarded runs of the layer-wise update (update_wide.cu): m = 65
# ends one sample into the second 64-sample TMA box, m = 1025 one sample into the second 1,024-sample partial row; 256 x 3 adds
# the middle layer.  They take that path whatever the impl switch says, so they run once.
UPDATE_GUARDS = {"False-1000": (False, 1000, 64, 2), "True-129": (True, 129, 64, 2), "False-4097": (False, 4097, 64, 2)}
UPDATE_GUARDS.update({f"{'cont' if c else 'disc'}{h}x{nl}-{m}": (c, m, h, nl) for h, nl in ((128, 2), (256, 3))
                      for c in (False, True) for m in (65, 1025)})


@pytest.mark.parametrize("impl", [0, 1, 2, 3])
@pytest.mark.parametrize("case", list(UPDATE_GUARDS))
def test_update_writes_stay_inside(impl, case):
    cont, m, hidden, layers = UPDATE_GUARDS[case]
    if hidden != 64 and impl != 1:
        pytest.skip("one kernel behind this shape")
    obs_dim, act_dim = (3, 1) if cont else (4, 2)
    _, named = random_policy(obs_dim, act_dim, hidden, layers, cont, seed=4)
    desc = kernels.policy_desc(obs_dim, act_dim, hidden, layers, cont)
    flat = torch.from_numpy(flat_from_named(named)).cuda()
    B = 5000
    g = torch.Generator().manual_seed(2)
    obs = (torch.randn(B, obs_dim, generator=g) * 0.5).cuda()
    act = (torch.randn(B, act_dim, generator=g) if cont else torch.randint(0, act_dim, (B,), generator=g).float()).cuda()
    oldlp = (-0.7 + 0.2 * torch.randn(B, generator=g)).cuda(); adv = torch.randn(B, generator=g).cuda()
    ret = torch.randn(B, generator=g).cuda(); vold = torch.randn(B, generator=g).cuda()
    L = _lib.lib()
    L.aur_ppo_update_set_impl(impl)
    try:
        up = kernels.Updater(desc, flat.clone())
        P = up.P
        gp, gg = Guarded((P,), torch.float32), Guarded((P + kernels.NUM_STATS,), torch.float32)
        gm1, gm2 = Guarded((P,), torch.float32, False), Guarded((P,), torch.float32, False)
        gws, gst = Guarded(tuple(up.workspace.shape), torch.float32, False), Guarded((kernels.NUM_STATS,), torch.float32)
        gidx = Guarded((m,), torch.int32)
        gp.t.copy_(flat)
        up.params, up.grads, up.exp_avg, up.exp_avg_sq, up.workspace, up.stats = gp.t, gg.t, gm1.t, gm2.t, gws.t, gst.t
        kernels.shuffle_indices(m, seed=1, stream_id=0, out=gidx.t)
        gidx.check("shuffle", True)
        idx = (gidx.t % B).contiguous()
        up.grad(obs, act, oldlp, adv, ret, vold, idx)
        up.apply(2.5e-4, 0.5)
        torch.cuda.synchronize()
        gg.check("grads", True); gst.check("stats", True); gp.check("params"); gm1.check("exp_avg"); gm2.check("exp_avg_sq")
        gws.check("workspace")
        assert torch.isfinite(gp.t).all() and torch.isfinite(gg.t).all()
    finally:
        L.aur_ppo_update_set_impl(1)


@pytest.mark.parametrize("P", [1, 2])
@pytest.mark.parametrize("B,H,Cin,Cout,pool", [(3, 8, 64, 64, True), (1, 16, 64, 200, False), (5, 8, 128, 256, True)])
def test_conv_and_wgrad_writes_stay_inside(B, H, Cin, Cout, pool, P):
    g = torch.Generator().manual_seed(B + H)
    Hb = H + 2
    Hn = H // 2 if pool else H
    with kernels.tc_precision(P):
        x = kernels.split_planes(torch.randn(B, Hb, Hb, Cin, generator=g).cuda(), P)
        w = kernels.split_planes((torch.randn(Cout, 9, Cin, generator=g) * 0.05).cuda(), P)
        bias = torch.zeros(Cout, device="cuda")
        out = Guarded((P, B, Hn + 2, Hn + 2, Cout), torch.bfloat16, False)
        arg = Guarded((B, Hn, Hn, Cout), torch.uint8) if pool else None
        kernels.conv3x3_bf16(x if P > 1 else x[0], w if P > 1 else w[0], bias, 2 if pool else 1, out.t if P > 1 else out.t[0], 1,
                             arg.t if pool else None)
        dy = kernels.split_planes((torch.randn(B, Hb, Hb, Cout, generator=g) * 0.1).cuda(), P)
        dw = Guarded((Cout, 9, Cin), torch.float32, False)
        rc = _lib.lib().aur_wgrad3x3_bf16(Cout, Cin, B * Hb * Hb, dy.data_ptr(), x.data_ptr(), -(Hb + 1), Hb, dw.t.data_ptr(), 0,
                                          kernels._stream())
        _lib.check(rc, "aur_wgrad3x3_bf16")
        a, b = kernels.split_planes(torch.randn(70, 72, generator=g).cuda(), P), kernels.split_planes(torch.randn(50, 72, generator=g).cuda(), P)
        c = Guarded((70, 50), torch.float32)
        rc = _lib.lib().aur_tc_gemm_bf16(70, 50, 72, a.data_ptr(), b.data_ptr(), c.t.data_ptr(), kernels._stream())
        _lib.check(rc, "aur_tc_gemm_bf16")
    torch.cuda.synchronize()
    out.check("conv out")
    dw.check("wgrad")
    c.check("gemm", True)
    if pool:
        arg.check("pool arg", False)
        assert int(arg.t.max()) <= 3
    assert float(out.t[:, :, 0].float().abs().max()) == 0 and float(out.t[:, :, :, 0].float().abs().max()) == 0      # halo rows / columns untouched
