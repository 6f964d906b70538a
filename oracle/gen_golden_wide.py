"""Golden vectors for the WIDE policy shapes (`--hidden_dim 128`, src/run_ppo.py:36) from the REFERENCE'S OWN CODE: the minibatch
step of ppo.py:220-269 around the reference's actor_critic + torch.optim.Adam(eps=1e-5), two consecutive steps, exactly as
oracle/gen_golden.py::update_cases does for the 64-wide headline shape.  Run in the build container only (/root/reference does
not exist on the GPU box):  python oracle/gen_golden_wide.py  ->  tests/golden/update_wide.npz

TEST INFRASTRUCTURE ONLY.  To keep the fixture small the initial parameters are NOT stored: they are gen_golden.fill_params'
closed form (i-th parameter tensor <- 0.1 sin(0.37 k + i)), which the test re-creates from the stored parameter names / shapes;
stored are the raw gradients of both steps, the statistics and the parameters after the second step.  The first step's gradients
are stored whole; of every hidden x hidden matrix, the second step's gradients and the final parameters keep a fixed sample of
their entries (sample_large), which keeps the file under 1 MB."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gen_golden import OUT, fill_params, import_reference  # noqa: E402

CASES = [  # tag, state_dim, action_dim, continuous, hidden, layers, minibatch
    ("disc128", 4, 2, False, 128, 2, 1300),        # two partial rows of the layer-wise path, the second ragged
    ("cont128", 3, (1,), True, 128, 2, 700),
    ("disc128x3", 4, 2, False, 128, 3, 500),
]
SAMPLED = 2048      # entries kept of a sampled matrix


def sample_large(out):
    """For every parameter of more than 4 * SAMPLED entries, keep SAMPLED of them (`{tag}_sample_<name>`: sorted flat indices,
    seed 0) in the second step's gradients and in the final parameters."""
    rng = np.random.default_rng(0)
    for tag, *_ in CASES:
        for n in out[f"{tag}_names"]:
            size = int(np.prod(out[f"{tag}_pshape_{n}"]))
            if size <= 4 * SAMPLED:
                continue
            idx = np.sort(rng.choice(size, SAMPLED, replace=False)).astype(np.uint16 if size <= 1 << 16 else np.int64)
            out[f"{tag}_sample_{n}"] = idx
            for key in (f"{tag}_s1_g_{n}", f"{tag}_final_p_{n}"):
                out[key] = out[key].reshape(-1)[idx]
    return out


def rollout_cases(ref_ac):
    """Log-probs / values of the reference's actor_critic.evaluate (models/actor_critic.py:31-51) on the observations a seeded
    rollout visits: the env trajectory under a fixed action tape is deterministic (the checker of oracle/envs.py replays it bit
    for bit), so the GPU rollout kernels at 128 / 256 units can be compared with the REFERENCE's numbers, not a restatement's."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle import envs as E
    out = {}
    for tag, kind, sd, ad, cont, hidden in [("cart128", E.CARTPOLE, 4, 2, False, 128), ("pend128", E.PENDULUM, 3, (1,), True, 128),
                                            ("cart256", E.CARTPOLE, 4, 2, False, 256)]:
        N, T = 96, 6
        m = ref_ac.actor_critic(sd, ad, hidden, 2, 0.0, cont)
        fill_params(m)
        rng = np.random.default_rng(5)
        actions = rng.normal(size=(T, N, 1)).astype(np.float32) if cont else rng.integers(0, 2, (T, N))
        cv = E.CVecEnv(kind, N, wrappers=cont, trig=E.TRIG_CR)
        cur, _ = cv.reset(list(range(N)))
        obs = np.zeros((T, N, sd), np.float32)
        for t in range(T):
            obs[t] = cur
            cur = cv.step(actions[t])[0]
        ot = torch.from_numpy(obs.reshape(-1, sd))
        at = torch.from_numpy(actions.reshape(-1, 1)) if cont else torch.from_numpy(actions.reshape(-1)).long()
        with torch.no_grad():
            _, lp, ent, v = m.evaluate(ot, at)
            nv = m.value(torch.from_numpy(cur))
        out[f"{tag}_names"] = np.array([n for n, _ in m.named_parameters()])
        for n, p in m.named_parameters():
            out[f"{tag}_pshape_{n}"] = np.array(p.shape)
        out[f"{tag}_shape"] = np.array([sd, int(np.prod(ad)) if cont else ad, hidden, 2, int(cont), N, T])
        for k, v_ in dict(actions=actions.astype(np.float32), obs=obs, logp=lp.numpy().reshape(T, N), value=v.numpy().reshape(T, N),
                          next_value=nv.numpy().reshape(N)).items():
            out[f"{tag}_{k}"] = v_
    return out


def main():
    _, ref_ac, _ = import_reference()
    np.savez_compressed(os.path.join(OUT, "rollout_wide.npz"), **rollout_cases(ref_ac))
    out = {}
    for tag, sd, ad, cont, hidden, nl, B in CASES:
        m = ref_ac.actor_critic(sd, ad, hidden, nl, 0.0, cont)
        fill_params(m)
        clip_coeff, ent_c, vf_c, mgn, lr = 0.2, 0.01, 0.5, 0.5, 2.5e-4
        opt = torch.optim.Adam(m.parameters(), lr=lr, eps=1e-5)
        g = torch.Generator().manual_seed(11)
        obs = torch.randn(B, sd, generator=g) * 0.5
        if cont:
            act = torch.randn(B, 1, generator=g)
            oldlp = -0.9 - 0.5 * act.flatten() ** 2 + 0.1 * torch.randn(B, generator=g)
        else:
            act = torch.randint(0, 2, (B,), generator=g).float()
            oldlp = -0.69 + 0.3 * torch.randn(B, generator=g)
        adv = torch.randn(B, generator=g) * 2
        ret = torch.randn(B, generator=g)
        vold = ret + 0.3 * torch.randn(B, generator=g)
        names = [n for n, _ in m.named_parameters()]
        out[f"{tag}_names"] = np.array(names)
        out[f"{tag}_shape"] = np.array([sd, int(np.prod(ad)) if cont else ad, hidden, nl, int(cont)])
        for n, p in m.named_parameters():
            out[f"{tag}_pshape_{n}"] = np.array(p.shape)
        for k, v_ in dict(obs=obs, act=act, oldlp=oldlp, adv=adv, ret=ret, vold=vold).items():
            out[f"{tag}_{k}"] = v_.numpy()
        out[f"{tag}_hyper"] = np.array([clip_coeff, ent_c, vf_c, mgn, lr])
        for step in range(2):
            _, newlogprob, entropy, newvalue = m.evaluate(obs, act)
            log_ratio = newlogprob - oldlp
            ratio = log_ratio.exp()
            with torch.no_grad():
                old_approx_kl = (-log_ratio).mean()
                approx_kl = ((ratio - 1) - log_ratio).mean()
                clipfrac = ((ratio - 1.0).abs() > clip_coeff).float().mean()
            mb_adv = (adv - adv.mean()) / (adv.std() + 1e-8)                      # ppo.py:239
            loss_one = -mb_adv * ratio
            loss_two = -mb_adv * torch.clamp(ratio, 1 - clip_coeff, 1 + clip_coeff)
            policy_loss = torch.max(loss_one, loss_two).mean()
            newvalue = newvalue.view(-1)
            v_loss_unclipped = (newvalue - ret) ** 2
            v_clipped = vold + torch.clamp(newvalue - vold, -clip_coeff, clip_coeff)
            v_loss_clipped = (v_clipped - ret) ** 2
            value_loss = 0.5 * torch.max(v_loss_unclipped, v_loss_clipped).mean()
            entropy_loss = entropy.mean()
            loss = policy_loss - ent_c * entropy_loss + value_loss * vf_c
            opt.zero_grad()
            loss.backward()
            for n, p in m.named_parameters():
                out[f"{tag}_s{step}_g_{n}"] = p.grad.detach().numpy().copy()
            gnorm = torch.nn.utils.clip_grad_norm_(m.parameters(), mgn)
            opt.step()
            out[f"{tag}_s{step}_stats"] = np.array([policy_loss.item(), value_loss.item(), entropy_loss.item(), loss.item(),
                                                    old_approx_kl.item(), approx_kl.item(), clipfrac.item(), gnorm.item()])
        for n, p in m.named_parameters():
            out[f"{tag}_final_p_{n}"] = p.detach().numpy().copy()
    path = os.path.join(OUT, "update_wide.npz")
    np.savez_compressed(path, **sample_large(out))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
