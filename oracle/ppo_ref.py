"""CPU restatement of the reference's PPO arithmetic -- TEST INFRASTRUCTURE ONLY.

Imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs; the product path never touches it.

Pinned: every function here is checked against tests/golden/*.npz, which
oracle/gen_golden.py produced by running the reference's own code
(tests/test_oracle_ppo.py).  Floating point work uses torch fp32 on the CPU,
the library the reference itself computes with; RefPolicy(dtype=torch.float64)
runs the same update in float64.

  gae / normal_advantage   ppo.py:125-142 / ppo.py:145-157
  MLP forward              nets/nets.py:19-53 (Linear-Tanh stacks)
  evaluate / value         models/actor_critic.py:31-51
  Categorical / Normal     torch.distributions as used at actor_critic.py:39-50
  squashed_sample          nets/nets.py:90-105 (PPOGaussianPolicyBase.sample)
  ppo_update_step          ppo.py:220-269 (+ clip_grad_norm_ + Adam(eps=1e-5))
  explained_variance       ppo.py:277-279
  lr_anneal                ppo.py:195-198
  philox4x32_10 / sampling the device sampler's counter-based stream, restated
                           so sampled rollouts can be replayed on the CPU; the
                           vectorised forms and normal4_f64 / categorical_icdf
                           restate every draw in float64
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch


# --------------------------------------------------------------------------- GAE
def gae(rewards, values, terminals, next_value, next_done, gamma: float, gae_lambda: float):
    """ppo.py:125-142.  All tensors fp32; sequential in t, same op order."""
    T = rewards.shape[0]
    advantages = torch.zeros_like(rewards)
    lastgaelam = 0
    for t in reversed(range(T)):
        if t == T - 1:
            nextnonterminal = 1.0 - next_done
            nextvalues = next_value
        else:
            nextnonterminal = 1.0 - terminals[t + 1]
            nextvalues = values[t + 1]
        delta = rewards[t] + gamma * nextvalues * nextnonterminal - values[t]
        advantages[t] = lastgaelam = delta + gamma * gae_lambda * nextnonterminal * lastgaelam
    returns = advantages + values
    return returns, advantages


def normal_advantage(rewards, values, terminals, next_value, next_done, gamma: float):
    """ppo.py:145-157."""
    T = rewards.shape[0]
    returns = torch.zeros_like(rewards)
    for t in reversed(range(T)):
        if t == T - 1:
            nextnonterminal = 1.0 - next_done
            next_return = next_value
        else:
            nextnonterminal = 1.0 - terminals[t + 1]
            next_return = returns[t + 1]
        returns[t] = rewards[t] + gamma * nextnonterminal * next_return
    advantages = returns - values
    return returns, advantages


# ------------------------------------------------------------------------- model
class RefPolicy:
    """Parameter container in the reference's naming: actor.net.{0,2,..}.{weight,bias},
    critic.net.{...}, optional actor_logstd [1,A] (models/actor_critic.py:8-26).
    dtype: float32 is the reference's own arithmetic; float64 gives the high-precision value that the fp32 kernels and the
    fp32 restatement are both measured against (ppo_loss, clip_grad_norm and RefAdam follow the parameters' dtype)."""

    def __init__(self, params: Dict[str, torch.Tensor], continuous: bool, dtype: torch.dtype = torch.float32):
        self.p = {k: (v if isinstance(v, torch.Tensor) else torch.from_numpy(np.asarray(v))).clone().to(dtype)
                  for k, v in params.items()}
        self.continuous = continuous

    def tensors(self) -> List[torch.Tensor]:
        return list(self.p.values())

    def requires_grad_(self, flag=True):
        for v in self.p.values():
            v.requires_grad_(flag)
        return self

    def _mlp(self, prefix: str, x):
        idx = sorted({int(k.split(".")[2]) for k in self.p if k.startswith(prefix + ".net.")})
        for j, i in enumerate(idx):
            x = torch.nn.functional.linear(x, self.p[f"{prefix}.net.{i}.weight"], self.p[f"{prefix}.net.{i}.bias"])
            if j != len(idx) - 1:
                x = torch.tanh(x)
        return x

    def value(self, state):
        return self._mlp("critic", state).flatten()

    def evaluate(self, state, action=None, generator=None):
        head = self._mlp("actor", state)
        if self.continuous:
            logstd = self.p["actor_logstd"].expand_as(head)
            std = torch.exp(logstd)
            if action is None:
                action = head + std * torch.randn(head.shape, generator=generator, dtype=head.dtype)
                action = action.detach()
            var = std ** 2
            log_scale = std.log()      # torch Normal: log(exp(logstd)), not logstd itself
            log_prob = (-((action - head) ** 2) / (2 * var) - log_scale - math.log(math.sqrt(2 * math.pi))).sum(1)
            entropy = (0.5 + 0.5 * math.log(2 * math.pi) + log_scale).sum(1)
        else:
            logits = head - head.logsumexp(dim=-1, keepdim=True)
            probs = torch.softmax(logits, dim=-1)
            if action is None:
                action = torch.multinomial(probs, 1, generator=generator).squeeze(-1)
            log_prob = logits.gather(-1, action.long().unsqueeze(-1)).squeeze(-1)
            min_real = torch.finfo(logits.dtype).min
            entropy = -(torch.clamp(logits, min=min_real) * probs).sum(-1)
        return action, log_prob, entropy, self._mlp("critic", state)


def squashed_sample(mean, log_std, action):
    """nets/nets.py:90-105 with `action` given: tanh-squashed Gaussian log-prob."""
    std = log_std.exp()
    y = torch.tanh(action)
    log_prob = -((action - mean) ** 2) / (2 * std ** 2) - std.log() - math.log(math.sqrt(2 * math.pi))
    log_prob = log_prob - torch.log((1 - y.pow(2)) + 1e-6)
    log_prob = log_prob.sum(1, keepdim=True)
    entropy = 0.5 + 0.5 * math.log(2 * math.pi) + std.log()
    return y, log_prob, torch.tanh(mean), entropy


# ------------------------------------------------------------------------ update
def ppo_loss(policy: RefPolicy, obs, act, oldlp, adv, ret, vold, clip_coeff=0.2, ent_c=0.01, vf_c=0.5,
             norm_adv=True, clip_vloss=True):
    """ppo.py:220-264: returns (loss, stats dict, newlogprob, newvalue)."""
    _, newlogprob, entropy, newvalue = policy.evaluate(obs, act)
    log_ratio = newlogprob - oldlp
    ratio = log_ratio.exp()
    with torch.no_grad():
        old_approx_kl = (-log_ratio).mean()
        approx_kl = ((ratio - 1) - log_ratio).mean()
        clipfrac = ((ratio - 1.0).abs() > clip_coeff).to(ratio.dtype).mean()
    mb_adv = adv
    if norm_adv:
        mb_adv = (mb_adv - mb_adv.mean()) / (mb_adv.std() + 1e-8)
    loss_one = -mb_adv * ratio
    loss_two = -mb_adv * torch.clamp(ratio, 1 - clip_coeff, 1 + clip_coeff)
    policy_loss = torch.max(loss_one, loss_two).mean()
    newvalue = newvalue.view(-1)
    if clip_vloss:
        v_loss_unclipped = (newvalue - ret) ** 2
        v_clipped = vold + torch.clamp(newvalue - vold, -clip_coeff, clip_coeff)
        v_loss_clipped = (v_clipped - ret) ** 2
        value_loss = 0.5 * torch.max(v_loss_unclipped, v_loss_clipped).mean()
    else:
        value_loss = 0.5 * ((newvalue - vold) ** 2).mean()  # reference quirk ppo.py:261
    entropy_loss = entropy.mean()
    loss = policy_loss - ent_c * entropy_loss + value_loss * vf_c
    stats = dict(policy_loss=policy_loss.item(), value_loss=value_loss.item(), entropy=entropy_loss.item(),
                 loss=loss.item(), old_approx_kl=old_approx_kl.item(), approx_kl=approx_kl.item(),
                 clipfrac=clipfrac.item())
    return loss, stats, newlogprob, newvalue


class RefAdam:
    """torch.optim.Adam(lr, betas=(0.9,0.999), eps, no weight decay), single-tensor form."""

    def __init__(self, tensors: Sequence[torch.Tensor], lr: float, eps: float = 1e-5):
        self.t = list(tensors)
        self.lr, self.eps, self.b1, self.b2 = lr, eps, 0.9, 0.999
        self.m = [torch.zeros_like(p) for p in self.t]
        self.v = [torch.zeros_like(p) for p in self.t]
        self.step_count = 0

    def step(self, grads: Sequence[torch.Tensor]):
        self.step_count += 1
        bc1 = 1 - self.b1 ** self.step_count
        bc2 = 1 - self.b2 ** self.step_count
        step_size = self.lr / bc1
        with torch.no_grad():
            for p, g, m, v in zip(self.t, grads, self.m, self.v):
                m.lerp_(g, 1 - self.b1)
                v.mul_(self.b2).addcmul_(g, g, value=1 - self.b2)
                denom = (v.sqrt() / math.sqrt(bc2)).add_(self.eps)
                p.addcdiv_(m, denom, value=-step_size)


def clip_grad_norm(grads: Sequence[torch.Tensor], max_norm: float) -> float:
    """torch.nn.utils.clip_grad_norm_: g *= min(1, max_norm / (norm + 1e-6))."""
    total = torch.linalg.vector_norm(torch.stack([torch.linalg.vector_norm(g) for g in grads]))
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
    for g in grads:
        g.mul_(coef)
    return total.item()


def ppo_update_step(policy: RefPolicy, opt: RefAdam, obs, act, oldlp, adv, ret, vold, max_grad_norm=0.5, **kw):
    """One minibatch step (ppo.py:220-269).  Returns (stats, raw grads, newlogp, newvalue)."""
    policy.requires_grad_(True)
    loss, stats, nlp, nv = ppo_loss(policy, obs, act, oldlp, adv, ret, vold, **kw)
    grads = torch.autograd.grad(loss, policy.tensors(), allow_unused=True)
    grads = [torch.zeros_like(p) if g is None else g.clone() for p, g in zip(policy.tensors(), grads)]
    raw = [g.clone() for g in grads]
    stats["grad_norm"] = clip_grad_norm(grads, max_grad_norm)
    policy.requires_grad_(False)
    opt.step(grads)
    return stats, raw, nlp.detach(), nv.detach()


def explained_variance(values: np.ndarray, returns: np.ndarray) -> float:
    """ppo.py:277-279 (NumPy population variance)."""
    var_y = np.var(returns)
    return float("nan") if var_y == 0 else float(1 - np.var(returns - values) / var_y)


def lr_anneal(lr: float, update: int, num_updates: int) -> float:
    """ppo.py:195-198."""
    return (1.0 - (update - 1.0) / num_updates) * lr


# ------------------------------------------------- device sampler, restated on CPU
_M0, _M1 = 0xD2511F53, 0xCD9E8D57
_W0, _W1 = 0x9E3779B9, 0xBB67AE85


def philox4x32_10(counter: Sequence[int], key: Sequence[int]) -> Tuple[int, int, int, int]:
    """Philox4x32-10 (Salmon et al., SC'11).  Known answer checked in tests."""
    c0, c1, c2, c3 = [int(c) & 0xFFFFFFFF for c in counter]
    k0, k1 = [int(k) & 0xFFFFFFFF for k in key]
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c3 ^ k1) & 0xFFFFFFFF, p0 & 0xFFFFFFFF
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def sampler_words(seed: int, env_id: int, step: int) -> Tuple[int, int, int, int]:
    """Counter layout of the device sampler: (env_lo, env_hi, step_lo, step_hi), key = seed."""
    return philox4x32_10((env_id & 0xFFFFFFFF, env_id >> 32, step & 0xFFFFFFFF, step >> 32),
                         (seed & 0xFFFFFFFF, seed >> 32))


def u01(word: int) -> np.float32:
    """24-bit uniform in [0,1): (w >> 8) * 2^-24."""
    return np.float32((word >> 8) * (1.0 / 16777216.0))


# Vectorised forms of the above, for checking every draw of a launch.  Each device sampler keys one Philox4x32-10 block
# by the 64-bit seed and builds its counter from two 64-bit ids and a dimension block (dims 4 blk .. 4 blk + 3):
#   rollouts, policy_evaluate:     (gid lo, gid hi, step lo, step hi ^ blk << 24)   gid = env_id0 + env or row0 + row
#   aur_squashed_gaussian_sample:  (row lo, row hi, stream lo, stream hi ^ blk << 24)
#   head_eval_kernel (facades):    (b, 0, stream lo, stream hi ^ blk << 24)          b < 2^31, so b hi = 0
_U32 = np.uint64(0xFFFFFFFF)


def philox4x32_10_np(c0, c1, c2, c3, k0, k1) -> np.ndarray:
    """philox4x32_10 over broadcast arrays of counter and key words -> uint32 [4, ...] (words c[0..3])."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*[np.asarray(x, dtype=np.uint64) & _U32 for x in (c0, c1, c2, c3, k0, k1)])
    k0, k1 = k0.copy(), k1.copy()
    m0, m1, w0, w1, s32 = np.uint64(_M0), np.uint64(_M1), np.uint64(_W0), np.uint64(_W1), np.uint64(32)
    for _ in range(10):
        p0, p1 = c0 * m0, c2 * m1
        c0, c1, c2, c3 = (p1 >> s32) ^ c1 ^ k0, p1 & _U32, (p0 >> s32) ^ c3 ^ k1, p0 & _U32
        k0 = (k0 + w0) & _U32
        k1 = (k1 + w1) & _U32
    return np.stack([c0, c1, c2, c3]).astype(np.uint32)


def sampler_counter(idx, stream, blk: int = 0):
    """The four counter words (idx lo, idx hi, stream lo, stream hi ^ blk << 24) of the table above."""
    idx, stream = np.asarray(idx, dtype=np.uint64), np.asarray(stream, dtype=np.uint64)
    return idx & _U32, idx >> np.uint64(32), stream & _U32, (stream >> np.uint64(32)) ^ np.uint64(blk << 24)


def sampler_words_np(seed: int, idx, stream, blk: int = 0) -> np.ndarray:
    """uint32 [4, ...]: the Philox block a device sampler draws for (idx, stream, dimension block blk) under `seed`."""
    return philox4x32_10_np(*sampler_counter(idx, stream, blk), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)


def normal4_f64(words: np.ndarray) -> np.ndarray:
    """Box-Muller of policy.cuh normal4 in float64: u = ((w >> 8) + 1/2) 2^-24 lies in (0, 1) for every word, and
    z = sqrt(-2 ln u1) (cos, sin)(2 pi u2), sqrt(-2 ln u3) (cos, sin)(2 pi u4).  words [4, ...] -> z [..., 4]."""
    u = ((np.asarray(words, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) + 0.5) * 2.0 ** -24
    ra, rb = np.sqrt(-2.0 * np.log(u[0])), np.sqrt(-2.0 * np.log(u[2]))
    return np.stack([ra * np.cos(2 * np.pi * u[1]), ra * np.sin(2 * np.pi * u[1]),
                     rb * np.cos(2 * np.pi * u[3]), rb * np.sin(2 * np.pi * u[3])], axis=-1)


def categorical_icdf(probs, u):
    """Inverse CDF of Categorical(probs): the first class k with u < P_0 + .. + P_k; a u at or past the total takes the last
    class with nonzero probability.  probs [n, A] float64, u [n] -> (class [n] int64, distance of u to the nearest interior
    CDF boundary [n]; inf when A = 1), so that a check can leave out draws closer to a boundary than a kernel's error."""
    probs = np.asarray(probs, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    cdf = np.cumsum(probs, axis=1)
    cls = (cdf <= u[:, None]).sum(axis=1)
    last_nz = probs.shape[1] - 1 - np.argmax(probs[:, ::-1] > 0, axis=1)
    cls = np.where(cls >= probs.shape[1], last_nz, cls)
    inner = cdf[:, :-1]
    margin = np.abs(inner - u[:, None]).min(axis=1) if inner.shape[1] else np.full(u.shape, np.inf)
    return cls.astype(np.int64), margin


# ------------------------------------------------- device minibatch shuffle, restated on CPU
SHUF_ROUNDS = 8


def _shuf_mix(v: np.ndarray) -> np.ndarray:
    v = (v * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF); v ^= v >> np.uint64(15)
    v = (v * np.uint64(0x85EBCA77)) & np.uint64(0xFFFFFFFF); v ^= v >> np.uint64(13)
    v = (v * np.uint64(0xC2B2AE3D)) & np.uint64(0xFFFFFFFF); v ^= v >> np.uint64(16)
    return v


def feistel_shuffle(n: int, seed: int, stream_id: int) -> np.ndarray:
    """aur_shuffle_indices (aur_ppo_b200/csrc/shuffle.cu), the device stand-in for `np.random.shuffle(b_inds)`
    (src/ppo.py:214-215): alternating unbalanced Feistel network over ceil(log2 n) bits with cycle walking -> int32
    permutation of [0, n)."""
    if n == 0:
        return np.zeros(0, np.int32)
    bits = 1
    while (1 << bits) < n:
        bits += 1
    wa = (bits + 1) // 2
    wb = max(bits - wa, 0)
    ma, mb = np.uint64((1 << wa) - 1), np.uint64((1 << wb) - 1)
    m32 = np.uint64(0xFFFFFFFF)
    keys = [np.uint64(philox4x32_10((r, stream_id & 0xFFFFFFFF, (stream_id >> 32) & 0xFFFFFFFF, 0x5AFE5EED),
                                    (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))[0]) for r in range(SHUF_ROUNDS)]

    def encrypt(x):
        L, R = x >> np.uint64(wb), x & mb
        for r in range(0, SHUF_ROUNDS, 2):
            t = L ^ (_shuf_mix((R + keys[r]) & m32) & ma)
            L, R = R, t
            t = L ^ (_shuf_mix((R + keys[r + 1]) & m32) & mb)
            L, R = R, t
        return (L << np.uint64(wb)) | R

    x = encrypt(np.arange(n, dtype=np.uint64))
    while True:
        bad = x >= np.uint64(n)
        if not bad.any():
            break
        x[bad] = encrypt(x[bad])
    return x.astype(np.int32)
