"""Shared helpers for the GPU parity tests."""
import numpy as np
import torch

from oracle import ppo_ref as R


def flat_from_named(named: dict) -> np.ndarray:
    """Canonical flat parameter order of include/aur_ppo.h from the reference's names."""
    def net(prefix):
        idx = sorted({int(k.split(".")[2]) for k in named if k.startswith(prefix + ".net.")})
        out = []
        for i in idx:
            out += [np.asarray(named[f"{prefix}.net.{i}.weight"]).ravel(), np.asarray(named[f"{prefix}.net.{i}.bias"]).ravel()]
        return out
    parts = net("actor") + net("critic")
    if "actor_logstd" in named:
        parts.append(np.asarray(named["actor_logstd"]).ravel())
    return np.concatenate(parts).astype(np.float32)


def golden_policy(golden_dir, tag, file="model.npz", prefix="p"):
    import os
    g = np.load(os.path.join(golden_dir, file))
    names = [str(n) for n in g[f"{tag}_names"]]
    named = {n: g[f"{tag}_{prefix}_{n}"] for n in names}
    return R.RefPolicy(named, continuous="actor_logstd" in names), named, g


def golden_flat(g, tag, key, names):
    """The golden arrays `{tag}_{key}_<name>` in flat_from_named order, and the mask of the full flat vector's entries they
    hold: a parameter stored as a sample of its entries (`{tag}_sample_<name>`, sorted flat indices) gives only those."""
    vals, mask = {}, {}
    for n in names:
        m = np.zeros(int(np.prod(g[f"{tag}_pshape_{n}"])), np.float32)
        v = g[f"{tag}_{key}_{n}"]
        if v.size == m.size:
            m[:] = 1
        else:
            m[g[f"{tag}_sample_{n}"]] = 1
        vals[n], mask[n] = v, m
    return flat_from_named(vals), flat_from_named(mask).astype(bool)


def random_policy(obs_dim, act_dim, hidden, num_layers, continuous, seed=0, scale=1.0):
    """Reference-shaped parameters with torch's default Linear init scale (deterministic)."""
    g = torch.Generator().manual_seed(seed)
    named = {}
    def net(prefix, out):
        dims = [obs_dim] + [hidden] * num_layers + [out]
        for li in range(len(dims) - 1):
            bound = scale / np.sqrt(dims[li])
            named[f"{prefix}.net.{2 * li}.weight"] = ((torch.rand(dims[li + 1], dims[li], generator=g) * 2 - 1) * bound).numpy()
            named[f"{prefix}.net.{2 * li}.bias"] = ((torch.rand(dims[li + 1], generator=g) * 2 - 1) * bound).numpy()
    net("actor", act_dim)
    net("critic", 1)
    if continuous:
        named["actor_logstd"] = (torch.rand(1, act_dim, generator=g) * 0.6 - 0.5).numpy()
    return R.RefPolicy(named, continuous), named
