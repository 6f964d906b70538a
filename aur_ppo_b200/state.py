"""The training-state file: everything a `ppo` or `ppo_population` run needs to continue bit for bit after its process stops.

One file per run, written by `torch.save` and holding only CPU tensors and plain Python values (str, int, float, bool, None,
lists, dicts), so it loads with `torch.load(path, weights_only=True)` and loading never runs pickled code (the policy
checkpoints `actor_critic_*.pt` are whole-module pickles and need weights_only=False).  Header keys: `format`, `version`, `kind`
("ppo" or "population").  The `fingerprint` is the run's configuration minus the keys that do not change what it computes; a
state is only loaded into a run whose fingerprint is equal (DESIGN.md section 13).
"""
from __future__ import annotations

import os
from typing import Dict, Iterable, Optional, Sequence, Tuple

import numpy as np
import torch

from ._lib import AurError

FORMAT, VERSION = "aur_ppo_training_state", 1
KINDS = ("ppo", "population")
# params keys that change nothing a run computes (logging, output files, placement)
NON_COMPUTE_KEYS = frozenset(("track", "capture_video", "exp_name", "tensorboard", "save", "device"))
_ABSENT = "<absent>"


def plain(v):
    """`v` with NumPy scalars turned into Python ones (the types weights_only loading accepts); AurError on anything else that
    is not a tensor, str, int, float, bool, None, list, tuple or dict."""
    if isinstance(v, np.generic):
        return v.item()
    if v is None or isinstance(v, (str, int, float, bool, torch.Tensor)):
        return v
    if isinstance(v, (list, tuple)):
        return type(v)(plain(x) for x in v)
    if isinstance(v, dict):
        return {plain(k): plain(x) for k, x in v.items()}
    raise AurError(f"training state: a value of type {type(v).__name__} cannot be stored (plain Python values and tensors only)")


def fingerprint(params: Dict, members: Optional[Sequence[Dict]] = None, pbt: Optional[Dict] = None) -> Dict:
    """What must be equal for a state to be loaded: the params entries that affect the computation; for a population
    (`members` given) also the member overrides and the PBT config (interval, fraction, keys, factors)."""
    fp = plain({k: v for k, v in params.items() if k not in NON_COMPUTE_KEYS})
    if members is None:
        return fp
    if pbt is not None:
        pbt = dict(interval=pbt["interval"], fraction=pbt["fraction"], keys=list(pbt["keys"]), factors=list(pbt["factors"]))
    return plain(dict(params=fp, members=[dict(m) for m in members], pbt=pbt))


def check_fingerprint(stored: Dict, current: Dict) -> None:
    """AurError naming every key whose value differs between a stored and the current fingerprint (nested dicts: `a.b`)."""
    diffs = []

    def walk(a, b, prefix):
        for k in sorted(set(a) | set(b), key=str):
            x, y = a.get(k, _ABSENT), b.get(k, _ABSENT)
            if isinstance(x, dict) and isinstance(y, dict):
                walk(x, y, f"{prefix}{k}.")
            elif x != y:
                diffs.append(f"{prefix}{k} (state: {x!r}, this run: {y!r})")

    walk(stored, current, "")
    if diffs:
        raise AurError("training state was saved by a run with a different configuration: " + "; ".join(diffs))


def env_tensors(envs) -> Dict[str, torch.Tensor]:
    """The device tensors of a DeviceVecEnv that carry over from one iteration to the next (norm: with the wrappers only)."""
    out = dict(phys=envs.phys, pcg=envs.pcg, elapsed=envs.elapsed, ep_return=envs.ep_return, ep_length=envs.ep_length,
               next_obs=envs.next_obs, next_done=envs.next_done)
    if envs.norm is not None:
        out["norm"] = envs.norm
    return out


def to_host(tensors: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    return {k: t.detach().cpu() for k, t in tensors.items()}


def history(values: Sequence, dtype) -> torch.Tensor:
    """An episode-history list as a CPU tensor (float64 holds every logged fp32 return exactly; `.tolist()` gives the list back).
    Pickling the list itself costs about five times as much once it holds a long run's episodes."""
    return torch.from_numpy(np.asarray(values, dtype=dtype).reshape(-1))


def fields(obj: Dict, names: Sequence[str]) -> Dict:
    """The entries `names` of a loaded state; AurError if one is missing (checked before anything is restored)."""
    missing = [n for n in names if n not in obj]
    if missing:
        raise AurError(f"training state lacks {missing}")
    return {n: obj[n] for n in names}


def write(path: str, kind: str, fp: Dict, body: Dict) -> None:
    """Write the state atomically: to `path + ".tmp"`, flushed and fsync'ed, then renamed over `path`.  If the process dies or
    torch.save raises on the way, the previous file at `path` is left as it was."""
    if kind not in KINDS:
        raise AurError(f"training state kind must be one of {KINDS} (got {kind!r})")
    obj = plain(dict(format=FORMAT, version=VERSION, kind=kind, fingerprint=fp, **body))
    tmp = path + ".tmp"
    try:
        with open(tmp, "wb") as f:
            torch.save(obj, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    except BaseException:
        try:
            os.remove(tmp)
        except OSError:
            pass
        raise
    # make the rename itself durable
    fd = os.open(os.path.dirname(os.path.abspath(path)), os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def read(path: str, kind: str, fp: Dict) -> Dict:
    """Load a state file (weights_only) and check its header and fingerprint against the run it is loaded into."""
    try:
        obj = torch.load(path, map_location="cpu", weights_only=True)
    except FileNotFoundError:
        raise AurError(f"training state {path!r} does not exist")
    except Exception as e:
        raise AurError(f"training state {path!r} is not a readable state file: {e}")
    if not isinstance(obj, dict) or obj.get("format") != FORMAT:
        raise AurError(f"{path!r} is not an aur_ppo training state (format {obj.get('format') if isinstance(obj, dict) else None!r})")
    if obj.get("version") != VERSION:
        raise AurError(f"training state {path!r} has version {obj.get('version')!r}; this build reads version {VERSION}")
    if obj.get("kind") != kind:
        raise AurError(f"training state {path!r} was saved by a {obj.get('kind')!r} run and cannot be loaded into a {kind!r} run")
    check_fingerprint(obj.get("fingerprint", {}), fp)
    if not isinstance(obj.get("iteration"), int) or obj["iteration"] < 1:
        raise AurError(f"training state {path!r} holds no completed iteration (iteration {obj.get('iteration')!r})")
    return obj


def restore(pairs: Iterable[Tuple[str, torch.Tensor, object]]) -> None:
    """Copy loaded tensors into the run's tensors in place, (name, destination, loaded).  Every shape and dtype is checked
    before the first copy, so a refused state changes nothing."""
    pairs = list(pairs)
    for name, dst, src in pairs:
        if not isinstance(src, torch.Tensor):
            raise AurError(f"training state: {name} is missing or not a tensor")
        if src.shape != dst.shape or src.dtype != dst.dtype:
            raise AurError(f"training state: {name} is {src.dtype} {tuple(src.shape)}, this run needs {dst.dtype} "
                           f"{tuple(dst.shape)}")
    for _, dst, src in pairs:
        dst.copy_(src)


def restore_env(envs, loaded: Dict) -> list:
    """The (name, destination, loaded) pairs of a DeviceVecEnv's state; a state with or without wrapper statistics that the
    env does not match is refused."""
    want = env_tensors(envs)
    extra = set(loaded) - set(want)
    if extra:
        raise AurError(f"training state has env tensors this run does not keep: {sorted(extra)}")
    return [(f"env.{k}", t, loaded.get(k)) for k, t in want.items()]
