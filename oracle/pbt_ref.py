"""Population-based training, restated in NumPy: the decision rule of include/aur_ppo.h ("population-based training",
steps 1-5) and the row / column copies of step 6 on host arrays.  tests/test_pbt_gpu.py compares aur_pop_pbt_step with
these, np.array_equal.

  1. member k is ranked when fitness[k] is not NaN (+-inf are ranked); n_valid = number of ranked members
  2. order = ranked members by fitness, highest first, ties (-0.0 == +0.0 included) to the lower index; rank[k] its position
     in order, -1 when not ranked
  3. n_sel = floor(q * n_valid) in fp64 (0 < q <= 0.5); n_sel == 0 changes nothing
  4. recipients: rank[k] >= n_valid - n_sel (the bottom n_sel); donors: the top n_sel
  5. recipient k: w = philox4x32_10((k, r lo, r hi, PHILOX_C3), (seed lo, seed hi)), donor = order[(w0 * n_sel) >> 32];
     the donor's six hyper-parameters are copied and field j with mask bit j is multiplied in fp64 by up if bit j of w1
     is set, else by down
  6. the recipient gets the donor's params / exp_avg / exp_avg_sq rows, Adam step count and rows 0 .. 2D + 3 of its env
     columns of the wrapper statistics `norm`; row 2D + 4 (the return accumulator) and everything else stays
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import numpy as np

from .ppo_ref import philox4x32_10

PHILOX_C3 = 0x50B7D0E5          # AUR_PBT_PHILOX_C3
HPARAM_FIELDS = ("learning_rate", "entropy_coeff", "clip_coeff", "value_coeff", "max_grad_norm", "target_kl")


def rank_members(fitness: Sequence[float]) -> Tuple[np.ndarray, np.ndarray]:
    """Steps 1-2 -> (rank [K] int32, order [n_valid] int32)."""
    f = [float(v) for v in fitness]
    ranked = [k for k, v in enumerate(f) if not math.isnan(v)]
    order = sorted(ranked, key=lambda k: (-f[k], k))       # -(-0.0) == -(+0.0): ties fall to the index
    rank = np.full(len(f), -1, dtype=np.int32)
    for pos, k in enumerate(order):
        rank[k] = pos
    return rank, np.array(order, dtype=np.int32)


def decide(fitness: Sequence[float], q: float, down: float, up: float, mask: int, seed: int, rnd: int,
           hparams: np.ndarray) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Steps 1-5 -> (rank [K] int32, donor [K] int32 (-1: not a recipient), hparams after the round [K][6] fp64)."""
    assert 0.0 < q <= 0.5 and 0 <= mask < 64
    rank, order = rank_members(fitness)
    n_valid = len(order)
    n_sel = math.floor(q * n_valid)
    donor = np.full(len(rank), -1, dtype=np.int32)
    hp = np.array(hparams, dtype=np.float64, copy=True)
    if n_sel == 0:
        return rank, donor, hp
    seed &= 0xFFFFFFFFFFFFFFFF
    for k in np.nonzero(rank >= n_valid - n_sel)[0]:
        w = philox4x32_10((int(k), rnd & 0xFFFFFFFF, (rnd >> 32) & 0xFFFFFFFF, PHILOX_C3), (seed & 0xFFFFFFFF, seed >> 32))
        d = int(order[(w[0] * n_sel) >> 32])
        donor[k] = d
        row = np.array(hparams[d], dtype=np.float64, copy=True)
        for j in range(6):
            if (mask >> j) & 1:
                row[j] = row[j] * (up if (w[1] >> j) & 1 else down)
        hp[k] = row
    return rank, donor, hp


def exploit(donor: np.ndarray, rows: Sequence[np.ndarray], steps: np.ndarray, norm: Optional[np.ndarray] = None,
            n_member: int = 0, obs_dim: int = 0) -> None:
    """Step 6 in place: rows are [K][P] arrays (params, exp_avg, exp_avg_sq), steps [K], norm [2 D + 5][K * n_member] or None.
    Donors are never recipients, so the copies do not depend on their order."""
    for k in np.nonzero(donor >= 0)[0]:
        d = int(donor[k])
        for r in rows:
            r[k] = r[d]
        steps[k] = steps[d]
        if norm is not None:
            n = n_member
            norm[:2 * obs_dim + 4, k * n:(k + 1) * n] = norm[:2 * obs_dim + 4, d * n:(d + 1) * n]
