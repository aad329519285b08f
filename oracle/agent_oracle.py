"""TEST INFRASTRUCTURE ONLY -- never imported by the product package.

CPU restatement of the reference's tabular agent (PKG/double_q_learning.py)
and of the three Trainer schedules on the hot path (PKG/trainer.py:88-138).
Random draws are explicit arguments (see oracle/philox.py for the contract).

``dtype`` selects the Q-table arithmetic:
  float64 -- the reference default (PKG/double_q_learning.py:38-40);
  float32 -- what the unmodified reference computes under NumPy >= 2 (NEP 50)
             when float32 tables are assigned through its public attributes;
             Python-float operands (alpha, gamma, reward) are then rounded to
             float32 and every operation is a float32 operation.  This is the
             bit-exact oracle for the device tables (SURVEY.md A.7).
"""
from __future__ import annotations

import math
from typing import Sequence, Tuple

import numpy as np

TABLE_SHAPE_TAIL = (3, 3, 3, 7, 3)
ALPHA_SATURATION = 1002   # (1/c)**0.51 <= alpha_min for c >= 1002 (probe, SURVEY.md A.5)


def state_id(s: Sequence[int]) -> int:
    return (((s[0] * 3 + s[1]) * 3 + s[2]) * 3 + s[3]) * 7 + s[4]


def state_from_id(i: int) -> Tuple[int, int, int, int, int]:
    t = i % 7; i //= 7
    a = i % 3; i //= 3
    v = i % 3; i //= 3
    p = i % 3; i //= 3
    return (i, p, v, a, t)


def alpha_of(count: float, alpha_min: float = 0.02949, omega: float = 0.51) -> float:
    """PKG/trainer.py:88-110 (count BEFORE the increment, quirk Q5)."""
    if count == 0:
        return alpha_min
    return float(np.max([np.float_power(1 / count, omega), alpha_min]))


def exploration_rate(episode: int, w: int) -> float:
    """PKG/trainer.py:112-126."""
    if w > 0:
        return 0.0
    if 0 <= episode <= 800:
        return 1.0
    return max(1 + (0.01 - 1) * (episode - 800) / (2000 - 800), 0.01)


SCALE_MODIFICATION = (0.8172650252856599, 0.8211253690681617, 0.8257273369742982, 0.8311571820651724)


def transfer_ratio(step: int, scale: Sequence[float] = SCALE_MODIFICATION) -> float:
    """PKG/trainer.py:128-138 (``scale`` = Trainer's scale_modification_value)."""
    if step < 1:
        return 1.0
    if step < len(scale) + 1:
        return scale[step - 1]
    raise ValueError(f"Transfer learning can be done up to the 5th curriculum step, {step} is invalid")


def explore_threshold(eps: float) -> int:
    """u24 < threshold  <=>  u24 * 2**-24 < eps  (exact: scaling by 2**24 is exact in float64)."""
    return int(math.ceil(eps * 2.0 ** 24))


class AgentOracle:
    def __init__(self, curriculum_steps: int = 5, dtype=np.float64, alpha_min=0.02949, omega=0.51, gamma=0.99):
        shape = (curriculum_steps,) + TABLE_SHAPE_TAIL
        self.dtype = np.dtype(dtype)
        self.qa = np.zeros(shape, self.dtype)
        self.qb = np.zeros(shape, self.dtype)
        self.count = np.zeros(shape, np.float64)
        self.alpha_min, self.omega, self.gamma = alpha_min, omega, gamma

    def predict(self, s) -> int:
        """PKG/double_q_learning.py:119-124."""
        return int(np.argmax(np.add(self.qa[tuple(s)], self.qb[tuple(s)]) / 2))

    def guess(self, s, eps: float, w_explore: int, w_action: int) -> int:
        """PKG/double_q_learning.py:110-117: both draws are always consumed (quirk Q4)."""
        explore = (int(w_explore) >> 8) < explore_threshold(eps)
        k = (int(w_action) * 3) >> 32
        return int(k if explore else self.predict(s))

    def alpha(self, sa) -> float:
        return alpha_of(self.count[tuple(sa)], self.alpha_min, self.omega)

    @staticmethod
    def target(q_snapshot, s_next, sa, reward, gamma, T):
        """reward + (gamma*q[s', argmax q[s']]) * [sa.p_bin != s'.p_bin]   (PKG/double_q_learning.py:136-143)."""
        row = q_snapshot[tuple(s_next)]
        q_next = row[int(np.argmax(row))]
        return T(reward) + (T(gamma) * q_next) * T(int(sa[1] != s_next[1]))

    def update(self, sa, s_next, alpha: float, reward: float, q_snapshot=None):
        """PKG/double_q_learning.py:91-108,126-146: count += 1, then table A either way (quirks Q1, Q2, Q3).
        ``q_snapshot`` (batched S1 semantics): table the bootstrap value is read from; default = live table."""
        T = self.dtype.type
        sa = tuple(sa)
        self.count[sa] += 1
        src = self.qa if q_snapshot is None else q_snapshot
        tgt = self.target(src, s_next, sa, reward, self.gamma, T)
        loss = T(alpha) * (tgt - self.qa[sa])
        self.qa[sa] += loss

    def transfer(self, step: int, ratio: float):
        """PKG/double_q_learning.py:77-89 (slot `step` from slot `step-1`; step 0 reads slot -1, quirk Q7)."""
        self.qa[step] = self.qa[step - 1] * ratio
        self.qb[step] = self.qb[step - 1] * ratio
