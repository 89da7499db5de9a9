"""CPU restatement of the reference's hand-written policies (TEST INFRASTRUCTURE -- never imported by
``madrl_b200``; only tests, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU legs may use it).

  * ``waterworld_action``    heuristics/waterworld.py:11-53  WaterworldHeuristicPolicy.sample_actions
  * ``pursuit_action``       heuristics/pursuit.py:18-50     PursuitHeuristicPolicy.sample_actions
  * ``pursuit_action_table`` the same decision tabulated per window cell (what the CUDA host code builds)
  * ``policy_draw``          the injected stream that stands in for ``action_space.sample()``

Pinned: ``tests/test_heuristics.py`` compares it with the actions the real classes (loaded through
``oracle/refshim.load_reference_heuristics``) took on the same inputs, recorded in ``tests/golden/ref_heuristics_*.npz``.
"""
import math

import numpy as np

from .philox import Stream, u32_to_range

LEFT, RIGHT, UP, DOWN, STAY = 0, 1, 2, 3, 4     # heuristics/pursuit.py:6-10
POLICY_TAG = 2                                   # stream family of the policy's own draws


def waterworld_action(obs_row, return_norm=False):
    """One agent's observation [7K+2(+1)] -> action [2] (heuristics/waterworld.py:25-50 with B = 1, the way
    the reference calls it: per agent, so the norm is the agent's own).  `return_norm`: also the norm the sum
    was divided by (a tiny one amplifies float32 rounding: the fp32 parity tests skip those rows)."""
    o = np.asarray(obs_row, dtype=np.float64)[None]
    K = o.shape[1] // 7                                                     # :26
    ang = np.linspace(0., 2. * np.pi, K + 1)[:-1]                           # :27
    vecs = np.c_[np.cos(ang), np.sin(ang)]                                  # :29
    ob = -np.sum(o[:, 0:K][..., None] * vecs[None], axis=1)                 # :31
    ev = np.sum(o[:, K:2 * K][..., None] * vecs[None], axis=1)              # :34
    po = -np.sum(o[:, 3 * K:4 * K][..., None] * vecs[None], axis=1)         # :37
    pu = np.sum(o[:, 5 * K:6 * K][..., None] * vecs[None], axis=1) / 2      # :40
    ev[o[:, 7 * K] > 0] *= 1.5                                              # :43
    po[o[:, 7 * K + 1] > 0] *= 1.5                                          # :44
    a = ob + ev + po + pu                                                   # :46
    n = np.linalg.norm(a)                                                   # :47
    out = (a / n)[0] if n > 0 else np.zeros(2)                              # :48-51
    return (out, n) if return_norm else out


def _direction(dx, dy):
    """heuristics/pursuit.py:33-48 for a target at offset (dx, dy) from the pursuer."""
    if dx == 0 and dy == 0:
        return STAY
    ang = math.atan2(dy, dx)
    ang = (ang + np.pi) % (2 * np.pi) - np.pi
    if -np.pi / 4 <= ang < np.pi / 4:
        return RIGHT
    if np.pi / 4 <= ang < 3 / 4. * np.pi:
        return UP
    if ang >= 3 / 4. * np.pi or ang < -3 / 4. * np.pi:
        return LEFT
    return DOWN


def _centre(R, py2_division):
    """`xs / 2` (heuristics/pursuit.py:23): integer division under Python 2, the reference's language."""
    return float(R // 2) if py2_division else R / 2


def pursuit_action_table(R, py2_division=True):
    """Action towards each window cell w = wx * R + wy, as the CUDA host code tabulates it."""
    c = _centre(R, py2_division)
    return np.array([_direction(w // R - c, w % R - c) for w in range(R * R)], dtype=np.int32)


def pursuit_action(obs_rr4, sample, py2_division=True):
    """One agent's (R, R, 4) observation -> action; `sample()` stands in for action_space.sample()
    (heuristics/pursuit.py:18-50)."""
    o = np.asarray(obs_rr4)
    if np.sum(o[..., 2]) > 0:                                               # :19,26
        x = y = _centre(o.shape[0], py2_division)                           # :21-23
        xev, yev = np.nonzero(o[..., 2])                                    # :27
        d = np.sqrt((xev - x) ** 2 + (yev - y) ** 2)                        # :28
        k = np.argmin(d)                                                    # :29
        return _direction(xev[k] - x, yev[k] - y)
    return sample()                                                         # :50


def policy_draw(seed, env_id, counter, q):
    """The policy's own draw for pursuer q deciding on an observation produced when the env's draw counter
    stood at `counter`: word 32*counter + q of the (seed, env_id, tag 2) stream, mapped to {0..4}."""
    return u32_to_range(Stream(seed, env_id, POLICY_TAG, 32 * int(counter) + int(q)).next_u32(), 0, 5)
