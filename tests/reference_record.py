"""The reference's side of the tests that compare this project with sisl/MADRL, stored under tests/golden/.

A test asks ``recorded(name, produce)`` for what the reference computed; it is read from
tests/golden/ref_<name>.npz, so the comparison runs on every machine.  ``produce()`` runs the reference
(through oracle/refshim.py) and returns a dict of arrays / strings; it only runs when the goldens are
re-recorded from a reference checkout:

    MADRL_REFERENCE_ROOT=<checkout> MADRL_RECORD_REFERENCE=1 python -m pytest tests -k <test>

TEST INFRASTRUCTURE (shared by the CPU tests; nothing here is imported by ``madrl_b200``).
"""
import hashlib
import json
import os

import numpy as np

from conftest import GOLDEN_DIR

RECORD = os.environ.get("MADRL_RECORD_REFERENCE") == "1"


def recorded(name, produce):
    path = os.path.join(GOLDEN_DIR, "ref_" + name + ".npz")
    if RECORD:
        np.savez_compressed(path, **{k: np.asarray(v) for k, v in produce().items()})
    with np.load(path, allow_pickle=False) as g:
        return {k: g[k] for k in g.files}


def digest(*xs):
    """8 bytes of SHA-256 over the shapes and float64 values of xs (-0.0 counts as 0.0, as in np.array_equal):
    equal digests stand for bitwise-equal values."""
    h = hashlib.sha256()
    for x in xs:
        a = np.ascontiguousarray(np.asarray(x, dtype=np.float64) + 0.0)
        h.update(repr(a.shape).encode() + a.tobytes())
    return np.frombuffer(h.digest()[:8], dtype=np.uint8)


def trace(env, actions, reset_after=lambda t: False):
    """reset(), then step(a) for every action, reset() again after a done step and wherever reset_after(t).
    `calls`: in call order, the digest of each reset()'s observation and of each step()'s observation and reward;
    dones, infos and the steps followed by a reset in full."""
    calls, done, info, resets = [digest(env.reset())], [], [], []
    for t, a in enumerate(actions):
        o, r, d, i = env.step(a)
        calls.append(digest(o, r))
        done.append(bool(d))
        info.append(i)
        if d or reset_after(t):
            resets.append(t)
            calls.append(digest(env.reset()))
    return dict(calls=np.array(calls), done=np.array(done), resets=np.array(resets, dtype=np.int64),
                info=json.dumps(info, default=lambda v: v.item()))


def assert_same_trace(got, want):
    """Every key of `got` equals the recorded one; the message names the first differing entry."""
    assert sorted(got) == sorted(want)
    for k in got:
        if k == "info":
            a, b = json.loads(str(got[k])), json.loads(str(want[k]))
            assert a == b, (k, next(t for t, (x, y) in enumerate(zip(a, b)) if x != y) if len(a) == len(b) else "length")
            continue
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.shape == b.shape, (k, a.shape, b.shape)
        if not np.array_equal(a, b):
            bad = np.nonzero((a != b).reshape(a.shape[0], -1).any(1))[0] if a.ndim else [None]
            raise AssertionError("%s differs first at entry %s" % (k, bad[0]))
