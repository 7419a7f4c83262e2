"""Reference runs recorded for the lock-step tests (tests/golden/make_lockstep.py -> tests/golden/lockstep/).

The tests that step the product in the reference's Gauss-Seidel order read that order from here: for every step the
reference's contact pool order after its pair update and narrow phase, as shape-pair keys, together with whatever the
test compares the product with (positions, angles, counts, query results)."""
from __future__ import annotations

import os

import numpy as np

LOCKSTEP_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lockstep")


def pool_keys(R, wid) -> np.ndarray:
    """The reference's live contacts in pool order (= its sequential solve order) as (min shape, max shape) keys."""
    _, ci = R.contacts(wid)
    live = ci[:, 0] == 1
    a, b = ci[live, 1].astype(np.uint64), ci[live, 2].astype(np.uint64)
    return (np.minimum(a, b) << np.uint64(32)) | np.maximum(a, b)


def reference_steps(R, wid, steps, dt, vel=4, pos=2, before_solve=None) -> list:
    """Step a reference world split at the stage boundaries; returns the pool-order keys of every step."""
    keys = []
    for step in range(steps):
        R.step_collide(wid)
        keys.append(pool_keys(R, wid))
        if before_solve is not None:
            before_solve(step)
        R.step_solve(wid, dt, vel, pos, True)
        R.step_finalize(wid)
    return keys


def pack_keys(keys: list, prefix: str = "") -> dict:
    off = np.zeros(len(keys) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(k) for k in keys])
    flat = np.concatenate(keys) if keys else np.zeros(0, np.uint64)
    return {prefix + "order_keys": flat.astype(np.uint64), prefix + "order_offsets": off}


class Run:
    """One recorded run: `keys(step)` is the reference's order of that step; other arrays by name."""

    def __init__(self, name: str, prefix: str = ""):
        self.g = np.load(os.path.join(LOCKSTEP_DIR, name + ".npz"))
        self.prefix = prefix

    def keys(self, step: int, prefix: str | None = None) -> np.ndarray:
        p = self.prefix if prefix is None else prefix
        k, off = self.g[p + "order_keys"], self.g[p + "order_offsets"]
        return np.ascontiguousarray(k[off[step]:off[step + 1]])

    def __getitem__(self, key):
        return self.g[key]


def save(name: str, arrays: dict) -> str:
    os.makedirs(LOCKSTEP_DIR, exist_ok=True)
    path = os.path.join(LOCKSTEP_DIR, name + ".npz")
    np.savez_compressed(path, **arrays)
    return path
