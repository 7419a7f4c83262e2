"""Regenerate tests/golden/stage/*.npz from the UNMODIFIED reference (oracle/_ref, built by `make -C oracle ref`).

    python tests/golden/make_stage_cases.py

The cases are those the solver-stage tests ask for: every test function of tests/test_oracle_cpu.py (the oracle pinned to
the reference) and tests/test_solver_stage_gpu.py (the device's wavefront schedule against the reference) is called with
each of its parameter sets while tests/stage_cases.py records every case it loads. The GPU tests stop at their first
device call (a stand-in device raises there); their case has been recorded by then. Each case is a scene stepped `warm`
times by the reference, then collided once; the rows its solver stage receives and what that stage returns are stored.
Free body slots and joint slots hold whatever the reference's pools left there: they are stored as zero rows, so that a
regeneration reproduces the files byte for byte.
"""
import inspect
import itertools
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import stage_cases  # noqa: E402
from helpers import body_rows_from_ref, contact_rows_from_ref, joint_rows_from_ref  # noqa: E402
from oracle import ref as refmod  # noqa: E402
from solver2d_b200 import device, scenes  # noqa: E402
from stage_cases import STAGE_DIR, STICKY, case_name  # noqa: E402

TEST_MODULES = ("test_oracle_cpu", "test_solver_stage_gpu")


class _NoDevice(Exception):
    pass


class _StandInDevice:
    def __getattr__(self, name):
        raise _NoDevice(name)


def record(R, recipe, solver, warm, vel, pos, warm_start, warm_iters, kw):
    wv, wp = warm_iters or (vel, pos)
    sc = getattr(scenes, recipe)(R, solver, **kw)
    for _ in range(warm):
        sc.step(1.0 / 60.0, wv, wp, True)
    R.step_collide(sc.world)
    bodies = body_rows_from_ref(*R.bodies(sc.world))
    contacts, slots = contact_rows_from_ref(*R.contacts(sc.world))
    joints = joint_rows_from_ref(*R.joints(sc.world))
    R.step_solve(sc.world, 1.0 / 60.0, vel, pos, warm_start)
    bf, _ = R.bodies(sc.world)
    cf, ci = R.contacts(sc.world)
    F, P = refmod.BODY_F, refmod.POINT_F
    free = (bodies["flags"] & 1) == 0
    bodies[free] = np.zeros(1, dtype=bodies.dtype)
    bodies["index"] = np.arange(len(bodies))
    joints[(joints["flags"] & 1) == 0] = np.zeros(1, dtype=joints.dtype)
    joints["index"] = np.arange(len(joints))
    # the reference's revolute joints never set collideConnected (the flag reads uninitialised memory); the solver stage
    # does not read it, so it is stored cleared
    joints["flags"] &= ~np.int32(device.JOINT_COLLIDE_CONNECTED)
    out = dict(bodies=bodies, contacts=contacts, joints=joints)
    out["out_body"] = np.concatenate([bf[:, F["origin"]:F["origin"] + 2], bf[:, F["position"]:F["position"] + 2],
                                      bf[:, F["rot"]:F["rot"] + 2], bf[:, F["v"]:F["v"] + 2], bf[:, F["w"]:F["w"] + 1]],
                                     axis=1).astype(np.float32)
    out["out_body"][free] = 0.0
    base = [refmod.CONTACT_F["points"] + refmod.POINT_STRIDE * j for j in range(2)]
    out["out_normal"] = np.stack([cf[slots, b + P["normalImpulse"]] for b in base], axis=1).astype(np.float32)
    out["out_tangent"] = np.stack([cf[slots, b + P["tangentImpulse"]] for b in base], axis=1).astype(np.float32)
    out["out_friction_persisted"] = ci[slots, refmod.CONTACT_I["frictionPersisted"]].astype(np.int32)
    if solver == "TGS_Sticky":
        for name in STICKY:
            out[name] = np.stack([cf[slots, b + P[name]:b + P[name] + 2] for b in base], axis=1).astype(np.float32)
    sc.destroy()
    return out


def _parameter_sets(fn):
    """Every keyword set pytest calls `fn` with (its parametrize marks, crossed)."""
    axes = []
    for mark in getattr(fn, "pytestmark", []):
        if mark.name != "parametrize":
            continue
        names, values = mark.args[0], mark.args[1]
        names = [n.strip() for n in names.split(",")] if isinstance(names, str) else list(names)
        axes.append([dict(zip(names, v if len(names) > 1 else (v,))) for v in values])
    for combo in itertools.product(*axes):
        kw = {}
        for part in combo:
            kw.update(part)
        yield kw


def main():
    R = refmod.load()
    os.makedirs(STAGE_DIR, exist_ok=True)
    names = set()

    def recorder(recipe, solver, warm, vel, pos, warm_start, warm_iters, kw):
        name = case_name(recipe, solver, warm, vel, pos, warm_start, warm_iters, **kw)
        if name not in names:
            names.add(name)
            np.savez_compressed(os.path.join(STAGE_DIR, name + ".npz"),
                                **record(R, recipe, solver, warm, vel, pos, warm_start, warm_iters, kw))

    stage_cases.recorder = recorder
    for module_name in TEST_MODULES:
        module = __import__(module_name)
        for fname, fn in sorted(vars(module).items()):
            if not fname.startswith("test_") or not callable(fn):
                continue
            for kw in _parameter_sets(fn):
                if "dev" in inspect.signature(fn).parameters:
                    kw["dev"] = _StandInDevice()
                try:
                    fn(**kw)
                except _NoDevice:
                    pass
    print(f"wrote {len(names)} cases to {STAGE_DIR}")


if __name__ == "__main__":
    main()
