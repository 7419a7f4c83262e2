"""Regenerate tests/golden/multistep/*.npy: per-step digests of the reference pipeline replayed in the device's order
(needs a CUDA device and the UNMODIFIED reference in oracle/_ref, built by `make -C oracle ref`).

    python tests/golden/make_multistep.py

For every case of tests/test_multistep_gpu.py and every step: the device state before the step is loaded into the
reference world, the reference runs its pair update and narrow phase, the device runs one s2World_Step, the plain-C oracle
replays the solver stage in the order the device reports, and the reference finalizes the oracle's result. The digest
(test_multistep_gpu.step_digest) of the reference's contact table, bodies and the oracle's impulses is stored; the device's
own digest must already equal it here, or nothing is written.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from helpers import body_rows_from_ref, contact_rows_from_ref, joint_rows_from_ref  # noqa: E402
from oracle import port  # noqa: E402
from oracle import ref as refmod  # noqa: E402
from solver2d_b200 import capi, device  # noqa: E402
from test_multistep_gpu import CASES, DT, MULTISTEP_DIR, device_step_digest, start, step_digest  # noqa: E402


def _load_bodies_into_ref(R, wid, rows):
    """Device body rows -> the reference world's bodies (state fields only; mass data and flags are construction-time)."""
    F = refmod.BODY_F
    bf, bi = R.bodies(wid)
    n = min(len(rows), bf.shape[0])
    valid = bi[:n, 0] == 1
    for name, col, width in (("origin", F["origin"], 2), ("position", F["position"], 2), ("rot", F["rot"], 2),
                             ("linearVelocity", F["v"], 2)):
        bf[:n, col:col + width][valid] = rows[name][:n][valid]
    bf[:n, F["w"]][valid] = rows["angularVelocity"][:n][valid]
    bf[:n, F["dp"]:F["dp"] + 2][valid] = 0.0
    bf[:n, F["force"]:F["force"] + 2][valid] = rows["force"][:n][valid]
    bf[:n, F["torque"]][valid] = rows["torque"][:n][valid]
    R.load_body_state(wid, bf)


def record(R, P, dev, name):
    recipe, solver, steps, vel, pos, kw, setup = CASES[name]
    O = port.load()
    sr = recipe(R, solver, **kw)
    sp, dw = start(dev, P, recipe, solver, kw, setup)
    ctx = device.make_context(solver, DT, vel, pos, True)
    F = refmod.BODY_F
    digests = []
    for step in range(steps):
        cap = R.capacities(sr.world)["bodyCap"]
        _load_bodies_into_ref(R, sr.world, dw.download_all_bodies(cap))
        R.step_collide(sr.world)

        sp.step(DT, vel, pos, True)

        bodies = body_rows_from_ref(*R.bodies(sr.world))
        cf, ci = R.contacts(sr.world)
        rows_slot, slots = contact_rows_from_ref(cf, ci)
        keys = (np.minimum(rows_slot["shapeA"], rows_slot["shapeB"]).astype(np.uint64) << np.uint64(32)) | \
            np.maximum(rows_slot["shapeA"], rows_slot["shapeB"]).astype(np.uint64)
        perm = np.argsort(keys, kind="stable")
        rows_key = rows_slot[perm]
        joints = joint_rows_from_ref(*R.joints(sr.world))
        order, _ = dw.solve_order(len(rows_key) + len(joints) + 16, max_groups=200000)
        ob, oc, oj = O.solve(capi.SOLVER[solver], bodies, rows_key, joints, ctx, order=order)

        # advance the reference world with the oracle's result
        bf, bi = R.bodies(sr.world)
        valid = bi[:, 0] == 1
        bf[:, F["position"]:F["position"] + 2][valid] = ob["position"][valid]
        bf[:, F["rot"]:F["rot"] + 2][valid] = ob["rot"][valid]
        bf[:, F["v"]:F["v"] + 2][valid] = ob["linearVelocity"][valid]
        bf[:, F["w"]][valid] = ob["angularVelocity"][valid]
        bf[:, F["dp"]:F["dp"] + 2][valid] = 0.0
        R.load_body_state(sr.world, bf)
        imp = np.zeros((cf.shape[0], 4), dtype=np.float32)
        imp[slots[perm], 0] = oc["points"]["normalImpulse"][:, 0]
        imp[slots[perm], 1] = oc["points"]["tangentImpulse"][:, 0]
        imp[slots[perm], 2] = oc["points"]["normalImpulse"][:, 1]
        imp[slots[perm], 3] = oc["points"]["tangentImpulse"][:, 1]
        R.load_contact_impulses(sr.world, imp)
        if len(oj):
            jimp = np.zeros((len(oj), 5), dtype=np.float32)
            jimp[:, 0:2] = oj["impulse"]
            jimp[:, 2] = oj["motorImpulse"]
            jimp[:, 3] = oj["lowerImpulse"]
            jimp[:, 4] = oj["upperImpulse"]
            R.load_joint_impulses(sr.world, jimp)
        R.step_finalize(sr.world)

        rf, ri = R.bodies(sr.world)
        ref_bodies = body_rows_from_ref(rf, ri)
        want = step_digest(rows_key["shapeA"], rows_key["shapeB"], rows_key["pointCount"], ri[:, 0] == 1, ref_bodies,
                           oc["points"]["normalImpulse"], oc["points"]["tangentImpulse"], (oj["flags"] & 1) == 1, oj)
        assert device_step_digest(dw) == want, f"{name} step {step}: device != reference pipeline"
        digests.append(np.frombuffer(want, dtype=np.uint8))
    sr.destroy()
    sp.destroy()
    return np.stack(digests)


def main():
    R = refmod.load()
    P = capi.Solver2D(device.LIB_PATH)
    dev = device.Device()
    os.makedirs(MULTISTEP_DIR, exist_ok=True)
    out = {name: record(R, P, dev, name) for name in CASES}
    for name, digests in out.items():
        np.save(os.path.join(MULTISTEP_DIR, name + ".npy"), digests)
    print(f"wrote {len(out)} cases to {MULTISTEP_DIR}")


if __name__ == "__main__":
    main()
