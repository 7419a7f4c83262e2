"""GPU end-to-end parity through the public C API: the SAME scene script drives the reference library and the product
library (solver2d_b200/capi.py binds both).

What is compared, stage by stage (SURVEY §8c):
* broad phase : the contact (shape-pair) set and the (A, B) order of every pair            -> must be identical
* narrow phase: every manifold after the first step (ids, anchors, separations, normal)   -> bit-exact
* full step, reference Gauss-Seidel order imposed (wavefront schedule + per-step order)   -> |dpos| <= 1e-4 m after
  600 steps on config 1 (north_star), in practice bit-exact
* full step, production colour schedule, free running                                       -> deviation is the order
  sensitivity of Gauss-Seidel itself (SURVEY §7 H1: 2.5e-3 m after 600 steps when the *reference* is re-ordered);
  bounded loosely here and reported.
"""
import ctypes as C
import os

import numpy as np
import pytest

import lockstep
from oracle import ref as refmod
from solver2d_b200 import capi, device, scenes

pytestmark = pytest.mark.gpu

DT = 1.0 / 60.0


@pytest.fixture(scope="module")
def product():
    return capi.Solver2D(device.LIB_PATH)


def _ref_pair_table(R, wid):
    cf, ci = R.contacts(wid)
    I = refmod.CONTACT_I
    slots = np.nonzero(ci[:, I["valid"]] == 1)[0]
    a, b = ci[slots, I["shapeA"]], ci[slots, I["shapeB"]]
    keys = (np.minimum(a, b).astype(np.uint64) << np.uint64(32)) | np.maximum(a, b).astype(np.uint64)
    return keys, a, b, slots, cf, ci


def _positions(lib, sc):
    return np.array([tuple(lib.s2Body_GetPosition(b)) for b in sc.bodies], dtype=np.float64)


def _angles(lib, sc):
    return np.array([lib.s2Body_GetAngle(b) for b in sc.bodies], dtype=np.float64)


FIRST_STEP = [(scenes.pyramid, dict(base_count=10)), (scenes.pyramid, dict(base_count=30)),
              (scenes.vertical_stack, dict(count=6, columns=3))]


def _first_step_name(recipe, kw):
    return "first_step_" + recipe.__name__ + "".join(f"_{k}{v}" for k, v in sorted(kw.items()))


def _reference_first_step(recipe, kw):
    """The reference's contact table after one step: shape pairs in pool order, point counts and ids, normals, and per
    point the anchors and separation (geometry is computed before the solver runs)."""
    def run(R):
        sr = recipe(R, "TGS_Soft", **kw)
        sr.step(DT, 4, 2, True)
        keys, a, b, slots, cf, ci = _ref_pair_table(R, sr.world)
        I = refmod.CONTACT_I
        out = dict(keys=keys, a=a, b=b, pointCount=ci[slots, I["pointCount"]], id0=ci[slots, I["id0"]],
                   id1=ci[slots, I["id1"]], normal=cf[slots, 1:3])
        for j in range(2):
            base = refmod.CONTACT_F["points"] + refmod.POINT_STRIDE * j
            out[f"point{j}"] = cf[slots, base:base + 5]  # localAnchorA, localAnchorB, separation
        sr.destroy()
        return out
    return run


@pytest.mark.parametrize("recipe,kw", FIRST_STEP)
def test_pairs_and_manifolds_first_step(product, dev, recipe, kw):
    P = product
    ref = lockstep.Run(_first_step_name(recipe, kw))
    sp = recipe(P, "TGS_Soft", **kw)
    sp.step(DT, 4, 2, True)
    keys, a, b = ref["keys"], ref["a"], ref["b"]
    dw = device.DeviceWorld.attach(dev, sp.world)
    rows = dw.download_contacts(len(keys) + 16)
    assert len(rows) == len(keys), "contact count differs"
    order = np.argsort(keys)
    dev_keys = (np.minimum(rows["shapeA"], rows["shapeB"]).astype(np.uint64) << np.uint64(32)) | \
        np.maximum(rows["shapeA"], rows["shapeB"]).astype(np.uint64)
    assert np.array_equal(dev_keys, keys[order]), "pair sets differ"
    assert np.array_equal(rows["shapeA"], a[order]) and np.array_equal(rows["shapeB"], b[order]), "(A,B) order differs"
    # manifolds (geometry is computed before the solver runs, so it is comparable after the full step)
    assert np.array_equal(rows["pointCount"], ref["pointCount"][order])
    two = rows["pointCount"] == 2
    assert np.array_equal(rows["points"]["id"][:, 0], ref["id0"][order])
    assert np.array_equal(rows["points"]["id"][two, 1], ref["id1"][order][two])
    ref_normal = np.ascontiguousarray(ref["normal"][order])
    assert np.array_equal(rows["normal"].view(np.uint32), ref_normal.view(np.uint32)), "normals not bit-exact"
    for j in range(2):
        pts = ref[f"point{j}"][order]
        live = rows["pointCount"] > j
        for name, off, width in (("localAnchorA", 0, 2), ("localAnchorB", 2, 2), ("separation", 4, 1)):
            ref_v = pts[:, off:off + width][live]
            dev_v = rows["points"][name][:, j][live].reshape(ref_v.shape)
            assert np.array_equal(np.ascontiguousarray(dev_v).view(np.uint32), np.ascontiguousarray(ref_v).view(np.uint32)), \
                f"{name}[{j}] not bit-exact"
    sp.destroy()


def _config1_golden():
    """The reference's config-1 trajectory (tests/golden/pyramid10_tgs_soft.npz, tests/golden/make_golden.py): its contact
    pool order of every step and the bodies after steps 1, 10, 60 and 600."""
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pyramid10_tgs_soft.npz"))


def test_config1_600_steps_reference_order(product, dev):
    """north_star criterion: per-body |dpos| <= 1e-4 m vs the reference after 600 steps on config 1 (Pyramid, 55 boxes,
    TGS_Soft, 4 sub-steps), with the reference's Gauss-Seidel order imposed through the validation schedule."""
    P = product
    g = _config1_golden()
    keys, off = g["order_keys"], g["order_offsets"]
    sp = scenes.pyramid(P, "TGS_Soft", base_count=10)
    dw = device.DeviceWorld.attach(dev, sp.world)
    dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    worst = 0.0
    for step in range(600):
        dw.set_contact_order(np.ascontiguousarray(keys[off[step]:off[step + 1]]))  # pool order of the reference = its sequential solve order
        sp.step(DT, 4, 2, True)
        if step in (0, 9, 59, 599):
            d = np.abs(g[f"origin_step{step + 1}"].astype(np.float64) - _positions(P, sp)).max()
            worst = max(worst, d)
    dpos = np.abs(g["origin_step600"].astype(np.float64) - _positions(P, sp)).max()
    rot = g["rot_step600"].astype(np.float64)
    dang = np.abs(np.arctan2(rot[:, 0], rot[:, 1]) - _angles(P, sp)).max()
    print(f"config1 reference-order: max|dpos| = {dpos:.3e} m, max|dangle| = {dang:.3e} rad, worst sampled {worst:.3e}")
    assert dpos <= 1e-4 and dang <= 1e-4
    sp.destroy()


def test_config1_600_steps_color_schedule(product):
    P = product
    g = _config1_golden()
    sp = scenes.pyramid(P, "TGS_Soft", base_count=10)
    for _ in range(600):
        sp.step(DT, 4, 2, True)
    dpos = np.abs(g["origin_step600"].astype(np.float64) - _positions(P, sp)).max()
    print(f"config1 colour schedule, free running: max|dpos| = {dpos:.3e} m")
    # order sensitivity of Gauss-Seidel (the reference re-ordered against itself: 2.5e-3 m, SURVEY §7 H1)
    assert dpos < 2e-2
    # the reference's contact count after step 600 = its live contacts of that step
    assert g["order_offsets"][600] - g["order_offsets"][599] == P.s2World_GetStatistics(sp.world).contactCount
    sp.destroy()


def _falling_boxes(lib):
    sc = scenes.vertical_stack(lib, "TGS_Soft", count=5, columns=4)
    # throw the top boxes sideways so pairs are created and destroyed
    for k, bid in enumerate(sc.bodies[1:]):
        if k % 5 >= 3:
            lib.s2Body_SetLinearVelocity(bid, capi.Vec2(3.0 if k % 2 else -3.0, 1.0))
    return sc


def _reference_falling_boxes(R):
    sr = _falling_boxes(R)
    out = lockstep.pack_keys(lockstep.reference_steps(R, sr.world, 120, DT))
    out["positions"] = _positions(R, sr)
    sr.destroy()
    return out


def test_falling_boxes_pair_set_tracks_reference(product, dev):
    """Proxies leave their fat AABBs while falling: the device pair pass must create / destroy the same contacts."""
    P = product
    ref = lockstep.Run("falling_boxes")
    sp = _falling_boxes(P)
    dw = device.DeviceWorld.attach(dev, sp.world)
    dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    passes = 0
    for step in range(120):
        keys = ref.keys(step)
        dw.set_contact_order(keys)
        sp.step(DT, 4, 2, True)
        rows = dw.download_contacts(len(keys) + 64)
        dev_keys = (np.minimum(rows["shapeA"], rows["shapeB"]).astype(np.uint64) << np.uint64(32)) | \
            np.maximum(rows["shapeA"], rows["shapeB"]).astype(np.uint64)
        assert np.array_equal(np.sort(keys), dev_keys), f"pair set differs at step {step}"
    passes = dw.counters().pairPassCount
    assert passes > 3
    dpos = np.abs(ref["positions"] - _positions(P, sp)).max()
    assert dpos <= 1e-4, dpos
    sp.destroy()


def test_device_atan2_bit_equal_to_libm(dev):
    """Joint-limit rows read the joint angle through atan2f: the device restatement (include/solver2d/atan2_f32.h) must
    return the bits of the host C library the reference links against. 400k inputs on the GPU vs libm."""
    import ctypes as C
    import ctypes.util
    from test_host_cpu import _atan2_inputs
    y, x = _atan2_inputs(200_000, 5)
    out = np.empty_like(y)
    dev.lib.s2b_eval_atan2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    dev.lib.s2b_eval_atan2(y.ctypes.data, x.ctypes.data, out.ctypes.data, len(y))
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.atan2f.restype = C.c_float
    libm.atan2f.argtypes = [C.c_float, C.c_float]
    want = np.array([libm.atan2f(float(a), float(b)) for a, b in zip(y, x)], np.float32)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(out), nan)
    assert np.array_equal(out[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _bulk_force(step, n):
    f = np.zeros((n, 2), dtype=np.float32)
    f[:, 0] = 3.0 * np.sin(0.3 * step + np.arange(n))
    f[:, 1] = 1.5
    return f


def _reference_bulk_force(R):
    """The reference driven by per-body forces on every third box, with a force and a state edit on some steps."""
    sr = scenes.pyramid(R, "TGS_Soft", base_count=9)
    pushed = list(range(1, len(sr.bodies), 3))

    def forces(step):
        for k, (fx, fy) in zip(pushed, _bulk_force(step, len(pushed))):
            R.s2Body_ApplyForceToCenter(sr.bodies[k], capi.Vec2(float(fx), float(fy)))
        if step % 7 == 3:
            R.s2Body_ApplyForceToCenter(sr.bodies[pushed[0]], capi.Vec2(0.5, 0.25))
            R.s2Body_SetLinearVelocity(sr.bodies[pushed[1]], capi.Vec2(0.1, -0.2))

    out = lockstep.pack_keys(lockstep.reference_steps(R, sr.world, 40, DT, before_solve=forces))
    out["positions"] = _positions(R, sr)
    out["angles"] = _angles(R, sr)
    sr.destroy()
    return out


def test_bulk_force_and_transform_paths_equal_per_body_api(product, dev):
    """s2World_ApplyForcesToCenters / s2World_GetBodyTransforms (device-side add + 16 B/body read-back) against the
    per-body calls they stand for, and against the reference driven by the same per-body forces (order-preserving
    schedule, so the comparison with the reference is bit-exact too)."""
    import ctypes as C
    P = product
    ref = lockstep.Run("bulk_force")
    L = P.lib
    L.s2World_ApplyForcesToCenters.argtypes = [capi.WorldId, C.c_void_p, C.c_void_p, C.c_int32]
    L.s2World_GetBodyTransforms.restype = C.c_int32
    L.s2World_GetBodyTransforms.argtypes = [capi.WorldId, C.c_void_p, C.c_int32]
    sa = scenes.pyramid(P, "TGS_Soft", base_count=9)   # per-body API
    sb = scenes.pyramid(P, "TGS_Soft", base_count=9)   # bulk API
    dws = [device.DeviceWorld.attach(dev, s.world) for s in (sa, sb)]
    for dw in dws:
        dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    pushed = list(range(1, len(sa.bodies), 3))
    idx = np.array([sb.bodies[k].index for k in pushed], dtype=np.int32)
    for step in range(40):
        f = _bulk_force(step, len(pushed))
        keys = ref.keys(step)
        for dw in dws:
            dw.set_contact_order(keys)
        for k, (fx, fy) in zip(pushed, f):
            P.s2Body_ApplyForceToCenter(sa.bodies[k], capi.Vec2(float(fx), float(fy)))
        L.s2World_ApplyForcesToCenters(sb.world, idx.ctypes.data, f.ctypes.data, len(idx))
        if step % 7 == 3:
            # a per-body force and a state edit AFTER the bulk call must not drop the bulk force of those bodies
            for sc in (sa, sb):
                P.s2Body_ApplyForceToCenter(sc.bodies[pushed[0]], capi.Vec2(0.5, 0.25))
                P.s2Body_SetLinearVelocity(sc.bodies[pushed[1]], capi.Vec2(0.1, -0.2))
        sa.step(DT, 4, 2, True)
        sb.step(DT, 4, 2, True)
    cap = dws[1].counters().bodyCapacity
    xf = np.zeros((cap, 4), dtype=np.float32)
    assert len(sb.bodies) <= L.s2World_GetBodyTransforms(sb.world, xf.ctypes.data, cap) <= cap
    pa = _positions(P, sa)
    pr = ref["positions"]
    pb = np.array([xf[b.index, :2] for b in sb.bodies], dtype=np.float64)
    assert np.array_equal(pa, pb), "bulk and per-body paths differ"
    assert np.array_equal(pa, pr), f"public API with forces differs from the reference: {np.abs(pa - pr).max()}"
    ang_b = np.arctan2(xf[[b.index for b in sb.bodies], 2].astype(np.float64), xf[[b.index for b in sb.bodies], 3].astype(np.float64))
    assert np.abs(ang_b - ref["angles"]).max() < 1e-6
    for s in (sa, sb):
        s.destroy()


@pytest.mark.parametrize("solver", ["TGS_Soft", "PGS_NGS_Block", "XPBD"])
def test_graph_replay_gives_the_same_bits(product, dev, solver):
    """The solver stage is replayed as a CUDA graph while its inputs' shapes and addresses stand still. Same scene with
    and without it: identical bits; and the replay really happens."""
    P = product
    sa = scenes.joint_contact_stress(P, solver, bridges=2, planks=16, grid=6)
    sb = scenes.joint_contact_stress(P, solver, bridges=2, planks=16, grid=6)
    da = device.DeviceWorld.attach(dev, sa.world)
    db = device.DeviceWorld.attach(dev, sb.world)
    da.set_graph(True)
    db.set_graph(False)
    for _ in range(60):
        sa.step(DT, 4, 2, True)
        sb.step(DT, 4, 2, True)
    assert np.array_equal(_positions(P, sa), _positions(P, sb))
    assert np.array_equal(_angles(P, sa), _angles(P, sb))
    assert da.counters().graphReplays > 10 and db.counters().graphReplays == 0
    sa.destroy()
    sb.destroy()


def test_colour_kernel_probe_and_row_built_world(dev):
    """scenes.pyramid_rows builds the same kind of world the API does (contacts appear, colours form), and the per-colour
    kernel probe returns a time for a non-empty colour."""
    import ctypes as C
    bodies, shapes = scenes.pyramid_rows(40)
    dw = dev.create_world(7)
    dw.upload_bodies(bodies, len(bodies))
    dw.upload_shapes(shapes, len(shapes))
    ctx = device.make_context("TGS_Soft", DT, 4, 2, True)
    for _ in range(3):
        dw.step(ctx)
    c = dw.counters()
    assert c.contactCount == 3 * 820 - 40 - 39 - 1 or c.contactCount > 2000  # ~3 contacts per box
    assert 4 <= c.groupCount <= 16
    n = C.c_int(0)
    ms = dev.lib.s2b_time_color_kernel(dw.h, C.byref(ctx), 3, C.byref(n))
    assert ms > 0.0 and n.value > 100
    dw.destroy()


def _reference_tumbler(R):
    sr = scenes.tumbler(R, "TGS_Soft", grid=18, half_extent=4.0)
    out = lockstep.pack_keys(lockstep.reference_steps(R, sr.world, 90, DT))
    out["positions"] = _positions(R, sr)
    out["angles"] = _angles(R, sr)
    out["final_contacts"] = np.array(len(_ref_pair_table(R, sr.world)[0]))
    sr.destroy()
    return out


def test_tumbler_large_proxies_reference_order(product, dev):
    """A motorised container whose four walls span the scene (their proxies take the leaf-side 'large mover' query of the
    broad phase, are touched by dozens of boxes -> serial overflow group, and carry a motor joint): 90 steps through the
    public API with the reference's Gauss-Seidel order imposed must reproduce the reference bit for bit."""
    P = product
    ref = lockstep.Run("tumbler")
    sp = scenes.tumbler(P, "TGS_Soft", grid=18, half_extent=4.0)
    dw = device.DeviceWorld.attach(dev, sp.world)
    dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    for step in range(90):
        dw.set_contact_order(ref.keys(step))
        sp.step(DT, 4, 2, True)
    c = dw.counters()
    assert c.constraintCount > 100, "the boxes must have reached the walls"
    assert np.array_equal(ref["positions"], _positions(P, sp))
    assert np.array_equal(ref["angles"], _angles(P, sp))
    rows = dw.download_contacts(int(ref["final_contacts"]) + 16)
    assert len(rows) == int(ref["final_contacts"])
    sp.destroy()


def _reference_field(R):
    sr = scenes.pyramid_field(R, "TGS_Soft", count=4, base_count=6)
    out = lockstep.pack_keys(lockstep.reference_steps(R, sr.world, 60, DT))
    out["positions"] = _positions(R, sr)
    sr.destroy()
    return out


def test_batched_worlds_field_reference_order(product, dev):
    """Config 5 in small: several independent pyramid worlds batched into one s2World (disconnected islands). Through the
    public API with the reference's order imposed: bit-identical to the reference stepping the same field; and the worlds
    really are independent (no pair ever forms between two of them)."""
    P = product
    ref = lockstep.Run("field")
    sp = scenes.pyramid_field(P, "TGS_Soft", count=4, base_count=6)
    dw = device.DeviceWorld.attach(dev, sp.world)
    dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    for step in range(60):
        dw.set_contact_order(ref.keys(step))
        sp.step(DT, 4, 2, True)
    assert np.array_equal(ref["positions"], _positions(P, sp))
    rows = dw.download_contacts(4096)
    per_world = 1 + 6 * 7 // 2
    assert np.array_equal(rows["bodyA"] // per_world, rows["bodyB"] // per_world), "a contact spans two worlds"
    sp.destroy()


# what tests/golden/make_lockstep.py records from the reference: name -> run(R) -> arrays
REFERENCE_RUNS = {_first_step_name(r, kw): _reference_first_step(r, kw) for r, kw in FIRST_STEP}
REFERENCE_RUNS.update(falling_boxes=_reference_falling_boxes, bulk_force=_reference_bulk_force, tumbler=_reference_tumbler,
                      field=_reference_field)
