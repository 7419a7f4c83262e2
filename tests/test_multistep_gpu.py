"""GPU: TIGHT multi-step parity of the free-running PRODUCTION path (public C API, colour schedule, persisted colours,
contact-table merges, feature-id impulse matching, CUDA-graph replay with the schedule skipped while the live constraint
set stands) — every step, every body, every manifold impulse, tolerance 0.

Gauss-Seidel is order sensitive, so the device cannot be compared with the free-running reference directly (SURVEY §7 H1).
Instead every step is checked on its own against the reference pipeline fed with the device's state and order:

    device state before the step  ->  loaded into the unmodified reference world (oracle/_ref, s2ref_load_body_state)
    reference stages 1-3          ->  s2ref_step_collide: pair update, narrow phase, impulse matching   (world.c:123-168)
    device                        ->  one s2World_Step through the public API
    solver stage                  ->  the plain-C oracle (pinned bit for bit to the reference, tests/test_oracle_cpu.py)
                                      replayed in the order the device reports for THIS step
    reference stage 4             ->  s2ref_step_finalize on the oracle's result                         (world.c:258-301)
    compare                       ->  bodies (position, rotation, velocities, origin) and manifold / joint impulses, bitwise

The reference world is advanced with the oracle's result (bodies and warm-start impulses), so its broad phase, contact pool
and manifold ids evolve exactly as if the reference had solved in the device's order. tests/golden/make_multistep.py runs
that pipeline and stores, for every step, a SHA-256 digest of what it produced (tests/golden/multistep/); the tests compute
the same digest from what the device produced and compare, step by step."""
import hashlib
import os

import numpy as np
import pytest

from solver2d_b200 import capi, device, scenes

pytestmark = pytest.mark.gpu
DT = 1.0 / 60.0
MULTISTEP_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "multistep")


@pytest.fixture(scope="module")
def product():
    return capi.Solver2D(device.LIB_PATH)


def step_digest(shape_a, shape_b, point_count, body_valid, bodies, normal, tangent, joint_valid, joints) -> bytes:
    """Digest of one step's compared results: the contact table (shape pairs in key order, point counts), every valid body
    (position, rotation, velocities, origin), the impulses of the live manifolds and of the valid joints."""
    h = hashlib.sha256()

    def put(a, dtype):
        h.update(np.ascontiguousarray(a, dtype=dtype).tobytes())
    for a in (shape_a, shape_b, point_count):
        put(a, np.int32)
    for name in ("position", "rot", "linearVelocity", "origin", "angularVelocity"):
        put(bodies[name][body_valid], np.float32)
    live = np.asarray(point_count) > 0
    put(normal[live], np.float32)
    put(tangent[live], np.float32)
    for name in ("impulse", "motorImpulse", "lowerImpulse", "upperImpulse"):
        put(joints[name][joint_valid], np.float32)
    return h.digest()


def device_step_digest(dw) -> bytes:
    c = dw.counters()
    got = dw.download_contacts(c.contactCount + 64)
    post = dw.download_all_bodies(c.bodyCapacity)
    joints = dw.download_joints(c.jointCapacity)
    return step_digest(got["shapeA"], got["shapeB"], got["pointCount"], (post["flags"] & 1) == 1, post,
                       got["points"]["normalImpulse"], got["points"]["tangentImpulse"], (joints["flags"] & 1) == 1, joints)


def start(dev, P, recipe, solver, kw, setup=None):
    """The product's scene, pushed to the device now (s2World_Step would do it): the first step is checked like any other."""
    sp = recipe(P, solver, **kw)
    dev.lib.s2World_Flush.restype = None
    dev.lib.s2World_Flush.argtypes = [capi.WorldId]
    dev.lib.s2World_Flush(sp.world)
    dw = device.DeviceWorld.attach(dev, sp.world)
    if setup is not None:
        setup(dw)
    return sp, dw


def _run(P, dev, name, min_replays=0):
    recipe, solver, steps, vel, pos, kw, setup = CASES[name]
    want = np.load(os.path.join(MULTISTEP_DIR, name + ".npy"))
    assert want.shape == (steps, 32)
    sp, dw = start(dev, P, recipe, solver, kw, setup)
    for step in range(steps):
        sp.step(DT, vel, pos, True)
        got = np.frombuffer(device_step_digest(dw), dtype=np.uint8)
        assert np.array_equal(got, want[step]), \
            f"{solver} step {step}: device != reference pipeline replayed in the device's order"
    c = dw.counters()
    assert c.graphReplays >= min_replays, f"the solver stage was replayed as a graph only {c.graphReplays} times"
    sp.destroy()
    return c


def _falling_boxes(lib, solver, **kw):
    sc = scenes.vertical_stack(lib, solver, count=5, columns=4)
    for k, bid in enumerate(sc.bodies[1:]):
        if k % 5 >= 3:
            lib.s2Body_SetLinearVelocity(bid, capi.Vec2(3.0 if (k // 5) % 2 == 0 else -3.0, 1.0))
    return sc


def _kinematic_platforms(lib, solver, **kw):
    import ctypes as C
    world = lib.create_world(solver)
    sc = scenes.Scene(lib, world, name="kinematic_platforms")
    h, base = 0.5, 16
    box = lib.s2MakeSquare(h)
    sd = scenes.default_shape_def()
    sd.density = 1.0
    for k in range(4):
        x0 = k * 30.0
        bd = scenes.default_body_def()
        bd.type = capi.KINEMATIC_BODY
        bd.position = capi.Vec2(x0, -1.0)
        bd.linearVelocity = capi.Vec2(0.6 if k % 2 == 0 else -0.4, 0.0)
        gid = lib.s2CreateBody(world, C.byref(bd))
        plat = lib.s2MakeBox(0.5 * base + 2.0, 1.0)
        lib.s2CreatePolygonShape(gid, C.byref(sd), C.byref(plat))
        sc.bodies.append(gid)
        bd = scenes.default_body_def()
        bd.type = capi.DYNAMIC_BODY
        for i in range(base):
            y = (2.0 * i + 1.0) * h
            for j in range(i, base):
                x = (i + 1.0) * h + 2.0 * (j - i) * h - h * base
                bd.position = capi.Vec2(x0 + x, y)
                bid = lib.s2CreateBody(world, C.byref(bd))
                lib.s2CreatePolygonShape(bid, C.byref(sd), C.byref(box))
                sc.bodies.append(bid)
    return sc


def _force_regions(dw):
    dw.set_regions(2)


VARIANTS = ["PGS", "PGS_NGS", "PGS_NGS_Block", "PGS_Soft", "SoftStep", "TGS_NGS", "XPBD"]
# name -> (recipe, solver, steps, velocity iterations, relax iterations, recipe kwargs, device setup)
CASES = {
    "config1": (scenes.pyramid, "TGS_Soft", 120, 4, 2, dict(base_count=10), None),
    "pyramid_5k": (scenes.pyramid, "TGS_Soft", 60, 4, 2, dict(base_count=100), None),
    "joints_and_contacts": (scenes.joint_contact_stress, "TGS_Soft", 90, 4, 2, dict(bridges=3, planks=24, grid=9), None),
    "falling_boxes": (_falling_boxes, "TGS_Soft", 120, 4, 2, {}, None),
    "kinematic_platforms": (_kinematic_platforms, "TGS_Soft", 40, 4, 2, {}, _force_regions),
}
CASES.update({f"variant_{s.lower()}": (scenes.pyramid, s, 40, 4, 2, dict(base_count=20), None) for s in VARIANTS})


def test_config1_every_step_bit_exact(product, dev):
    """BASELINE config 1 (Pyramid, 55 boxes, TGS_Soft, 4 sub-steps), 120 free-running steps."""
    c = _run(product, dev, "config1", min_replays=60)
    assert c.constraintCount > 100


def test_pyramid_5k_every_step_bit_exact(product, dev):
    """5 050 boxes / ~15 000 contact constraints, 60 free-running steps: several thread blocks, contact-table changes while
    the pile settles, graph replays with the schedule skipped in between."""
    c = _run(product, dev, "pyramid_5k")
    assert c.constraintCount > 14000


def test_joints_and_contacts_every_step_bit_exact(product, dev):
    """Bridges (revolute chains) with boxes dropped on them: joints and contacts in one colouring, contacts appearing and
    disappearing every few steps."""
    c = _run(product, dev, "joints_and_contacts")
    assert c.jointCount == 75


@pytest.mark.parametrize("solver", VARIANTS)
def test_variants_every_step_bit_exact(product, dev, solver):
    c = _run(product, dev, f"variant_{solver.lower()}")
    assert c.constraintCount > 300


def test_falling_boxes_every_step_bit_exact(product, dev):
    """Boxes thrown sideways: proxies leave their fat AABBs, pairs are created and destroyed, manifolds gain and lose
    points — the schedule is rebuilt on exactly the steps the device flags."""
    c = _run(product, dev, "falling_boxes")
    assert c.pairPassCount > 5


def test_kinematic_platforms_under_regions_every_step_bit_exact(product, dev):
    """Piles standing on KINEMATIC platforms that slide sideways, region-local schedule forced. A kinematic body conflicts
    with nothing (no constraint moves it) but its pose changes every sub-step, integrated by the block that owns it: a
    constraint that reads it from another block's region-local phase would race with that pass. Such constraints have to
    run in the device-wide steps (s2bClassifyItemsKernel)."""
    c = _run(product, dev, "kinematic_platforms")
    assert c.regionCount >= 3 and c.cutCount >= 40
