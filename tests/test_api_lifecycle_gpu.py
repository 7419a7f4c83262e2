"""GPU: the object model behind the public API against the unmodified reference — bodies, shapes and joints created and
destroyed mid-run (slot and proxy-id reuse), state edits, impulses, mouse-joint targets, s2World_QueryAABB, s2Shape_TestPoint
and s2World_Draw. The same scripted session is played on both libraries; with the reference's Gauss-Seidel order imposed
(validation schedule) every body must stay bit-identical after every phase."""
import ctypes as C

import numpy as np
import pytest

import lockstep
from solver2d_b200 import capi, device, scenes
from solver2d_b200.capi import Capsule, Circle, Vec2, default_body_def, default_mouse_def, default_revolute_def, default_shape_def

pytestmark = pytest.mark.gpu
DT = 1.0 / 60.0


class Color(C.Structure):
    _fields_ = [("r", C.c_float), ("g", C.c_float), ("b", C.c_float), ("a", C.c_float)]


class Box(C.Structure):
    _fields_ = [("lowerBound", Vec2), ("upperBound", Vec2)]


VP = C.POINTER(Vec2)
DRAW_SIGS = [
    ("DrawPolygon", C.CFUNCTYPE(None, VP, C.c_int, Color, C.c_void_p)),
    ("DrawSolidPolygon", C.CFUNCTYPE(None, VP, C.c_int, Color, C.c_void_p)),
    ("DrawRoundedPolygon", C.CFUNCTYPE(None, VP, C.c_int, C.c_float, Color, Color, C.c_void_p)),
    ("DrawCircle", C.CFUNCTYPE(None, Vec2, C.c_float, Color, C.c_void_p)),
    ("DrawSolidCircle", C.CFUNCTYPE(None, Vec2, C.c_float, Vec2, Color, C.c_void_p)),
    ("DrawCapsule", C.CFUNCTYPE(None, Vec2, Vec2, C.c_float, Color, C.c_void_p)),
    ("DrawSolidCapsule", C.CFUNCTYPE(None, Vec2, Vec2, C.c_float, Color, C.c_void_p)),
    ("DrawSegment", C.CFUNCTYPE(None, Vec2, Vec2, Color, C.c_void_p)),
    ("DrawTransform", C.CFUNCTYPE(None, capi.Transform, C.c_void_p)),
    ("DrawPoint", C.CFUNCTYPE(None, Vec2, C.c_float, Color, C.c_void_p)),
    ("DrawString", C.CFUNCTYPE(None, Vec2, C.c_char_p, C.c_void_p)),
]


class DebugDraw(C.Structure):
    _fields_ = [(n, t) for n, t in DRAW_SIGS] + [("dynamicBodyColor", Color)] + \
        [(n, C.c_bool) for n in ("drawShapes", "drawJoints", "drawAABBs", "drawMass", "drawContactPoints", "drawContactNormals",
                                 "drawContactImpulses", "drawFrictionImpulses")] + [("context", C.c_void_p)]


def _draw_log(lib, world):
    """Play s2World_Draw into a list of (primitive, rounded numbers)."""
    log = []

    def rec(name):
        def f(*args):
            vals = []
            for a in args[:-1]:
                if isinstance(a, Vec2):
                    vals += [a.x, a.y]
                elif isinstance(a, (float, int)):
                    vals.append(float(a))
                elif isinstance(a, capi.Transform):
                    vals += [a.p.x, a.p.y, a.q.s, a.q.c]
                elif isinstance(a, Color):
                    vals += [a.r, a.g, a.b]
                elif hasattr(a, "contents"):
                    n = args[1]
                    for k in range(n):
                        vals += [a[k].x, a[k].y]
            log.append((name, tuple(np.float32(v).item() for v in vals)))
        return f

    dd = DebugDraw()
    keep = []
    for name, sig in DRAW_SIGS:
        cb = sig(rec(name))
        keep.append(cb)
        setattr(dd, name, cb)
    dd.dynamicBodyColor = Color(0.5, 0.6, 0.7, 1.0)
    dd.drawShapes = True
    dd.drawJoints = True
    dd.drawAABBs = True
    dd.drawMass = True
    lib.lib.s2World_Draw.argtypes = [capi.WorldId, C.POINTER(DebugDraw)]
    lib.lib.s2World_Draw.restype = None
    lib.lib.s2World_Draw(world, C.byref(dd))
    return log


QUERY_CB = C.CFUNCTYPE(C.c_bool, capi.ShapeId, C.c_void_p)


def _query(lib, world, lo, hi):
    found = []

    def cb(shape_id, ctx):
        found.append((shape_id.index, shape_id.revision))
        return True
    fn = QUERY_CB(cb)
    lib.lib.s2World_QueryAABB.argtypes = [capi.WorldId, Box, QUERY_CB, C.c_void_p]
    lib.lib.s2World_QueryAABB.restype = None
    lib.lib.s2World_QueryAABB(world, Box(Vec2(*lo), Vec2(*hi)), fn, None)
    return sorted(found)


class Session:
    """One library's side of the scripted session."""

    def __init__(self, lib, solver):
        self.lib = lib
        self.world = lib.create_world(solver)
        self.bodies = {}
        self.shapes = {}
        self.joints = {}

    def body(self, name, kind, pos, shape, angle=0.0):
        lib = self.lib
        bd = default_body_def()
        bd.type = kind
        bd.position = Vec2(*pos)
        bd.angle = angle
        bid = lib.s2CreateBody(self.world, C.byref(bd))
        sd = default_shape_def()
        if shape[0] == "box":
            poly = lib.s2MakeBox(shape[1], shape[2])
            sid = lib.s2CreatePolygonShape(bid, C.byref(sd), C.byref(poly))
        elif shape[0] == "circle":
            c = Circle(Vec2(0.0, 0.0), shape[1])
            sid = lib.s2CreateCircleShape(bid, C.byref(sd), C.byref(c))
        else:
            cap = Capsule(Vec2(-shape[1], 0.0), Vec2(shape[1], 0.0), shape[2])
            sid = lib.s2CreateCapsuleShape(bid, C.byref(sd), C.byref(cap))
        self.bodies[name] = bid
        self.shapes[name] = sid
        return bid

    def revolute(self, name, a, b, pivot, **kw):
        lib = self.lib
        jd = default_revolute_def()
        jd.bodyIdA = self.bodies[a]
        jd.bodyIdB = self.bodies[b]
        jd.localAnchorA = lib.s2Body_GetLocalPoint(self.bodies[a], Vec2(*pivot))
        jd.localAnchorB = lib.s2Body_GetLocalPoint(self.bodies[b], Vec2(*pivot))
        for k, v in kw.items():
            setattr(jd, k, v)
        self.joints[name] = lib.s2CreateRevoluteJoint(self.world, C.byref(jd))

    def mouse(self, name, a, b, target):
        md = default_mouse_def()
        md.bodyIdA = self.bodies[a]
        md.bodyIdB = self.bodies[b]
        md.target = Vec2(*target)
        md.hertz = 4.0
        md.dampingRatio = 0.8
        self.joints[name] = self.lib.s2CreateMouseJoint(self.world, C.byref(md))

    def state(self):
        names = sorted(self.bodies)
        return np.array([tuple(self.lib.s2Body_GetPosition(self.bodies[n])) + (self.lib.s2Body_GetAngle(self.bodies[n]),)
                         for n in names], dtype=np.float64)


def _script(s: Session, phase: int):
    """The edits of each phase (identical calls on both libraries)."""
    L = s.lib
    if phase == 0:
        s.body("ground", capi.STATIC_BODY, (0.0, -1.0), ("box", 30.0, 1.0))
        for i in range(6):
            for j in range(5):
                kind = ("box", 0.5, 0.4) if (i + j) % 3 == 0 else (("circle", 0.45) if (i + j) % 3 == 1 else ("capsule", 0.4, 0.25))
                s.body(f"b{i}_{j}", capi.DYNAMIC_BODY, (-6.0 + 2.2 * j + 0.3 * (i % 2), 0.6 + 1.3 * i), kind, angle=0.1 * (i - j))
        s.body("arm", capi.DYNAMIC_BODY, (8.0, 4.0), ("box", 1.5, 0.2))
        s.revolute("hinge", "ground", "arm", (6.5, 4.0), enableLimit=True, lowerAngle=-0.6, upperAngle=0.9, enableMotor=True,
                   motorSpeed=1.0, maxMotorTorque=50.0)
        s.body("kin", capi.KINEMATIC_BODY, (-10.0, 3.0), ("box", 1.0, 0.3))
        L.s2Body_SetLinearVelocity(s.bodies["kin"], Vec2(1.5, 0.0))
    elif phase == 1:
        # destroy bodies in the middle of the pile (their contacts, shapes and proxies go), then reuse the slots
        for n in ("b1_2", "b2_2", "b3_1"):
            L.s2DestroyBody(s.bodies.pop(n))
            s.shapes.pop(n)
        s.body("new0", capi.DYNAMIC_BODY, (-1.5, 9.0), ("box", 0.6, 0.6))
        s.body("new1", capi.DYNAMIC_BODY, (1.0, 10.0), ("circle", 0.5))
        s.mouse("drag", "ground", "b5_4", (4.0, 9.0))
        L.s2Body_ApplyLinearImpulse(s.bodies["b4_0"], Vec2(3.0, 1.0), L.s2Body_GetPosition(s.bodies["b4_0"]))
    elif phase == 2:
        L.s2MouseJoint_SetTarget(s.joints["drag"], Vec2(-3.0, 8.0))
        L.s2RevoluteJoint_SetMotorSpeed(s.joints["hinge"], -2.0)
        L.s2Body_SetAngularVelocity(s.bodies["new0"], 3.0)
        s.body("late", capi.DYNAMIC_BODY, (8.0, 6.0), ("capsule", 0.5, 0.2))
        s.revolute("link", "arm", "late", (9.5, 4.0), collideConnected=False)
    elif phase == 3:
        L.s2DestroyJoint(s.joints.pop("drag"))
        L.s2RevoluteJoint_EnableLimit(s.joints["hinge"], False)
        L.s2DestroyJoint(s.joints.pop("link"))  # joints must go before their bodies (reference src/body.c:82-83)
        L.s2DestroyBody(s.bodies.pop("late"))
        s.shapes.pop("late")
        s.body("again", capi.DYNAMIC_BODY, (0.0, 12.0), ("box", 0.4, 0.4))


QUERY_BOXES = (((-7.0, -0.5), (0.0, 4.0)), ((-30.0, -3.0), (30.0, 30.0)), ((7.0, 3.0), (10.0, 7.0)))
TEST_POINTS = ((0.1, 0.5), (-3.0, 1.0), (8.0, 4.0))


def _draw_entries(log) -> np.ndarray:
    """A draw log as sorted strings (primitive and the exact bits of its numbers)."""
    return np.array(sorted(name + ":" + ",".join(float(v).hex() for v in vals) for name, vals in log))


def _session_readback(lib, s: Session, phase: int) -> dict:
    """What the scripted-session test compares after a phase."""
    out = {f"p{phase}_state": s.state(), f"p{phase}_contacts": np.array(lib.s2World_GetStatistics(s.world).contactCount)}
    for k, (lo, hi) in enumerate(QUERY_BOXES):
        out[f"p{phase}_query{k}"] = np.array(_query(lib, s.world, lo, hi), dtype=np.int64).reshape(-1, 2)
    out[f"p{phase}_test_point"] = np.array([[lib.s2Shape_TestPoint(s.shapes[name], Vec2(*pt)) for pt in TEST_POINTS]
                                            for name in sorted(s.shapes)[:12]], dtype=bool)
    out[f"p{phase}_draw"] = _draw_entries(_draw_log(lib, s.world))
    return out


def _reference_session(solver):
    def run(R):
        sr = Session(R, solver)
        out = {}
        for phase in range(4):
            _script(sr, phase)
            out.update(lockstep.pack_keys(lockstep.reference_steps(R, sr.world, 45, DT), prefix=f"p{phase}_"))
            out.update(_session_readback(R, sr, phase))
        R.s2DestroyWorld(sr.world)
        return out
    return run


@pytest.mark.parametrize("solver", ["TGS_Soft", "PGS_NGS_Block"])
def test_scripted_session_matches_reference(dev, solver):
    ref = lockstep.Run(f"session_{solver.lower()}")
    P = capi.Solver2D(device.LIB_PATH)
    sp = Session(P, solver)
    dw = None
    for phase in range(4):
        _script(sp, phase)
        if dw is None:
            dw = device.DeviceWorld.attach(dev, sp.world)
            dw.set_schedule(device.SCHEDULE_WAVEFRONT)
        for step in range(45):
            dw.set_contact_order(ref.keys(step, prefix=f"p{phase}_"))
            P.step(sp.world, DT, 4, 2, True)
        got = _session_readback(P, sp, phase)
        a, b = ref[f"p{phase}_state"], got[f"p{phase}_state"]
        assert np.array_equal(a, b), f"phase {phase}: bodies differ, max {np.abs(a - b).max()}"
        assert int(ref[f"p{phase}_contacts"]) == int(got[f"p{phase}_contacts"])
        # queries and debug draw read the same state back
        for k in range(len(QUERY_BOXES)):
            assert np.array_equal(ref[f"p{phase}_query{k}"], got[f"p{phase}_query{k}"])
        assert np.array_equal(ref[f"p{phase}_test_point"], got[f"p{phase}_test_point"])
        dr, dp = ref[f"p{phase}_draw"], got[f"p{phase}_draw"]
        assert len(dr) == len(dp) and len(dr) > 20
        assert np.array_equal(dr, dp), "s2World_Draw output differs"
    P.s2DestroyWorld(sp.world)


def _edge_case_session(lib):
    s = Session(lib, "TGS_Soft")
    s.body("ground", capi.STATIC_BODY, (0.0, -1.0), ("box", 40.0, 1.0))
    for i in range(8):
        s.body(f"a{i}", capi.DYNAMIC_BODY, (-3.0 + 0.9 * i, 0.6 + 0.05 * i), ("box", 0.4, 0.4))
    return s


def _grow(s):
    for k in range(300):
        s.body(f"g{k}", capi.DYNAMIC_BODY, (-15.0 + 0.11 * k, 3.0 + 1.1 * (k % 7)), ("circle", 0.3) if k % 2 else ("box", 0.3, 0.3))


# (steps, dt, velocity iterations, relax iterations) of each run; the pools grow before the last one
EDGE_RUNS = ((20, DT, 4, 2), (3, 0.0, 4, 2), (10, DT, 4, 0), (40, DT, 4, 2))


def _reference_edge_cases(R):
    sr = _edge_case_session(R)
    out = {}
    for k, (steps, dt, vel, pos) in enumerate(EDGE_RUNS):
        if k == len(EDGE_RUNS) - 1:
            _grow(sr)
        out.update(lockstep.pack_keys(lockstep.reference_steps(R, sr.world, steps, dt, vel, pos), prefix=f"r{k}_"))
        out[f"r{k}_state"] = sr.state()
    out["body_count"] = np.array(R.s2World_GetStatistics(sr.world).bodyCount)
    R.s2DestroyWorld(sr.world)
    return out


def test_edge_cases_match_reference(dev):
    """Empty world, a paused step (dt = 0: reference src/world.c:176-183 still runs the solver with inv_dt = 0), growth of
    every pool after the world has been stepped (device columns re-allocated, solver graph re-captured), and a step with
    zero relax iterations — all against the reference, reference order imposed."""
    ref = lockstep.Run("edge_cases")
    P = capi.Solver2D(device.LIB_PATH)
    # 1. an empty world steps (and reads back) without complaint
    we = P.create_world("TGS_Soft")
    P.step(we, DT, 4, 2, True)
    assert P.s2World_GetStatistics(we).bodyCount == 0
    P.s2DestroyWorld(we)

    sp = _edge_case_session(P)
    dw = device.DeviceWorld.attach(dev, sp.world)
    dw.set_schedule(device.SCHEDULE_WAVEFRONT)
    # 20 steps, 3 paused, 10 without relax iterations, then (2.) pools grow well past their initial capacity after stepping
    for k, (steps, dt, vel, pos) in enumerate(EDGE_RUNS):
        if k == len(EDGE_RUNS) - 1:
            _grow(sp)
        for step in range(steps):
            dw.set_contact_order(ref.keys(step, prefix=f"r{k}_"))
            P.step(sp.world, dt, vel, pos, True)
        a, b = ref[f"r{k}_state"], sp.state()
        assert np.array_equal(a, b), f"run {k}: max {np.abs(a - b).max()}"
    assert P.s2World_GetStatistics(sp.world).bodyCount == int(ref["body_count"]) == 309
    P.s2DestroyWorld(sp.world)


def _recreate_script(lib):
    """Rest a stack, then replace the second box of the middle column by a new one at the same place, at rest; returns
    the contact count and the new box's height over the next 30 steps."""
    sc = scenes.vertical_stack(lib, "TGS_Soft", count=4, columns=3)
    for _ in range(40):
        sc.step(DT, 4, 2, True)
    victim = sc.bodies[1 + 4 + 1]
    pos = lib.s2Body_GetPosition(victim)
    lib.s2DestroyBody(victim)
    bd = default_body_def()
    bd.type = capi.DYNAMIC_BODY
    bd.position = Vec2(pos.x, pos.y)
    bid = lib.s2CreateBody(sc.world, C.byref(bd))
    sd = default_shape_def()
    box = lib.s2MakeSquare(0.5)
    lib.s2CreatePolygonShape(bid, C.byref(sd), C.byref(box))
    sc.bodies[1 + 4 + 1] = bid
    counts, ys = [], []
    for _ in range(30):
        sc.step(DT, 4, 2, True)
        counts.append(lib.s2World_GetStatistics(sc.world).contactCount)
        ys.append(lib.s2Body_GetPosition(bid).y)
    sc.destroy()
    return counts, ys


def _reference_recreated(R):
    counts, ys = _recreate_script(R)
    return dict(counts=np.array(counts, dtype=np.int64), ys=np.array(ys, dtype=np.float64))


def test_body_recreated_in_the_same_slot_at_the_same_place(dev):
    """A resting box is destroyed and a new one is created where it stood: the new body re-uses the body and shape slots
    (and the proxy id) of the old one, so the contact table still holds the OLD shape's pairs under the same keys when the
    next pair pass runs. The pass has to drop those and report the pairs of the new shape in the same pass (the reference
    removes the keys on destroy and re-creates the contacts on its next update); otherwise the new box has no contacts
    until it leaves its fat AABB and sinks into its neighbours."""
    ref = lockstep.Run("body_recreated")
    cr, yr = ref["counts"].tolist(), ref["ys"].tolist()
    cp, yp = _recreate_script(capi.Solver2D(device.LIB_PATH))
    assert cp == cr, f"contact counts after re-creating the body: device {cp[:6]}... reference {cr[:6]}..."
    assert max(abs(a - b) for a, b in zip(yr, yp)) < 2e-3, "the re-created box does not rest where the reference's does"
    assert min(yp) > yr[0] - 0.02, "the re-created box sank into its neighbour"


# what tests/golden/make_lockstep.py records from the reference: name -> run(R) -> arrays
REFERENCE_RUNS = {f"session_{s.lower()}": _reference_session(s) for s in ("TGS_Soft", "PGS_NGS_Block")}
REFERENCE_RUNS.update(edge_cases=_reference_edge_cases, body_recreated=_reference_recreated)
