"""CPU: the product library loads without a GPU, exports every symbol the headers declare, and its host-side geometry and
narrow-phase code (csrc/shared/s2_collide.h — the SAME source the CUDA narrow-phase kernel compiles) is bit-identical to
the unmodified reference on seeded inputs (its outputs recorded in tests/golden/host_vectors_ref.npz by
tests/golden/make_host_vectors.py). No world is created here: s2CreateWorld needs a CUDA device by design."""
import ctypes as C
import re

import numpy as np
import pytest

import os

from solver2d_b200 import capi, device

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def product():
    return capi.Solver2D(device.LIB_PATH)


def test_library_exports_every_declared_symbol(product):
    assert product.missing == []
    lib = C.CDLL(device.LIB_PATH)
    header = open(os.path.join(ROOT, "include", "s2b_device.h")).read()
    declared = re.findall(r"^S2B_API [^;(]*?(s2b_\w+)\(", header, flags=re.M)
    assert len(declared) >= 35
    for name in declared + device.ABI_SYMBOLS:
        assert hasattr(lib, name), name
    ext = open(os.path.join(ROOT, "include", "solver2d_b200.h")).read()
    for name in re.findall(r"^S2B_API [^;(]*?(s2World_\w+)\(", ext, flags=re.M):
        assert hasattr(lib, name), name
    for variant in ("Jacobi", "PGS", "PGS_NGS", "PGS_NGS_Block", "PGS_Soft", "TGS_Soft", "TGS_Sticky", "TGS_NGS", "XPBD",
                    "SoftStep"):
        assert hasattr(lib, f"s2Solve_{variant}")


def test_row_struct_sizes_match_numpy_mirrors():
    lib = C.CDLL(device.LIB_PATH)
    out = (C.c_int32 * 6)()
    lib.s2b_abi_sizes(out)
    assert list(out)[:4] == [device.BODY_ROW.itemsize, device.SHAPE_ROW.itemsize, device.JOINT_ROW.itemsize,
                             device.CONTACT_ROW.itemsize]
    assert out[4] == C.sizeof(device.StepContext) and out[5] == C.sizeof(device.Counters)


GOLDEN = os.path.join(ROOT, "tests", "golden", "host_vectors_ref.npz")


def _poly(p) -> np.ndarray:
    """A polygon as the compared fields: count, radius, then its vertices and normals (unused slots zero)."""
    out = np.zeros(2 + 32, dtype=np.float32)
    out[0], out[1] = p.count, p.radius
    for i in range(p.count):
        out[2 + 2 * i:4 + 2 * i] = (p.vertices[i].x, p.vertices[i].y)
        out[18 + 2 * i:20 + 2 * i] = (p.normals[i].x, p.normals[i].y)
    return out


def _raw(struct) -> np.ndarray:
    return np.frombuffer(bytes(struct), dtype=np.uint8).copy()


def box_with_radius(L, hx, hy):
    """What s2MakeRoundedBox(hx, hy, 0.1) stands for: a box polygon with a 0.1 radius."""
    p = L.s2MakeBox(hx, hy)
    p.radius = 0.1
    return p


def polygon_factory_outputs(L, rounded_box=None) -> np.ndarray:
    """Box / offset box / rounded box / capsule factories, their mass data and a polygon AABB on seeded inputs, as bytes.
    The rounded box comes from L's s2MakeRoundedBox unless `rounded_box(L, hx, hy)` builds it."""
    rng = np.random.default_rng(7)
    out = []
    for _ in range(50):
        hx, hy = rng.uniform(0.05, 3.0, 2)
        ang = rng.uniform(-3, 3)
        c = capi.Vec2(*rng.uniform(-2, 2, 2))
        out.append(_poly(L.s2MakeBox(hx, hy)).view(np.uint8))
        a = L.s2MakeOffsetBox(hx, hy, c, ang)
        out.append(_poly(a).view(np.uint8))
        for dens in (1.0, 20.0):
            out.append(_raw(L.s2ComputePolygonMass(C.byref(a), dens)))
        rb = rounded_box(L, hx, hy) if rounded_box is not None else L.s2MakeRoundedBox(hx, hy, 0.1)
        out.append(_raw(L.s2ComputePolygonMass(C.byref(rb), 2.0)))
        p1, p2 = capi.Vec2(*rng.uniform(-1, 1, 2)), capi.Vec2(*rng.uniform(1.5, 3, 2))
        out.append(_poly(L.s2MakeCapsule(p1, p2, 0.3)).view(np.uint8))
        cap = capi.Capsule(p1, p2, 0.3)
        out.append(_raw(L.s2ComputeCapsuleMass(C.byref(cap), 1.5)))
        xf = capi.Transform(c, capi.Rot(np.float32(np.sin(ang)), np.float32(np.cos(ang))))
        out.append(_raw(L.s2ComputePolygonAABB(C.byref(a), xf)))
    return np.concatenate(out)


def hull_outputs(L) -> np.ndarray:
    """Quickhull on seeded point sets (welded / collinear inputs among them) and the polygon made from each hull."""
    rng = np.random.default_rng(11)
    out = []
    for trial in range(200):
        n = int(rng.integers(3, 9))
        pts = (capi.Vec2 * n)(*[capi.Vec2(*rng.uniform(-1.5, 1.5, 2)) for _ in range(n)])
        if trial % 5 == 0:  # welded / collinear inputs
            pts[1] = capi.Vec2(pts[0].x + 0.001, pts[0].y)
        h = L.s2ComputeHull(pts, n)
        row = np.zeros(1 + 16, dtype=np.float32)
        row[0] = h.count
        for i in range(h.count):
            row[1 + 2 * i:3 + 2 * i] = (h.points[i].x, h.points[i].y)
        out.append(row)
        out.append(_poly(L.s2MakePolygon(C.byref(h))) if h.count >= 3 else np.zeros(34, np.float32))
    return np.concatenate(out)


def _manifold(m) -> np.ndarray:
    """pointCount, then (normal, per point: anchors, separation, id) when it has points; the compared fields only."""
    out = np.zeros(3 + 2 * 6, dtype=np.float32)
    out[0] = m.pointCount
    if m.pointCount:
        out[1:3] = (m.normal.x, m.normal.y)
        for i in range(m.pointCount):
            p = m.points[i]
            out[3 + 6 * i:8 + 6 * i] = (p.localAnchorA.x, p.localAnchorA.y, p.localAnchorB.x, p.localAnchorB.y, p.separation)
            out[8 + 6 * i:9 + 6 * i] = np.array([p.id], dtype=np.int32).view(np.float32)
    return out


def manifold_outputs(L) -> np.ndarray:
    """All nine shape-pair manifold functions (reference src/contact.c:139-154) on random near-contact configurations,
    with the GJK cache carried over several perturbed calls as a persistent contact does: (trials, 3, 9 + 5, 15)."""
    rng = np.random.default_rng(2024)

    def xf(x, y, ang):
        return capi.Transform(capi.Vec2(x, y), capi.Rot(np.float32(np.sin(ang)), np.float32(np.cos(ang))))

    out = np.zeros((400, 3, 14, 15), dtype=np.float32)
    for trial in range(400):
        boxA = L.s2MakeBox(*rng.uniform(0.3, 1.2, 2))
        pts = (capi.Vec2 * 6)(*[capi.Vec2(*rng.uniform(-0.8, 0.8, 2)) for _ in range(6)])
        hull = L.s2ComputeHull(pts, 6)
        polyB = L.s2MakePolygon(C.byref(hull)) if hull.count >= 3 else L.s2MakeBox(0.5, 0.4)
        polyB.radius = 0.05 if trial % 3 == 0 else 0.0
        circ = capi.Circle(capi.Vec2(*rng.uniform(-0.2, 0.2, 2)), float(rng.uniform(0.2, 0.6)))
        circ2 = capi.Circle(capi.Vec2(0.0, 0.0), float(rng.uniform(0.2, 0.6)))
        cap = capi.Capsule(capi.Vec2(-0.5, 0.0), capi.Vec2(0.5, float(rng.uniform(-0.2, 0.2))), float(rng.uniform(0.1, 0.4)))
        cap2 = capi.Capsule(capi.Vec2(0.0, -0.4), capi.Vec2(0.1, 0.5), 0.25)
        seg = capi.Segment(capi.Vec2(-1.0, 0.0), capi.Vec2(1.0, float(rng.uniform(-0.3, 0.3))))
        d = rng.uniform(0.6, 1.9)
        th = rng.uniform(0, 2 * np.pi)
        cache = [capi.DistanceCache() for _ in range(5)]
        for it in range(3):  # persistent cache across slightly moved poses
            A = xf(*rng.uniform(-0.01, 0.01, 2), rng.uniform(-0.02, 0.02) + 0.3 * trial)
            B = xf(d * np.cos(th) + rng.uniform(-0.01, 0.01), d * np.sin(th) + rng.uniform(-0.01, 0.01), rng.uniform(-3, 3) if it == 0 else 0.1 * it)
            ms = [
                L.s2CollideCircles(C.byref(circ), A, C.byref(circ2), B),
                L.s2CollideCapsuleAndCircle(C.byref(cap), A, C.byref(circ), B),
                L.s2CollideSegmentAndCircle(C.byref(seg), A, C.byref(circ), B),
                L.s2CollidePolygonAndCircle(C.byref(boxA), A, C.byref(circ), B),
                L.s2CollidePolygons(C.byref(boxA), A, C.byref(polyB), B, C.byref(cache[0])),
                L.s2CollideCapsules(C.byref(cap), A, C.byref(cap2), B, C.byref(cache[1])),
                L.s2CollidePolygonAndCapsule(C.byref(boxA), A, C.byref(cap), B, C.byref(cache[2])),
                L.s2CollideSegmentAndCapsule(C.byref(seg), A, C.byref(cap), B, C.byref(cache[3])),
                L.s2CollideSegmentAndPolygon(C.byref(seg), A, C.byref(polyB), B, C.byref(cache[4])),
            ]
            for k, m in enumerate(ms):
                out[trial, it, k] = _manifold(m)
            for k, cc in enumerate(cache):
                out[trial, it, 9 + k, 0] = cc.count
                out[trial, it, 9 + k, 1:4] = list(bytes(cc.indexA))[:3]
                out[trial, it, 9 + k, 4:7] = list(bytes(cc.indexB))[:3]
    return out


def _golden(key):
    return np.load(GOLDEN)[key]


def test_polygon_factories_and_mass_match_reference(product):
    want = _golden("polygon_factories")
    got = polygon_factory_outputs(product)
    assert got.shape == want.shape and np.array_equal(got, want)


def test_hull_matches_reference(product):
    want = _golden("hull")
    got = hull_outputs(product)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_manifold_functions_match_reference_bitwise(product):
    want = _golden("manifolds")
    got = manifold_outputs(product)
    bad = np.nonzero((got.view(np.uint32) != want.view(np.uint32)).any(axis=-1))
    assert len(bad[0]) == 0, f"first mismatch: trial {bad[0][0]} iter {bad[1][0]} function/cache {bad[2][0]}"
    assert (want[:, :, :9, 0] > 0).sum() > 1500  # the sweep actually produced contacts


def _atan2_inputs(n, seed):
    rng = np.random.default_rng(seed)
    # (sin, cos)-like pairs as s2RelativeAngle produces them, raw bit patterns, and the special values
    a = rng.uniform(-np.pi, np.pi, n)
    y = [np.sin(a).astype(np.float32), rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32).view(np.float32),
         np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, 1e-40, -1e-40, 3e38, 0.4375, 0.6875, 1.1875, 2.4375] * 13, np.float32)]
    x = [np.cos(a).astype(np.float32), rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32).view(np.float32),
         np.repeat(np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, 1e-40, -1e-40, 3e38, 0.4375, 0.6875, 1.1875, 2.4375],
                            np.float32), 13)]
    return np.concatenate(y), np.concatenate(x)


def test_device_atan2_restatement_equals_libm_on_host():
    """include/solver2d/atan2_f32.h (what the kernels call) against the C library atan2f the reference is linked with."""
    import ctypes.util
    lib = C.CDLL(device.LIB_PATH)
    lib.s2Atan2Device.restype = C.c_float
    lib.s2Atan2Device.argtypes = [C.c_float, C.c_float]
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.atan2f.restype = C.c_float
    libm.atan2f.argtypes = [C.c_float, C.c_float]
    y, x = _atan2_inputs(150000, 11)
    mine = np.array([lib.s2Atan2Device(float(a), float(b)) for a, b in zip(y, x)], np.float32)
    want = np.array([libm.atan2f(float(a), float(b)) for a, b in zip(y, x)], np.float32)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(mine), nan)
    assert np.array_equal(mine[~nan].view(np.uint32), want[~nan].view(np.uint32))
