"""GPU: the pair pass against brute force. The contact table's shape pairs are compared with every overlapping pair of fat
AABBs that the pair rules allow, computed with numpy from the boxes the device reports. The scenes use only what these
rules cover: default filters, no joints between shapes, one shape per body, static, kinematic and dynamic bodies. A pair
is allowed when its shapes are on different bodies and at least one of the bodies is dynamic.

The leaf counts 1, 2, 15, 16, 17 and 257 sit on the boundaries of the 16-wide hierarchy; the bar scenes put more
scene-sized leaves into the world than the large-leaf list holds (64), so some stay in the hierarchy and some do not."""
import ctypes as C

import numpy as np
import pytest

from solver2d_b200 import capi, device, scenes

pytestmark = pytest.mark.gpu
DT = 1.0 / 60.0


class Built:
    def __init__(self, lib):
        self.lib = lib
        self.world = lib.create_world("TGS_Soft")
        self.types = {}  # shape slot -> body type
        self.bodies = []

    def add(self, body_type, x, y, poly, velocity=(0.0, 0.0), angle=0.0):
        bd = scenes.default_body_def()
        bd.type = body_type
        bd.position = capi.Vec2(x, y)
        bd.angle = angle
        bd.linearVelocity = capi.Vec2(*velocity)
        bid = self.lib.s2CreateBody(self.world, C.byref(bd))
        sd = scenes.default_shape_def()
        sd.density = 1.0
        sid = self.lib.s2CreatePolygonShape(bid, C.byref(sd), C.byref(poly))
        self.types[sid.index] = body_type
        self.bodies.append(bid)

    def step(self):
        self.lib.s2World_Step(self.world, DT, 4, 2, True)

    def destroy(self):
        self.lib.s2DestroyWorld(self.world)


def _attach(dev, b):
    b.lib.lib.s2World_Flush.restype = None
    b.lib.lib.s2World_Flush.argtypes = [capi.WorldId]
    b.lib.lib.s2World_Flush(b.world)
    return device.DeviceWorld.attach(dev, b.world)


def _dynamic_mask(b, cap):
    dyn = np.zeros(cap, dtype=bool)
    for slot, t in b.types.items():
        dyn[slot] = t == capi.DYNAMIC_BODY
    return dyn


def _overlapping(fat, valid):
    """Keys (lo << 32 | hi) of every pair of valid shapes whose fat boxes overlap (closed test, as s2AABB_Overlaps)."""
    ids = np.nonzero(valid)[0]
    box = fat[ids]
    order = np.argsort(box[:, 0], kind="stable")
    box, ids = box[order], ids[order]
    n = len(ids)
    hi = np.searchsorted(box[:, 0], box[:, 2], side="right")
    counts = np.maximum(hi - np.arange(n) - 1, 0)
    first = np.repeat(np.arange(n), counts)
    start = np.repeat(np.cumsum(counts) - counts, counts)
    second = first + 1 + (np.arange(counts.sum()) - start)
    keep = (box[second, 1] <= box[first, 3]) & (box[first, 1] <= box[second, 3])
    a, c = ids[first[keep]].astype(np.uint64), ids[second[keep]].astype(np.uint64)
    return (np.minimum(a, c) << np.uint64(32)) | np.maximum(a, c)


def _split(keys):
    return (keys >> np.uint64(32)).astype(np.int64), (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)


def _allowed(keys, dynamic):
    a, c = _split(keys)
    return keys[dynamic[a] | dynamic[c]]


def _table(dw):
    rows = dw.download_contacts(dw.counters().contactCount + 64)
    a, c = rows["shapeA"].astype(np.uint64), rows["shapeB"].astype(np.uint64)
    keys = (np.minimum(a, c) << np.uint64(32)) | np.maximum(a, c)
    assert len(np.unique(keys)) == len(keys), "a pair is in the table twice"
    return np.sort(keys)


def _check_first_step(dev, b):
    dw = _attach(dev, b)
    _, fat, flags = dw.download_shape_boxes()
    valid = (flags & 1) != 0
    assert valid.sum() == len(b.types)
    dw.update_pairs()
    expected = np.sort(_allowed(_overlapping(fat, valid), _dynamic_mask(b, len(fat))))
    got = _table(dw)
    missing = np.setdiff1d(expected, got)
    extra = np.setdiff1d(got, expected)
    assert len(missing) == 0 and len(extra) == 0, (f"{len(missing)} pairs missing (first {_split(missing[:4])}), "
                                                   f"{len(extra)} extra (first {_split(extra[:4])})")
    return len(got)


def _rows_of_boxes(lib, b, n, rows=3, pitch=0.9):
    box = lib.s2MakeSquare(0.5)
    cols = (n + rows - 1) // rows
    for k in range(n):
        b.add(capi.DYNAMIC_BODY, pitch * (k % cols), pitch * (k // cols), box)


@pytest.mark.parametrize("leaves", [1, 2, 15, 16, 17, 257])
def test_first_step_table_at_fanout_boundaries(dev, leaves):
    lib = capi.Solver2D(device.LIB_PATH)
    b = Built(lib)
    _rows_of_boxes(lib, b, leaves)
    pairs = _check_first_step(dev, b)
    assert leaves < 2 or pairs > 0
    b.destroy()


def test_first_step_table_pyramid_447(dev):
    lib = capi.Solver2D(device.LIB_PATH)
    sc = scenes.pyramid(lib, "TGS_Soft", base_count=447)
    b = Built.__new__(Built)
    b.lib, b.world, b.bodies = lib, sc.world, sc.bodies
    # one shape per body, in creation order: the ground first
    b.types = {k: (capi.STATIC_BODY if k == 0 else capi.DYNAMIC_BODY) for k in range(len(sc.bodies))}
    pairs = _check_first_step(dev, b)
    assert pairs > 100000
    b.destroy()


def _pile_with_bars(lib, bars, bar_type, velocity=(0.0, 0.0), grid=(40, 25)):
    """A grid of boxes crossed by `bars` long thin bars of one body type, at spread heights and slight angles."""
    b = Built(lib)
    box = lib.s2MakeSquare(0.4)
    gx, gy = grid
    for i in range(gy):
        for j in range(gx):
            b.add(capi.DYNAMIC_BODY, 1.0 * j, 1.0 * i, box)
    bar = lib.s2MakeBox(0.5 * gx + 2.0, 0.1)
    for k in range(bars):
        b.add(bar_type, 0.5 * gx, (gy - 1) * (k + 0.5) / bars, bar, velocity=velocity, angle=0.01 * (k % 7 - 3))
    return b


def test_first_step_table_more_static_bars_than_the_large_list(dev):
    lib = capi.Solver2D(device.LIB_PATH)
    b = _pile_with_bars(lib, 80, capi.STATIC_BODY)
    _check_first_step(dev, b)
    b.destroy()


def test_first_step_table_kinematic_bar_through_a_pile(dev):
    lib = capi.Solver2D(device.LIB_PATH)
    b = _pile_with_bars(lib, 1, capi.KINEMATIC_BODY, velocity=(0.0, 3.0))
    _check_first_step(dev, b)
    b.destroy()


def _tumbler(lib):
    sc = scenes.tumbler(lib, "TGS_Soft", grid=40, half_extent=10.0)
    b = Built.__new__(Built)
    b.lib, b.world, b.bodies = lib, sc.world, sc.bodies
    # four wall shapes on the container (dynamic), then one box per body; the static anchor body has no shape
    b.types = {k: capi.DYNAMIC_BODY for k in range(4 + 40 * 40)}
    return b


def _free_running(dev, b, same_body, steps=40):
    """table_{k+1} == (table_k & overlapping(fat_k)) | {allowed overlapping pairs in fat_k with >= 1 mover}, movers being
    the shapes whose fat box changed between steps k-1 and k."""
    dw = _attach(dev, b)
    fats, tables = [], []
    for _ in range(steps):
        b.step()
        _, fat, flags = dw.download_shape_boxes()
        fats.append((fat.copy(), (flags & 1) != 0))
        tables.append(_table(dw))
    dynamic = _dynamic_mask(b, len(fats[0][0]))
    for k in range(1, steps - 1):
        fat, valid = fats[k]
        moved = np.any(fat != fats[k - 1][0], axis=1)
        overlapping = np.sort(_overlapping(fat, valid))
        survivors = np.intersect1d(tables[k], overlapping)
        candidates = _allowed(overlapping, dynamic)
        a, c = _split(candidates)
        candidates = candidates[(moved[a] | moved[c]) & ~same_body(a, c)]
        expected = np.union1d(survivors, candidates)
        got = tables[k + 1]
        assert np.array_equal(expected, got), (f"step {k + 1}: {len(np.setdiff1d(expected, got))} missing, "
                                               f"{len(np.setdiff1d(got, expected))} extra")
    return dw.counters().treeHeight


def test_free_running_kinematic_bar_sweep(dev):
    lib = capi.Solver2D(device.LIB_PATH)
    b = _pile_with_bars(lib, 1, capi.KINEMATIC_BODY, velocity=(0.0, 3.0))
    assert _free_running(dev, b, lambda a, c: np.zeros(len(a), dtype=bool)) >= 2
    b.destroy()


def test_free_running_tumbler(dev):
    lib = capi.Solver2D(device.LIB_PATH)
    b = _tumbler(lib)
    assert _free_running(dev, b, lambda a, c: (a < 4) & (c < 4)) >= 2
    b.destroy()
