"""ctypes binding of the device C ABI (include/s2b_device.h) — the inner drop-in boundary.

Used by the stage-level parity tests and by bench.py to drive the CUDA pipeline directly (the public ``s2*`` API in
capi.py goes through the same entry points from host C). Rows are numpy structured arrays whose dtypes mirror the
C row structs field for field.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsolver2d.so")

BODY_ROW = np.dtype([
    ("index", "<i4"), ("flags", "<i4"), ("origin", "<f4", 2), ("position", "<f4", 2), ("rot", "<f4", 2),
    ("linearVelocity", "<f4", 2), ("angularVelocity", "<f4"), ("localCenter", "<f4", 2), ("mass", "<f4"),
    ("invMass", "<f4"), ("I", "<f4"), ("invI", "<f4"), ("force", "<f4", 2), ("torque", "<f4"),
    ("linearDamping", "<f4"), ("angularDamping", "<f4"), ("gravityScale", "<f4"),
], align=True)

SHAPE_ROW = np.dtype([
    ("index", "<i4"), ("flags", "<i4"), ("body", "<i4"), ("proxyKey", "<i4"), ("categoryBits", "<u4"),
    ("maskBits", "<u4"), ("groupIndex", "<i4"), ("friction", "<f4"), ("aabb", "<f4", 4), ("fatAABB", "<f4", 4),
    ("radius", "<f4"), ("count", "<i4"), ("vertices", "<f4", 16), ("normals", "<f4", 16),
], align=True)

JOINT_ROW = np.dtype([
    ("index", "<i4"), ("flags", "<i4"), ("bodyA", "<i4"), ("bodyB", "<i4"), ("localOriginAnchorA", "<f4", 2),
    ("localOriginAnchorB", "<f4", 2), ("referenceAngle", "<f4"), ("lowerAngle", "<f4"), ("upperAngle", "<f4"),
    ("maxMotorTorque", "<f4"), ("motorSpeed", "<f4"), ("hertz", "<f4"), ("dampingRatio", "<f4"), ("target", "<f4", 2),
    ("impulse", "<f4", 2), ("motorImpulse", "<f4"), ("lowerImpulse", "<f4"), ("upperImpulse", "<f4"),
], align=True)

CONTACT_POINT = np.dtype([
    ("localAnchorA", "<f4", 2), ("localAnchorB", "<f4", 2), ("separation", "<f4"), ("normalImpulse", "<f4"),
    ("tangentImpulse", "<f4"), ("frictionAnchorA", "<f4", 2), ("frictionAnchorB", "<f4", 2),
    ("frictionNormalA", "<f4", 2), ("frictionNormalB", "<f4", 2), ("id", "<i4"), ("persisted", "<i4"),
], align=True)

CONTACT_ROW = np.dtype([
    ("shapeA", "<i4"), ("shapeB", "<i4"), ("bodyA", "<i4"), ("bodyB", "<i4"), ("pointCount", "<i4"),
    ("frictionPersisted", "<i4"), ("friction", "<f4"), ("normal", "<f4", 2), ("points", CONTACT_POINT, 2),
    ("cacheCount", "<i4"), ("cacheIndexA", "u1", 4), ("cacheIndexB", "u1", 4), ("cacheMetric", "<f4"),
], align=True)


class StepContext(C.Structure):
    _fields_ = [("dt", C.c_float), ("inv_dt", C.c_float), ("h", C.c_float), ("inv_h", C.c_float),
                ("iterations", C.c_int32), ("extraIterations", C.c_int32), ("warmStart", C.c_int32)]


class Counters(C.Structure):
    _fields_ = [("bodyCapacity", C.c_int32), ("shapeCapacity", C.c_int32), ("jointCapacity", C.c_int32),
                ("contactCount", C.c_int32), ("constraintCount", C.c_int32), ("jointCount", C.c_int32),
                ("groupCount", C.c_int32), ("overflowCount", C.c_int32), ("treeHeight", C.c_int32),
                ("movedCount", C.c_int32), ("pairPassCount", C.c_int32), ("kernelLaunches", C.c_int32),
                ("graphReplays", C.c_int32), ("graphCaptures", C.c_int32), ("scratchBytes", C.c_int64),
                ("regionCount", C.c_int32), ("cutCount", C.c_int32), ("cutGroupCount", C.c_int32), ("recolouredCount", C.c_int32),
                ("largeLeafCount", C.c_int32), ("pairRebuildCount", C.c_int32)]


SCHEDULE_COLOR, SCHEDULE_WAVEFRONT = 0, 1
ROW_VALID = 0x1
SHAPE_MOVED = 0x10
JOINT_ENABLE_LIMIT, JOINT_ENABLE_MOTOR, JOINT_COLLIDE_CONNECTED = 0x10, 0x20, 0x40

# symbols declared in include/s2b_device.h (checked by the CPU test-suite against the built library)
ABI_SYMBOLS = [
    "s2b_world_create", "s2b_world_destroy", "s2b_set_gravity", "s2b_set_schedule", "s2b_set_max_colors",
    "s2b_set_persistent", "s2b_upload_bodies", "s2b_upload_shapes", "s2b_upload_joints", "s2b_upload_contacts",
    "s2b_upload_joint_pairs", "s2b_mark_pairs_dirty", "s2b_set_contact_order", "s2b_update_pairs",
    "s2b_update_contacts", "s2b_solve", "s2b_finalize", "s2b_step", "s2b_sync", "s2b_download_bodies",
    "s2b_download_all_bodies", "s2b_download_shape_boxes", "s2b_download_joints", "s2b_download_contacts",
    "s2b_download_solve_order", "s2b_download_islands", "s2b_prefetch_pairs", "s2b_get_counters", "s2b_pack_body_state", "s2b_timed_steps", "s2b_last_stage_ms",
    "s2b_flush_l2", "s2b_time_color_kernel", "s2b_version", "s2b_abi_sizes", "s2b_upload_forces", "s2b_host_alloc",
    "s2b_host_free", "s2b_sync_body_state", "s2b_set_warm_gather", "s2b_eval_atan2", "s2b_set_dataflow", "s2b_set_regions", "s2b_set_graph", "s2b_get_stream", "s2b_add_forces", "s2b_download_transforms",
]


def make_context(solver: str, dt: float, vel_iters: int, pos_iters: int, warm_start: bool = True) -> StepContext:
    """Step context exactly as s2World_Step builds it (reference src/world.c:171-202), in float32 arithmetic."""
    from .capi import SUBSTEPPING
    f = np.float32
    ctx = StepContext()
    ctx.dt = dt
    ctx.iterations = vel_iters
    ctx.extraIterations = pos_iters
    ctx.warmStart = 1 if warm_start else 0
    dt32 = f(dt)
    inv_dt = f(1.0) / dt32 if dt32 > 0 else f(0.0)
    ctx.inv_dt = float(inv_dt)
    if solver in SUBSTEPPING:
        ctx.h = float(dt32 / f(vel_iters))
        ctx.inv_h = float(inv_dt * f(vel_iters))
    else:
        ctx.h = float(dt32)
        ctx.inv_h = float(inv_dt)
    return ctx


class Device:
    """The loaded product library, device-ABI view."""

    def __init__(self, path: str = LIB_PATH):
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} is missing: build it with `python -m solver2d_b200.build` — there is no CPU fallback")
        self.lib = L = C.CDLL(path)
        vp = C.c_void_p
        L.s2b_world_create.restype = vp
        L.s2b_world_create.argtypes = [C.c_int, C.c_int]
        L.s2b_world_destroy.argtypes = [vp]
        L.s2b_set_gravity.argtypes = [vp, C.c_float, C.c_float]
        for name in ("s2b_set_schedule", "s2b_set_max_colors", "s2b_set_persistent", "s2b_set_warm_gather", "s2b_set_dataflow", "s2b_set_regions", "s2b_set_graph"):
            getattr(L, name).argtypes = [vp, C.c_int]
        for name in ("s2b_upload_bodies", "s2b_upload_shapes", "s2b_upload_joints"):
            getattr(L, name).argtypes = [vp, vp, C.c_int, C.c_int]
        L.s2b_upload_contacts.argtypes = [vp, vp, C.c_int]
        L.s2b_upload_joint_pairs.argtypes = [vp, vp, C.c_int, vp, C.c_int]
        L.s2b_set_contact_order.argtypes = [vp, vp, C.c_int]
        for name in ("s2b_mark_pairs_dirty", "s2b_update_pairs", "s2b_update_contacts", "s2b_finalize", "s2b_sync",
                     "s2b_flush_l2"):
            getattr(L, name).argtypes = [vp]
        L.s2b_solve.argtypes = [vp, C.c_int, C.POINTER(StepContext)]
        L.s2b_step.argtypes = [vp, C.c_int, C.POINTER(StepContext)]
        L.s2b_download_bodies.argtypes = [vp, vp, C.c_int]
        L.s2b_download_all_bodies.argtypes = [vp, vp, C.c_int]
        L.s2b_download_shape_boxes.argtypes = [vp, vp, vp, vp, C.c_int]
        L.s2b_download_joints.argtypes = [vp, vp, C.c_int]
        L.s2b_download_contacts.restype = C.c_int
        L.s2b_download_contacts.argtypes = [vp, vp, C.c_int]
        L.s2b_download_solve_order.restype = C.c_int
        L.s2b_download_solve_order.argtypes = [vp, vp, C.c_int, vp, C.c_int, vp]
        L.s2b_get_counters.argtypes = [vp, C.POINTER(Counters)]
        L.s2b_pack_body_state.argtypes = [vp, C.c_int, C.c_int, vp]
        L.s2b_timed_steps.restype = C.c_float
        L.s2b_timed_steps.argtypes = [vp, C.c_int, C.POINTER(StepContext), C.c_int]
        L.s2b_last_stage_ms.argtypes = [vp, C.POINTER(C.c_float)]
        L.s2b_time_color_kernel.restype = C.c_float
        L.s2b_time_color_kernel.argtypes = [vp, C.POINTER(StepContext), C.c_int, C.POINTER(C.c_int)]
        L.s2b_version.restype = C.c_char_p

    def create_world(self, solver_type: int, device: int = -1) -> "DeviceWorld":
        return DeviceWorld(self, solver_type, device)


class DeviceWorld:
    def __init__(self, dev: Device, solver_type: int, device: int = -1):
        self.dev = dev
        self.L = dev.lib
        self.solver_type = solver_type
        self.h = self.L.s2b_world_create(device, solver_type)
        self.body_cap = self.shape_cap = self.joint_cap = 0

    @classmethod
    def attach(cls, dev: Device, world_id) -> "DeviceWorld":
        """Device view of a world created through the public API (s2World_GetDevice, include/solver2d_b200.h)."""
        fn = dev.lib.s2World_GetDevice
        fn.restype = C.c_void_p
        from .capi import WorldId
        fn.argtypes = [WorldId]
        self = cls.__new__(cls)
        self.dev = dev
        self.L = dev.lib
        self.solver_type = -1
        self.h = fn(world_id)
        self.owned = False
        c = Counters()
        self.L.s2b_get_counters(self.h, C.byref(c))
        self.body_cap, self.shape_cap, self.joint_cap = c.bodyCapacity, c.shapeCapacity, c.jointCapacity
        return self

    def destroy(self):
        if self.h and getattr(self, "owned", True):
            self.L.s2b_world_destroy(self.h)
        self.h = None

    # -- uploads ------------------------------------------------------------------------------------------------
    def upload_bodies(self, rows: np.ndarray, capacity: int):
        rows = np.ascontiguousarray(rows, dtype=BODY_ROW)
        self.body_cap = max(self.body_cap, capacity)
        self.L.s2b_upload_bodies(self.h, rows.ctypes.data, len(rows), capacity)

    def upload_shapes(self, rows: np.ndarray, capacity: int):
        rows = np.ascontiguousarray(rows, dtype=SHAPE_ROW)
        self.shape_cap = max(self.shape_cap, capacity)
        self.L.s2b_upload_shapes(self.h, rows.ctypes.data, len(rows), capacity)

    def upload_joints(self, rows: np.ndarray, capacity: int):
        rows = np.ascontiguousarray(rows, dtype=JOINT_ROW)
        self.joint_cap = max(self.joint_cap, capacity)
        self.L.s2b_upload_joints(self.h, rows.ctypes.data, len(rows), capacity)

    def upload_contacts(self, rows: np.ndarray):
        rows = np.ascontiguousarray(rows, dtype=CONTACT_ROW)
        self.L.s2b_upload_contacts(self.h, rows.ctypes.data, len(rows))

    def upload_joint_pairs(self, block_keys: np.ndarray, destroy_keys: np.ndarray | None = None):
        block = np.ascontiguousarray(np.sort(block_keys.astype(np.uint64)))
        destroy = block if destroy_keys is None else np.ascontiguousarray(np.sort(destroy_keys.astype(np.uint64)))
        self.L.s2b_upload_joint_pairs(self.h, block.ctypes.data, len(block), destroy.ctypes.data, len(destroy))

    def set_contact_order(self, keys: np.ndarray):
        keys = np.ascontiguousarray(keys.astype(np.uint64))
        self.L.s2b_set_contact_order(self.h, keys.ctypes.data, len(keys))

    # -- stages -------------------------------------------------------------------------------------------------
    def set_schedule(self, schedule: int):
        self.L.s2b_set_schedule(self.h, schedule)

    def set_persistent(self, enable: bool):
        self.L.s2b_set_persistent(self.h, 1 if enable else 0)

    def set_graph(self, enable: bool):
        self.L.s2b_set_graph(self.h, 1 if enable else 0)

    def set_dataflow(self, enable: bool):
        self.L.s2b_set_dataflow(self.h, 1 if enable else 0)

    def set_regions(self, mode):
        """Region-local schedule of the persistent kernel: 0 / False never, 1 when the cut set needs few colours (default),
        2 / True always. See DESIGN.md §3.1."""
        self.L.s2b_set_regions(self.h, 2 if mode is True else (0 if mode is False else int(mode)))

    def set_warm_gather(self, enable: bool):
        self.L.s2b_set_warm_gather(self.h, 1 if enable else 0)

    def set_max_colors(self, n: int):
        self.L.s2b_set_max_colors(self.h, n)

    def update_pairs(self):
        self.L.s2b_update_pairs(self.h)

    def update_contacts(self):
        self.L.s2b_update_contacts(self.h)

    def solve(self, ctx: StepContext, solver_type: int | None = None):
        self.L.s2b_solve(self.h, self.solver_type if solver_type is None else solver_type, C.byref(ctx))

    def finalize(self):
        self.L.s2b_finalize(self.h)

    def step(self, ctx: StepContext):
        self.L.s2b_step(self.h, self.solver_type, C.byref(ctx))

    def sync(self):
        self.L.s2b_sync(self.h)

    def timed_steps(self, ctx: StepContext, steps: int) -> float:
        return float(self.L.s2b_timed_steps(self.h, self.solver_type, C.byref(ctx), steps))

    def stage_ms(self):
        out = (C.c_float * 4)()
        self.L.s2b_last_stage_ms(self.h, out)
        return list(out)

    def flush_l2(self):
        self.L.s2b_flush_l2(self.h)

    # -- downloads ----------------------------------------------------------------------------------------------
    def download_all_bodies(self, capacity: int | None = None) -> np.ndarray:
        cap = self.body_cap if capacity is None else capacity
        rows = np.zeros(cap, dtype=BODY_ROW)
        self.L.s2b_download_all_bodies(self.h, rows.ctypes.data, cap)
        return rows

    def download_joints(self, capacity: int | None = None) -> np.ndarray:
        cap = self.joint_cap if capacity is None else capacity
        rows = np.zeros(cap, dtype=JOINT_ROW)
        self.L.s2b_download_joints(self.h, rows.ctypes.data, cap)
        return rows

    def download_contacts(self, max_count: int) -> np.ndarray:
        rows = np.zeros(max(max_count, 1), dtype=CONTACT_ROW)
        n = self.L.s2b_download_contacts(self.h, rows.ctypes.data, max_count)
        return rows[:n]

    def download_shape_boxes(self, capacity: int | None = None):
        cap = self.shape_cap if capacity is None else capacity
        aabb = np.zeros((cap, 4), dtype=np.float32)
        fat = np.zeros((cap, 4), dtype=np.float32)
        flags = np.zeros(cap, dtype=np.int32)
        self.L.s2b_download_shape_boxes(self.h, aabb.ctypes.data, fat.ctypes.data, flags.ctypes.data, cap)
        return aabb, fat, flags

    def islands(self, capacity: int | None = None):
        """(labels, count): labels[i] = island of body slot i (smallest body slot of the island, -1 for free slots)."""
        cap = self.body_cap if capacity is None else capacity
        labels = np.full(max(cap, 1), -1, dtype=np.int32)
        self.L.s2b_download_islands.restype = C.c_int
        self.L.s2b_download_islands.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        n = self.L.s2b_download_islands(self.h, labels.ctypes.data, cap)
        return labels[:cap], int(n)

    def solve_order(self, max_items: int, max_groups: int = 70000):
        """(items, group_sizes): items >= 0 contact slot, < 0 joint slot (-1 - k), in the order the last solve visited them."""
        items = np.zeros(max(max_items, 1), dtype=np.int32)
        sizes = np.zeros(max_groups, dtype=np.int32)
        groups = C.c_int(0)
        n = self.L.s2b_download_solve_order(self.h, items.ctypes.data, max_items, sizes.ctypes.data, max_groups,
                                            C.byref(groups))
        return items[:n], sizes[:groups.value]

    def counters(self) -> Counters:
        c = Counters()
        self.L.s2b_get_counters(self.h, C.byref(c))
        return c
