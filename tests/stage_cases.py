"""Solver-stage cases recorded from the unmodified reference (tests/golden/make_stage_cases.py -> tests/golden/stage/).

A case is one scene stepped `warm` times by the reference, then ONE step split at the stage boundaries: the rows the
reference hands its solver stage (bodies and joints by pool slot, contacts in pool order = its Gauss-Seidel order) and
what its solver stage returns (body state, stored impulses). Tests feed the rows to the oracle or the device and compare
the result with the reference's, bit for bit, without needing the reference itself."""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np

STAGE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "stage")

# out_body columns
OUT_BODY = dict(origin=(0, 2), position=(2, 4), rot=(4, 6), linearVelocity=(6, 8), angularVelocity=(8, 9))
STICKY = ("frictionAnchorA", "frictionAnchorB", "frictionNormalA", "frictionNormalB")


def case_name(recipe: str, solver: str, warm: int, vel: int, pos: int, warm_start: bool = True, warm_iters=None, **kw) -> str:
    """`warm` steps with `warm_iters` = (vel, pos) iterations (default: the case's own), warm starting on; then the split
    step with (vel, pos) and `warm_start`. `kw` are the scene recipe's arguments."""
    params = "".join(f"_{k}{v}" for k, v in sorted(kw.items()))
    wi = "" if warm_iters is None or tuple(warm_iters) == (vel, pos) else f"_wi{warm_iters[0]}x{warm_iters[1]}"
    return f"{recipe}{params}_{solver.lower()}_w{warm}{wi}_i{vel}x{pos}" + ("" if warm_start else "_cold")


@dataclass
class StageCase:
    solver: str
    vel: int
    pos: int
    warm_start: bool
    bodies: np.ndarray       # device BODY_ROW, every body slot
    contacts: np.ndarray     # device CONTACT_ROW, live contacts in the reference's pool order
    joints: np.ndarray       # device JOINT_ROW, every joint slot
    out_body: np.ndarray     # (body slots, 9) float32: origin, position, rot, v, w after the reference's solver stage
    out_normal: np.ndarray   # (contacts, 2) float32 normal impulse of both points after the solver stage
    out_tangent: np.ndarray  # (contacts, 2) float32 tangent impulse
    out_friction_persisted: np.ndarray  # (contacts,) int32
    out_sticky: dict         # TGS_Sticky only: name -> (contacts, 2, 2) float32

    def out(self, name: str) -> np.ndarray:
        a, b = OUT_BODY[name]
        return self.out_body[:, a:b] if b - a > 1 else self.out_body[:, a]


# set by tests/golden/make_stage_cases.py: called with every case a test asks for, before it is loaded
recorder = None


def load_case(recipe: str, solver: str, warm: int, vel: int, pos: int, warm_start: bool = True, warm_iters=None,
              **kw) -> StageCase:
    if recorder is not None:
        recorder(recipe, solver, warm, vel, pos, warm_start, warm_iters, kw)
    g = np.load(os.path.join(STAGE_DIR, case_name(recipe, solver, warm, vel, pos, warm_start, warm_iters, **kw) + ".npz"))
    return StageCase(solver, vel, pos, warm_start, g["bodies"], g["contacts"], g["joints"], g["out_body"], g["out_normal"],
                     g["out_tangent"], g["out_friction_persisted"], {n: g[n] for n in STICKY if n in g.files})
