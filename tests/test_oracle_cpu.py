"""CPU: pin the plain-C restatement (oracle/s2o_solver.c) against the UNMODIFIED reference, bit for bit, in the
reference's own constraint order. The reference ships no tests or golden vectors of its own (SURVEY §4), so this — and the
committed fixtures recorded from it (tests/golden, tests/golden/make_stage_cases.py) — is what the oracle's parity claim
rests on. Each case feeds the oracle the rows the reference's solver stage received and compares with what it returned."""
import numpy as np
import pytest

from helpers import bit_equal
from oracle import port
from solver2d_b200 import capi, device
from stage_cases import STICKY, load_case

DT = 1.0 / 60.0


def _pin(recipe, solver, warm_steps, vel, pos, warm_start=True, **kw):
    case = load_case(recipe, solver, warm_steps, vel, pos, warm_start, **kw)
    O = port.load()
    bodies, contacts, joints = case.bodies, case.contacts, case.joints
    ctx = device.make_context(solver, DT, vel, pos, warm_start)
    ob, oc, oj = O.solve(capi.SOLVER[solver], bodies, contacts, joints, ctx)

    valid = (bodies["flags"] & 1) == 1
    for name in ("position", "rot", "linearVelocity", "angularVelocity"):
        assert bit_equal(ob[name][valid], case.out(name)[valid]), name
    for j in range(2):
        live = oc["pointCount"] > j
        assert bit_equal(oc["points"]["normalImpulse"][:, j][live], case.out_normal[:, j][live])
        assert bit_equal(oc["points"]["tangentImpulse"][:, j][live], case.out_tangent[:, j][live])
        if solver == "TGS_Sticky":
            for name in STICKY:
                assert bit_equal(oc["points"][name][:, j][live], case.out_sticky[name][:, j][live]), name
    if solver == "TGS_Sticky":
        live = oc["pointCount"] > 0
        assert np.array_equal(oc["frictionPersisted"][live], case.out_friction_persisted[live])
    return len(contacts), int((joints["flags"] & 1).sum())


@pytest.mark.parametrize("base,warm", [(10, 0), (10, 25), (30, 3)])
def test_tgs_soft_pyramid_pinned(base, warm):
    nc, nj = _pin("pyramid", "TGS_Soft", warm, 4, 2, base_count=base)
    assert nc > 0


def test_tgs_soft_no_warmstart_no_relax_pinned():
    _pin("pyramid", "TGS_Soft", 10, 3, 0, warm_start=False, base_count=12)


def test_tgs_soft_bridge_joints_pinned():
    nc, nj = _pin("bridge", "TGS_Soft", 20, 4, 2, count=40)
    assert nj == 41


def test_tgs_soft_mixed_shapes_pinned():
    nc, nj = _pin("mixed_shapes", "TGS_Soft", 120, 4, 2)
    assert nc > 20


def test_oracle_order_changes_result():
    """Sanity: the order hook really changes the Gauss-Seidel result (otherwise the colour-schedule check is vacuous)."""
    O = port.load()
    case = load_case("pyramid", "TGS_Soft", 20, 4, 2, base_count=10)
    bodies, contacts, joints = case.bodies, case.contacts, case.joints
    ctx = device.make_context("TGS_Soft", DT, 4, 2, True)
    a, _, _ = O.solve(7, bodies, contacts, joints, ctx)
    order = np.arange(len(contacts), dtype=np.int32)[::-1]
    b, _, _ = O.solve(7, bodies, contacts, joints, ctx, order=order)
    assert not bit_equal(a["linearVelocity"], b["linearVelocity"])


VARIANTS = ["Jacobi", "PGS", "PGS_NGS", "PGS_NGS_Block", "PGS_Soft", "SoftStep", "TGS_Sticky", "TGS_Soft", "TGS_NGS", "XPBD"]


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_pyramid_pinned(solver):
    # the reference's Jacobi variant blows a pyramid apart within five steps (its own behaviour): pin it early
    warm = 2 if solver == "Jacobi" else 40
    nc, _ = _pin("pyramid", solver, warm, 4, 2, base_count=10)
    assert nc > 50


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_cold_start_pinned(solver):
    _pin("pyramid", solver, 2 if solver == "Jacobi" else 30, 3, 1, warm_start=False, base_count=8)


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_bridge_pinned(solver):
    _, nj = _pin("bridge", solver, 12, 4, 2, count=30)
    assert nj == 31


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_limits_motors_mouse_pinned(solver):
    nc, nj = _pin("limited_chains", solver, 40, 4, 2)
    assert nj == 19 and nc > 20


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_mixed_shapes_pinned(solver):
    nc, _ = _pin("mixed_shapes", solver, 100, 4, 2)
    assert nc > 20
