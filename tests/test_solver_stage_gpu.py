"""GPU parity of the solver stage (s2Solve_* on the device) against the unmodified reference.

Each case: a scene stepped by the reference, then ONE step split at the stage boundaries, recorded in tests/golden/stage:
the bodies + manifolds (pool order) the reference's solver stage received -> a device world -> solver stage ->
compare per-body state and stored impulses with what the reference's solver stage returned.

* WAVEFRONT schedule preserves the reference's sequential Gauss-Seidel order; the kernels are compiled with
  -fmad=false, so the result must be BIT-EXACT (tolerance 0).
* COLOR schedule solves in colour-major order; the reference run in pool order differs by the order sensitivity of
  Gauss-Seidel itself (SURVEY §7 H1), so this file only bounds it loosely; the tight check of the COLOR schedule
  is against the order-permuted oracle in test_solver_color_gpu.py.
"""
import numpy as np
import pytest

from helpers import bit_equal
from solver2d_b200 import capi, device
from stage_cases import load_case

pytestmark = pytest.mark.gpu

DT = 1.0 / 60.0


def _one_case(dev, recipe, solver, warm_steps, vel_iters, pos_iters, schedule, persistent, warm_start=True, warm_iters=None,
              **kw):
    """The rows the reference's solver stage received (tests/golden/stage) -> a device world -> solver stage -> compare
    per-body state and stored impulses with what the reference's stage returned."""
    case = load_case(recipe, solver, warm_steps, vel_iters, pos_iters, warm_start, warm_iters, **kw)
    dw = dev.create_world(capi.SOLVER[solver])
    dw.upload_bodies(case.bodies, len(case.bodies))
    dw.upload_joints(case.joints, len(case.joints))
    dw.upload_contacts(case.contacts)
    dw.set_schedule(schedule)
    if persistent is not None:
        dw.set_persistent(persistent)
    ctx = device.make_context(solver, DT, vel_iters, pos_iters, warm_start)

    dw.solve(ctx)
    rows = dw.download_all_bodies(len(case.bodies))
    contacts = dw.download_contacts(len(case.contacts))
    counters = dw.counters()
    valid = (case.bodies["flags"] & 1) == 1
    diff = {key: float(np.abs(rows[name][valid] - case.out(name)[valid]).max()) if valid.any() else 0.0
            for key, name in (("pos", "position"), ("rot", "rot"), ("v", "linearVelocity"), ("w", "angularVelocity"),
                              ("origin", "origin"))}

    # stored impulses, same (pool) order on both sides
    ref_imp, ref_timp = case.out_normal, case.out_tangent
    dev_imp = contacts["points"]["normalImpulse"]
    dev_timp = contacts["points"]["tangentImpulse"]
    two = np.stack([contacts["pointCount"] > 0, contacts["pointCount"] > 1], axis=1) if len(contacts) else None
    diff["impulse"] = float(np.abs(ref_imp - dev_imp).max()) if len(contacts) else 0.0
    exact = (bit_equal(rows["position"][valid], case.out("position")[valid])
             and bit_equal(rows["linearVelocity"][valid], case.out("linearVelocity")[valid])
             and bit_equal(rows["angularVelocity"][valid], case.out("angularVelocity")[valid])
             and bit_equal(rows["rot"][valid], case.out("rot")[valid])
             and bit_equal(ref_imp, dev_imp)
             and (two is None or bit_equal(ref_timp[two], dev_timp[two])))
    if solver == "TGS_Sticky" and len(contacts):
        live = contacts["pointCount"] > 0
        exact = exact and bool(np.array_equal(contacts["frictionPersisted"][live], case.out_friction_persisted[live]))
    dw.destroy()
    return diff, exact, counters


@pytest.mark.parametrize("persistent", [True, False])
@pytest.mark.parametrize("base,warm", [(10, 0), (10, 30), (40, 5)])
def test_tgs_soft_wavefront_bit_exact(dev, base, warm, persistent):
    diff, exact, counters = _one_case(dev, "pyramid", "TGS_Soft", warm, 4, 2, device.SCHEDULE_WAVEFRONT,
                                      persistent, base_count=base)
    assert counters.constraintCount > 0
    assert exact, f"not bit-exact: {diff}"
    assert max(diff.values()) == 0.0


@pytest.mark.parametrize("persistent", [True, False])
def test_tgs_soft_color_close(dev, persistent):
    diff, exact, counters = _one_case(dev, "pyramid", "TGS_Soft", 30, 4, 2, device.SCHEDULE_COLOR,
                                      persistent, base_count=20)
    assert 1 <= counters.groupCount <= 16
    assert counters.overflowCount == 0
    # one step of a different Gauss-Seidel order on a settled pyramid: SURVEY §7 H1 measured ~3e-4 m
    assert diff["pos"] < 2e-3 and diff["v"] < 0.2, diff


def test_tgs_soft_no_warm_start_and_no_relax(dev):
    diff, exact, counters = _one_case(dev, "pyramid", "TGS_Soft", 10, 3, 0, device.SCHEDULE_WAVEFRONT, None,
                                      warm_start=False, warm_iters=(4, 2), base_count=12)
    assert max(v for k, v in diff.items() if k != "impulse") == 0.0


VARIANTS = ["Jacobi", "PGS", "PGS_NGS", "PGS_NGS_Block", "PGS_Soft", "SoftStep", "TGS_Sticky", "TGS_Soft", "TGS_NGS", "XPBD"]


@pytest.mark.parametrize("persistent", [True, False])
@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_wavefront_bit_exact_pyramid(dev, solver, persistent):
    warm = 2 if solver == "Jacobi" else 30  # the reference's Jacobi blows a pyramid apart within five steps
    diff, exact, counters = _one_case(dev, "pyramid", solver, warm, 4, 2, device.SCHEDULE_WAVEFRONT,
                                      persistent, base_count=12)
    assert counters.constraintCount > 50
    assert exact, f"{solver} not bit-exact: {diff}"


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_wavefront_bit_exact_joints(dev, solver):
    diff, exact, counters = _one_case(dev, "limited_chains", solver, 40, 4, 2, device.SCHEDULE_WAVEFRONT, True)
    assert counters.jointCount == 19
    assert exact, f"{solver} not bit-exact: {diff}"


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_wavefront_bit_exact_cold_mixed(dev, solver):
    diff, exact, counters = _one_case(dev, "mixed_shapes", solver, 100, 3, 1, device.SCHEDULE_WAVEFRONT, True,
                                      warm_start=False)
    assert counters.constraintCount > 20
    assert exact, f"{solver} not bit-exact: {diff}"
