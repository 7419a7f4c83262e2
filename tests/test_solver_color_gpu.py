"""GPU: the PRODUCTION schedule (device graph colouring + persistent cooperative kernel) against the order-permuted
oracle. The device reports the Gauss-Seidel order it used (colour-major); the plain-C oracle — pinned bit for bit to the
unmodified reference in tests/test_oracle_cpu.py — replays the solver stage in exactly that order. Tolerance: 0 (bit-exact),
because the kernels are compiled without FMA contraction. The rows both solve are those the product's own pipeline hands
its solver stage after `warm` steps of the scene through the public API."""
import numpy as np
import pytest

from helpers import bit_equal
from oracle import port
from solver2d_b200 import capi, device, scenes

pytestmark = pytest.mark.gpu
DT = 1.0 / 60.0


def _collided_rows(dev, recipe, solver, warm, vel, pos, **kw):
    """Step the scene `warm` times through the public API, then run stages 1-3 of the next step (pair update, narrow phase,
    impulse matching) and read back what the solver stage would receive: body and joint rows by slot, live contacts."""
    P = capi.Solver2D(device.LIB_PATH)
    sc = recipe(P, solver, **kw)
    for _ in range(warm):
        sc.step(DT, vel, pos, True)
    P.lib.s2World_Flush.restype = None
    P.lib.s2World_Flush.argtypes = [capi.WorldId]
    P.lib.s2World_Flush(sc.world)
    dw = device.DeviceWorld.attach(dev, sc.world)
    dw.update_pairs()
    dw.update_contacts()
    c = dw.counters()
    bodies = dw.download_all_bodies(c.bodyCapacity)
    contacts = dw.download_contacts(c.contactCount + 64)
    joints = dw.download_joints(c.jointCapacity)
    sc.destroy()
    return bodies, contacts, joints


def _case(dev, recipe, solver, warm, vel, pos, persistent, max_colors=None, warm_start=True, warm_gather=True, dataflow=False,
          regions=True, **kw):
    O = port.load()
    bodies, contacts, joints = _collided_rows(dev, recipe, solver, warm, vel, pos, **kw)
    ctx = device.make_context(solver, DT, vel, pos, warm_start)

    dw = dev.create_world(capi.SOLVER[solver])
    dw.upload_bodies(bodies, len(bodies))
    dw.upload_joints(joints, len(joints))
    dw.upload_contacts(contacts)
    dw.set_schedule(device.SCHEDULE_COLOR)
    dw.set_persistent(persistent)
    dw.set_warm_gather(warm_gather)
    dw.set_dataflow(dataflow)
    dw.set_regions(regions)
    if max_colors is not None:
        dw.set_max_colors(max_colors)
    dw.solve(ctx)
    got = dw.download_all_bodies(len(bodies))
    got_contacts = dw.download_contacts(len(contacts))
    got_joints = dw.download_joints(len(joints))
    order, group_sizes = dw.solve_order(len(contacts) + len(joints))
    counters = dw.counters()
    dw.destroy()

    # validity of the schedule: within a parallel group no movable body appears twice
    movable = (bodies["invMass"] != 0) | (bodies["invI"] != 0)
    parallel_groups = len(group_sizes) - (1 if counters.overflowCount > 0 else 0)
    is_contact = order >= 0
    if len(contacts):
        ends_a = np.where(is_contact, contacts["bodyA"][np.where(is_contact, order, 0)], -1)
        ends_b = np.where(is_contact, contacts["bodyB"][np.where(is_contact, order, 0)], -1)
    else:
        ends_a = np.full(len(order), -1)
        ends_b = np.full(len(order), -1)
    if len(joints):
        jslot = np.where(is_contact, 0, -1 - order)
        jtype = (joints["flags"][jslot] >> 1) & 7
        ends_a = np.where(is_contact, ends_a, np.where(jtype == 1, -1, joints["bodyA"][jslot]))  # a mouse joint acts on B only
        ends_b = np.where(is_contact, ends_b, joints["bodyB"][jslot])
    group_of = np.repeat(np.arange(len(group_sizes)), group_sizes)
    assert len(group_of) == len(order)
    both = np.concatenate([np.stack([group_of, ends_a], 1), np.stack([group_of, ends_b], 1)])
    both = both[(both[:, 1] >= 0) & (both[:, 0] < parallel_groups)]
    both = both[movable[both[:, 1]]]
    packed = both[:, 0].astype(np.int64) * (len(bodies) + 1) + both[:, 1]
    uniq, cnt = np.unique(packed, return_counts=True)
    assert (cnt == 1).all(), f"a movable body appears twice in a parallel group: group {uniq[cnt > 1][0] // (len(bodies) + 1)}"

    ob, oc, oj = O.solve(capi.SOLVER[solver], bodies, contacts, joints, ctx, order=order)
    valid = (bodies["flags"] & 1) == 1
    report = {}
    for name in ("position", "rot", "linearVelocity", "angularVelocity"):
        g = np.ascontiguousarray(got[name][valid]).reshape(int(valid.sum()), -1)
        o = np.ascontiguousarray(ob[name][valid]).reshape(int(valid.sum()), -1)
        bad = np.nonzero((g.view(np.uint32) != o.view(np.uint32)).any(axis=1))[0]
        if len(bad):
            report[name] = dict(count=len(bad), first=np.nonzero(valid)[0][bad[:8]].tolist(),
                                maxabs=float(np.abs(g[bad] - o[bad]).max()))
    assert not report, f"{solver}: device != permuted oracle: {report}"
    live = contacts["pointCount"] > 0
    assert bit_equal(got_contacts["points"]["normalImpulse"][live], oc["points"]["normalImpulse"][live])
    assert bit_equal(got_contacts["points"]["tangentImpulse"][live], oc["points"]["tangentImpulse"][live])
    if solver == "TGS_Sticky":
        assert np.array_equal(got_contacts["frictionPersisted"][live], oc["frictionPersisted"][live])
        for name in ("frictionAnchorA", "frictionAnchorB", "frictionNormalA", "frictionNormalB"):
            for j in range(2):
                has = contacts["pointCount"] > j
                assert bit_equal(got_contacts["points"][name][:, j][has], oc["points"][name][:, j][has]), name
    jlive = (joints["flags"] & 1) == 1
    for name in ("impulse", "motorImpulse", "lowerImpulse", "upperImpulse"):
        assert bit_equal(got_joints[name][jlive], oj[name][jlive]), name
    return counters


@pytest.mark.parametrize("persistent", [True, False])
@pytest.mark.parametrize("base,warm", [(10, 30), (40, 10)])
def test_color_schedule_matches_permuted_oracle(dev, base, warm, persistent):
    c = _case(dev, scenes.pyramid, "TGS_Soft", warm, 4, 2, persistent, base_count=base)
    assert c.overflowCount == 0 and 2 <= c.groupCount <= 16


def test_color_schedule_with_overflow_group(dev):
    # force constraints into the serial overflow group by allowing only 3 colours
    c = _case(dev, scenes.pyramid, "TGS_Soft", 20, 4, 2, True, max_colors=3, base_count=15)
    assert c.overflowCount > 0 and c.groupCount <= 3


def test_color_schedule_joints_and_contacts(dev):
    c = _case(dev, scenes.joint_contact_stress, "TGS_Soft", 90, 4, 2, True, bridges=3, planks=24, grid=9)
    assert c.jointCount == 75 and c.constraintCount > 20


VARIANTS = ["Jacobi", "PGS", "PGS_NGS", "PGS_NGS_Block", "PGS_Soft", "SoftStep", "TGS_Sticky", "TGS_Soft", "TGS_NGS", "XPBD"]


@pytest.mark.parametrize("persistent", [True, False])
@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_color_pyramid(dev, solver, persistent):
    warm = 2 if solver == "Jacobi" else 30  # the reference's Jacobi blows a pyramid apart within five steps
    c = _case(dev, scenes.pyramid, solver, warm, 4, 2, persistent, base_count=16)
    assert c.constraintCount > 100 and c.overflowCount == 0


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_color_limits_motors_mouse(dev, solver):
    c = _case(dev, scenes.limited_chains, solver, 40, 4, 2, True)
    assert c.jointCount == 19 and c.constraintCount > 20


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_color_mixed_shapes_with_overflow(dev, solver):
    c = _case(dev, scenes.mixed_shapes, solver, 100, 4, 2, True, max_colors=2)
    assert c.constraintCount > 20 and c.overflowCount > 0


@pytest.mark.parametrize("solver", VARIANTS)
def test_variant_color_cold_start(dev, solver):
    warm = 2 if solver == "Jacobi" else 20
    c = _case(dev, scenes.joint_contact_stress, solver, warm, 3, 1, False, warm_start=False, bridges=2, planks=16,
              grid=6)
    assert c.jointCount == 34


@pytest.mark.parametrize("solver", ["TGS_Soft", "SoftStep", "TGS_NGS"])
def test_grouped_warm_start_path_still_matches(dev, solver):
    """The per-sub-step warm start runs as a per-body gather by default; the grouped constraint passes it replaces
    must give the same bits (both are compared with the permuted oracle)."""
    c = _case(dev, scenes.limited_chains, solver, 40, 4, 2, True, warm_gather=False)
    assert c.jointCount == 19
    c = _case(dev, scenes.pyramid, solver, 30, 4, 2, True, warm_gather=False, max_colors=3, base_count=14)
    assert c.overflowCount > 0


@pytest.mark.parametrize("solver", VARIANTS)
def test_device_wide_colour_steps_still_match(dev, solver):
    """The persistent kernel runs the constraints interior to a block's region between block barriers and only the cut set
    in device-wide steps (default). With regions off every colour is one device-wide step; both orders are replayed by
    the oracle bit for bit."""
    c = _case(dev, scenes.limited_chains, solver, 40, 4, 2, True, regions=False)
    assert c.jointCount == 19 and c.regionCount == 0
    warm = 2 if solver == "Jacobi" else 30
    c = _case(dev, scenes.pyramid, solver, warm, 4, 2, True, regions=False, max_colors=3, base_count=14)
    assert c.overflowCount > 0


def test_region_schedule_has_a_cut_set(dev):
    """A pyramid large enough for several blocks: most constraints are interior to a region, the rest form a cut set with
    only a few colours (= device-wide steps per sweep)."""
    c = _case(dev, scenes.pyramid, "TGS_Soft", 5, 4, 2, True, base_count=60)
    assert c.regionCount >= 4 and 0 < c.cutCount < c.constraintCount // 2 and 1 <= c.cutGroupCount <= 8


@pytest.mark.parametrize("solver", VARIANTS)
def test_ticketed_passes_match(dev, solver):
    """Experimental schedule: Gauss-Seidel passes synchronised by per-body tickets instead of one grid barrier per
    colour. Must give the same bits as the default (both are compared with the permuted oracle)."""
    c = _case(dev, scenes.limited_chains, solver, 40, 4, 2, True, dataflow=True)
    assert c.jointCount == 19
    warm = 2 if solver == "Jacobi" else 30
    c = _case(dev, scenes.pyramid, solver, warm, 4, 2, True, dataflow=True, max_colors=3, base_count=14)
    assert c.overflowCount > 0


@pytest.mark.parametrize("base,vel", [(300, 8), (447, 4)])
def test_full_size_configs_match_permuted_oracle(dev, base, vel):
    """BASELINE.json's full sizes — config 2 (45 150 boxes, 134 850 constraints, 8 sub-steps) and the headline workload
    (100 128 boxes, 299 490 constraints, 4 sub-steps): one solver stage of the production schedule against the oracle
    replayed in the device's colour order, every body, tolerance 0."""
    c = _case(dev, scenes.pyramid, "TGS_Soft", 3, vel, 2, True, base_count=base)
    assert c.constraintCount == 3 * (base * (base + 1) // 2) - 2 * base + (base - 1) - (base - 1) or c.constraintCount > 100000
    assert c.overflowCount == 0 and c.groupCount <= 16
    # every box touches six others: six colours is the optimum; greedy leaves a few dozen stragglers in a seventh, which the
    # Kempe-chain pass recolours (s2bKempeKernel) — and the oracle has just replayed the result bit for bit
    print(f"pyramid {base}: colours {c.groupCount}, recoloured by Kempe chains {c.recolouredCount}")
    assert c.groupCount <= 7


# ---- BASELINE.json configs 3, 4, 5 at their full sizes: one solver stage of the production schedule against the oracle
# replayed in the device's order, every body and every impulse, tolerance 0 ----------------------------------------------

@pytest.mark.parametrize("solver", ["PGS", "PGS_NGS", "TGS_NGS", "XPBD", "Jacobi", "TGS_Soft"])
def test_config3_tumbler_full_size(dev, solver):
    """Config 3: the solver-variant sweep on the 10 000-box motorised tumbler, after the boxes have fallen against the
    container (a hub body with hundreds of contacts: overflow group, block-wide warm-start gather)."""
    # the lattice needs ~1.7 s to reach the container floor and ~4 s to pile up; the reference's Jacobi variant blows a
    # pile apart, so it is sampled while the pile forms
    warm = 150 if solver == "Jacobi" else 240
    c = _case(dev, scenes.tumbler, solver, warm, 4, 2, True, grid=100)
    print(f"config 3 {solver}: contact constraints {c.constraintCount}, colours {c.groupCount}, overflow {c.overflowCount}")
    assert c.jointCount == 1 and c.constraintCount > (500 if solver == "Jacobi" else 9000)


def test_config4_joints_and_contacts_full_size(dev):
    """Config 4: 25 bridges x 160 planks = 4 025 revolute joints with the 73 x 73 box lattice landed on them."""
    c = _case(dev, scenes.joint_contact_stress, "TGS_Soft", 420, 4, 2, True)
    print(f"config 4: joints {c.jointCount}, contact constraints {c.constraintCount}, colours {c.groupCount}, overflow {c.overflowCount}")
    assert c.jointCount == 4025 and c.constraintCount > 8000


def test_config5_field_full_size(dev):
    """Config 5: 256 independent 1 035-box pyramid worlds batched into one constraint graph (264 960 boxes)."""
    c = _case(dev, scenes.pyramid_field, "TGS_Soft", 2, 4, 2, True, count=256, base_count=45)
    assert c.constraintCount > 700000 and c.overflowCount == 0


def test_kempe_pass_reaches_six_colours_on_the_headline_pyramid(dev):
    """The bench workload through the public API: greedy colouring leaves 36 of 299 490 constraints in a seventh colour, the
    Kempe-chain pass moves them into the six below (every box touches six others: the optimum), and the colours persist."""
    P = capi.Solver2D(device.LIB_PATH)
    sc = scenes.pyramid(P, "TGS_Soft", base_count=447)
    dw = device.DeviceWorld.attach(dev, sc.world)
    for _ in range(3):
        sc.step(DT, 4, 2, True)
    c = dw.counters()
    sc.destroy()
    assert c.constraintCount > 290000 and c.overflowCount == 0
    assert c.groupCount == 6 and c.recolouredCount >= 30
