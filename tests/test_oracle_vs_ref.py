"""Oracle pinned against the reference itself: against its recorded runs (tests/golden/reference_runs.npz) everywhere, and against
a reference build (oracle/_ref) where one was made.  Larger than the golden fixtures."""
import numpy as np
import pytest

import reference_golden
import scenes
from conftest import have_ref
from parity_util import perturb

needs_ref = pytest.mark.skipif(not (have_ref("f32") and have_ref("f64")), reason="oracle/_ref not built (no /root/reference here)")

CASES = {
    "cfg1": lambda m: scenes.cfg1(m, 50),
    "cloth_xpbd_64": lambda m: scenes.cfg2(m, 64, 8),
    "cloth_fem_dihedral": lambda m: scenes.cloth(m, 30, 30, 2, 1, fem=(1000.0, 1000.0, 500.0, 0.3, 0.3)),
    "cfg3_small": lambda m: scenes.cfg3(m, 14, 5, 5),
    "bar_xpbd": lambda m: scenes.bar(m, 10, 4, 4, 6, k=1e5, vol_k=1e5),
    "bar_strain": lambda m: scenes.bar(m, 10, 4, 4, 4, k=1.0),
    "bar_femx_1step": lambda m: scenes.bar(m, 7, 4, 4, 3, k=1.0e4, sub_steps=2, max_iter=3),
}


def steps_of(name):
    return 1 if name.endswith("1step") else 3  # XPBD-FEM amplifies rounding differences chaotically after a step


@pytest.mark.parametrize("name", sorted(CASES))
def test_structure_and_trajectory(name, cpu_libs):
    """The reference's side is the recorded run of tests/golden/reference_runs.npz (same builder, perturbation and steps)."""
    for prec, tol in (("f64", 1e-9), ("f32", 5e-5)):
        key = "oracle_vs_ref/%s/%s/" % (name, prec)
        o = cpu_libs.CpuPbd("oracle", prec)
        CASES[name](o)
        to, bo, po, _ = o.constraints()
        reference_golden.assert_structure(key, to, bo, *o.groups())
        p_ref, p_got, p_scale = reference_golden.sampled(key, "params", po, reference_golden.PARAM_ROWS)
        assert np.abs(p_got - p_ref).max() <= tol * p_scale
        perturb([o], 0.01)
        o.step(steps_of(name))
        x_ref, x_got, x_scale = reference_golden.sampled(key, "x", o.get("x"))
        err = np.abs(x_got - x_ref).max() / x_scale
        limit = tol
        if prec == "f32" and name in ("cfg1", "cloth_xpbd_64"):
            limit = 3e-3  # isometric bending in fp32: both sides are inside the reference's own cancellation noise
        if prec == "f32" and name == "bar_femx_1step":
            limit = 2e-3  # sqrt(2U') constraint near the rest state: ill-conditioned in fp32 (reference fp32 vs fp64 differ by 7e-5 here)
        assert err <= limit, (name, prec, err)


@needs_ref
def test_thread_count_does_not_change_results(cpu_libs):
    """Colours make the parallel Gauss-Seidel deterministic (SURVEY.md F6)."""
    r = cpu_libs.CpuPbd("ref", "f32")
    out = []
    for threads in (1, 4):
        r.reset(); r.set_threads(threads)
        scenes.cfg1(r, 40)
        r.step(5)
        out.append(r.get("x"))
    assert (out[0] == out[1]).all()


def test_reference_side_adapter_is_built_and_fails_loudly_without_a_gpu():
    """oracle/_ref/libpbdref_gpu_*.so = the unmodified reference + integration/GpuTimeStepController.h (the PBD::TimeStep subclass
    that binds libpbd_b200.so).  Here (no GPU) installing it must fail with the engine's "no CUDA device" message, never fall
    back to a CPU path; the GPU parity of the adapter is tests/test_gpu_parity.py::test_reference_side_adapter."""
    import torch
    from oracle import pyoracle
    for precision in ("f32", "f64"):
        if not pyoracle.available("refgpu", precision):
            pytest.skip("oracle/_ref/libpbdref_gpu_%s.so not built (no /root/reference here)" % precision)
        m = pyoracle.CpuPbd("refgpu", precision)
        scenes.cloth(m, 6, 6, 4, 3, dist_k=1e5, bend_k=100.0)
        if torch.cuda.is_available():
            m.use_gpu_timestep(0, 0)
            m.step(1)
            assert m.gpu_error() == ""
        else:
            with pytest.raises(RuntimeError, match="no CUDA device"):
                m.use_gpu_timestep(0, 0)
            x0 = m.get("x").copy()
            m.step(1)  # the reference's own TimeStepController is still installed and still works
            assert np.abs(m.get("x") - x0).max() > 0


CONTACT_STEPS = 110
CHECKPOINTS = (40, 60, 80, 100, 110)  # fp64: velocities compared along the free run (the first contacts appear around step 35)
LOCKSTEP_STEPS = (60, 90)             # fp32: single steps from the reference's state


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_contact_path_restatement_is_pinned_to_the_reference(precision, cpu_libs):
    """The C restatement of the contact path (oracle/pbd_oracle.c: distance functions, collisionTest, contact initialisation, velocity-level
    solve) against the reference's DistanceFieldCollisionDetection + ParticleRigidBodyContactConstraint in the same precision, as recorded
    in tests/golden/reference_runs.npz: 110 steps of a cloth falling onto all six analytic shapes -- the same contact list after every
    step, and velocities that agree to rounding (the two sides evaluate the same formulas in the same precision).  In fp64 the velocities
    are compared along the free run; in fp32, whose rounding differences grow over a free run, after single steps taken from the
    reference's state."""
    # Real = float: the reference takes the torus' ring distance from a float norm (Vector2r(x, z).norm(), DistanceFieldCollisionDetection.cpp:635);
    # the central differences of approximateNormal (eps = 1e-6) then differentiate rounding noise and the normal is off by percent in a
    # rounding-dependent direction -- nothing to pin there, so the float run leaves the torus out (the double run has all six shapes)
    orc = cpu_libs.CpuPbd("oracle", precision)
    scenes.on_recorded_colliders(orc, "cloth_all_shapes" if precision == "f64" else "cloth_no_torus_f32")
    key = "contact_run/%s/" % precision
    counts = reference_golden.get(key + "counts"); pairs = [tuple(q) for q in reference_golden.get(key + "pairs").tolist()]
    starts = np.concatenate([[0], np.cumsum(counts, dtype=np.int64)])
    events = 0; worst_dv = 0.0; grazing = 0

    def compare_contacts(step):
        a = set(pairs[starts[step - 1]:starts[step]])  # the reference's contacts of this step
        po, bo, _ = orc.oracle_contacts()
        c = set(zip(po.tolist(), bo.tolist()))
        if a != c:  # only a contact whose signed distance is at the rounding level may be on one side only (never in fp64)
            assert precision == "f32" and len(a ^ c) <= 2, "step %d: contact lists differ: %s" % (step, sorted(a ^ c))
        return a, a ^ c

    def velocity_error(step, one_sided):
        v_ref, v_got, _ = reference_golden.sampled(key, "v%d" % step, orc.get("v"))
        dv = np.abs(v_got - v_ref).max(axis=1)
        dv[np.isin(reference_golden.sample_rows(orc.num_particles()), [q for q, _ in one_sided])] = 0.0
        return float(dv.max())

    tol_v = 1e-9 if precision == "f64" else 5e-3  # float: the penalty impulse (stiffness 100 x depth) amplifies the rounding of the positions; a flipped contact would be 0.1 - 2 m/s
    for step in range(1, CONTACT_STEPS + 1):
        orc.step(1)
        a, one_sided = compare_contacts(step)
        grazing += len(one_sided); events += len(a)
        if precision == "f64" and step in CHECKPOINTS:
            worst_dv = max(worst_dv, velocity_error(step, one_sided))
    if precision == "f32":
        for step in LOCKSTEP_STEPS:
            orc.set("x", reference_golden.get(key + "x_before%d" % step)); orc.set("v", reference_golden.get(key + "v_before%d" % step))
            orc.step(1)
            _, one_sided = compare_contacts(step)
            grazing += len(one_sided)
            worst_dv = max(worst_dv, velocity_error(step, one_sided))
    print("contact restatement, %s: %d contact events, %d grazing, worst |dv| %.2e" % (precision, events, grazing, worst_dv))
    assert events > 2000 and grazing <= 4 and worst_dv <= tol_v
