"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU checkers on identical seeded scenes.

Tolerance (north_star): <= 1e-4 relative on particle positions after the configured iterations.  The engine is fp32;
the checker is the fp64 build of the CPU restatement (== the reference's default precision, SURVEY.md F4) and, when the
prebuilt oracle/_ref travelled to this box, the unmodified reference itself.  Scenes with IsometricBending are gated
against fp64 only: the fp32 reference is dominated by cancellation noise there (DESIGN.md "Parity").
"""
import numpy as np
import pytest

import reference_golden
import scenes
from parity_util import perturb, rel_position_error, rel_displacement_error
from conftest import have_ref

pytestmark = pytest.mark.gpu

TOL = 1e-4       # relative on positions (north_star)
TOL_DISP = 5e-3  # relative to the distance the particles moved in the test (measured 1e-4 ... 1.4e-3)

SCENES = {
    # name: (builder, perturbation amplitude, steps)
    "cloth_distance": (lambda m: scenes.cloth(m, 24, 24, 1, 0, dist_k=1.0, max_iter=5), 0.02, 3),
    "cloth_distance_xpbd": (lambda m: scenes.cloth(m, 24, 24, 4, 0, dist_k=1.0e5, max_iter=5), 0.02, 3),
    "cloth_isobending": (lambda m: scenes.cloth(m, 24, 24, 1, 2, bend_k=0.5, max_iter=5), 0.02, 3),
    "cloth_isobending_xpbd": (lambda m: scenes.cloth(m, 24, 24, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=5), 0.02, 3),
    "cloth_dihedral": (lambda m: scenes.cloth(m, 24, 24, 1, 1, bend_k=0.5, max_iter=5), 0.02, 3),
    "cloth_femtriangle": (lambda m: scenes.cloth(m, 24, 24, 2, 0, fem=(1000.0, 1000.0, 500.0, 0.3, 0.3), max_iter=5), 0.02, 3),
    "cloth_straintriangle": (lambda m: scenes.cloth(m, 24, 24, 3, 0, max_iter=5), 0.02, 3),
    "cfg1_50x50": (lambda m: scenes.cfg1(m, 50), 0.01, 2),
    "bar_distance_volume": (lambda m: scenes.bar(m, 9, 4, 4, 1, k=1.0, sub_steps=2, max_iter=3), 0.01, 3),
    "bar_femtet": (lambda m: scenes.bar(m, 9, 4, 4, 2, k=1.0e6, sub_steps=2, max_iter=3), 0.01, 3),
    # XPBD-FEM (C = sqrt(2U')) amplifies rounding differences chaotically: the reference's own fp32 and fp64 builds differ
    # by 7e-5 relative after ONE step of this scene and by O(1) after three (DESIGN.md "Parity"); one step, E = 1e4.
    "bar_femtet_xpbd": (lambda m: scenes.bar(m, 7, 4, 4, 3, k=1.0e4, sub_steps=2, max_iter=3), 0.01, 1),
    "bar_straintet": (lambda m: scenes.bar(m, 9, 4, 4, 4, k=1.0, sub_steps=2, max_iter=3), 0.01, 3),
    "bar_shapematching": (lambda m: scenes.bar(m, 9, 4, 4, 5, k=0.5, sub_steps=2, max_iter=3), 0.02, 3),
    "bar_distance_volume_xpbd": (lambda m: scenes.bar(m, 9, 4, 4, 6, k=1.0e5, vol_k=1.0e5, sub_steps=2, max_iter=3), 0.01, 3),
    "bar_fem_plus_volume": (lambda m: scenes.bar(m, 9, 4, 4, 2, k=1.0e6, extra_volume=True, sub_steps=3, max_iter=2), 0.01, 3),
    # cfg4 without rigid bodies: cloth (FEMTriangle + IsometricBending) and a tet solid (FEMTet) in one model
    "mixed_cloth_solid": (lambda m: scenes.mixed(m), 0.01, 3),
    "mixed_cloth_solid_distance_volume": (lambda m: scenes.mixed(m, cloth_method=1, bending_method=1, solid_method=1, max_iter=3), 0.01, 3),
}


def _run(name, mode, cpu_libs, checker_kind):
    from positionbaseddynamics_b200.model import HostModel
    build, amp, steps = SCENES[name]
    gpu = HostModel(); cpu = cpu_libs.CpuPbd(checker_kind, "f64")
    build(gpu); build(cpu)
    # identical structure first (integers: exact)
    tg, bg, _, _ = gpu.constraints(); tc, bc, _, _ = cpu.constraints()
    assert (tg == tc).all() and (bg == bc).all()
    og, ig = gpu.groups(); oc, ic = cpu.groups()
    assert (og == oc).all() and (ig == ic).all()
    x_start = perturb([gpu, cpu], amp)
    gpu.time_step().set_mode(mode)
    gpu.step(steps); cpu.step(steps)
    xg, xc = gpu.get("x"), cpu.get("x")
    vg, vc = gpu.get("v"), cpu.get("v")
    assert np.isfinite(xg).all()
    e_pos = rel_position_error(xg, xc)
    e_disp = rel_displacement_error(xg, xc, x_start)
    e_vel = float(np.abs(vg - vc).max() / max(np.abs(vc).max(), 1e-30))
    print("%s mode=%d checker=%s: rel pos %.2e, rel disp %.2e, rel vel %.2e" % (name, mode, checker_kind, e_pos, e_disp, e_vel))
    tol = 5e-4 if name == "bar_femtet_xpbd" else TOL  # see the comment at the scene definition
    assert e_pos <= tol, (name, e_pos)
    if name != "bar_femtet_xpbd":
        assert e_disp <= TOL_DISP, (name, e_disp)
    gpu.close()
    return xg


@pytest.mark.parametrize("name", sorted(SCENES))
def test_scene_vs_oracle_f64(name, cpu_libs):
    _run(name, 0, cpu_libs, "oracle")


@pytest.mark.parametrize("name", sorted(SCENES))
def test_scene_vs_reference_f64(name):
    """The same gates as _run, with the reference's recorded fp64 run of the scene (tests/golden/reference_runs.npz) as the checker:
    structure bit for bit, positions on the recorded sample of particles, relative to the scales of the whole run."""
    from positionbaseddynamics_b200.model import HostModel
    build, amp, steps = SCENES[name]
    key = "gpu_parity/%s/" % name
    gpu = HostModel()
    build(gpu)
    tg, bg, _, _ = gpu.constraints()
    reference_golden.assert_structure(key, tg, bg, *gpu.groups())
    perturb([gpu], amp)
    gpu.time_step().set_mode(0)
    gpu.step(steps)
    xg = gpu.get("x")
    assert np.isfinite(xg).all()
    x_ref, x_got, x_scale = reference_golden.sampled(key, "x", xg)
    d = np.abs(x_got.astype(np.float64) - x_ref).max()
    e_pos, e_disp = d / x_scale, d / reference_golden.get(key + "disp_scale")
    print("%s vs recorded reference: rel pos %.2e, rel disp %.2e" % (name, e_pos, e_disp))
    assert e_pos <= (5e-4 if name == "bar_femtet_xpbd" else TOL), (name, e_pos)
    if name != "bar_femtet_xpbd":
        assert e_disp <= TOL_DISP, (name, e_disp)
    gpu.close()


def test_mode_switch_keeps_state_bitwise():
    """Switching to the resident mode permutes every particle array on the device (tile-major order) and back; the simulation
    state must survive both moves bit for bit and the uploads/downloads in between must address the right particles."""
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    nx = 40
    hm = HostModel()
    hm.add_regular_triangle_model(nx, nx, (0, 0, 0), np.eye(3), (4.0, 4.0))
    for i in (0, nx - 1):
        hm.set_mass(i, 0.0)
    hm.add_cloth_constraints(0, 4, 1e5)   # Distance_XPBD on the edges
    hm.add_bending_constraints(0, 3, 50.0)  # IsometricBending_XPBD
    types, bodies, params, nb = hm.constraints()
    x = hm.get("x"); mass, _ = hm.masses()

    def run(schedule):
        eng = _capi.Engine(0)
        eng.set_particles(x, mass)
        eng.add_flat(types, bodies, params)
        eng.color_first_fit()
        eng.set_params(dt=0.005, sub_steps=2, max_iter=5)
        for mode, steps in schedule:
            eng.set_mode(mode); eng.step(steps); eng.sync()
            v = eng.get_attr(_capi.ATTR_V); eng.set_attr(_capi.ATTR_V, v)  # round trip through the host in the current layout
        out = eng.get_attr(_capi.ATTR_X), eng.get_attr(_capi.ATTR_V), eng.get_attr(_capi.ATTR_OLDX)
        eng.close()
        return out
    a = run([(_capi.MODE_GRAPH, 6)])
    b = run([(_capi.MODE_GRAPH, 2), (_capi.MODE_RESIDENT, 2), (_capi.MODE_LAUNCH, 1), (_capi.MODE_RESIDENT, 1)])
    for u, w in zip(a, b):
        assert np.isfinite(u).all() and (u == w).all()


ADAPTER_SCENES = ["cloth_isobending_xpbd", "cloth_femtriangle", "cloth_dihedral", "bar_fem_plus_volume", "bar_straintet", "bar_shapematching",
                  "mixed_cloth_solid", "cfg4_small_with_rig"]


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ADAPTER_SCENES)
def test_reference_side_adapter(name, precision, cpu_libs):
    """The drop-in proper.  integration/GpuTimeStepController.h -- the PBD::TimeStep subclass a maintainer adds to the reference --
    is compiled inside a build of the unmodified reference (oracle/_ref/libpbdref_gpu_*.so, both Real = float and Real = double) and
    installed with Simulation::setTimeStep.  The REFERENCE builds the scene, initialises the constraints and colours them; the
    adapter flattens the model through its public members and steps it with libpbd_b200.so.  A twin scene stepped by the
    reference's own TimeStepController (fp64) is the yardstick."""
    _reference_side_adapter(name, precision, 0, cpu_libs)


@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", ADAPTER_SCENES)
def test_reference_side_adapter_auto_mode(name, precision, cpu_libs):
    """test_reference_side_adapter with the adapter in PBD_MODE_AUTO, the default of a user: the resident kernel for the cloth and
    FEM scenes, the graph mode for the others."""
    _reference_side_adapter(name, precision, 4, cpu_libs)


def _reference_side_adapter(name, precision, mode, cpu_libs):
    from oracle import pyoracle
    if not (pyoracle.available("refgpu", precision) and have_ref("f64")):
        pytest.skip("prebuilt oracle/_ref/libpbdref_gpu_%s.so not present on this box" % precision)
    if name == "cfg4_small_with_rig":
        build, amp, steps = (lambda m: scenes.cfg4(m, n_cloth=32, bar_dims=(7, 4, 4))), 0.0, 6
    else:
        build, amp, steps = SCENES[name]
    gpu = cpu_libs.CpuPbd("refgpu", precision); cpu = cpu_libs.CpuPbd("ref", "f64")
    build(gpu); build(cpu)
    gpu.use_gpu_timestep(0, mode)
    x_start = perturb([gpu, cpu], amp) if amp else cpu.get("x")
    gpu.step(steps); cpu.step(steps)
    assert gpu.gpu_error() == ""
    xg, xc = gpu.get("x"), cpu.get("x")
    assert np.isfinite(xg).all()
    e_pos = rel_position_error(xg, xc)
    print("adapter %s Real=%s mode %d: rel pos %.2e" % (name, precision, mode, e_pos))
    assert e_pos <= TOL, (name, e_pos)
    assert abs(gpu.time() - cpu.time()) < 1e-6       # TimeManager advanced like TimeStepController.cpp:239
    if name == "cfg4_small_with_rig":
        assert np.abs(gpu.rigid_bodies()[:, :7] - cpu.rigid_bodies()[:, :7]).max() <= 1e-4
    assert np.abs(xg - x_start).max() > 1e-4         # the step did something


def _engine_from(hm, with_rb=False):
    from positionbaseddynamics_b200 import _capi
    types, bodies, params, _ = hm.constraints()
    mass, _ = hm.masses()
    eng = _capi.Engine(0)
    eng.set_particles(hm.get("x"), mass, x0=hm.get("x0"))
    if with_rb:
        rb = hm.rigid_bodies()
        eng.set_rigid_bodies(np.ones(len(rb)), rb[:, :3], rb[:, 3:7], np.ones((len(rb), 3)))
    eng.add_flat(types, bodies, params)
    return eng


@pytest.mark.parametrize("name", sorted(SCENES) + ["cfg4_small_with_rig"])
def test_device_colouring_is_the_reference_first_fit(name):
    """SURVEY 8 f-3: the colouring computed on the GPU (wavefronts over the insertion-order dependency DAG) must reproduce the
    sequential greedy first fit exactly: same groups, same order inside the groups, as the host model mirror (which the CPU
    tests pin to the reference's initConstraintGroups) and as the engine's host colouring."""
    from positionbaseddynamics_b200.model import HostModel
    hm = HostModel()
    rig = name == "cfg4_small_with_rig"
    if rig:
        scenes.cfg4(hm, n_cloth=32, bar_dims=(7, 4, 4))
    else:
        SCENES[name][0](hm)
    hm.init_groups()
    off_ref, ids_ref = hm.groups()
    eng = _engine_from(hm, with_rb=rig)
    eng.color_first_fit()
    off_h, ids_h = eng.groups()
    ms, fronts = eng.color_first_fit_device()
    off_d, ids_d = eng.groups()
    assert fronts > 0
    assert (off_h == off_ref).all() and (ids_h == ids_ref).all()
    assert len(off_d) == len(off_ref) and (off_d == off_ref).all() and (ids_d == ids_ref).all()
    eng.step(1); eng.sync()  # and the groups are accepted by the flattening (valid colouring check)
    eng.close()


def test_device_colouring_more_than_128_colours():
    """A star: 200 distance constraints sharing particle 0 need 200 colours; the used-colour sets start at 128 bits and grow."""
    from positionbaseddynamics_b200 import _capi
    n = 201
    x = np.zeros((n, 3), np.float32); x[:, 0] = np.arange(n)
    eng = _capi.Engine(0)
    eng.set_particles(x, np.ones(n, np.float32))
    b = np.stack([np.zeros(n - 1, np.uint32), np.arange(1, n, dtype=np.uint32)], axis=1)
    eng.add_constraints(_capi.DISTANCE, b, np.stack([np.arange(1, n, dtype=np.float32), np.ones(n - 1, np.float32)], axis=1))
    eng.color_first_fit_device()
    off, ids = eng.groups()
    assert len(off) - 1 == n - 1 and (ids == np.arange(n - 1)).all()
    eng.close()


def _kat_engine(x, w, cases, dt, mode, clusters=None):
    """One engine holding `cases` = [(type, params row)], case j on particles 4j..4j+3: one step of 1 substep x 1 iteration without
    gravity.  Returns the corrections [len(cases), 4, 3] and the multipliers by case (NaN for non-XPBD types)."""
    import os
    from positionbaseddynamics_b200 import _capi
    if clusters:
        os.environ["PBD_B200_CLUSTERS"] = clusters
    try:
        eng = _capi.Engine(0)
        try:
            mass = np.where(w != 0, 1.0 / np.where(w != 0, w, 1.0), 0.0).astype(np.float32)
            eng.set_particles(x, mass)
            for j, (t, p) in enumerate(cases):
                eng.add_constraints(t, np.arange(4 * j, 4 * j + _capi.num_bodies(t)), p[:_capi.num_params(t)])
            eng.color_first_fit()
            eng.set_params(dt=float(dt), sub_steps=1, max_iter=1, gravity=(0, 0, 0))
            eng.set_mode(mode)
            eng.step(1); eng.sync()
            got = (eng.get_attr(_capi.ATTR_X).astype(np.float64) - x.astype(np.float64)).reshape(-1, 4, 3)
            lam = np.full(len(cases), np.nan)
            for t in (_capi.DISTANCE_XPBD, _capi.ISOBENDING_XPBD, _capi.VOLUME_XPBD, _capi.FEMTET_XPBD):
                if any(c[0] == t for c in cases):
                    vals, ids = eng.lambdas(t); lam[ids] = vals
        finally:
            eng.close()
    finally:
        os.environ.pop("PBD_B200_CLUSTERS", None)
    return got, lam


def _known_answers(mode, clusters=None):
    import os
    from positionbaseddynamics_b200 import _capi
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kat_f64.npz"))
    T = d["solve_type"]; X = d["solve_x"]; W = d["solve_w"]; P = d["solve_p"]; DT = d["solve_dt"]
    ok = d["solve_lam0"] == 0.0  # the engine zeroes lambda at the first sweep of a substep, like the constraint classes do
    # FEM: the constraint classes derive handleInversion from the current volume (Constraints.cpp:1795-1798); keep the
    # golden cases whose recorded flag agrees with that rule
    for i in range(len(T)):
        if T[i] in (_capi.FEMTET, _capi.FEMTET_XPBD):
            x = X[i]; vol = np.dot(np.cross(x[1] - x[0], x[2] - x[0]), x[3] - x[0]) / 6.0
            ok[i] &= (bool(d["solve_hinv"][i]) == bool(vol / P[i][0] < 0.2))
    worst = {}; worst_lam = 0.0
    for dt in np.unique(DT):
        sel = np.nonzero(ok & (DT == dt))[0]
        x = X[sel].reshape(-1, 3).astype(np.float32)
        w = W[sel].reshape(-1)
        got, lam = _kat_engine(x, w, [(int(T[i]), P[i]) for i in sel], dt, mode, clusters)
        for j, i in enumerate(sel):
            ref = d["solve_corr"][i].copy()
            if not d["solve_res"][i]:
                ref[:] = 0.0
            ref[W[i] == 0] = 0.0  # corrections are applied to dynamic particles only
            sc = max(np.abs(ref).max(), 1e-3)
            err = np.abs(got[j] - ref).max() / sc
            worst[int(T[i])] = max(worst.get(int(T[i]), 0.0), err)
            # fp32 kernels vs fp64 reference answers on O(1) stencils a few units from the origin
            assert err <= 5e-4, (int(T[i]), int(i), err, got[j], ref)
            if not np.isnan(lam[j]):  # XPBD: the multiplier after the solve
                e_lam = abs(lam[j] - d["solve_lam1"][i]) / max(abs(d["solve_lam1"][i]), 1e-3)
                worst_lam = max(worst_lam, e_lam)
                assert e_lam <= 5e-4, (int(T[i]), int(i), e_lam, lam[j], d["solve_lam1"][i])
    print("GPU known answers (mode %d%s), worst relative error per type:" % (mode, ", clusters " + clusters if clusters else ""),
          {_capi.TYPE_NAMES[k]: "%.1e" % v for k, v in sorted(worst.items())}, "multipliers %.1e" % worst_lam)
    assert len(worst) == 13


def test_known_answers_against_reference_golden():
    """Per-function known answers: the golden inputs/outputs recorded from the reference's stateless solve_* functions
    (tests/golden/kat_f64.npz) replayed through the CUDA kernels.  Every case becomes one constraint on four private
    particles (one colour, no coupling), gravity off, 1 substep x 1 iteration, so x_after - x_before is the correction."""
    from positionbaseddynamics_b200 import _capi
    _known_answers(_capi.MODE_LAUNCH)


@pytest.mark.parametrize("mode", ["graph", "resident", "resident_4x1", "jacobi"])
def test_known_answers_through_every_mode(mode):
    """The known answers of test_known_answers_against_reference_golden through the other execution paths: the graph mode, the
    resident kernel (its default shape, one cluster; and 4 independent CTAs, where stencils split between CTAs run as X items through
    global memory) and the Jacobi mode, which equals Gauss-Seidel here because no two cases share a particle."""
    from positionbaseddynamics_b200 import _capi
    m, clusters = {"graph": (_capi.MODE_GRAPH, None), "resident": (_capi.MODE_RESIDENT, None),
                   "resident_4x1": (_capi.MODE_RESIDENT, "4x1"), "jacobi": (_capi.MODE_JACOBI, None)}[mode]
    _known_answers(m, clusters)


def test_known_answers_full_q_bending(cpu_libs):
    """IsometricBending with a Q that is not of the rank-one form (a user-modified Q): the full-Q projection (layout variant 1) of the
    launch, graph and Jacobi modes against the fp64 checker's solver on the same parameter row; the resident mode refuses it."""
    import os
    from positionbaseddynamics_b200 import _capi
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kat_f64.npz"))
    T = d["solve_type"]
    sel = np.nonzero(np.isin(T, (_capi.ISOBENDING, _capi.ISOBENDING_XPBD)) & (d["solve_lam0"] == 0.0))[0]
    rng = np.random.RandomState(31)
    rows = []
    for i in sel:
        p = d["solve_p"][i].copy()
        Q = p[1:17].reshape(4, 4)
        S = rng.uniform(-1.0, 1.0, (4, 4)); S = 0.5 * (S + S.T)
        p[1:17] = (Q + 0.3 * np.abs(Q).max() * S).reshape(-1)
        rows.append(p.astype(np.float32).astype(np.float64))  # what the engine sees, exactly
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    worst = 0.0
    for dt in np.unique(d["solve_dt"][sel]):
        js = [j for j, i in enumerate(sel) if d["solve_dt"][i] == dt]
        x = d["solve_x"][sel[js]].reshape(-1, 3).astype(np.float32)
        w = d["solve_w"][sel[js]].reshape(-1)
        cases = [(int(T[sel[j]]), rows[j]) for j in js]
        ref = []
        for k, j in enumerate(js):
            res, corr, lam = cpu.kat_solve(cases[k][0], x[4 * k:4 * k + 4].astype(np.float64), w[4 * k:4 * k + 4], rows[j], dt=float(dt))
            corr = corr if res else np.zeros((4, 3))
            corr[w[4 * k:4 * k + 4] == 0] = 0.0
            ref.append((corr, lam))
        for mode in (_capi.MODE_LAUNCH, _capi.MODE_GRAPH, _capi.MODE_JACOBI):
            got, lam = _kat_engine(x, w, cases, dt, mode)
            for k in range(len(js)):
                corr, lam_ref = ref[k]
                err = np.abs(got[k] - corr).max() / max(np.abs(corr).max(), 1e-3)
                worst = max(worst, err)
                assert err <= 5e-4, (mode, cases[k][0], err, got[k], corr)
                if cases[k][0] == _capi.ISOBENDING_XPBD:
                    assert abs(lam[k] - lam_ref) <= 5e-4 * max(abs(lam_ref), 1e-3), (mode, lam[k], lam_ref)
        with pytest.raises(_capi.PbdError):
            _kat_engine(x, w, cases, dt, _capi.MODE_RESIDENT)
    print("full-Q IsometricBending known answers: worst relative error %.1e" % worst)


def test_engine_level_drop_in(cpu_libs):
    """The drop-in seam: a model built by the CPU side (stand-in for a reference SimulationModel) is flattened into the
    engine-level C ABI (pbd_set_particles / pbd_add_constraints / pbd_set_groups / pbd_step) -- INTEGRATION.md."""
    from positionbaseddynamics_b200 import _capi
    cpu = cpu_libs.CpuPbd("ref" if have_ref("f64") else "oracle", "f64")
    scenes.cloth(cpu, 20, 20, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=4)
    perturb([cpu], 0.02)
    types, bodies, params, _ = cpu.constraints()
    off, ids = cpu.groups()
    mass, _ = cpu.masses()
    eng = _capi.Engine(0)
    eng.set_particles(cpu.get("x"), mass, x0=cpu.get("x0"), v=cpu.get("v"))
    eng.add_flat(types, bodies, params)
    eng.set_groups(off, ids)
    eng.set_params(dt=0.005, sub_steps=1, max_iter=4)
    eng.step(3); eng.sync()
    cpu.step(3)
    e = rel_position_error(eng.get_attr(_capi.ATTR_X), cpu.get("x"))
    print("engine-level drop-in: rel pos %.2e" % e)
    assert e <= TOL
    # multipliers come back per constraint, keyed by the reference's insertion index
    lam, lam_ids = eng.lambdas(_capi.DISTANCE_XPBD)
    assert len(lam) == int((types == _capi.DISTANCE_XPBD).sum()) and np.isfinite(lam).all()
    st = eng.stats()
    assert st.projections == len(types) * 1 * 4 * 3 and st.kernel_launches > 0
    eng.close()


def test_first_fit_in_engine_matches_reference_groups(cpu_libs):
    from positionbaseddynamics_b200 import _capi
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    scenes.bar(cpu, 7, 4, 4, 2, extra_volume=True)
    types, bodies, params, _ = cpu.constraints()
    off, ids = cpu.groups()
    mass, _ = cpu.masses()
    eng = _capi.Engine(0)
    eng.set_particles(cpu.get("x"), mass)
    eng.add_flat(types, bodies, params)
    eng.color_first_fit()
    eng._nc = len(types)
    off2, ids2 = eng.groups()
    assert (off == off2).all() and (ids == ids2).all()
    eng.close()


def test_inverted_tets_take_the_svd_branch(cpu_libs):
    """FEMTet with collapsed/inverted elements exercises svdWithInversionHandling (MathFunctions.cpp:261-388)."""
    from positionbaseddynamics_b200.model import HostModel
    gpu = HostModel(); cpu = cpu_libs.CpuPbd("oracle", "f64")
    for m in (gpu, cpu):
        scenes.bar(m, 5, 3, 3, 2, k=1.0e6, sub_steps=1, max_iter=2)
    x = np.asarray(cpu.get("x")).copy()
    # squash the bar through itself along y: many tets end up with negative volume
    x[:, 1] = -0.6 * x[:, 1]
    m, w = cpu.masses()
    x[w == 0] = np.asarray(cpu.get("x"))[w == 0]
    for mdl in (gpu, cpu):
        mdl.set("x", x.astype(np.float32))
    gpu.step(1); cpu.step(1)
    e = rel_position_error(gpu.get("x"), cpu.get("x"))
    print("inverted tets: rel pos %.2e" % e)
    assert np.isfinite(gpu.get("x")).all()
    assert e <= 1e-3  # the Jacobi eigen-solver in fp32 vs fp64 on near-degenerate F: looser, stated
    gpu.close()


def test_second_order_velocity_update_and_pinned_particles(cpu_libs):
    from positionbaseddynamics_b200.model import HostModel
    gpu = HostModel(); cpu = cpu_libs.CpuPbd("oracle", "f64")
    for m in (gpu, cpu):
        scenes.cloth(m, 16, 16, 1, 0, max_iter=3, sub_steps=2, vel_method=1)
    perturb([gpu, cpu], 0.02)
    gpu.step(4); cpu.step(4)
    assert rel_position_error(gpu.get("x"), cpu.get("x")) <= TOL
    assert np.abs(gpu.get("v") - cpu.get("v")).max() <= 1e-3 * max(np.abs(cpu.get("v")).max(), 1.0)
    assert np.abs(gpu.get("lastX") - cpu.get("lastX")).max() <= 1e-4 * 10
    # pinned corners never move
    assert (gpu.get("x")[0] == gpu.get("x0")[0]).all() and (gpu.get("x")[15] == gpu.get("x0")[15]).all()
    gpu.close()


def test_degenerate_inputs_take_the_reference_branches(cpu_libs):
    """The early-outs of the reference's solvers (SURVEY 8a, "branches the kernel must keep"): both particles static (wSum == 0),
    coincident particles (d <= eps / zero gradient), stiffness 0 (XPBD alpha = 0; PBD volume k == 0 skip), a constraint between a
    static and a dynamic particle, a flat (zero-volume) tetrahedron.  Every constraint sits on its own particles; GPU and fp64
    checker must agree and stay finite."""
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    pts = np.array([[0, 0, 0], [1, 0, 0],            # 0-1   both static, stretched distance
                    [0, 1, 0], [0, 1, 0],            # 2-3   coincident
                    [0, 2, 0], [1.5, 2, 0],          # 4-5   XPBD distance with stiffness 0
                    [0, 3, 0], [1.2, 3, 0],          # 6-7   static + dynamic
                    [0, 4, 0], [1, 4, 0], [0, 5, 0], [1, 5, 0],        # 8-11  flat tetrahedron (volume constraints)
                    [0, 6, 0], [1, 6, 0], [0, 7, 0], [0.3, 6.4, 0.8],  # 12-15 volume constraint with stiffness 0
                    ], dtype=np.float64)
    tris = np.array([[0, 1, 2]], dtype=np.uint32)  # a triangle model only provides the particles' container
    gpu = HostModel(); cpu = cpu_libs.CpuPbd("oracle", "f64")
    for m in (gpu, cpu):
        m.add_triangle_model(pts, np.array([[0, 1, 2], [3, 4, 5], [6, 7, 8], [9, 10, 11], [12, 13, 14], [13, 14, 15]], dtype=np.uint32))
        for i in (0, 1, 6):
            m.set_mass(i, 0.0)
        assert m.add_constraint(_capi.DISTANCE, [0, 1], [1.0])
        assert m.add_constraint(_capi.DISTANCE_XPBD, [2, 3], [1.0e5])
        assert m.add_constraint(_capi.DISTANCE_XPBD, [4, 5], [0.0])
        assert m.add_constraint(_capi.DISTANCE, [6, 7], [1.0])
        m.add_constraint(_capi.VOLUME, [8, 9, 10, 11], [1.0])
        m.add_constraint(_capi.VOLUME_XPBD, [8, 9, 10, 11], [1.0e5])
        assert m.add_constraint(_capi.VOLUME, [12, 13, 14, 15], [0.0])
        m.set_params(dt=0.005, sub_steps=2, max_iter=3)
    # stretch / compress away from the rest state so that the non-degenerate parts of the solvers are active
    x = gpu.get("x").astype(np.float64)
    x[1] += [0.5, 0, 0]; x[5] += [0.3, 0, 0]; x[7] += [0.4, 0, 0]; x[15] += [0.1, 0.1, 0.1]
    gpu.set("x", x); cpu.set("x", x)
    assert gpu.num_constraints() == cpu.num_constraints()
    gpu.step(3); cpu.step(3)
    xg, xc = gpu.get("x"), cpu.get("x")
    assert np.isfinite(xg).all() and np.isfinite(xc).all()
    assert rel_position_error(xg, xc) <= TOL
    assert (xg[0] == x[0].astype(np.float32)).all() and (xg[1] == x[1].astype(np.float32)).all() and (xg[6] == x[6].astype(np.float32)).all()
    gpu.close()


def test_empty_and_constraint_free_models():
    from positionbaseddynamics_b200.model import HostModel
    m = HostModel()
    m.set_params(sub_steps=2, max_iter=2)
    m.step(1)  # no particles, no constraints: a no-op that must not fail
    m.add_regular_triangle_model(4, 4, scale=(1, 1))
    m.step(2)  # free fall, no constraints
    x, x0 = m.get("x"), m.get("x0")
    t = 2 * 0.005
    # semi-implicit Euler with 2 substeps of h=0.0025: y drop = g h^2 (1+2+3+4)
    h = 0.0025
    expect = -9.81 * h * h * 10
    assert np.allclose(x[:, 1] - x0[:, 1], expect, rtol=1e-4, atol=5e-7), (x[:, 1] - x0[:, 1], expect)  # fp32 ulp of x (~1) is 6e-8
    m.close()


def test_rigid_body_coupling_scene(cpu_libs):
    """SURVEY.md 8f-1 / cfg4: cloth + tet solid + the 12-body coupling rig (BallJoint, RigidBodyParticleBallJoint) inside
    the coloured sweep; particles AND rigid-body state against the fp64 checker."""
    from positionbaseddynamics_b200.model import HostModel
    kind = "ref" if have_ref("f64") else "oracle"
    gpu = HostModel(); cpu = cpu_libs.CpuPbd(kind, "f64")
    for m in (gpu, cpu):
        scenes.cfg4(m, 20, (6, 4, 3))
    for _ in range(4):
        gpu.step(5); cpu.step(5)
    e = rel_position_error(gpu.get("x"), cpu.get("x"))
    rg, rc = gpu.rigid_bodies().astype(np.float64), cpu.rigid_bodies()
    e_rb_x = np.abs(rg[:, :3] - rc[:, :3]).max() / np.abs(rc[:, :3]).max()
    e_rb_q = np.abs(rg[:, 3:7] - rc[:, 3:7]).max()
    print("coupling (%s): particles rel %.2e, rigid-body x rel %.2e, q abs %.2e, |omega| max %.3f" % (kind, e, e_rb_x, e_rb_q, np.abs(rc[:, 10:]).max()))
    assert e <= TOL and e_rb_x <= TOL and e_rb_q <= 1e-4
    assert np.abs(rc[:, 7:]).max() > 1e-3  # the rig actually moves
    # static anchors (mass 0) never move
    assert (rg[0, :3] == np.array([-5.0, 0.0, -5.0])).all()
    gpu.close()


def test_engine_level_drop_in_with_rigid_bodies(cpu_libs):
    """The C-ABI call sequence of INTEGRATION.md for a coupled model: pbd_set_rigid_bodies before the joints are added."""
    from positionbaseddynamics_b200 import _capi
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    scenes.cfg4(cpu, 16, (5, 3, 3))
    types, bodies, params, _ = cpu.constraints()
    off, ids = cpu.groups()
    mass, _ = cpu.masses()
    rb = cpu.rigid_bodies(); rb0 = rb.copy()
    eng = _capi.Engine(0)
    eng.set_particles(cpu.get("x"), mass, x0=cpu.get("x0"))
    rb_mass = [0.0 if i % 3 == 0 else 1.0 for i in range(12)]
    inertia = [scenes.box_inertia(1.0, 0.5, 0.5, 0.5) if i % 3 == 0 else scenes.box_inertia(1.0, 0.4, 2.0, 0.4) for i in range(12)]
    eng.set_rigid_bodies(rb_mass, rb[:, :3], rb[:, 3:7], inertia)
    eng.add_flat(types, bodies, params)
    eng.set_groups(off, ids)
    eng.set_params(dt=0.005, sub_steps=5, max_iter=1)
    eng.step(6); eng.sync(); cpu.step(6)
    assert rel_position_error(eng.get_attr(_capi.ATTR_X), cpu.get("x")) <= TOL
    assert np.abs(eng.get_rigid_bodies()[:, :7] - cpu.rigid_bodies()[:, :7]).max() <= 1e-4
    # the resident cluster kernel runs the joints inside its colour phases: same bits as the graph mode
    x_graph, rb_graph = eng.get_attr(_capi.ATTR_X), eng.get_rigid_bodies()
    eng2 = _capi.Engine(0)
    eng2.set_particles(cpu.get("x0"), mass, x0=cpu.get("x0"))
    eng2.set_rigid_bodies(rb_mass, rb0[:, :3], rb0[:, 3:7], inertia)
    eng2.add_flat(types, bodies, params)
    eng2.set_groups(off, ids)
    eng2.set_params(dt=0.005, sub_steps=5, max_iter=1)
    eng2.set_mode(_capi.MODE_RESIDENT)
    eng2.step(6); eng2.sync()
    assert (eng2.get_attr(_capi.ATTR_X) == x_graph).all()
    assert (eng2.get_rigid_bodies() == rb_graph).all()
    eng2.close()
    eng.close()


def test_jacobi_comparison_mode():
    """PBD_MODE_JACOBI (north_star: "a Jacobi path uses atomicAdd for comparison"): colours ignored, corrections accumulated with
    float4 atomicAdd and averaged.  Not the reference's algorithm, so no parity gate; checked for what it must do: (1) on constraints
    that share no particle it equals the Gauss-Seidel result up to rounding, (2) on a cloth it reduces the constraint violation that a
    projection-free step leaves, and stays finite."""
    from positionbaseddynamics_b200 import _capi
    # (1) 512 disjoint distance constraints, stretched by 10 %
    n = 1024
    x = np.zeros((n, 3), np.float32); x[:, 0] = np.arange(n) * 1.0; x[1::2, 0] += 0.1
    b = np.arange(n, dtype=np.uint32).reshape(-1, 2)
    out = []
    for mode in (_capi.MODE_GRAPH, _capi.MODE_JACOBI):
        eng = _capi.Engine(0)
        eng.set_particles(x, np.ones(n, np.float32))
        eng.add_constraints(_capi.DISTANCE, b, np.stack([np.ones(n // 2, np.float32), np.full(n // 2, 0.5, np.float32)], axis=1))
        eng.color_first_fit(); eng.set_params(dt=0.005, sub_steps=1, max_iter=3, gravity=(0, 0, 0)); eng.set_mode(mode)
        eng.step(2); eng.sync(); out.append(eng.get_attr(_capi.ATTR_X).copy()); eng.close()
    assert np.abs(out[0] - out[1]).max() <= 2e-6
    assert np.abs(out[0] - x).max() > 1e-2  # the constraints did pull the pairs together
    # (2) cloth: violation of the distance constraints after 3 steps with and without projections
    from positionbaseddynamics_b200.model import HostModel
    def violation(mode, constraints=True):
        m = HostModel()
        m.add_regular_triangle_model(24, 24, t=(0, 1, 0), R=scenes.RX90, scale=(10.0, 10.0))
        m.set_mass(0, 0.0); m.set_mass(23, 0.0)
        m.add_cloth_constraints(0, 4, dist_k=1.0e5)
        types, bodies, params, _ = m.constraints()
        rest = params[:, 0].copy(); pairs = bodies[:, :2].astype(np.int64)
        if not constraints:
            m.close(); m = HostModel()
            m.add_regular_triangle_model(24, 24, t=(0, 1, 0), R=scenes.RX90, scale=(10.0, 10.0))
            m.set_mass(0, 0.0); m.set_mass(23, 0.0)
        m.set_params(dt=0.005, sub_steps=1, max_iter=10)
        perturb([m], 0.05)
        m.time_step().set_mode(mode)
        m.step(3)
        xx = m.get("x").astype(np.float64); m.close()
        assert np.isfinite(xx).all()
        return np.abs(np.linalg.norm(xx[pairs[:, 0]] - xx[pairs[:, 1]], axis=1) - rest).mean()
    v_free = violation(_capi.MODE_GRAPH, constraints=False)
    v_gs = violation(_capi.MODE_GRAPH)
    v_jac = violation(_capi.MODE_JACOBI)
    print("mean |d - rest|: no projections %.3e, Gauss-Seidel %.3e, Jacobi %.3e" % (v_free, v_gs, v_jac))
    assert v_gs < 0.2 * v_free and v_jac < 0.6 * v_free


def test_adapter_refuses_models_with_collision_objects(cpu_libs):
    """TimeStepController.cpp:189-196 (collision detection + velocityConstraintProjection over the contacts): the GPU path covers
    DistanceFieldCollisionDetection with static analytic bodies (tests/test_gpu_contacts.py); with any other collision detection
    GpuTimeStepController must refuse the model with lastError() instead of silently simulating it without contacts."""
    from oracle import pyoracle
    if not pyoracle.available("refgpu", "f32"):
        pytest.skip("prebuilt oracle/_ref/libpbdref_gpu_f32.so not present on this box")
    gpu = cpu_libs.CpuPbd("refgpu", "f32")
    scenes.cloth(gpu, 12, 12, 1, 2, dist_k=1.0, bend_k=0.01, max_iter=3)
    gpu.use_gpu_timestep(0, 0)
    gpu.step(1)
    assert gpu.gpu_error() == ""
    x1 = gpu.get("x").copy()
    assert gpu.attach_collision_object() == 1
    gpu.step(1)
    assert "collision" in gpu.gpu_error() and "CPU TimeStepController" in gpu.gpu_error()
    assert (gpu.get("x") == x1).all()  # nothing was stepped


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_adapter_notices_parameter_setters_and_mass_edits(precision, cpu_libs):
    """ADVICE round 1: SimulationModel::setClothStiffness and ParticleData::setMass after the first step do not clear
    m_groupsInitialized; the reference reads the values on every solve, so the adapter has to notice them itself (sentinel
    signature of the constraint parameters, per-step mass comparison).  Twin on the reference's own TimeStepController (fp64)."""
    from oracle import pyoracle
    if not (pyoracle.available("refgpu", precision) and have_ref("f64")):
        pytest.skip("prebuilt oracle/_ref/libpbdref_gpu_%s.so not present on this box" % precision)
    gpu = cpu_libs.CpuPbd("refgpu", precision); cpu = cpu_libs.CpuPbd("ref", "f64")
    for m in (gpu, cpu):
        scenes.cloth(m, 20, 20, 1, 2, dist_k=1.0, bend_k=0.01, max_iter=4)
    gpu.use_gpu_timestep(0, 0)
    x_start = perturb([gpu, cpu], 0.02)
    gpu.step(2); cpu.step(2)
    for m in (gpu, cpu):
        m.set_cloth_stiffness(0.05)   # every DistanceConstraint::m_stiffness
        m.set_mass(210, 0.0)          # pin a particle in the middle of the sheet
    x_mid = cpu.get("x").copy(); xg_mid = gpu.get("x").copy()
    gpu.step(6); cpu.step(6)
    assert gpu.gpu_error() == "", gpu.gpu_error()
    xg, xc = gpu.get("x"), cpu.get("x")
    e = rel_position_error(xg, xc)
    print("adapter after setClothStiffness + setMass, Real=%s: rel pos %.2e" % (precision, e))
    assert e <= TOL
    assert np.abs(xc[210] - x_mid[210]).max() == 0.0 and np.abs(xg[210] - xg_mid[210]).max() == 0.0  # the pinned particle stopped, on both sides
    old_c = cpu.get("oldX").copy()
    # the edits matter: a twin that ignored them is off by far more than the tolerance
    ign = cpu_libs.CpuPbd("ref", "f64")
    scenes.cloth(ign, 20, 20, 1, 2, dist_k=1.0, bend_k=0.01, max_iter=4)
    ign.set("x", x_start); ign.step(8)
    assert rel_position_error(ign.get("x"), xc) > 10 * TOL  # 2.3e-3 (the checkers share one library instance: xc was copied before)
    # history comes back on demand (second-order velocity update of another TimeStep would read it)
    assert gpu.download_history() == 0
    assert rel_position_error(gpu.get("oldX"), old_c) <= TOL


def test_auto_mode_picks_resident_where_it_pays_and_falls_back():
    """PBD_MODE_AUTO (the default): cloth / FEM models run in the resident mode, models with rigid coupling in graph mode, and a model
    the resident mode refuses (IsometricBending with a user-modified, non-rank-one Q) falls back to the graph mode without an error.
    The bits never depend on the choice."""
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel

    def engine_of(hm, with_rb=False, edit=None):
        types, bodies, params, _ = hm.constraints()
        if edit is not None:
            params = params.copy(); edit(types, params)
        mass, _ = hm.masses()
        eng = _capi.Engine(0)
        eng.set_particles(hm.get("x"), mass)
        if with_rb:
            rb = hm.rigid_bodies()
            eng.set_rigid_bodies([0.0 if i % 3 == 0 else 1.0 for i in range(len(rb))], rb[:, :3], rb[:, 3:7],
                                 [scenes.box_inertia(1.0, 0.5, 0.5, 0.5) if i % 3 == 0 else scenes.box_inertia(1.0, 0.4, 2.0, 0.4) for i in range(len(rb))])
        eng.add_flat(types, bodies, params)
        eng.color_first_fit()
        eng.set_params(dt=0.005, sub_steps=1, max_iter=4)
        return eng

    def run(hm, mode, **kw):
        eng = engine_of(hm, **kw)
        if mode is not None:
            eng.set_mode(mode)
        assert eng.get_mode()[0] == (_capi.MODE_AUTO if mode is None else mode)
        eng.step(3); eng.sync()
        out = eng.get_attr(_capi.ATTR_X).copy(), eng.get_mode()[1]
        eng.close()
        return out

    cloth = HostModel(); scenes.cloth(cloth, 24, 24, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=4)
    perturb([cloth], 0.02)
    xa, active = run(cloth, None)
    assert active == _capi.MODE_RESIDENT
    assert (xa == run(cloth, _capi.MODE_GRAPH)[0]).all()

    rig = HostModel(); scenes.cfg4(rig, n_cloth=16, bar_dims=(5, 3, 3))
    xr, active = run(rig, None, with_rb=True)
    assert active == _capi.MODE_GRAPH
    assert (xr == run(rig, _capi.MODE_RESIDENT, with_rb=True)[0]).all()  # the resident kernel runs joints too when asked to

    def spoil_q(types, params):  # one bending constraint gets a Q that is not of the rank-one form
        i = int(np.nonzero(types == _capi.ISOBENDING_XPBD)[0][0])
        params[i, 1] += 0.5
    xq, active = run(cloth, None, edit=spoil_q)
    assert active == _capi.MODE_GRAPH and np.isfinite(xq).all()
    assert (xq == run(cloth, _capi.MODE_GRAPH, edit=spoil_q)[0]).all()
    with pytest.raises(_capi.PbdError):
        run(cloth, _capi.MODE_RESIDENT, edit=spoil_q)


def test_adapter_device_authoritative_state(cpu_libs):
    """GpuTimeStepController::setHostStateAuthoritative(false): no per-step upload of x and v (the model still receives the result
    of every step).  Without host edits the trajectory is bit-identical to the default policy; a host edit is picked up after
    invalidateState()."""
    from oracle import pyoracle
    if not pyoracle.available("refgpu", "f32"):
        pytest.skip("prebuilt oracle/_ref/libpbdref_gpu_f32.so not present on this box")
    outs = []
    for authoritative in (True, False):
        gpu = cpu_libs.CpuPbd("refgpu", "f32")
        scenes.cloth(gpu, 16, 16, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=4)
        gpu.use_gpu_timestep(0, 0)
        gpu.set_host_state_authoritative(authoritative)
        perturb([gpu], 0.02)
        gpu.step(4)
        x = gpu.get("x").copy()
        x[100, 1] += 0.05           # a host edit between steps
        gpu.set("x", x)
        if not authoritative:
            gpu.invalidate_state()
        gpu.step(2)
        assert gpu.gpu_error() == "", gpu.gpu_error()
        outs.append(gpu.get("x").copy())
    assert np.isfinite(outs[0]).all() and (outs[0] == outs[1]).all()


def test_pipelined_host_step_equals_blocking():
    """pbd_step_host_async / pbd_step_host_wait (three streams, two staging slots): same results as the blocking pbd_step_host, for
    independent frames (every call uploads its own x, v) and for a trajectory (uploads skipped, every frame downloaded)."""
    import torch
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    def make():
        m = HostModel()
        scenes.cloth(m, 48, 40, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=5)
        types, bodies, params, _ = m.constraints()
        off, ids = m.groups()
        mass, _ = m.masses()
        eng = _capi.Engine(0)
        eng.set_particles(m.get("x0"), mass)
        eng.add_flat(types, bodies, params)
        eng.set_groups(off, ids)
        eng.set_params(dt=0.005, sub_steps=1, max_iter=5)
        m.close()
        return eng
    a, b = make(), make()
    rng = np.random.default_rng(5)
    x0 = a.get_attr(_capi.ATTR_X).copy()
    frames = [np.ascontiguousarray(x0 + rng.uniform(-0.02, 0.02, x0.shape).astype(np.float32)) for _ in range(5)]
    v0 = np.zeros_like(x0)
    pin = lambda arr: torch.from_numpy(arr).pin_memory().numpy()
    fin = [pin(f) for f in frames]; vin = pin(v0)
    out_blocking = []
    for f in fin:
        xo = np.empty_like(x0); a.step_host(1, f, vin, xo); out_blocking.append(xo)
    outs = [pin(np.empty_like(x0)) for _ in fin]
    for k, f in enumerate(fin):
        b.step_host_async(1, f, vin, outs[k])
        b.step_host_wait(1)
    b.step_host_wait(0)
    for k in range(len(fin)):
        assert (outs[k] == out_blocking[k]).all(), "frame %d differs" % k
    # trajectory: device state authoritative, every frame downloaded while the next one is computed
    traj_blocking = []
    for _ in range(6):
        xo = np.empty_like(x0); a.step_host(1, None, None, xo); traj_blocking.append(xo)
    traj = [pin(np.empty_like(x0)) for _ in range(6)]
    for k in range(6):
        b.step_host_async(1, None, None, traj[k])
    b.step_host_wait(0)
    for k in range(6):
        assert (traj[k] == traj_blocking[k]).all(), "trajectory frame %d differs" % k
    assert np.abs(traj[5] - traj[0]).max() > 1e-4  # it moved
    a.close(); b.close()
