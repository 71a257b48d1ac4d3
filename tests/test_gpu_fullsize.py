"""Parity at BASELINE.json's full sizes: direct comparison with the fp64 CPU checker where it finishes in seconds, plus
size-independent properties of the path (fixed point at rest, translation invariance, mode/replica determinism,
pinned particles, free fall)."""
import numpy as np
import pytest

import scenes
from parity_util import perturb, rel_position_error, assert_parity, assert_gate_rejects
from conftest import have_ref

pytestmark = pytest.mark.gpu


def _gpu(build, mode=4):
    """The scene on a GPU time step; the default is PBD_MODE_AUTO, what a user and bench.py run (the resident kernel for cfg2, cfg3
    and cfg5); the bitwise tests below hold the other modes to it."""
    from positionbaseddynamics_b200.model import HostModel
    m = HostModel(); build(m); m.time_step().set_mode(mode)
    return m


def _particles_only(kind):
    """The scene's particles, pins and time-step parameters WITHOUT any constraint: stepping it integrates and updates velocities
    only -- what an engine whose projection kernels did nothing would produce (negative control of the parity gate)."""
    from positionbaseddynamics_b200.model import HostModel
    m = HostModel()
    if kind in ("cfg2", "cfg5"):
        n = 1000 if kind == "cfg2" else 500
        m.add_regular_triangle_model(n, n, t=(0, 1, 0), R=scenes.RX90, scale=(10.0, 10.0))
        m.set_mass(0, 0.0); m.set_mass(n - 1, 0.0)
        m.set_params(dt=0.005, sub_steps=1, max_iter=20)
    elif kind == "cfg3":
        w, h, d = 101, 21, 21
        m.add_regular_tet_model(w, h, d, t=(5, 0, 0), R=np.eye(3), scale=(10.0, 1.5, 1.5))
        for j in range(h):
            for k in range(d):
                m.set_mass(j * d + k, 0.0)
        m.set_params(dt=0.005, sub_steps=10, max_iter=5)
    return m


def _full_size_case(name, build, amp, steps, cpu, control=None):
    """Perturbed start state (seeded, identical fp32 values on both sides), `steps` steps, then the discriminating gate:
    <= 1e-4 of the scene size AND <= 5e-3 of the largest displacement; the untouched start state and a projection-free step must
    both FAIL the same gate."""
    gpu = _gpu(build)
    build(cpu)
    assert gpu.num_constraints() == cpu.num_constraints()
    og, ig = gpu.groups(); oc, ic = cpu.groups()
    assert (og == oc).all() and (ig == ic).all()
    x_start = perturb([gpu, cpu], amp)
    gpu.step(steps); cpu.step(steps)
    xg, xc = gpu.get("x"), cpu.get("x")
    e_pos, e_disp = assert_parity(xg, xc, x_start, what=name)
    moved = np.abs(np.asarray(xc, dtype=np.float64) - x_start).max()
    print("%s full size, perturbed by %.1e: rel pos %.2e, rel to displacement %.2e (max displacement %.3e, abs err %.2e)"
          % (name, amp, e_pos, e_disp, moved, np.abs(xg - xc).max()))
    assert_gate_rejects(x_start, xc, x_start, what=name + " / untouched start state")
    if control is not None:
        twin = _particles_only(control)
        twin.set("x", x_start)
        twin.step(steps)
        assert_gate_rejects(twin.get("x"), xc, x_start, what=name + " / step without projections")
        twin.close()
    return gpu, og


def test_cfg2_full_size_two_steps_vs_fp64(cpu_libs):
    """cfg2 at the benchmark size (1,000,000 particles, 5,988,006 constraints, 20 iterations): structure equal to the
    checker's bit for bit; from a perturbed state (20 % of the edge length) positions within 1e-4 relative and within 5e-3 of the
    displacement after 2 steps.  fp64 checker = the unmodified reference when the prebuilt oracle/_ref is on this box, else the
    C restatement."""
    kind = "ref" if have_ref("f64") else "oracle"
    cpu = cpu_libs.CpuPbd(kind, "f64"); cpu.set_threads(16)
    gpu, og = _full_size_case("cfg2", lambda m: scenes.cfg2(m, 1000, 20), 2.0e-3, 2, cpu, control="cfg2")
    assert gpu.num_constraints() == 5988006
    assert list(np.diff(og))[:4] == [500000, 499999, 499499, 498004]
    xg = gpu.get("x")
    # pinned corners (particles 0 and 999) never move
    assert (xg[0] == gpu.get("x0")[0]).all() and (xg[999] == gpu.get("x0")[999]).all()
    gpu.close()


def test_cfg5_size_two_steps_vs_fp64(cpu_libs):
    """cfg5's per-GPU scene (500x500 cloth, 1,494,006 constraints, XPBD 1 x 20) against the fp64 checker, perturbed."""
    kind = "ref" if have_ref("f64") else "oracle"
    cpu = cpu_libs.CpuPbd(kind, "f64"); cpu.set_threads(16)
    gpu, og = _full_size_case("cfg5", lambda m: scenes.cfg2(m, 500, 20), 4.0e-3, 2, cpu, control="cfg5")
    assert gpu.num_constraints() == 748001 + 746005
    gpu.close()


def test_cfg3_full_size_one_step_vs_fp64(cpu_libs):
    """cfg3 at the benchmark size (200,000 tets, FEMTet E=1e6 + Volume, 10 substeps x 5 iterations): one step from a perturbed state."""
    cpu = cpu_libs.CpuPbd("oracle", "f64"); cpu.set_threads(16)
    gpu, og = _full_size_case("cfg3", scenes.cfg3, 4.0e-3, 1, cpu, control="cfg3")
    assert gpu.num_constraints() == 400000 and len(og) - 1 == 74
    gpu.close()


def test_rest_state_without_gravity_is_a_fixed_point():
    """Idempotence: with g = 0 every constraint of an undeformed scene is satisfied, so the step must not move anything
    (XPBD multipliers stay 0, PBD corrections vanish or fall under the reference's eps early-outs)."""
    for build in (lambda m: scenes.cfg2(m, 300, 5), lambda m: scenes.cfg3(m, 31, 9, 9)):
        gpu = _gpu(build)
        gpu.set_params(**dict(gpu._params, gravity=(0.0, 0.0, 0.0)))
        gpu.step(3)
        d = np.abs(gpu.get("x") - gpu.get("x0")).max()
        print("fixed point drift", d)
        assert d <= 2e-6
        assert np.abs(gpu.get("v")).max() <= 1e-3
        gpu.close()


def test_translation_invariance_large_cloth():
    """Shifting the whole scene shifts the result: the rank-1 bending form and the distance constraints only see
    differences of positions.  (The reference's fp32 absolute-position bending evaluation violates this at O(1e-3).)"""
    res = []
    for shift in (np.zeros(3), np.array([37.0, -11.0, 23.0])):
        gpu = _gpu(lambda m: scenes.cfg2(m, 400, 10))
        x = gpu.get("x") + shift.astype(np.float32)
        gpu.set("x", x); gpu.set("oldX", x); gpu.set("lastX", x)
        gpu.step(3)
        res.append(gpu.get("x").astype(np.float64) - shift)
        gpu.close()
    err = np.abs(res[0] - res[1]).max()
    print("translation invariance: max deviation %.2e" % err)
    assert err <= 5e-5  # fp32 ulp at |x| ~ 50 is 4e-6; a few ulps accumulate over 3 steps x 10 sweeps


def test_modes_and_layouts_agree_at_scale():
    """Graph, resident (default shape: one CTA per SM with X items through global memory; one cluster of 8 / 16 CTAs with early and
    late items over DSMEM; 37 independent CTAs) and plain-launch execution of a 300x300 XPBD cloth (540k constraints): bit-identical."""
    import os
    out = []
    for mode, clusters in ((0, None), (1, None), (2, None), (1, "1x8"), (1, "1x16"), (1, "37x1")):
        if clusters: os.environ["PBD_B200_CLUSTERS"] = clusters
        try:
            gpu = _gpu(lambda m: scenes.cfg2(m, 300, 8), mode)
            gpu.step(3)
            out.append((gpu.get("x").copy(), gpu.get("v").copy())); gpu.close()
        finally:
            os.environ.pop("PBD_B200_CLUSTERS", None)
    for o in out[1:]:
        assert (out[0][0] == o[0]).all() and (out[0][1] == o[1]).all()


def test_resident_mode_full_size_cfg2_bitwise():
    """cfg2 at full size in the resident mode: one CTA per SM, ~6,300 particles per tile in shared memory, ~7 % of the
    particles global-homed with their constraints ordered across the CTAs by the X counter.  Must reproduce the graph mode bit
    for bit, positions and velocities."""
    res = []
    for mode in (0, 1):
        gpu = _gpu(lambda m: scenes.cfg2(m, 1000, 20), mode)
        gpu.step(2)
        res.append((gpu.get("x").copy(), gpu.get("v").copy())); gpu.close()
    assert np.isfinite(res[0][0]).all()
    assert (res[0][0] == res[1][0]).all() and (res[0][1] == res[1][1]).all()


def test_resident_mode_cfg3_cfg4_bitwise():
    """cfg3 (FEMTet + Volume, one 16-CTA cluster) and cfg4 (cloth + solid + rigid coupling rig) in the resident mode against the graph mode."""
    for build in (scenes.cfg3, scenes.cfg4):
        res = []
        for mode in (0, 1):
            gpu = _gpu(build, mode)
            perturb([gpu], 2.0e-3)
            gpu.step(2)
            res.append((gpu.get("x").copy(), gpu.get("v").copy(), gpu.rigid_bodies().copy())); gpu.close()
        assert np.isfinite(res[0][0]).all()
        for a, b in zip(res[0], res[1]):
            assert (a == b).all()


def test_free_fall_of_an_unpinned_sheet_is_rigid():
    """Without pinned particles an undeformed cloth in free fall stays undeformed: every particle drops by the same
    g h^2 k(k+1)/2 and no constraint injects energy."""
    from positionbaseddynamics_b200.model import HostModel
    m = HostModel()
    m.add_regular_triangle_model(200, 200, t=(0, 5, 0), R=scenes.RX90, scale=(4, 4))
    m.add_cloth_constraints(0, 4, dist_k=1e5); m.add_bending_constraints(0, 3, 100.0)
    m.set_params(dt=0.005, sub_steps=2, max_iter=5)
    m.step(4)
    d = m.get("x") - m.get("x0")
    h = 0.0025; k = 8
    # fp32: ulp(5.0) = 4.8e-7 per update, 8 substeps, and the constraints react to that rounding noise
    assert np.abs(d[:, 1] - (-9.81 * h * h * k * (k + 1) / 2)).max() <= 2e-5
    assert np.abs(d[:, 0]).max() <= 1e-5 and np.abs(d[:, 2]).max() <= 1e-5
    m.close()


def test_cfg4_full_size_vs_fp64(cpu_libs):
    """cfg4 at the benchmark size: 224x224 cloth (FEMTriangle + IsometricBending) + 51x21x11 tet block (FEMTet) + the rigid
    coupling rig, 5 substeps x 1 iteration; two steps from a perturbed state against the fp64 checker (particles and rigid bodies)."""
    cpu = cpu_libs.CpuPbd("oracle", "f64"); cpu.set_threads(16)
    rb_start = None
    gpu, og = _full_size_case("cfg4", scenes.cfg4, 1.0e-2, 2, cpu)
    rg, rc = gpu.rigid_bodies().astype(np.float64)[:, :7], cpu.rigid_bodies()[:, :7]
    erb = np.abs(rg - rc).max()
    print("cfg4 full size: %d constraints, %d colours, rigid bodies abs %.2e" % (gpu.num_constraints(), len(og) - 1, erb))
    assert erb <= 1e-4
    gpu.close()


def test_device_colouring_cfg2_full_size():
    """Exact first-fit colouring of cfg2 (5,988,006 constraints, 27 colours) on the GPU equals the host colouring; prints both times."""
    import time
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    hm = HostModel(); scenes.cfg2(hm, 1000, 20)
    types, bodies, params, _ = hm.constraints()
    mass, _ = hm.masses()
    eng = _capi.Engine(0)
    eng.set_particles(hm.get("x"), mass)
    eng.add_flat(types, bodies, params)
    t0 = time.perf_counter(); eng.color_first_fit(); t_host = time.perf_counter() - t0
    off_h, ids_h = eng.groups()
    t0 = time.perf_counter(); ms, fronts = eng.color_first_fit_device(); t_dev = time.perf_counter() - t0
    off_d, ids_d = eng.groups()
    print("cfg2 colouring: host %.1f ms, device %.1f ms on the GPU (%.1f ms incl. host CSR build, upload and readback), %d wavefronts, %d colours"
          % (t_host * 1e3, ms, t_dev * 1e3, fronts, len(off_d) - 1))
    assert len(off_d) - 1 == 27
    assert (off_d == off_h).all() and (ids_d == ids_h).all()
    eng.close(); hm.close()
