"""Every execution mode and resident-kernel shape against the fp64 checker, on every constraint type.

The parity tests pin the graph mode; the resident cluster kernel (what PBD_MODE_AUTO runs for cloth, FEM and "light" models) and
its launch shapes are held to the fp64 C restatement here, configuration by configuration:
  * the modes LAUNCH, GRAPH, RESIDENT and AUTO;
  * RESIDENT with the cluster shape forced (PBD_B200_CLUSTERS "GxC": G clusters of C CTAs), which reaches the X items of G x 1
    layouts (LocalXAcc), the DSMEM paths of 1 x C and both at once in G x C;
  * RESIDENT at every block size PBD_B200_RTHREADS accepts (sizes a mask is not instantiated for are clamped to one it is);
  * the per-engine knobs of the per-bucket kernels (particle layout, colour merging, gather cache policy, bucket sort).
Each configuration must pass the position gates of parity_util, gates on the velocities and oldX, keep pinned particles bit for
bit, and reproduce the graph mode bit for bit in x, v, oldX and the XPBD multipliers (matched by insertion id, so that a
permutation bug of the resident layouts cannot hide).

The Jacobi comparison mode is held to an fp64 restatement of its own algorithm (jacobi_reference below), which is itself checked
on the CPU against the Gauss-Seidel checker where the two must agree.
"""
import ctypes as C
import os

import numpy as np
import pytest

import scenes
from parity_util import assert_parity, perturb, rel_position_error, rel_displacement_error
from test_gpu_parity import SCENES as PARITY_SCENES

DISTANCE, DISTANCE_XPBD, DIHEDRAL, ISOBENDING, ISOBENDING_XPBD, FEMTRIANGLE, STRAINTRIANGLE, VOLUME, VOLUME_XPBD, \
    FEMTET, FEMTET_XPBD, STRAINTET, SHAPEMATCHING = range(13)
XPBD_TYPES = (DISTANCE_XPBD, ISOBENDING_XPBD, VOLUME_XPBD, FEMTET_XPBD)
NBODIES = [2, 2, 4, 4, 4, 3, 3, 4, 4, 4, 4, 4, 4]
MODE_GRAPH, MODE_RESIDENT, MODE_LAUNCH, MODE_JACOBI, MODE_AUTO = 0, 1, 2, 3, 4


# ---- scenes: the parity scenes plus shapes and materials they do not reach ------------------------------------------------------
def _hetero_light(m):
    """Distance_XPBD on the edges with per-edge k in [1e3, 1e6] and FEMTriangle on the faces with per-face moduli: the light mask."""
    nx, ny = 15, 13
    m.add_regular_triangle_model(nx, ny, t=(0, 1, 0), R=scenes.RX90, scale=(6.0, 5.0))
    m.set_mass(0, 0.0); m.set_mass(nx - 1, 0.0)
    rng = np.random.RandomState(11)
    for e in m.tri_edges(0):
        assert m.add_constraint(DISTANCE_XPBD, [int(e[0]), int(e[1])], [float(rng.randint(1, 1001) * 1000)])
    for f in m.tri_faces(0):  # every value is exact in fp32, so both sides see the same material
        assert m.add_constraint(FEMTRIANGLE, [int(v) for v in f], [float(rng.randint(500, 2001)), float(rng.randint(500, 2001)),
                                                                    float(rng.randint(250, 1001)), rng.randint(1, 8) / 16.0, rng.randint(1, 8) / 16.0])
    m.set_params(dt=0.005, sub_steps=2, max_iter=4)


def _hetero_fem(m):
    """FEMTet with per-tet E and nu, then Volume_XPBD with per-tet k, on a 7x3x4 bar: the FEM mask."""
    w, h, d = 7, 3, 4
    m.add_regular_tet_model(w, h, d, t=(5, 0, 0), R=np.eye(3), scale=(6.0, 1.2, 1.5))
    for j in range(h):
        for k in range(d):
            m.set_mass(j * d + k, 0.0)
    rng = np.random.RandomState(12)
    tets = m.tet_tets(0)
    for t in tets:
        assert m.add_constraint(FEMTET, [int(v) for v in t], [float(rng.randint(100, 1001) * 1000), rng.randint(10, 25) / 64.0])
    for t in tets:
        assert m.add_constraint(VOLUME_XPBD, [int(v) for v in t], [float(rng.randint(1, 101) * 1000)])
    m.set_params(dt=0.005, sub_steps=2, max_iter=3)


def _hetero_all(m):
    """StrainTriangle on the faces with per-face stiffnesses and normalisation flags: only the everything-mask covers it."""
    nx, ny = 13, 11
    m.add_regular_triangle_model(nx, ny, t=(0, 1, 0), R=scenes.RX90, scale=(5.0, 4.0))
    m.set_mass(0, 0.0); m.set_mass(nx - 1, 0.0)
    rng = np.random.RandomState(13)
    for f in m.tri_faces(0):
        assert m.add_constraint(STRAINTRIANGLE, [int(v) for v in f], [rng.randint(4, 17) / 8.0, rng.randint(4, 17) / 8.0, rng.randint(2, 9) / 8.0,
                                                                       float(rng.randint(0, 2)), float(rng.randint(0, 2))])
    m.set_params(dt=0.005, sub_steps=1, max_iter=5)


EXTRA_SCENES = {
    # odd particle count on the deep-pipeline cloth-XPBD kernel, two substeps
    "cloth_23x25_xpbd": (lambda m: scenes.cloth(m, 23, 25, 4, 3, dist_k=1.0e5, bend_k=100.0, sub_steps=2, max_iter=5), 0.02, 3),
    # second-order velocity update (lastX) on the light mask
    "cloth_17x19_second_order": (lambda m: scenes.cloth(m, 17, 19, 2, 1, bend_k=0.5, fem=(1000.0, 1000.0, 500.0, 0.3, 0.3), sub_steps=3, max_iter=4,
                                                        vel_method=1), 0.02, 3),
    # odd particle count on the everything-mask (StrainTet with normalised stretch)
    "bar_7x3x5_straintet_norm": (lambda m: scenes.bar(m, 7, 3, 5, 4, k=1.0, sub_steps=2, max_iter=3, norm_stretch=True), 0.01, 3),
    "hetero_light": (_hetero_light, 0.02, 3),
    "hetero_fem": (_hetero_fem, 0.01, 3),
    "hetero_all": (_hetero_all, 0.02, 3),
}
SCENES = dict(PARITY_SCENES, **EXTRA_SCENES)

# bar_femtet_xpbd: XPBD-FEM amplifies rounding chaotically; test_gpu_parity.py gates it at 5e-4 without the displacement bound
TOL_POS = {"bar_femtet_xpbd": 5e-4}
TOL_DISP = {"bar_femtet_xpbd": np.inf}
# velocities: max |v - v_ref| / max |v_ref|; oldX as a velocity: max |oldX - oldX_ref| / (h max |v_ref|).  fp32 rounding of the positions
# reaches them divided by the substep h.  Worst over every scene and configuration, measured on a B200 (1000 W): velocity 9.2e-3
# (cloth_dihedral), oldX 1.1e-2 (mixed_cloth_solid, h = 1 ms); the second-order update (1.5 x - 2 oldX + 0.5 lastX) / h doubles the
# amplification: 4.8e-2 / 2.0e-2 (cloth_17x19_second_order).  Gates: about 3x the worst.  A step without projections is off by 0.6 - 1.1.
TOL_VEL = 3e-2
TOL_VEL_SCENE = {"cloth_17x19_second_order": 0.15}
# multipliers: max |lambda - lambda_ref| / max |lambda_ref| over the XPBD constraints; worst measured 5.5e-3 (hetero_fem)
TOL_LAM = 2e-2

ENV_KNOBS = ("PBD_B200_CLUSTERS", "PBD_B200_RTHREADS", "PBD_B200_LAYOUT", "PBD_B200_MERGE", "PBD_B200_GATHER")
CONFIGS = {
    # name: (mode, environment, bucket sort)
    "launch": (MODE_LAUNCH, {}, True),
    "graph": (MODE_GRAPH, {}, True),
    "resident": (MODE_RESIDENT, {}, True),
    "auto": (MODE_AUTO, {}, True),
    "graph_layout_linear": (MODE_GRAPH, {"PBD_B200_LAYOUT": "linear"}, True),
    "graph_merge_0": (MODE_GRAPH, {"PBD_B200_MERGE": "0"}, True),
    "graph_gather_cg": (MODE_GRAPH, {"PBD_B200_GATHER": "cg"}, True),
    "graph_no_bucket_sort": (MODE_GRAPH, {}, False),
}
for _shape in ("1x1", "1x4", "1x16", "4x1", "37x1", "2x4"):
    CONFIGS["resident_" + _shape] = (MODE_RESIDENT, {"PBD_B200_CLUSTERS": _shape}, True)
for _threads in ("256", "512", "640", "768"):  # each mask runs the sizes it is instantiated for; the others are clamped to one
    CONFIGS["resident_threads_" + _threads] = (MODE_RESIDENT, {"PBD_B200_RTHREADS": _threads}, True)


# ---- the fp64 checker's run of a scene, once per module ---------------------------------------------------------------------
def _oracle_lambdas(cpu, n):
    """m_lambda of every constraint of the checker's model, by insertion index."""
    get = cpu.f("get_constraint")
    b = np.zeros(4, np.uint32); p = np.zeros(24); lam = C.c_double(0.0); out = np.zeros(n)
    for i in range(n):
        get(C.c_uint(i), b.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), C.byref(lam))
        out[i] = lam.value
    return out


def _projection_free(x_start, w, prm, steps):
    """What a step that skipped every projection computes (fp64): integration and velocity update only."""
    x = x_start.astype(np.float64); v = np.zeros_like(x); old = x.copy(); last = x.copy()
    dyn = np.asarray(w) != 0
    h = prm["dt"] / prm["sub_steps"]; g = np.asarray(prm["gravity"], np.float64)
    for _ in range(steps * prm["sub_steps"]):
        last = old.copy(); old = x.copy()
        v[dyn] += g * h; x[dyn] += v[dyn] * h
        if prm["vel_method"] == 0:
            v[dyn] = (x[dyn] - old[dyn]) / h
        else:
            v[dyn] = (1.5 * x[dyn] - 2.0 * old[dyn] + 0.5 * last[dyn]) / h
    return x, v, old


class Case:
    pass


_CASES = {}


def _case(name, cpu_libs):
    """Structure (host model == checker, bit for bit), the seeded start state and the checker's fp64 run of scene `name`."""
    if name in _CASES:
        return _CASES[name]
    from positionbaseddynamics_b200.model import HostModel
    build, amp, steps = SCENES[name]
    hm = HostModel(); cpu = cpu_libs.CpuPbd("oracle", "f64")
    build(hm); build(cpu)
    c = Case()
    c.types, c.bodies, c.params, _ = hm.constraints()
    tc, bc, _, _ = cpu.constraints()
    assert (c.types == tc).all() and (c.bodies == bc).all()
    c.off, c.ids = hm.groups()
    oc, ic = cpu.groups()
    assert (c.off == oc).all() and (c.ids == ic).all()
    c.mass, c.w = hm.masses()
    c.x0 = hm.get("x0")
    c.prm = dict(hm._params); c.steps = steps
    c.x_start = perturb([hm, cpu], amp)
    for attr in ("oldX", "lastX"):
        cpu.set(attr, c.x_start)
    cpu.set("v", np.zeros_like(c.x_start))
    cpu.step(steps)
    c.x_ref, c.v_ref, c.old_ref = cpu.get("x"), cpu.get("v"), cpu.get("oldX")
    c.lam_ref = _oracle_lambdas(cpu, len(c.types))
    c.h = c.prm["dt"] / c.prm["sub_steps"]
    c.twin = _projection_free(c.x_start, c.w, c.prm, steps)
    hm.close()
    _CASES[name] = c
    return c


def _errors(c, x, v, old):
    v_scale = max(np.abs(c.v_ref).max(), 1e-30)
    e_vel = float(np.abs(np.asarray(v, np.float64) - c.v_ref).max() / v_scale)
    e_old = float(np.abs(np.asarray(old, np.float64) - c.old_ref).max() / (c.h * v_scale))
    return e_vel, e_old


def _velocity_gate(name):
    return TOL_VEL_SCENE.get(name, TOL_VEL)


def _position_gate(c, name, x, what):
    return assert_parity(x, c.x_ref, c.x_start, tol_pos=TOL_POS.get(name, 1e-4), tol_disp=TOL_DISP.get(name, 5e-3), what=what)


def _position_gate_fails(c, name, x):
    try:
        _position_gate(c, name, x, "")
    except AssertionError:
        return True
    return False


# ---- GPU runs -------------------------------------------------------------------------------------------------------------
def _run_engine(c, mode, env=None, bucket_sort=True):
    """x, v, oldX, the XPBD multipliers by insertion id (NaN for other types) and the active mode after `steps` steps."""
    from positionbaseddynamics_b200 import _capi
    env = env or {}
    os.environ.update(env)  # read when the engine is created (layout, merge, gather) and when it flattens (clusters, threads)
    try:
        eng = _capi.Engine(0)
        try:
            eng.set_particles(c.x_start, c.mass, x0=c.x0, v=np.zeros_like(c.x_start))
            eng.set_attr(_capi.ATTR_OLDX, c.x_start); eng.set_attr(_capi.ATTR_LASTX, c.x_start)
            eng.add_flat(c.types, c.bodies, c.params)
            eng.set_groups(c.off, c.ids)
            p = c.prm
            eng.set_params(dt=p["dt"], sub_steps=p["sub_steps"], max_iter=p["max_iter"], vel_method=p["vel_method"], gravity=p["gravity"])
            if not bucket_sort:
                eng.set_bucket_sort(0)
            eng.set_mode(mode)
            eng.step(c.steps); eng.sync()
            x, v, old = eng.get_attr(_capi.ATTR_X), eng.get_attr(_capi.ATTR_V), eng.get_attr(_capi.ATTR_OLDX)
            lam = np.full(len(c.types), np.nan, np.float32)
            for t in XPBD_TYPES:
                if (c.types == t).any():
                    vals, ids = eng.lambdas(t)
                    assert len(ids) == int((c.types == t).sum()) and (c.types[ids] == t).all()
                    lam[ids] = vals
            active = eng.get_mode()[1]
        finally:
            eng.close()
    finally:
        for k in env:
            os.environ.pop(k, None)
    return x, v, old, lam, active


_GRAPH = {}


def _graph_run(name, c):
    if name not in _GRAPH:
        _GRAPH[name] = _run_engine(c, MODE_GRAPH)
    return _GRAPH[name]


def _check_config(name, config, c, out):
    x, v, old, lam, _ = out
    what = "%s / %s" % (name, config)
    e_pos, e_disp = _position_gate(c, name, x, what)
    e_vel, e_old = _errors(c, x, v, old)
    xp = ~np.isnan(lam)
    e_lam = float(np.abs(lam[xp] - c.lam_ref[xp]).max() / max(np.abs(c.lam_ref[xp]).max(), 1e-30)) if xp.any() else 0.0
    print("MATRIX %-34s %-22s pos %.2e disp %.2e vel %.2e oldX %.2e lambda %.2e" % (name, config, e_pos, e_disp, e_vel, e_old, e_lam))
    tol_v = _velocity_gate(name)
    assert e_vel <= tol_v, "%s: velocity error %.3e > %.1e" % (what, e_vel, tol_v)
    assert e_old <= tol_v, "%s: oldX error %.3e > %.1e" % (what, e_old, tol_v)
    assert e_lam <= TOL_LAM, "%s: multiplier error %.3e > %.1e" % (what, e_lam, TOL_LAM)
    pinned = np.asarray(c.w) == 0
    assert (x[pinned] == c.x_start[pinned]).all(), what + ": a pinned particle moved"
    xg, vg, og, lg, _ = _graph_run(name, c)
    assert (x == xg).all() and (v == vg).all() and (old == og).all(), what + ": differs from the graph mode"
    assert np.array_equal(lam, lg, equal_nan=True), what + ": multipliers differ from the graph mode"


@pytest.mark.gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("name", sorted(SCENES))
def test_mode_matrix(name, config, cpu_libs):
    c = _case(name, cpu_libs)
    mode, env, bucket_sort = CONFIGS[config]
    out = _run_engine(c, mode, env, bucket_sort)
    _check_config(name, config, c, out)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_gates_reject_untouched_and_projection_free_states(name, cpu_libs):
    """Negative controls of the matrix's gates: the start state and a step without projections fail the position gate, and the
    projection-free twin fails the velocity gate."""
    c = _case(name, cpu_libs)
    assert _position_gate_fails(c, name, c.x_start), name + ": the start state passes the position gate"
    tx, tv, told = c.twin
    assert _position_gate_fails(c, name, tx), name + ": the projection-free twin passes the position gate"
    e_vel, e_old = _errors(c, tx, tv, told)
    print("%s projection-free twin: rel pos %.2e, rel disp %.2e, vel %.2e" % (name, rel_position_error(tx, c.x_ref),
                                                                             rel_displacement_error(tx, c.x_ref, c.x_start), e_vel))
    assert e_vel > _velocity_gate(name), name + ": the projection-free twin passes the velocity gate"


@pytest.mark.gpu
def test_resident_refuses_rigid_coupling_across_clusters():
    """The resident kernel integrates the rigid bodies on CTA 0 and runs their joints inside one cluster; more than one cluster is
    refused with PbdError (AUTO falls back to the graph mode)."""
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    hm = HostModel(); scenes.cfg4(hm, n_cloth=16, bar_dims=(5, 3, 3))
    types, bodies, params, _ = hm.constraints()
    mass, _ = hm.masses(); rb = hm.rigid_bodies()

    def run(mode):
        eng = _capi.Engine(0)
        try:
            eng.set_particles(hm.get("x"), mass)
            eng.set_rigid_bodies([0.0 if i % 3 == 0 else 1.0 for i in range(len(rb))], rb[:, :3], rb[:, 3:7], np.ones((len(rb), 3)))
            eng.add_flat(types, bodies, params)
            eng.color_first_fit()
            eng.set_params(dt=0.005, sub_steps=2, max_iter=1)
            eng.set_mode(mode)
            eng.step(1); eng.sync()
            return eng.get_attr(_capi.ATTR_X), eng.get_mode()[1]
        finally:
            eng.close()
    os.environ["PBD_B200_CLUSTERS"] = "4x1"
    try:
        with pytest.raises(_capi.PbdError, match="rigid-body coupling"):
            run(_capi.MODE_RESIDENT)
        x_auto, active = run(_capi.MODE_AUTO)
    finally:
        os.environ.pop("PBD_B200_CLUSTERS", None)
    assert active == _capi.MODE_GRAPH
    assert (x_auto == run(_capi.MODE_GRAPH)[0]).all()
    hm.close()


# ---- the Jacobi comparison mode ---------------------------------------------------------------------------------------------
def jacobi_reference(cpu, types, bodies, params, w, x_start, prm, steps):
    """fp64 restatement of PBD_MODE_JACOBI (engine.cu enqueue_step_jacobi): per sweep every constraint is projected from the
    positions at the start of the sweep (cpu.kat_solve, the checker's solver of that type, with lambda kept per constraint and zeroed
    at the first sweep of a substep); every dynamic particle of a constraint counts once, whether or not the solver moved it; after all
    types each particle moves by the average of its corrections.  Returns x, v, oldX and the multipliers."""
    types = np.asarray(types); params = np.asarray(params, np.float64); w = np.asarray(w, np.float64)
    assert not np.isin(types, (SHAPEMATCHING, 13, 14)).any(), "restated for the particle constraint types with a plain correction"
    x = np.asarray(x_start, np.float64).copy(); v = np.zeros_like(x); old = x.copy(); last = x.copy()
    lam = np.zeros(len(types))
    h = prm["dt"] / prm["sub_steps"]; g = np.asarray(prm["gravity"], np.float64)
    dyn = w != 0
    order = [i for t in range(13) for i in np.nonzero(types == t)[0]]  # one pass per type, like the launches
    for _ in range(steps * prm["sub_steps"]):
        last = old.copy(); old = x.copy()
        v[dyn] += g * h; x[dyn] += v[dyn] * h
        for it in range(prm["max_iter"]):
            delta = np.zeros_like(x); cnt = np.zeros(len(x))
            for i in order:
                t = int(types[i]); nb = NBODIES[t]; b = bodies[i, :nb].astype(np.int64)
                X = np.zeros((4, 3)); X[:nb] = x[b]
                W = np.zeros(4); W[:nb] = w[b]
                hinv = False
                if t in (FEMTET, FEMTET_XPBD):  # the constraint classes' handleInversion rule (current volume over rest volume)
                    vol = -np.dot(X[3] - X[0], np.cross(X[2] - X[0], X[1] - X[0])) / 6.0
                    hinv = vol / params[i, 0] < 0.2
                res, corr, l = cpu.kat_solve(t, X, W, params[i], dt=h, handle_inversion=hinv, lam=0.0 if it == 0 else lam[i])
                if t in XPBD_TYPES:
                    lam[i] = l
                for k in range(nb):
                    if W[k] != 0:
                        if res:
                            delta[b[k]] += corr[k]
                        cnt[b[k]] += 1
            moved = cnt > 0
            x[moved] += delta[moved] / cnt[moved, None]
        if prm["vel_method"] == 0:
            v[dyn] = (x[dyn] - old[dyn]) / h
        else:
            v[dyn] = (1.5 * x[dyn] - 2.0 * old[dyn] + 0.5 * last[dyn]) / h
    return x, v, old, lam


def _disjoint_scene(m):
    """Every constraint on particles of its own (one colour): Jacobi and Gauss-Seidel are the same algorithm here."""
    rng = np.random.RandomState(21)
    pts, groups = [], []

    def block(shape):
        base = len(pts)
        for p in shape:
            pts.append(np.asarray(p, np.float64) + [3.0 * len(groups), 0.0, 0.0])
        groups.append(list(range(base, base + len(shape))))
        return groups[-1]
    quad = [(0.5, 0.8, 0.0), (0.5, -0.8, 0.1), (0.0, 0.0, 0.0), (1.0, 0.0, 0.0)]
    tet = [(0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), (0.0, 0.0, 1.0)]
    spec = []
    for _ in range(6):
        spec.append((DISTANCE_XPBD, block([(0, 0, 0), (1, 0, 0)]), [float(rng.randint(1, 1001) * 1000)]))
        spec.append((DISTANCE, block([(0, 0, 0), (1, 0.2, 0)]), [rng.randint(1, 9) / 8.0]))
        spec.append((ISOBENDING_XPBD, block(quad), [float(rng.randint(1, 200))]))
        spec.append((DIHEDRAL, block(quad), [rng.randint(1, 9) / 8.0]))
        spec.append((FEMTRIANGLE, block(quad[:3]), [1000.0, 1000.0, 500.0, 0.25, 0.25]))
        spec.append((VOLUME_XPBD, block(tet), [float(rng.randint(1, 101) * 1000)]))
        spec.append((FEMTET, block(tet), [float(rng.randint(100, 1001) * 1000), 0.3125]))
    faces = np.array([g[:3] for g in groups if len(g) >= 3], np.uint32)
    m.add_triangle_model(np.array(pts), faces)
    m.set_mass(groups[0][0], 0.0); m.set_mass(groups[2][2], 0.0)  # a static particle in a distance and in a bending constraint
    for t, b, u in spec:
        assert m.add_constraint(t, b, u)
    m.set_params(dt=0.005, sub_steps=2, max_iter=3)


def test_jacobi_reference_equals_gauss_seidel_on_disjoint_constraints(cpu_libs):
    """The restatement of the Jacobi mode against the fp64 checker's Gauss-Seidel step where the two algorithms coincide."""
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    _disjoint_scene(cpu)
    types, bodies, params, _ = cpu.constraints()
    _, w = cpu.masses()
    x_start = perturb([cpu], 0.05).astype(np.float64)
    prm = dict(dt=0.005, sub_steps=2, max_iter=3, vel_method=0, gravity=(0.0, -9.81, 0.0))
    xj, vj, oj, lj = jacobi_reference(cpu, types, bodies, params, w, x_start, prm, 2)
    cpu.set("x", x_start); cpu.set("oldX", x_start); cpu.set("lastX", x_start); cpu.set("v", np.zeros_like(x_start))
    cpu.step(2)
    xc, vc = cpu.get("x"), cpu.get("v")
    err = np.abs(xj - xc).max()
    print("Jacobi restatement vs Gauss-Seidel on disjoint constraints: max |dx| %.1e, max |dv| %.1e" % (err, np.abs(vj - vc).max()))
    assert err <= 1e-12 * max(1.0, np.abs(xc).max()) and np.abs(vj - vc).max() <= 1e-9 * max(1.0, np.abs(vc).max())
    assert np.abs(xc - x_start).max() > 1e-3  # the projections moved the particles
    assert np.abs(lj[types == DISTANCE_XPBD]).max() > 0.0


@pytest.mark.gpu
def test_jacobi_mode_against_fp64_restatement(cpu_libs):
    """PBD_MODE_JACOBI on a 24x24 Distance_XPBD + IsometricBending_XPBD cloth against jacobi_reference: the usual position gates
    plus velocities and multipliers; the start state, the projection-free twin and the Gauss-Seidel answer must fail the gate."""
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    build = lambda m: scenes.cloth(m, 24, 24, 4, 3, dist_k=1.0e5, bend_k=100.0, max_iter=5)
    steps = 3
    hm = HostModel(); cpu = cpu_libs.CpuPbd("oracle", "f64")
    build(hm); build(cpu)
    types, bodies, params, _ = cpu.constraints()
    tg, bg, pg, _ = hm.constraints()
    assert (tg == types).all() and (bg == bodies).all()
    _, w = cpu.masses()
    mass, _ = hm.masses()
    x_start = perturb([hm, cpu], 0.02)
    prm = dict(hm._params)
    xr, vr, orf, lr = jacobi_reference(cpu, types, bodies, params, w, x_start, prm, steps)
    eng = _capi.Engine(0)
    eng.set_particles(x_start, mass, x0=hm.get("x0"))
    eng.add_flat(tg, bg, pg)
    eng.color_first_fit()
    eng.set_params(dt=prm["dt"], sub_steps=prm["sub_steps"], max_iter=prm["max_iter"])
    eng.set_mode(_capi.MODE_JACOBI)
    eng.step(steps); eng.sync()
    x, v = eng.get_attr(_capi.ATTR_X), eng.get_attr(_capi.ATTR_V)
    lam = np.zeros(len(types))
    for t in (DISTANCE_XPBD, ISOBENDING_XPBD):
        vals, ids = eng.lambdas(t); lam[ids] = vals
    eng.close()
    e_pos, e_disp = assert_parity(x, xr, x_start, what="Jacobi mode")
    e_vel = np.abs(v - vr).max() / np.abs(vr).max()
    e_lam = np.abs(lam - lr).max() / np.abs(lr).max()
    print("Jacobi mode vs fp64 restatement: rel pos %.2e, rel disp %.2e, vel %.2e, lambda %.2e" % (e_pos, e_disp, e_vel, e_lam))
    assert e_vel <= TOL_VEL and e_lam <= TOL_LAM
    # negative controls: the gate tells Jacobi from doing nothing, from skipping the projections and from Gauss-Seidel
    for bad, what in ((x_start, "start state"), (_projection_free(x_start, w, prm, steps)[0], "projection-free twin")):
        with pytest.raises(AssertionError):
            assert_parity(bad, xr, x_start, what=what)
    cpu.set("x", x_start); cpu.set("oldX", x_start); cpu.set("lastX", x_start); cpu.set("v", np.zeros_like(x_start))
    cpu.step(steps)
    with pytest.raises(AssertionError):
        assert_parity(cpu.get("x"), xr, x_start, what="Gauss-Seidel")
    hm.close()
