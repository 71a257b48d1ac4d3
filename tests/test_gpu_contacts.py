"""Contact path (SURVEY.md section 8 row f-4, the data-parallel part): particles of a cloth against analytic distance fields on static
rigid bodies + the velocity-level contact solve, against the UNMODIFIED reference's DistanceFieldCollisionDetection,
ParticleRigidBodyContactConstraint and TimeStepController::velocityConstraintProjection.  The checker is the fp64 C restatement of the
contact path (oracle/pbd_oracle.c), which tests/test_oracle_vs_ref.py pins to the reference's recorded runs, set up with the rigid bodies
and collision objects the reference built for the same scene (tests/scenes.py:on_recorded_colliders)."""
import numpy as np
import pytest

import scenes
from parity_util import rel_position_error

pytestmark = pytest.mark.gpu
TOL = 1.0e-4
ALL_SHAPES = ("box", "sphere", "torus", "cylinder", "hollow_sphere", "hollow_box")


def _engine_from(cpu, colliders=None):
    """The call sequence of INTEGRATION.md: a model built on the CPU side is handed to the engine through the C ABI; `colliders` =
    (models, rigid) as CpuPbd.collision_objects() returns them."""
    from positionbaseddynamics_b200 import _capi
    types, bodies, params, _ = cpu.constraints()
    off, ids = cpu.groups()
    mass, _ = cpu.masses()
    rb = cpu.rigid_bodies()
    eng = _capi.Engine(0)
    eng.set_particles(cpu.get("x"), mass, x0=cpu.get("x0"), v=cpu.get("v"))
    eng.set_rigid_bodies([0.0] * len(rb), rb[:, :3], rb[:, 3:7], [(1.0, 1.0, 1.0)] * len(rb))
    eng.add_flat(types, bodies, params)
    eng.set_groups(off, ids)
    if colliders is not None:
        models, rigid = colliders
        pcs = [_capi.ParticleCollider(o, c, r, f) for (o, c, r, f) in models]
        rcs = []
        for d in rigid:
            rc = _capi.RigidCollider()
            rc.shape, rc.body = int(d[0]), int(d[1])
            rc.dim[:] = [float(v) for v in d[2:5]]; rc.thickness = float(d[5]); rc.invert_sdf = int(d[6])
            rc.restitution, rc.friction = float(d[7]), float(d[8])
            rc.R[:] = [float(v) for v in d[9:18]]; rc.v1[:] = [float(v) for v in d[18:21]]; rc.v2[:] = [float(v) for v in d[21:24]]
            rc.aabb_min[:] = [float(v) for v in d[24:27]]; rc.aabb_max[:] = [float(v) for v in d[27:30]]
            rcs.append(rc)
        eng.set_colliders(pcs, rcs)
        eng.set_contact_params(tolerance=0.05, stiffness=100.0, max_iter_v=5)
        eng.record_contacts(1 << 14)
    return eng


def _lockstep(step_gpu, get_gpu, cpu, steps, contacts_gpu=None):
    """Per-step parity from identical states.  A contact event (a particle crossing the tolerance shell, |dv| ~ 1 m/s) that happens one
    step earlier or later in fp32 than in fp64 changes the trajectory by orders of magnitude more than any rounding, so a free-running
    fp32 trajectory cannot be held against the fp64 one over hundreds of contact events; instead the GPU state is re-synchronised with the
    checker's before every step and each step is compared on its own: positions to 1e-4 (relative), velocities -- which is all a
    contact changes -- to 2e-3 m/s, the contact list exactly.  A particle whose signed distance is within 1e-5 of the threshold may
    legitimately be a contact on one side only; such grazing cases are counted (and bounded), everything else must agree."""
    grazing = 0; events = 0; worst_dv = 0.0; worst_x = 0.0; bodies = set()
    for k in range(steps):
        x, v = cpu.get("x").copy(), cpu.get("v").copy()
        step_gpu(x, v); cpu.step(1)
        xg, vg = get_gpu()
        xc, vc = cpu.get("x"), cpu.get("v")
        p, b, info = cpu.oracle_contacts()
        events += len(p); bodies |= set(b.tolist())
        worst_x = max(worst_x, rel_position_error(xg, xc))
        assert rel_position_error(xg, xc) <= TOL  # positions of a step do not depend on its contacts
        dv = np.abs(vg - vc).max(axis=1)
        bad = np.nonzero(dv > 2.0e-3)[0]
        ref_pairs = set(zip(p.tolist(), b.tolist()))
        if contacts_gpu is not None:
            got, found = contacts_gpu()
            gpu_pairs = set((c.particle, c.body) for c in got)
            depth_ref = {(int(pp), int(bb)): float(np.dot(info[i, 6:9], info[i, 0:3] - info[i, 3:6])) for i, (pp, bb) in enumerate(zip(p, b))}
            depth_gpu = {(c.particle, c.body): c.dist for c in got}
            for pair in ref_pairs ^ gpu_pairs:  # on one side only: must be a grazing contact
                d = depth_ref.get(pair, depth_gpu.get(pair))
                assert abs(d) < 1.0e-5, "step %d: contact %s (depth %.3e) on one side only" % (k, pair, d)
                grazing += 1
            one_sided = set(pp for pp, _ in ref_pairs ^ gpu_pairs)
            assert all(int(i) in one_sided for i in bad), "step %d: velocities differ at particles %s" % (k, bad)
            by_pair = {(c.particle, c.body): c for c in got}
            for i, pair in enumerate(zip(p.tolist(), b.tolist())):
                if pair in by_pair:
                    c = by_pair[pair]
                    assert np.abs(np.array(c.cp1[:]) - info[i, 3:6]).max() <= 1e-4 and np.abs(np.array(c.normal[:]) - info[i, 6:9]).max() <= 1e-4
        else:
            grazing += len(bad)  # the adapter keeps no contact list on the host: bounded below
        worst_dv = max(worst_dv, float(np.delete(dv, bad).max()))
    return events, bodies, grazing, worst_x, worst_dv


@pytest.mark.parametrize("mode", [0, 1])
def test_contact_path_vs_reference(mode, cpu_libs):
    """Cloth dropped onto a floor box, a sphere, a torus, a cylinder, a hollow sphere and a hollow box (every analytic distance field of
    DistanceFieldCollisionDetection; rotated bodies exercise the local frames), 150 steps in lockstep with the fp64 checker: the same
    contact list with matching contact points and normals, positions within 1e-4 and velocities within 2e-3 m/s after every step."""
    from positionbaseddynamics_b200 import _capi
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    colliders = scenes.on_recorded_colliders(cpu, "cloth_all_shapes")
    cpu.init_groups()
    eng = _engine_from(cpu, colliders)
    eng.set_params(dt=0.005, sub_steps=1, max_iter=4)
    eng.set_mode(mode)
    n = cpu.num_particles()
    xo = np.zeros((n, 3), np.float32); vo = np.zeros((n, 3), np.float32)
    def step_gpu(x, v):
        eng.step_host(1, x.astype(np.float32), v.astype(np.float32), xo, vo)
    events, bodies, grazing, worst_x, worst_dv = _lockstep(step_gpu, lambda: (xo, vo), cpu, 150, contacts_gpu=lambda: eng.contacts())
    print("lockstep, mode %d: %d contact events on bodies %s, %d grazing, worst rel pos %.2e, worst |dv| %.2e m/s" % (mode, events, sorted(bodies), grazing, worst_x, worst_dv))
    assert events > 2000 and len(bodies) >= 5 and grazing <= 3
    # free-running for the first 40 steps (the first contacts appear around step 35): still inside the tolerance
    cpu2 = cpu_libs.CpuPbd("oracle", "f64")
    colliders = scenes.on_recorded_colliders(cpu2, "cloth_all_shapes")
    cpu2.init_groups()
    eng2 = _engine_from(cpu2, colliders)
    eng2.set_params(dt=0.005, sub_steps=1, max_iter=4); eng2.set_mode(mode)
    eng2.step(40); eng2.sync(); cpu2.step(40)
    assert len(cpu2.oracle_contacts()[0]) > 0 and rel_position_error(eng2.get_attr(_capi.ATTR_X), cpu2.get("x")) <= TOL
    eng.close(); eng2.close()


def test_tet_model_contacts_with_substeps(cpu_libs):
    """A tet model as the particle side (TetModelCollisionObjectType + rigid body: collisionDetectionRBSolid as well), two substeps per
    step: the contacts are detected and solved once per step, after the substeps (TimeStepController.cpp:189-196)."""
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    colliders = scenes.on_recorded_colliders(cpu, "bar")
    cpu.init_groups()
    eng = _engine_from(cpu, colliders)
    eng.set_params(dt=0.005, sub_steps=2, max_iter=3)
    n = cpu.num_particles()
    xo = np.zeros((n, 3), np.float32); vo = np.zeros((n, 3), np.float32)
    def step_gpu(x, v):
        eng.step_host(1, x.astype(np.float32), v.astype(np.float32), xo, vo)
    events, bodies, grazing, worst_x, worst_dv = _lockstep(step_gpu, lambda: (xo, vo), cpu, 200, contacts_gpu=lambda: eng.contacts())
    print("tet bar, 2 substeps: %d contact events on bodies %s, %d grazing, worst rel pos %.2e, worst |dv| %.2e m/s" % (events, sorted(bodies), grazing, worst_x, worst_dv))
    assert events > 300 and len(bodies) >= 2 and grazing <= 3
    eng.close()


def test_contacts_matter_and_colliders_are_validated(cpu_libs):
    """Negative control: the same engine without the colliders leaves the tolerance by orders of magnitude; a collider on a dynamic body
    is refused."""
    from positionbaseddynamics_b200 import _capi
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    scenes.on_recorded_colliders(cpu, "cloth_box_sphere_torus")
    cpu.init_groups()
    eng = _engine_from(cpu)
    eng.set_params(dt=0.005, sub_steps=1, max_iter=4)
    eng.step(120); eng.sync(); cpu.step(120)
    assert rel_position_error(eng.get_attr(_capi.ATTR_X), cpu.get("x")) > 100 * TOL
    rb = cpu.rigid_bodies()
    eng.set_rigid_bodies([0.0, 2.0, 0.0], rb[:, :3], rb[:, 3:7], [(1.0, 1.0, 1.0)] * 3)
    rc = _capi.RigidCollider(); rc.shape = _capi.SHAPE_SPHERE; rc.body = 1; rc.dim[0] = 1.0
    with pytest.raises(_capi.PbdError, match="static colliders only"):
        eng.set_colliders([_capi.ParticleCollider(0, 576, 0.5, 0.1)], [rc])
    eng.close()


@pytest.mark.parametrize("precision", ["f32", "f64"])
def test_adapter_runs_the_contact_path(precision, cpu_libs):
    """The reference-side adapter with the reference's own DistanceFieldCollisionDetection attached (TimeStep::setCollisionDetection,
    as Demos/DistanceFieldDemos/ClothCollisionDemo.cpp:162-181): GpuTimeStepController reads the collision objects, the engine detects
    and solves the contacts; twin on the fp64 checker."""
    from oracle import pyoracle
    if not pyoracle.available("refgpu", precision):
        pytest.skip("prebuilt oracle/_ref/libpbdref_gpu_%s.so not present on this box" % precision)
    gpu = cpu_libs.CpuPbd("refgpu", precision); cpu = cpu_libs.CpuPbd("oracle", "f64")
    scenes.cloth_on_colliders(gpu, 24, shapes=ALL_SHAPES)
    scenes.on_recorded_colliders(cpu, "cloth_all_shapes")
    gpu.use_gpu_timestep(0, 0)
    gpu.set_contact_params(stiffness=100.0, max_iter_v=5)  # the parameter lives in the time step: set it on the installed one
    def step_gpu(x, v):
        gpu.set("x", x); gpu.set("v", v)   # host state is authoritative: uploaded by the adapter before the step
        gpu.step(1)
        assert gpu.gpu_error() == "", gpu.gpu_error()
    events, bodies, grazing, worst_x, worst_dv = _lockstep(step_gpu, lambda: (gpu.get("x"), gpu.get("v")), cpu, 120)
    print("adapter + contact path, Real=%s: %d contact events, %d grazing, worst rel pos %.2e, worst |dv| %.2e m/s" % (precision, events, grazing, worst_x, worst_dv))
    assert events > 1500 and len(bodies) >= 5 and grazing <= 3
    # a dynamic collision body is refused, nothing is stepped
    x1 = gpu.get("x").copy()
    gpu.set_rigid_body_mass(1, 3.0)
    gpu.step(1)
    assert "dynamic collision object" in gpu.gpu_error()
    assert (gpu.get("x") == x1).all()


def test_host_mirror_contact_path(cpu_libs):
    """The same scene through the host mirror of the reference's interface (C++ SimulationModel / TimeStepController /
    DistanceFieldCollisionDetection of csrc/host/pbd_model.h, driven through include/pbd_b200_model.h): addCollisionBox / Sphere / Torus on static
    bodies, addCollisionObjectWithoutGeometry for the cloth, TimeStep::setCollisionDetection -- in lockstep with the fp64 checker."""
    from positionbaseddynamics_b200 import _capi, model as hm_mod
    cpu = cpu_libs.CpuPbd("oracle", "f64")
    scenes.on_recorded_colliders(cpu, "cloth_box_sphere_torus")
    hm = hm_mod.HostModel()
    hm.add_regular_triangle_model(24, 24, t=(-2.5, 2.2, -2.5), R=scenes.RX90, scale=(5.0, 5.0))
    hm.add_cloth_constraints(0, 4, dist_k=1.0e5)
    hm.add_bending_constraints(0, 3, 100.0)
    hm.set_params(dt=0.005, sub_steps=1, max_iter=4)
    rot = np.array([[0.9553365, -0.2955202, 0.0], [0.2955202, 0.9553365, 0.0], [0.0, 0.0, 1.0]])
    qz = (float(np.cos(0.15)), 0.0, 0.0, float(np.sin(0.15)))  # 0.3 rad about z = `rot`
    cd = hm_mod.CollisionDetection(); cd.set_tolerance(0.05)
    spec = [((0.0, -0.5, 0.0), (1, 0, 0, 0), (20.0, 1.0, 20.0), _capi.SHAPE_BOX, (20.0, 1.0, 20.0), 0.2),
            ((-0.8, 1.2, -0.6), (1, 0, 0, 0), (1.6, 1.6, 1.6), _capi.SHAPE_SPHERE, (0.8,), 0.1),
            ((1.2, 1.0, 0.8), qz, (2.4, 0.8, 2.4), _capi.SHAPE_TORUS, (0.8, 0.4), 0.1)]
    for x, q, scale, shape, dims, friction in spec:
        i = hm.add_rigid_body(0.0, x, (1.0, 1.0, 1.0), q)
        hm.set_contact_coefficients(0, i, 0.6, friction)
        cd.add_shape(i, hm_mod.RIGID_BODY_COLLISION_OBJECT, shape, dims, 0.05, vertices=scenes.BOX_VERTS * np.array(scale))
    hm.set_contact_coefficients(1, 0, 0.5, 0.1)
    cd.add_object_without_geometry(0, hm_mod.TRIANGLE_MODEL_COLLISION_OBJECT, True)
    hm.set_contact_stiffness_particle_rigid_body(100.0)
    ts = hm.time_step(device=0)
    ts.set_collision_detection(hm, cd)
    def step_gpu(x, v):
        hm.set("x", x); hm.set("v", v); hm.step(1)
    events, seen, grazing, worst_x, worst_dv = _lockstep(step_gpu, lambda: (hm.get("x"), hm.get("v")), cpu, 120)
    print("host mirror + contact path: %d contact events on bodies %s, %d grazing, worst rel pos %.2e, worst |dv| %.2e m/s" % (events, sorted(seen), grazing, worst_x, worst_dv))
    assert events > 1000 and len(seen) >= 2 and grazing <= 3  # the floor box is not reached within 120 steps
    # a dynamic collision body is refused with the reference-style bool + error
    hm.set_rigid_body_mass(1, 2.0)
    with pytest.raises(hm_mod.PbdError, match="dynamic collision object"):
        hm.step(1)
    hm.close(); cd.close()
