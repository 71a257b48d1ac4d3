"""The pyPBD-named facade: scene construction in the reference's own call style (pyPBD/examples/cloth_model.py:18-124)."""
import math
import numpy as np
import pytest


def _build():
    import positionbaseddynamics_b200.pypbd as pbd
    pbd.Simulation._current = None
    sim = pbd.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
    a = math.pi / 2
    R = [[1, 0, 0], [0, math.cos(a), -math.sin(a)], [0, math.sin(a), math.cos(a)]]
    model.addRegularTriangleModel(20, 20, [0, 1, 0], R, [10, 10])
    pd = model.getParticles()
    pd.setMass(0, 0.0); pd.setMass(19, 0.0)
    tm = model.getTriangleModels()[0]
    model.addClothConstraints(tm, 4, 1.0e5, 1.0, 1.0, 1.0, 0.3, 0.3, False, False)
    model.addBendingConstraints(tm, 3, 100.0)
    return pbd, sim, model


def test_scene_construction_matches_oracle(cpu_libs):
    import scenes
    pbd, sim, model = _build()
    o = cpu_libs.CpuPbd("oracle", "f64")
    scenes.cloth(o, 20, 20, 4, 3, dist_k=1e5, bend_k=100.0)
    groups = model.getConstraintGroups()
    off, ids = o.groups()
    assert len(groups) == len(off) - 1 and all((groups[g] == ids[off[g]:off[g + 1]]).all() for g in range(len(groups)))
    assert model.numConstraints() == o.num_constraints()
    assert model.getTriangleModels()[0].getParticleMesh().numFaces() == 2 * 19 * 19
    pd = model.getParticles()
    assert pd.size() == 400 and pd.getMass(0) == 0.0 and pd.getInvMass(1) == 1.0
    assert np.allclose(pd.getVertices(), o.get("x"), atol=1e-6)
    pd.setPosition(5, [1, 2, 3]); assert (pd.getPosition(5) == [1, 2, 3]).all()
    c = model.getConstraints()[0]
    assert c["type"] == "Distance_XPBD" and len(c["bodies"]) == 2


@pytest.mark.gpu
def test_step_through_facade(cpu_libs):
    import scenes
    from parity_util import rel_position_error
    pbd, sim, model = _build()
    ts = sim.getTimeStep()
    ts.setValueUInt(pbd.TimeStepController.NUM_SUB_STEPS, 1)
    ts.setValueUInt(pbd.TimeStepController.MAX_ITERATIONS, 5)
    pbd.TimeManager.getCurrent().setTimeStepSize(0.005)
    o = cpu_libs.CpuPbd("oracle", "f64")
    scenes.cloth(o, 20, 20, 4, 3, dist_k=1e5, bend_k=100.0, sub_steps=1, max_iter=5)
    for _ in range(5):
        ts.step(model)
    o.step(5)
    assert rel_position_error(model.getParticles().getVertices(), o.get("x")) <= 1e-4
    assert abs(pbd.TimeManager.getCurrent().getTime() - 0.025) < 1e-6
    sim.reset()
    assert np.allclose(model.getParticles().getVertices(), o.get("x0"), atol=1e-6)


def test_builders_return_the_model_like_pypbd_and_refuse_collision_meshes():
    """pyPBD's addRegular*Model / add*Model return the new model (SimulationModelModule.cpp:98-229) and take testMesh; the
    reference's example scripts use both."""
    import positionbaseddynamics_b200.pypbd as pbd
    pbd.Simulation._current = None
    sim = pbd.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
    tri = model.addRegularTriangleModel(4, 4, [0, 0, 0], np.eye(3), [1, 1], testMesh=False)
    tet = model.addRegularTetModel(3, 3, 3, testMesh=False)
    assert tri.getIndexOffset() == 0 and tri.getParticleMesh().numFaces() == 18
    assert tet.getIndexOffset() == 16 and tet.getParticleMesh().numTets() == 40
    tri2 = model.addTriangleModel([[0, 0, 0], [1, 0, 0], [0, 1, 0]], [0, 1, 2])
    assert tri2.getIndexOffset() == 16 + 27 and tri2.getParticleMesh().numFaces() == 1
    with pytest.raises(pbd.PbdError):
        model.addRegularTriangleModel(4, 4, testMesh=True)
    pbd.Logger.addConsoleSink(pbd.LogLevel.INFO)
    pbd.Timing.reset(); pbd.Timing.printAverageTimes()


@pytest.mark.gpu
def test_example_scripts_run():
    """examples/cloth_model.py and beam_model.py (headless counterparts of the reference's pyPBD examples): pinned particles stay,
    everything stays finite, the cloth falls."""
    import importlib.util, os
    import positionbaseddynamics_b200.pypbd as pbd
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples")
    out = {}
    for name in ("cloth_model", "beam_model"):
        pbd.Simulation._current = None
        spec = importlib.util.spec_from_file_location(name, os.path.join(root, name + ".py"))
        mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
        out[name] = mod.main(frames=2)
        assert np.isfinite(out[name]).all()
        pd = pbd.Simulation.getCurrent().getModel().getParticles()
        pinned = [i for i in range(pd.size()) if pd.getMass(i) == 0.0]
        assert len(pinned) == (2 if name == "cloth_model" else 25)
        for i in pinned:                                   # static particles never move
            assert (out[name][i] == np.asarray(pd.getPosition0(i), dtype=np.float32)).all()
        assert out[name][:, 1].min() < -1e-3               # the rest sags under gravity
    assert pbd.Timing.averageStepMs() > 0.0
    # examples/cloth_collision.py (Demos/DistanceFieldDemos/ClothCollisionDemo.cpp in pyPBD names): the cloth ends up draped over the
    # torus and resting on the floor, not below it
    pbd.Simulation._current = None
    spec = importlib.util.spec_from_file_location("cloth_collision", os.path.join(root, "cloth_collision.py"))
    mod = importlib.util.module_from_spec(spec); spec.loader.exec_module(mod)
    x = mod.main(frames=50)
    assert np.isfinite(x).all() and x[:, 1].min() > -0.2 and x[:, 1].max() > 1.5


CUBE_V = np.array([[-0.5, -0.5, -0.5], [0.5, -0.5, -0.5], [0.5, 0.5, -0.5], [-0.5, 0.5, -0.5],
                   [-0.5, -0.5, 0.5], [0.5, -0.5, 0.5], [0.5, 0.5, 0.5], [-0.5, 0.5, 0.5]])
CUBE_F = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [1, 2, 6], [1, 6, 5], [0, 4, 7], [0, 7, 3]])


def test_mass_properties_and_rigid_body_facade():
    """pyPBD's addRigidBody(density, vertices, mesh, ...) derives mass, centre of mass and principal inertia from the mesh
    (RigidBody::determineMassProperties); checked against the closed forms of a box and of a tetrahedron."""
    import positionbaseddynamics_b200.pypbd as pbd
    w, h, d = 0.4, 2.0, 0.6
    m, c, J = pbd.mass_properties(CUBE_V * [w, h, d] + [1.0, -2.0, 3.0], CUBE_F, 2.5)
    assert np.isclose(m, 2.5 * w * h * d) and np.allclose(c, [1.0, -2.0, 3.0])
    assert np.allclose(J, np.diag([m / 12 * (h * h + d * d), m / 12 * (w * w + d * d), m / 12 * (w * w + h * h)]), atol=1e-12)
    tet_v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1.0]]); tet_f = np.array([[0, 2, 1], [0, 1, 3], [0, 3, 2], [1, 2, 3]])
    m, c, J = pbd.mass_properties(tet_v, tet_f, 6.0)
    assert np.isclose(m, 1.0) and np.allclose(c, [0.25, 0.25, 0.25])
    assert np.isclose(J[0, 0], 6.0 * (1 / 60 + 1 / 60) - 2 * 0.25 ** 2)          # int(y^2 + z^2) about the origin, shifted to the centre of mass
    pbd.Simulation._current = None
    sim = pbd.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
    a = model.addRigidBody(1.0, CUBE_V, CUBE_F, translation=[-5.0, 0.0, -5.0], scale=[0.5, 0.5, 0.5], testMesh=False, generateCollisionObject=False)
    a.setMass(0.0)
    b = model.addRigidBody(1.0, CUBE_V, CUBE_F, [-5.0, 1.0, -5.0], scale=[w, h, d])
    assert a.getMass() == 0.0 and np.isclose(b.getMass(), w * h * d) and np.allclose(b.getPosition(), [-5.0, 1.0, -5.0])
    assert np.isclose(np.linalg.norm(b.getRotation()), 1.0) and len(model.getRigidBodies()) == 2
    tri = model.addRegularTriangleModel(4, 4, [0, 0, 0], np.eye(3), [1, 1])
    assert model.addBallJoint(0, 1, [-5.0, 0.0, -5.0]) and model.addRigidBodyParticleBallJoint(1, 0)
    assert model.numConstraints() == 2
    with pytest.raises(pbd.PbdError):
        model.addRigidBody(1.0, CUBE_V, CUBE_F, generateCollisionObject=True)


def coupling_example_model():
    """(example module, model) of examples/rigid_body_cloth_coupling.py, built through the facade."""
    import importlib.util, os
    import positionbaseddynamics_b200.pypbd as pbd
    pbd.Simulation._current = None
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples")
    spec = importlib.util.spec_from_file_location("rigid_body_cloth_coupling", os.path.join(root, "rigid_body_cloth_coupling.py"))
    ex = importlib.util.module_from_spec(spec); spec.loader.exec_module(ex)
    return ex, ex.buildModel()


def coupling_example_on_cpu(ref, ex, host):
    """The example's scene on a CPU checker, given the same bodies (mass, position, principal inertia, rotation) as the facade's."""
    ref.add_regular_triangle_model(ex.nCols, ex.nRows, [-5, 4, -5], ex.rotation_x(np.pi * 0.5), [ex.clothWidth, ex.clothHeight])
    ref.add_cloth_constraints(0, 2, 1.0, 1.0, 1.0, 1.0, 0.3, 0.3)
    ref.add_bending_constraints(0, 2, 0.01)
    rb = host.rigid_bodies()
    dims = {0: (0.5, 0.5, 0.5)}
    for i in range(len(rb)):
        mass = host.rigid_body_mass(i)
        w, h, d = (0.5, 0.5, 0.5) if i % 3 == 0 else (ex.width, ex.height, ex.depth)
        m = w * h * d
        inertia = np.sort([m / 12 * (h * h + d * d), m / 12 * (w * w + d * d), m / 12 * (w * w + h * h)])  # principal moments, ascending like eigh
        ref.add_rigid_body(mass, rb[i, 0:3], inertia, rb[i, 3:7])
    for chain in range(4):
        base = 3 * chain; x, z = rb[base, 0], rb[base, 2]
        ref.add_ball_joint(base, base + 1, [x, 0.0, z]); ref.add_ball_joint(base + 1, base + 2, [x, 2.0, z])
    for body, particle in ((2, 0), (5, ex.nCols - 1), (8, ex.nRows * ex.nCols - 1), (11, (ex.nRows - 1) * ex.nCols)):
        ref.add_rb_particle_ball_joint(body, particle)
    ref.set_params(dt=0.005, sub_steps=3, max_iter=1)


@pytest.mark.gpu
def test_coupling_example_against_the_reference():
    """examples/rigid_body_cloth_coupling.py (pyPBD-style construction incl. mesh-derived mass properties) stepped on the GPU, against
    the unmodified reference given the same bodies (coupling_example_on_cpu): its recorded run, tests/golden/reference_runs.npz."""
    import positionbaseddynamics_b200.pypbd as pbd
    import reference_golden as rg
    _, model = coupling_example_model()
    host = model._host
    assert rg.get("coupling_example/num_constraints") == model.numConstraints()
    sim = pbd.Simulation.getCurrent()
    for _ in range(6):
        sim.getTimeStep().step(model)
    xg = model.getParticles().getVertices()
    x_ref, x_got, x_scale = rg.sampled("coupling_example/", "x", xg)
    err = np.abs(x_got - x_ref).max() / x_scale
    print("coupling example vs reference: rel pos %.2e" % err)
    assert err <= 1e-4
    assert np.abs(host.rigid_bodies()[:, :3] - rg.get("coupling_example/rb_x")).max() <= 1e-4


def _quat_to_matrix(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


RB_R0 = np.array([[np.cos(0.3), -np.sin(0.3), 0], [np.sin(0.3), np.cos(0.3), 0], [0, 0, 1.0]])
RB_VERTS = CUBE_V + [0.1, 0.2, 0.3]          # off-centre: the body frame has to move to the centre of mass
RB_SCALES = ([0.4, 2.0, 0.6], [1.0, 1.0, 3.0])


def test_facade_rigid_body_matches_the_reference_init():
    """addRigidBody(density, vertices, mesh, translation, rotation, scale) against the unmodified reference's
    RigidBody::initBody(density, ...) (Utils/VolumeIntegration.cpp + principal-axes transform), as recorded in
    tests/golden/reference_runs.npz: mass, principal moments, position and the world-space inertia tensor (the principal frame
    itself is only defined up to signs / degenerate subspaces)."""
    import positionbaseddynamics_b200.pypbd as pbd
    import reference_golden as rg
    R0, verts = RB_R0, RB_VERTS
    for k, scale in enumerate(RB_SCALES):
        props = rg.get("facade_rigid_body/%d/props" % k)
        pbd.Simulation._current = None
        sim = pbd.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
        rb = model.addRigidBody(2.0, verts, CUBE_F, translation=[1.0, 2.0, 3.0], rotation=R0, scale=scale)
        assert np.isclose(rb.getMass(), props[0], rtol=1e-6)
        assert np.allclose(rb.getPosition(), props[4:7], rtol=1e-6, atol=1e-6)
        # principal moments: recompute the facade's from its stored body (model.py keeps them; compare through the world tensor)
        mass, com, J = pbd.mass_properties(verts * np.asarray(scale), CUBE_F, 2.0)
        assert np.allclose(np.sort(np.linalg.eigvalsh(J)), np.sort(props[1:4]), rtol=1e-9)
        Rr = _quat_to_matrix(props[7:11]); Jw_ref = Rr @ np.diag(props[1:4]) @ Rr.T
        w, V = np.linalg.eigh(J); Rf = _quat_to_matrix(rb.getRotation().astype(np.float64)); Jw_fac = Rf @ np.diag(w) @ Rf.T
        assert np.allclose(Jw_fac, Jw_ref, rtol=1e-5, atol=1e-6), (Jw_fac, Jw_ref)
        assert np.allclose(Jw_ref, R0 @ J @ R0.T, rtol=1e-9, atol=1e-12)


def test_compiled_pybind_module_builds_the_same_model():
    """The compiled pybind11 module (csrc/pybind/pypbd_module.cpp, north_star "pyPBD via pybind") exposes the pyPBD names over the
    same C++ host mirror: scene construction, constraint counts and colour groups equal the ctypes facade's (no GPU needed until
    getTimeStep())."""
    import importlib, math, os, sys
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "positionbaseddynamics_b200")
    sys.path.insert(0, pkg)
    try:
        native = importlib.import_module("pypbd_b200")
    finally:
        sys.path.remove(pkg)
    from positionbaseddynamics_b200 import pypbd as facade
    R = np.array([[1, 0, 0], [0, math.cos(math.pi / 2), -math.sin(math.pi / 2)], [0, math.sin(math.pi / 2), math.cos(math.pi / 2)]])
    sim = native.Simulation.getCurrent(); sim.initDefault(); m1 = sim.getModel()
    m2 = facade.SimulationModel()
    for m in (m1, m2):
        tm = m.addRegularTriangleModel(30, 20, (0, 1, 0), R, (6.0, 4.0))
        pd = m.getParticles(); pd.setMass(0, 0.0); pd.setMass(29, 0.0)
        m.addClothConstraints(tm, 4, 1.0e5, 1.0, 1.0, 1.0, 0.3, 0.3, False, False)
        m.addBendingConstraints(tm, 3, 100.0)
        tt = m.addRegularTetModel(5, 4, 3, (0, 3, 0), np.eye(3), (2.0, 1.0, 1.0))
        m.addSolidConstraints(tt, 2, 1.0e6, 0.3, 1.0, False, False)
    assert m1.numConstraints() == m2.numConstraints() > 0
    g1, g2 = m1.getConstraintGroups(), m2.getConstraintGroups()
    assert len(g1) == len(g2) and all((np.asarray(a) == np.asarray(b)).all() for a, b in zip(g1, g2))
    assert (m1.getParticles().getVertices() == m2.getParticles().getVertices()).all()
    assert m1.getParticles().getInvMass(0) == 0.0 and m1.getParticles().getMass(5) == 1.0
    assert native.TimeStepController.NUM_SUB_STEPS == facade.TimeStepController.NUM_SUB_STEPS
    assert m1.getTriangleModels()[0].getParticleMesh().numFaces() == 2 * 29 * 19
    c1, c2 = m1.getConstraints(), m2.getConstraints()
    assert all((c1[i]["bodies"] == c2[i]["bodies"]).all() for i in range(0, len(c1), 97))


@pytest.mark.gpu
def test_compiled_pybind_module_steps_like_the_facade():
    """The reference's cloth example flow (pyPBD/examples/cloth_model.py:18-124) through the compiled module: same bits as the ctypes
    facade, and the getVertices() view follows the device state."""
    import importlib, os, sys
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "positionbaseddynamics_b200")
    sys.path.insert(0, pkg)
    try:
        native = importlib.import_module("pypbd_b200")
    finally:
        sys.path.remove(pkg)
    pbd, sim2, model2 = _build()
    a = math.pi / 2
    R = [[1, 0, 0], [0, math.cos(a), -math.sin(a)], [0, math.sin(a), math.cos(a)]]
    sim = native.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
    tm = model.addRegularTriangleModel(20, 20, [0, 1, 0], R, [10, 10])
    pd = model.getParticles(); pd.setMass(0, 0.0); pd.setMass(19, 0.0)
    model.addClothConstraints(tm, 4, 1.0e5, 1.0, 1.0, 1.0, 0.3, 0.3, False, False)
    model.addBendingConstraints(tm, 3, 100.0)
    for s, mdl, mod in ((sim, model, native), (sim2, model2, pbd)):
        ts = s.getTimeStep()
        ts.setValueUInt(mod.TimeStepController.NUM_SUB_STEPS, 1); ts.setValueUInt(mod.TimeStepController.MAX_ITERATIONS, 5)
        mod.TimeManager.getCurrent().setTimeStepSize(0.005)
        for _ in range(4):
            ts.step(mdl)
    x1 = np.array(model.getParticles().getVertices()); x2 = np.array(model2.getParticles().getVertices())
    assert np.isfinite(x1).all() and (x1 == x2).all()
    assert abs(native.TimeManager.getCurrent().getTime() - 0.02) < 1e-6
    assert (x1[0] == [0.0, 1.0, 0.0]).all() or np.allclose(x1[0], model.getParticles().getPosition0(0))  # pinned corner


def test_collision_registry_in_both_python_surfaces():
    """DistanceFieldCollisionDetection with the reference's add* signatures (pyPBD/CollisionDetectionModule.cpp) in the compiled module and in
    the ctypes facade: construction and bookkeeping need no GPU."""
    import importlib, os, sys
    import positionbaseddynamics_b200.pypbd as pbd
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "positionbaseddynamics_b200")
    sys.path.insert(0, pkg)
    try:
        native = importlib.import_module("pypbd_b200")
    finally:
        sys.path.remove(pkg)
    for mod, rigid in ((native, native.CollisionDetection.CollisionObject.RigidBodyCollisionObjectType), (pbd, pbd.CollisionObject.RigidBodyCollisionObjectType)):
        cd = mod.DistanceFieldCollisionDetection(); cd.init()
        assert abs(cd.getTolerance() - 0.01) < 1e-7   # CollisionDetection.cpp:25
        cd.setTolerance(0.05)
        box = np.array([[-1, -1, -1], [1, 1, 1.0]])
        cd.addCollisionBox(0, rigid, box, 2, [2.0, 2.0, 2.0])
        cd.addCollisionSphere(1, rigid, None, 0, 0.5, True, False)
        cd.addCollisionTorus(2, rigid, None, 0, [1.0, 0.25])
        cd.addCollisionCylinder(3, rigid, None, 0, [0.5, 2.0])
        cd.addCollisionHollowSphere(4, rigid, None, 0, 1.0, 0.1)
        cd.addCollisionHollowBox(5, rigid, None, 0, [1.0, 1.0, 1.0], 0.1)
        cd.addCollisionObjectWithoutGeometry(0, 1, None, 0, True)
        assert cd.numCollisionObjects() == 7 and abs(cd.getTolerance() - 0.05) < 1e-7


@pytest.mark.gpu
def test_compiled_pybind_module_runs_the_contact_path():
    """Cloth dropped on a static sphere through the compiled module (the flow of Demos/DistanceFieldDemos/ClothCollisionDemo.cpp in pyPBD
    names): the sheet wraps the sphere instead of falling through it, and a dynamic collision body is refused with an exception."""
    import importlib, os, sys
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "positionbaseddynamics_b200")
    sys.path.insert(0, pkg)
    try:
        native = importlib.import_module("pypbd_b200")
    finally:
        sys.path.remove(pkg)
    a = math.pi / 2
    R = [[1, 0, 0], [0, math.cos(a), -math.sin(a)], [0, math.sin(a), math.cos(a)]]
    def run(with_collider):
        model = native.SimulationModel()
        tm = model.addRegularTriangleModel(30, 30, [-1.5, 1.5, -1.5], R, [3.0, 3.0])
        model.addClothConstraints(tm, 4, 1.0e5, 1.0, 1.0, 1.0, 0.3, 0.3, False, False)
        model.addBendingConstraints(tm, 3, 100.0)
        rb = model.addRigidBody(0.0, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
        ts = native.TimeStepController(0)
        ts.setValueUInt(native.TimeStepController.NUM_SUB_STEPS, 1); ts.setValueUInt(native.TimeStepController.MAX_ITERATIONS, 5)
        cd = native.DistanceFieldCollisionDetection(); cd.setTolerance(0.05)
        if with_collider:
            T = native.CollisionDetection.CollisionObject
            cd.addCollisionSphere(rb, T.RigidBodyCollisionObjectType, None, 0, 1.0)
            cd.addCollisionObjectWithoutGeometry(0, T.TriangleModelCollisionObjectType, None, 0, True)
            ts.setCollisionDetection(model, cd)
        for _ in range(200):
            ts.step(model)
        return np.array(model.getParticles().getVertices()).copy(), model, ts
    x_free, _, _ = run(False)
    x_hit, model, ts = run(True)
    r_free = np.linalg.norm(x_free, axis=1).min(); r_hit = np.linalg.norm(x_hit, axis=1).min()
    print("closest particle to the sphere centre: %.3f without the collider, %.3f with it (radius 1)" % (r_free, r_hit))
    assert x_free[:, 1].max() < -1.0                     # fell straight through
    assert r_hit > 0.9 and x_hit[:, 1].max() > 0.5       # held up by the sphere
    model.getRigidBodies()[0]  # the body object is reachable
    # dynamic collision body: refused
    model2 = native.SimulationModel()
    tm = model2.addRegularTriangleModel(10, 10, [-1.5, 1.5, -1.5], R, [3.0, 3.0])
    model2.addClothConstraints(tm, 4, 1.0e5, 1.0, 1.0, 1.0, 0.3, 0.3, False, False)
    rb = model2.addRigidBody(2.0, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))
    cd = native.DistanceFieldCollisionDetection()
    cd.addCollisionSphere(rb, 0, None, 0, 1.0); cd.addCollisionObjectWithoutGeometry(0, 1, None, 0, True)
    ts2 = native.TimeStepController(0); ts2.setCollisionDetection(model2, cd)
    with pytest.raises(RuntimeError, match="dynamic collision object"):
        ts2.step(model2)
