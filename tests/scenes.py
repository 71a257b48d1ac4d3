"""Deterministic benchmark/parity scenes (SURVEY.md section 8d), expressed against the common builder
surface shared by the CPU checkers (oracle.pyoracle.CpuPbd) and the product's host model
(positionbaseddynamics_b200.SimulationModel facade): add_regular_triangle_model / add_regular_tet_model /
set_mass / add_cloth_constraints / add_bending_constraints / add_solid_constraints / add_constraint /
set_params.  Scene definitions follow Demos/ClothDemo/main.cpp:132-162 and Demos/BarDemo/main.cpp:130-166.
"""
import math
import numpy as np

RX90 = np.array([[1, 0, 0], [0, math.cos(math.pi / 2), -math.sin(math.pi / 2)],
                 [0, math.sin(math.pi / 2), math.cos(math.pi / 2)]], dtype=np.float64)

VOLUME = 7  # flat type code


def cloth(m, nx, ny, cloth_method=1, bending_method=2, dist_k=1.0, bend_k=0.01, sub_steps=1, max_iter=5,
          dt=0.005, vel_method=0, size=10.0, fem=(1.0, 1.0, 1.0, 0.3, 0.3)):
    """ClothDemo (Demos/ClothDemo/main.cpp:132-162): nx x ny sheet, corners 0 and nx-1 pinned."""
    m.add_regular_triangle_model(nx, ny, t=(0, 1, 0), R=RX90, scale=(size, size))
    m.set_mass(0, 0.0)
    m.set_mass(nx - 1, 0.0)
    m.add_cloth_constraints(0, cloth_method, dist_k=dist_k, xx=fem[0], yy=fem[1], xy=fem[2], pxy=fem[3], pyx=fem[4])
    m.add_bending_constraints(0, bending_method, bend_k)
    m.set_params(dt=dt, sub_steps=sub_steps, max_iter=max_iter, vel_method=vel_method)


def cfg1(m, n=50):
    """cfg1: ClothDemo 50x50, Distance + IsometricBending (PBD), 1 substep x 5 iterations."""
    cloth(m, n, n, cloth_method=1, bending_method=2, dist_k=1.0, bend_k=0.01, sub_steps=1, max_iter=5)


def cfg2(m, n=1000, max_iter=20):
    """cfg2: n x n cloth, Distance_XPBD (k=1e5) + IsometricBending_XPBD (k=100), 1 substep x 20 iterations."""
    cloth(m, n, n, cloth_method=4, bending_method=3, dist_k=1.0e5, bend_k=100.0, sub_steps=1, max_iter=max_iter)


def bar(m, w, h, d, solid_method=2, k=1.0e6, nu=0.3, vol_k=1.0, extra_volume=False, sub_steps=10, max_iter=5,
        dt=0.005, scale=(10.0, 1.5, 1.5), norm_stretch=False):
    """BarDemo (Demos/BarDemo/main.cpp:130-166): w x h x d regular tet bar, slab i == 0 fixed."""
    m.add_regular_tet_model(w, h, d, t=(5, 0, 0), R=np.eye(3), scale=scale)
    for j in range(h):
        for kk in range(d):
            m.set_mass(j * d + kk, 0.0)  # i == 0 slab: index i*h*d + j*d + k
    m.add_solid_constraints(0, solid_method, k=k, nu=nu, vol_k=vol_k, norm_stretch=norm_stretch)
    if extra_volume:
        for t in m.tet_tets(0):
            m.add_constraint(VOLUME, [int(v) for v in t], [vol_k])
    m.set_params(dt=dt, sub_steps=sub_steps, max_iter=max_iter)


def cfg3(m, w=101, h=21, d=21):
    """cfg3: 101x21x21 bar = 200,000 tets, FEMTet (E=1e6, nu=0.3) + one Volume constraint per tet, 10 x 5."""
    bar(m, w, h, d, solid_method=2, k=1.0e6, nu=0.3, vol_k=1.0, extra_volume=True, sub_steps=10, max_iter=5)


def mixed(m, n_cloth=24, bar_dims=(7, 4, 4), cloth_method=2, bending_method=2, solid_method=2, sub_steps=5, max_iter=1):
    """cfg4 without the rigid bodies: a cloth and a tet solid in ONE model (two particle ranges, constraint types
    interleaved in the colour groups), the scene shape of Demos/CouplingDemos/RigidBodyClothCouplingDemo.cpp:151-289.
    Defaults are the reference's: cloth method 2 (FEMTriangle), 5 substeps x 1 iteration (TimeStepController.cpp:28-30)."""
    m.add_regular_triangle_model(n_cloth, n_cloth, t=(0, 1, 0), R=RX90, scale=(5.0, 5.0))
    m.add_regular_tet_model(bar_dims[0], bar_dims[1], bar_dims[2], t=(2.5, 3.0, 2.5), R=np.eye(3), scale=(2.0, 0.6, 0.6))
    m.set_mass(0, 0.0); m.set_mass(n_cloth - 1, 0.0)
    off = n_cloth * n_cloth
    for j in range(bar_dims[1]):
        for k in range(bar_dims[2]):
            m.set_mass(off + j * bar_dims[2] + k, 0.0)
    m.add_cloth_constraints(0, cloth_method, dist_k=1.0, xx=1000.0, yy=1000.0, xy=500.0, pxy=0.3, pyx=0.3)
    m.add_bending_constraints(0, bending_method, 0.01)
    m.add_solid_constraints(0, solid_method, k=1.0e6 if solid_method in (2, 3) else 1.0, nu=0.3, vol_k=1.0)
    m.set_params(dt=0.005, sub_steps=sub_steps, max_iter=max_iter)


def box_inertia(mass, w, h, d):
    """computeInertiaTensorBox (Demos/CouplingDemos/RigidBodyClothCouplingDemo.cpp:140-146)."""
    return (mass / 12.0 * (h * h + d * d), mass / 12.0 * (w * w + d * d), mass / 12.0 * (w * w + h * h))


def coupling_rig(m, n_cols, n_rows, half=5.0):
    """The 12-body / 8-BallJoint / 4-RigidBodyParticleBallJoint rig of RigidBodyClothCouplingDemo.cpp:151-289: four chains
    (static anchor + two dynamic boxes) at the corners, the top box of each chain pinned to a cloth corner particle.
    Must be called after the cloth (particle indices 0, n_cols-1, n_rows*n_cols-1, (n_rows-1)*n_cols)."""
    width, height, depth = 0.4, 2.0, 0.4  # demo globals (RigidBodyClothCouplingDemo.cpp:33-35)
    corners = [(-half, -half), (half, -half), (half, half), (-half, half)]
    for cx, cz in corners:
        r0 = m.add_rigid_body(0.0, (cx, 0.0, cz), box_inertia(1.0, 0.5, 0.5, 0.5))
        r1 = m.add_rigid_body(1.0, (cx, 1.0, cz), box_inertia(1.0, width, height, depth))
        r2 = m.add_rigid_body(1.0, (cx, 3.0, cz), box_inertia(1.0, width, height, depth))
        m.add_ball_joint(r0, r1, (cx, 0.0, cz))
        m.add_ball_joint(r1, r2, (cx, 2.0, cz))
    for rb, particle in zip((2, 5, 8, 11), (0, n_cols - 1, n_rows * n_cols - 1, (n_rows - 1) * n_cols)):
        m.add_rb_particle_ball_joint(rb, particle)


def cfg4(m, n_cloth=224, bar_dims=(51, 21, 11), cloth_method=2, with_rig=True, sub_steps=5, max_iter=1):
    """cfg4: 224x224 cloth (99,458 triangles; FEMTriangle + IsometricBending) + 51x21x11 tet block (50,000 tets, FEMTet) +
    the rigid coupling rig; reference defaults 5 substeps x 1 iteration (SURVEY.md section 8)."""
    m.add_regular_triangle_model(n_cloth, n_cloth, t=(-5, 4, -5), R=RX90, scale=(10.0, 10.0))
    m.add_regular_tet_model(bar_dims[0], bar_dims[1], bar_dims[2], t=(0.0, 7.0, 0.0), R=np.eye(3), scale=(4.0, 1.5, 1.0))
    off = n_cloth * n_cloth
    for j in range(bar_dims[1]):
        for k in range(bar_dims[2]):
            m.set_mass(off + j * bar_dims[2] + k, 0.0)
    m.add_cloth_constraints(0, cloth_method, dist_k=1.0, xx=1000.0, yy=1000.0, xy=500.0, pxy=0.3, pyx=0.3)
    m.add_bending_constraints(0, 2, 0.01)
    m.add_solid_constraints(0, 2, k=1.0e6, nu=0.3)
    if with_rig:
        coupling_rig(m, n_cloth, n_cloth)
    m.set_params(dt=0.005, sub_steps=sub_steps, max_iter=max_iter)


def projections_per_step(num_constraints, sub_steps, max_iter):
    return num_constraints * sub_steps * max_iter


# ---- contact path: the geometry of Demos/DistanceFieldDemos/ClothCollisionDemo.cpp (cloth dropped onto static distance-field bodies) ----
BOX_VERTS = np.array([[-0.5, -0.5, -0.5], [0.5, -0.5, -0.5], [0.5, 0.5, -0.5], [-0.5, 0.5, -0.5],
                      [-0.5, -0.5, 0.5], [0.5, -0.5, 0.5], [0.5, 0.5, 0.5], [-0.5, 0.5, 0.5]], dtype=np.float64)
BOX_FACES = np.array([[0, 2, 1], [0, 3, 2], [4, 5, 6], [4, 6, 7], [0, 1, 5], [0, 5, 4], [2, 3, 7], [2, 7, 6], [0, 4, 7], [0, 7, 3], [1, 2, 6], [1, 6, 5]], dtype=np.uint32)


def cloth_on_colliders(m, n=24, tolerance=0.05, max_iter=4, sub_steps=1, shapes=("box", "sphere", "torus")):
    """Reference builds only (m = CpuPbd "ref"/"refgpu").  A (n x n) XPBD cloth above a static floor box, a static sphere and a static torus,
    each a rigid body whose mesh is a unit cube scaled to the shape's bounding box (the mesh only feeds the AABB and the mass properties)."""
    m.add_regular_triangle_model(n, n, t=(-2.5, 2.2, -2.5), R=RX90, scale=(5.0, 5.0))
    m.add_cloth_constraints(0, 4, dist_k=1.0e5)
    m.add_bending_constraints(0, 3, 100.0)
    m.set_params(dt=0.005, sub_steps=sub_steps, max_iter=max_iter)
    bodies = []
    rot = np.array([[0.9553365, -0.2955202, 0.0], [0.2955202, 0.9553365, 0.0], [0.0, 0.0, 1.0]])  # 0.3 rad about z: exercises R, v1, v2
    if "box" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(0.0, -0.5, 0.0), R=np.eye(3), scale=(20.0, 1.0, 20.0)); bodies.append((i, 0, (20.0, 1.0, 20.0)))
    if "sphere" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(-0.8, 1.2, -0.6), R=np.eye(3), scale=(1.6, 1.6, 1.6)); bodies.append((i, 1, (0.8,)))
    if "torus" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(1.2, 1.0, 0.8), R=rot, scale=(2.4, 0.8, 2.4)); bodies.append((i, 2, (0.8, 0.4)))
    if "cylinder" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(-1.0, 1.0, 1.2), R=rot, scale=(1.0, 1.6, 1.0)); bodies.append((i, 3, (0.5, 1.6)))
    if "hollow_sphere" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(1.0, 1.3, -1.2), R=np.eye(3), scale=(1.4, 1.4, 1.4)); bodies.append((i, 4, (0.6,)))
    if "hollow_box" in shapes:
        i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(0.2, 1.1, -1.5), R=rot, scale=(1.2, 1.0, 1.0)); bodies.append((i, 5, (1.1, 0.9, 0.9)))
    m.use_distance_field_cd(tolerance)
    for i, shape, dims in bodies:
        m.set_rigid_body_mass(i, 0.0)
        m.add_rigid_collider(i, shape, dims, thickness=0.05, restitution=0.6, friction=0.1 if shape else 0.2)
    m.add_model_collider(0, 0, restitution=0.5, friction=0.1)
    m.set_contact_params(stiffness=100.0, max_iter_v=5)
    return bodies


def bar_on_colliders(m, tolerance=0.05, sub_steps=2, max_iter=3):
    """Reference builds only.  A small FEM tet bar (no pinned particles) dropped onto a static sphere and a static cylinder above a floor box:
    the tet-model branch of the contact path (DistanceFieldCollisionDetection.cpp:139-152), two substeps per step."""
    m.add_regular_tet_model(9, 4, 4, t=(0.0, 2.0, 0.0), R=np.eye(3), scale=(3.0, 0.6, 0.6))
    m.add_solid_constraints(0, 2, k=1.0e5, nu=0.3)
    m.set_params(dt=0.005, sub_steps=sub_steps, max_iter=max_iter)
    rot = np.array([[0.9553365, -0.2955202, 0.0], [0.2955202, 0.9553365, 0.0], [0.0, 0.0, 1.0]])
    bodies = []
    i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(0.0, -0.5, 0.0), R=np.eye(3), scale=(20.0, 1.0, 20.0)); bodies.append((i, 0, (20.0, 1.0, 20.0)))
    i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(-0.7, 1.0, 0.0), R=np.eye(3), scale=(1.0, 1.0, 1.0)); bodies.append((i, 1, (0.5,)))
    i, _ = m.add_rigid_body_mesh(1.0, BOX_VERTS, BOX_FACES, x=(0.9, 0.9, 0.0), R=rot, scale=(0.8, 1.2, 0.8)); bodies.append((i, 3, (0.4, 1.2)))
    m.use_distance_field_cd(tolerance)
    for i, shape, dims in bodies:
        m.set_rigid_body_mass(i, 0.0)
        m.add_rigid_collider(i, shape, dims, restitution=0.6, friction=0.2)
    m.add_model_collider(1, 0, restitution=0.4, friction=0.3)
    m.set_contact_params(stiffness=100.0, max_iter_v=5)
    return bodies


CONTACT_SCENES = {
    # name: (precision of the reference build, builder on a reference build); the reference's setup of each is recorded under
    # contacts/<name>/ in tests/golden/reference_runs.npz
    "cloth_all_shapes": ("f64", lambda m: cloth_on_colliders(m, 24, shapes=("box", "sphere", "torus", "cylinder", "hollow_sphere", "hollow_box"))),
    "cloth_no_torus_f32": ("f32", lambda m: cloth_on_colliders(m, 24, shapes=("box", "sphere", "cylinder", "hollow_sphere", "hollow_box"))),
    "cloth_box_sphere_torus": ("f64", lambda m: cloth_on_colliders(m, 24, shapes=("box", "sphere", "torus"))),
    "bar": ("f64", bar_on_colliders),
}


def on_recorded_colliders(m, name):
    """The C restatement (m = CpuPbd "oracle") set up as CONTACT_SCENES[name] sets up a reference build: the same particle model and
    constraints, and the reference's rigid bodies and collision objects as recorded.  Returns (models, rigid) in the form of
    CpuPbd.collision_objects(), what an adapter passes to pbd_set_colliders."""
    import reference_golden
    p = "contacts/%s/" % name
    if name == "bar":
        m.add_regular_tet_model(9, 4, 4, t=(0.0, 2.0, 0.0), R=np.eye(3), scale=(3.0, 0.6, 0.6))
        m.add_solid_constraints(0, 2, k=1.0e5, nu=0.3)
        m.set_params(dt=0.005, sub_steps=2, max_iter=3)
    else:
        m.add_regular_triangle_model(24, 24, t=(-2.5, 2.2, -2.5), R=RX90, scale=(5.0, 5.0))
        m.add_cloth_constraints(0, 4, dist_k=1.0e5)
        m.add_bending_constraints(0, 3, 100.0)
        m.set_params(dt=0.005, sub_steps=1, max_iter=4)
    for row in reference_golden.get(p + "rigid_bodies"):
        m.add_rigid_body(0.0, row[:3], (1.0, 1.0, 1.0), row[3:7])
    models = [(int(o), int(c), float(r), float(f)) for o, c, r, f in reference_golden.get(p + "models")]
    rigid = list(reference_golden.get(p + "rigid"))
    m.set_colliders(models, rigid)
    m.set_oracle_contact_params(tolerance=0.05, stiffness=100.0, max_iter_v=5)
    return models, rigid
