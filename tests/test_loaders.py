"""Mesh import with the reference's names (SURVEY.md section 8 row f-4, import part): Utilities::TetGenLoader / OBJLoader semantics
(Utils/TetGenLoader.cpp, Utils/OBJLoader.h) on small committed files, and on the reference's own data/models/armadillo_4k mesh,
whose tet model is then built by the host mirror and held against the reference's."""
import os
import numpy as np

import positionbaseddynamics_b200.pypbd as pbd

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "meshes")
X = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1]], dtype=np.float32)
T = np.array([0, 1, 2, 3, 1, 2, 3, 4], dtype=np.uint32)


def test_tet_formats():
    for x, t in (pbd.TetGenLoader.loadTetgenModel(os.path.join(HERE, "tiny.node"), os.path.join(HERE, "tiny.ele")),
                 pbd.TetGenLoader.loadTetFile(os.path.join(HERE, "tiny.tet")),
                 pbd.TetGenLoader.loadMSHModel(os.path.join(HERE, "tiny.msh"))):   # 1-based in the file, 0-based in memory
        assert x.dtype == np.float32 and t.dtype == np.uint32
        assert (x == X).all() and (t == T).all()


def test_obj_loader():
    x, normals, tex, faces = pbd.OBJLoader.loadObj(os.path.join(HERE, "tiny.obj"), (2.0, 1.0, 3.0))
    assert (x == np.array([[0, 0, 0], [2, 0, 0], [2, 1, 0], [0, 1, 0]], dtype=np.float32)).all()   # per-axis scale on the positions
    assert normals.shape == (1, 3) and tex.shape == (4, 2) and len(faces) == 2
    assert faces[1].posIndices == [0, 2, 3] and faces[1].texIndices == [0, 2, 3] and faces[1].normalIndices == [0, 0, 0]
    vd, mesh = pbd.OBJLoader.loadObjToMesh(os.path.join(HERE, "tiny.obj"), (1.0, 1.0, 1.0))
    assert vd.size() == 4 and mesh.numFaces() == 2 and (mesh.getFaces() == [0, 1, 2, 0, 2, 3]).all()
    # the loaded mesh goes straight into the model (pyPBD/examples/bunny_cloth.py style)
    pbd.Simulation._current = None
    sim = pbd.Simulation.getCurrent(); sim.initDefault(); model = sim.getModel()
    tm = model.addTriangleModel(vd.getVertices(), mesh.getFaces())
    assert tm.getParticleMesh().numFaces() == 2 and tm.getParticleMesh().numEdges() == 5


def test_armadillo_tet_model_like_the_reference(tmp_path, cpu_libs):
    """The reference's armadillo_4k mesh (as its TetGen loader reads it, tests/golden/reference_runs.npz) written back in TetGen format,
    loaded, and built into a tet model by the host mirror and the C restatement: the same colouring and edges as the reference's model."""
    import reference_golden as rg
    x_ref, t_ref = rg.get("armadillo/x"), rg.get("armadillo/tets")
    node, ele = str(tmp_path / "armadillo_4k.node"), str(tmp_path / "armadillo_4k.ele")
    with open(node, "w") as f:
        f.write("%d  3  0  0\n" % len(x_ref) + "".join("%4d    %r  %r  %r\n" % ((i,) + tuple(map(float, p))) for i, p in enumerate(x_ref)))
    with open(ele, "w") as f:
        f.write("%d  4  0\n" % len(t_ref) + "".join("%5d     %d  %d  %d  %d\n" % ((i,) + tuple(map(int, q))) for i, q in enumerate(t_ref)))
    x, t = pbd.TetGenLoader.loadTetgenModel(node, ele)
    assert x.shape == (1180, 3) and len(t) == 4 * 3717
    assert (x == x_ref).all() and (t.reshape(-1, 4) == t_ref).all()
    from positionbaseddynamics_b200.model import HostModel
    hm = HostModel(); other = cpu_libs.CpuPbd("oracle", "f64")
    for m in (hm, other):
        m.add_tet_model(x, t.reshape(-1, 4))
        m.add_solid_constraints(0, 2, k=1.0e6, nu=0.3)
    hm.init_groups(); other.init_groups()
    assert hm.num_constraints() == other.num_constraints() == 3717
    types, bodies, _, _ = hm.constraints()
    rg.assert_structure("armadillo/", types, bodies, *hm.groups())     # the reference's colouring of the imported mesh
    off_b, ids_b = other.groups()
    off_a, ids_a = hm.groups()
    assert (off_a == off_b).all() and (ids_a == ids_b).all()
    assert (rg.digest(hm.tet_edges(0), np.uint32) == rg.get("armadillo/tet_edges")).all()
    assert (hm.tet_edges(0) == other.tet_edges(0)).all()
    hm.close()
