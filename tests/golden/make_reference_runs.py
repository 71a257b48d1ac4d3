#!/usr/bin/env python
"""Record what the tests that compare with the UNMODIFIED reference take from it (oracle/_ref, built by oracle/Makefile from the
reference sources) into tests/golden/reference_runs.npz, read by tests/reference_golden.py.  Needs the reference's source tree
(for its data/models) and the reference build made from it:

    make -C oracle ref REF=<reference source dir>
    python tests/golden/make_reference_runs.py <reference source dir>

Every record is produced by the same scene builders and parameters as the test that reads it."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import pyoracle  # noqa: E402
import reference_golden as rg  # noqa: E402
from parity_util import perturb  # noqa: E402


def put_structure(out, prefix, m):
    types, bodies, _, _ = m.constraints()
    out[prefix + "structure"] = rg.structure_digest(types, bodies, *m.groups())


def put_rows(out, prefix, name, a, scale, k=rg.SAMPLE_ROWS):
    out[prefix + name] = np.asarray(a)[rg.sample_rows(len(a), k)]
    out[prefix + name + "_scale"] = np.float64(scale)


def oracle_vs_ref(out):
    """tests/test_oracle_vs_ref.py::test_structure_and_trajectory"""
    import test_oracle_vs_ref as t
    for name in sorted(t.CASES):
        for prec in ("f64", "f32"):
            p = "oracle_vs_ref/%s/%s/" % (name, prec)
            r = pyoracle.CpuPbd("ref", prec)
            t.CASES[name](r)
            put_structure(out, p, r)
            _, _, params, _ = r.constraints()
            put_rows(out, p, "params", params, max(np.abs(params).max(), 1.0), rg.PARAM_ROWS)
            perturb([r], 0.01)
            r.step(t.steps_of(name))
            x = r.get("x")
            put_rows(out, p, "x", x, np.abs(x).max())


def gpu_scenes(out):
    """tests/test_gpu_parity.py::test_scene_vs_reference_f64"""
    import test_gpu_parity as t
    for name in sorted(t.SCENES):
        build, amp, steps = t.SCENES[name]
        p = "gpu_parity/%s/" % name
        r = pyoracle.CpuPbd("ref", "f64")
        build(r)
        put_structure(out, p, r)
        x_start = perturb([r], amp)
        r.step(steps)
        x = r.get("x")
        put_rows(out, p, "x", x, np.abs(x).max())
        out[p + "disp_scale"] = np.float64(np.abs(x - x_start).max())


def facade_rigid_body(out):
    """tests/test_pypbd_facade.py::test_facade_rigid_body_matches_the_reference_init"""
    import test_pypbd_facade as t
    for k, scale in enumerate(t.RB_SCALES):
        r = pyoracle.CpuPbd("ref", "f64")
        _, props = r.add_rigid_body_mesh(2.0, t.RB_VERTS, t.CUBE_F, x=(1.0, 2.0, 3.0), R=t.RB_R0, scale=scale)
        out["facade_rigid_body/%d/props" % k] = props


def coupling_example(out):
    """tests/test_pypbd_facade.py::test_coupling_example_against_the_reference"""
    import test_pypbd_facade as t
    import positionbaseddynamics_b200.pypbd as pbd

    class NoDevice:  # the example sets its substep count on the GPU time step; the reference side gets it from coupling_example_on_cpu
        def setValueUInt(self, *_):
            pass
    pbd.Simulation.getTimeStep = lambda self: NoDevice()
    ex, model = t.coupling_example_model()
    ref = pyoracle.CpuPbd("ref", "f64")
    t.coupling_example_on_cpu(ref, ex, model._host)
    out["coupling_example/num_constraints"] = np.int64(ref.num_constraints())
    ref.step(6)
    x = ref.get("x")
    put_rows(out, "coupling_example/", "x", x, np.abs(x).max())
    out["coupling_example/rb_x"] = ref.rigid_bodies()[:, :3]


def armadillo(out, src):
    """tests/test_loaders.py::test_armadillo_tet_model_like_the_reference: the reference's data/models/armadillo_4k.{node,ele}, as
    loaded, and the tet model the reference builds from them."""
    import positionbaseddynamics_b200.pypbd as pbd
    x, t = pbd.TetGenLoader.loadTetgenModel(os.path.join(src, "armadillo_4k.node"), os.path.join(src, "armadillo_4k.ele"))
    out["armadillo/x"] = x; out["armadillo/tets"] = t.reshape(-1, 4).astype(np.uint16)
    r = pyoracle.CpuPbd("ref", "f64")
    r.add_tet_model(x, t.reshape(-1, 4))
    r.add_solid_constraints(0, 2, k=1.0e6, nu=0.3)
    r.init_groups()
    put_structure(out, "armadillo/", r)
    out["armadillo/tet_edges"] = rg.digest(r.tet_edges(0), np.uint32)


def contact_scenes(out):
    """tests/scenes.py:on_recorded_colliders: the reference's rigid bodies and collision objects of every contact scene.  The GPU contact
    tests cover particle / rigid-body contacts only: none of the scenes may produce another kind within the tests' horizons."""
    import scenes
    for name, (prec, build) in scenes.CONTACT_SCENES.items():
        p = "contacts/%s/" % name
        r = pyoracle.CpuPbd("ref", prec)
        build(r)
        models, rigid = r.collision_objects()
        out[p + "rigid_bodies"] = r.rigid_bodies(); out[p + "models"] = np.array(models, np.float64); out[p + "rigid"] = np.array(rigid)
        for _ in range(200):
            r.step(1)
            assert r.contacts()[3:] == (0, 0), name


def contact_runs(out):
    """tests/test_oracle_vs_ref.py::test_contact_path_restatement_is_pinned_to_the_reference: the reference's free run of the scene, its
    contact list after every step, its velocities after the checkpoint steps and, in fp32, its state around the lockstep steps."""
    import scenes
    import test_oracle_vs_ref as t
    for prec, name in (("f64", "cloth_all_shapes"), ("f32", "cloth_no_torus_f32")):
        p = "contact_run/%s/" % prec
        r = pyoracle.CpuPbd("ref", prec)
        scenes.CONTACT_SCENES[name][1](r)
        counts, pairs = [], []
        for step in range(1, t.CONTACT_STEPS + 1):
            if prec == "f32" and step in t.LOCKSTEP_STEPS:
                out[p + "x_before%d" % step] = r.get("x").astype(np.float32); out[p + "v_before%d" % step] = r.get("v").astype(np.float32)
            r.step(1)
            pp, bb, _, _, _ = r.contacts()
            counts.append(len(pp)); pairs += list(zip(pp.tolist(), bb.tolist()))
            if (prec == "f64" and step in t.CHECKPOINTS) or (prec == "f32" and step in t.LOCKSTEP_STEPS):
                v = r.get("v")
                put_rows(out, p, "v%d" % step, v, np.abs(v).max())
        out[p + "counts"] = np.array(counts, np.uint16); out[p + "pairs"] = np.array(pairs, np.uint16)


def main():
    if not (pyoracle.available("ref", "f32") and pyoracle.available("ref", "f64")):
        raise SystemExit("oracle/_ref has no reference build: make -C oracle ref REF=<reference source dir>")
    ref_models = os.path.join(sys.argv[1], "data", "models")
    out = {}
    oracle_vs_ref(out); gpu_scenes(out); facade_rigid_body(out); coupling_example(out); armadillo(out, ref_models)
    contact_scenes(out); contact_runs(out)
    np.savez_compressed(rg.PATH, **out)
    print(rg.PATH, os.path.getsize(rg.PATH), "bytes")


if __name__ == "__main__":
    main()
