"""CPU-side guard of the contact kernel's arithmetic: csrc/contacts.cuh compiled for the host through a test-only shim (tests/host_shim/),
one simulated thread per particle, in lockstep with the fp64 C restatement of the contact path, which tests/test_oracle_vs_ref.py pins to
the unmodified reference, set up with the reference's recorded colliders.  The GPU parity tests proper are in tests/test_gpu_contacts.py;
this one runs without a GPU and is not a product path."""
import ctypes as C
import os
import subprocess
import numpy as np

import scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _RC(C.Structure):  # pbdk::RigidCollider
    _fields_ = [("shape", C.c_int), ("body", C.c_uint), ("dim", C.c_float * 3), ("thickness", C.c_float), ("invert", C.c_float), ("restitution", C.c_float),
                ("friction", C.c_float), ("R", C.c_float * 9), ("v1", C.c_float * 3), ("v2", C.c_float * 3), ("aabbMin", C.c_float * 3), ("aabbMax", C.c_float * 3)]


def test_contact_kernel_arithmetic_on_the_host(tmp_path, cpu_libs):
    from positionbaseddynamics_b200 import _capi
    so = str(tmp_path / "libcontacts_host.so")
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "tests", "host_shim"), "-I" + os.path.join(ROOT, "positionbaseddynamics_b200", "csrc"),
                           "-o", so, os.path.join(ROOT, "tests", "host_shim", "run_contacts.cpp")])
    lib = C.CDLL(so)
    m = cpu_libs.CpuPbd("oracle", "f64")
    models, rigid = scenes.on_recorded_colliders(m, "cloth_all_shapes")
    mass, _ = m.masses(); n = len(mass); h = 0.005
    rb = m.rigid_bodies(); nrb = len(rb)
    rbX = np.zeros((nrb, 4), np.float32); rbX[:, :3] = rb[:, :3]
    rbV = np.zeros((nrb, 4), np.float32); rbW = np.zeros((nrb, 4), np.float32)
    rcs = (_RC * len(rigid))()
    for k, d in enumerate(rigid):
        rc = rcs[k]; rc.shape = int(d[0]); rc.body = int(d[1]); rc.dim[:] = [float(v) for v in d[2:5]]; rc.thickness = float(d[5]); rc.invert = -1.0 if d[6] else 1.0
        rc.restitution = float(d[7]); rc.friction = float(d[8]); rc.R[:] = [float(v) for v in d[9:18]]; rc.v1[:] = [float(v) for v in d[18:21]]
        rc.v2[:] = [float(v) for v in d[21:24]]; rc.aabbMin[:] = [float(v) for v in d[24:27]]; rc.aabbMax[:] = [float(v) for v in d[27:30]]
    pcs = (_capi.ParticleCollider * 1)(_capi.ParticleCollider(*models[0]))
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    events = 0; worst = 0.0; bodies = set()
    m.step(30)  # free fall until just before the first contacts
    for step in range(70):
        x_old = m.get("x").copy()
        m.step(1)
        x_new, v_new = m.get("x").copy(), m.get("v").copy()
        p, b, info = m.oracle_contacts()
        v_pre = (x_new - x_old) / h  # velocityUpdateFirstOrder: what the contact solve starts from
        pos = np.zeros((n, 4), np.float32); pos[:, :3] = x_new; pos[:, 3] = np.where(mass != 0, 1.0 / np.where(mass != 0, mass, 1.0), 0.0)
        vel = np.zeros((n, 4), np.float32); vel[:, :3] = v_pre; vel[:, 3] = mass
        rec = (_capi.Contact * 4096)(); cnt = C.c_uint(0)
        lib.run_contacts(n, vp(pos), vp(vel), vp(rbX), vp(rbV), vp(rbW), len(rigid), C.cast(rcs, C.c_void_p), 1, C.cast(pcs, C.c_void_p),
                         C.c_float(0.05), C.c_float(100.0), 5, C.cast(rec, C.c_void_p), C.byref(cnt), 4096)
        got = sorted((rec[i].particle, rec[i].body) for i in range(cnt.value))
        assert got == sorted(zip(p.tolist(), b.tolist())), "step %d: contact lists differ" % step
        worst = max(worst, float(np.abs(vel[:, :3] - v_new).max()))
        events += len(p); bodies |= set(b.tolist())
    print("host shim: %d contact events on bodies %s, worst |dv| %.2e m/s" % (events, sorted(bodies), worst))
    assert events > 1500 and len(bodies) >= 4 and worst <= 2.0e-3
