#!/usr/bin/env python
"""bench.py -- constraint-projections/sec of the PBD/XPBD hot path (BASELINE.json metric) on N B200s.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W   (the reference's own CPU implementation, all host threads)

Workload (config.workload = "cfg2"): cloth sheet 1000x1000 particles, Distance_XPBD (k=1e5) + IsometricBending_XPBD
(k=100), 1 substep x 20 iterations, h = 0.005 -- BASELINE.json configs[1], the configuration the metric is quoted on.
A "step" is one TimeStepController::step over that scene; value = projections executed by all ranks / device time
(CUDA events on the engine's stream, max over ranks), state resident in HBM.  e2e = the same metric through the C ABI's
host-buffer calls: pinned host x,v in -> step -> host x out, EVERY step, wall clock incl. the copies; the headline uses the
pipelined call (pbd_step_host_async, copies of neighbouring steps overlap the kernels), e2e.blocking the blocking one.
Multi-GPU = independent scene replicas, one per rank (SURVEY.md section 8e, "replicas only"): weak scaling, no
data-path collective; torch.distributed (NCCL) only gathers the per-rank timings.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "constraint_projections_per_sec"
UNIT = "projections/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", type=int, default=1000, help="cloth is size x size particles (cfg2 = 1000)")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--mode", default="auto", choices=["auto", "graph", "resident", "launch", "jacobi"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 is the BASELINE.json metric configuration (default); cfg1/cfg3 are side measurements for DESIGN.md")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the side measurements of cfg1/cfg3/cfg4/cfg5 (default workload only)")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the state they computed (x, v and, if any, the rigid bodies) as DIR/<name>.npy")
    return ap.parse_args()


WORKLOAD = "cfg2"


def build_scene(m, size, iters):
    """Build the selected workload on any object with the common builder surface; returns (sub_steps, iterations)."""
    import scenes
    if WORKLOAD == "cfg1":
        scenes.cfg1(m, 50); return 1, 5
    if WORKLOAD == "cfg3":
        scenes.cfg3(m); return 10, 5
    if WORKLOAD == "cfg4":
        scenes.cfg4(m); return 5, 1
    if WORKLOAD == "cfg5":
        scenes.cfg2(m, 500, iters); return 1, iters  # one 500x500 cloth per GPU (run with --gpus 8)
    scenes.cfg2(m, size, iters); return 1, iters


def workload_config(size, iters, n_gpus):
    if WORKLOAD == "cfg1":
        return {"workload": "cfg1", "scene": "ClothDemo 50x50, Distance + IsometricBending (PBD)", "sub_steps": 1, "iterations": 5, "dt": 0.005,
                "replicas": n_gpus, "parallelism": "replica x%d" % n_gpus, "l2": "L2-resident working set; L2 flushed between timed steps: no (latency-bound config)"}
    if WORKLOAD == "cfg3":
        return {"workload": "cfg3", "scene": "tet bar 101x21x21 = 200,000 tets, FEMTet(E=1e6, nu=0.3) + Volume per tet", "sub_steps": 10, "iterations": 5,
                "dt": 0.005, "replicas": n_gpus, "parallelism": "replica x%d" % n_gpus, "l2": "L2-resident working set (~16 MB); latency-bound config"}
    if WORKLOAD == "cfg4":
        return {"workload": "cfg4", "scene": "224x224 cloth (FEMTriangle + IsometricBending) + 51x21x11 tet block (FEMTet) + 12 rigid bodies / 8 BallJoints / "
                                             "4 RigidBodyParticleBallJoints", "sub_steps": 5, "iterations": 1, "dt": 0.005, "replicas": n_gpus,
                "parallelism": "replica x%d" % n_gpus, "l2": "L2-resident working set; latency-bound config"}
    if WORKLOAD == "cfg5":
        return {"workload": "cfg5", "scene": "one 500x500 cloth per GPU, Distance_XPBD + IsometricBending_XPBD", "sub_steps": 1, "iterations": iters, "dt": 0.005,
                "replicas": n_gpus, "parallelism": "replica x%d" % n_gpus, "l2": "per-sweep constraint stream 48 MB: L2-resident"}
    return {"workload": "cfg2", "scene": "cloth %dx%d particles, Distance_XPBD(k=1e5)+IsometricBending_XPBD(k=100)" % (size, size),
            "sub_steps": 1, "iterations": iters, "dt": 0.005, "replicas": n_gpus, "parallelism": "replica x%d" % n_gpus,
            "l2": "inputs larger than L2: the per-sweep constraint stream (~192 MB at 1000x1000) exceeds the 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref when it was built, else the C restatement)
# ---------------------------------------------------------------------------------------------------------------
def cpu_arm(size, iters, steps, warmup):
    import scenes
    from oracle import pyoracle
    if pyoracle.available("ref", "f32"):
        path, march = pyoracle.best_ref_variant()
        kind, lib = "reference", pyoracle.CpuPbd("ref", "f32", path=path)
    else:
        if not pyoracle.available("oracle", "f32"):
            pyoracle.build(ref=False)
        kind, lib, march = "port", pyoracle.CpuPbd("oracle", "f32"), "-march=x86-64-v3"
    sub_steps, iters = build_scene(lib, size, iters)
    ncons = lib.num_constraints()
    lib.init_groups()
    # "all the host threads it can use": the reference forks/joins an OpenMP team per colour group, which stops scaling
    # long before 128 hardware threads; probe a few team sizes on one step each and keep the fastest for the timed run.
    ncpu = os.cpu_count() or 1
    cand = sorted({c for c in (8, 16, 32, 64, ncpu) if c <= ncpu})
    best, cores = None, ncpu
    lib.set_threads(1)
    t1 = lib.step(1)  # single-thread figure, reported next to the OpenMP one
    for c in cand:
        lib.set_threads(c)
        t = lib.step(1)
        if best is None or t < best:
            best, cores = t, c
    lib.set_threads(cores)
    if warmup > 1:
        lib.step(warmup - 1)
    secs = lib.step(steps)
    proj = ncons * sub_steps * iters * steps
    return {"value": proj / secs, "unit": UNIT, "cores": cores, "kind": kind, "ms_per_step": 1e3 * secs / steps,
            "sample": "%d step(s) of workload %s (%d constraints x %d substeps x %d iterations) after warm-up, fp32 build g++ -O3 %s -fopenmp, OMP threads=%d "
                      "(fastest of %s on %d hardware threads); 1 thread: %.3e projections/s"
                      % (steps, WORKLOAD, ncons, sub_steps, iters, march, cores, cand, ncpu, ncons * sub_steps * iters / t1)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs and prints the reference arm
    size = args.size
    # bound the run to a few minutes: a 1000x1000 step costs ~2.5 s on 8 cores; shrink the sample for long runs
    budget_steps = args.steps + args.warmup
    if budget_steps > 40:
        size = max(200, int(args.size * (40.0 / budget_steps) ** 0.5))
    r = cpu_arm(size, args.iters, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(size, args.iters, args.gpus),
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index; self.p = None

    def start(self):
        # NVML in a thread (a sample every ~2 ms: the timed region of the default run is only tens of milliseconds long);
        # nvidia-smi -lms as the fallback when NVML cannot be used
        self.samples = []; self.thread = None; self.stop_flag = False
        try:
            import pynvml, threading
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self.stop_flag:
                    try:
                        self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx, int(get_reasons(h))))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.thread = threading.Thread(target=loop, daemon=True); self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        try:
            return self._stop()
        except Exception as ex:  # never let the clock report break the measurement
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling failed: %s" % ex]}

    def _stop(self):
        if getattr(self, "thread", None) is not None:
            self.stop_flag = True; self.thread.join(timeout=2)
            sm = sorted(c for c, _, _ in self.samples)
            bits = 0
            for _, _, r in self.samples:
                bits |= r
            names = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))  # nvml.h nvmlClocksEventReason*
            return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": float(self.samples[0][1]) if self.samples else None,
                    "samples": len(sm), "reasons": sorted(n for n, b in names if bits & b), "source": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); out = ""
        sm, mx, reasons = [], [], set()
        for ln in out.strip().splitlines():
            f = [c.strip() for c in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


PER_PROJ_NAMES = {"Distance": 76.0, "Distance_XPBD": 84.0, "Dihedral": 148.0, "IsometricBending": 160.0, "IsometricBending_XPBD": 168.0, "FEMTriangle": 128.0,
                  "StrainTriangle": 124.0, "Volume": 148.0, "Volume_XPBD": 156.0, "FEMTet": 184.0, "FEMTet_XPBD": 192.0, "StrainTet": 180.0, "ShapeMatching": 240.0}


def make_engine(local, size, iters):
    """Scene (host model mirror, C++) -> engine through the C ABI.  Returns (engine, info)."""
    import scenes as _sc
    from positionbaseddynamics_b200 import _capi
    from positionbaseddynamics_b200.model import HostModel
    t0 = time.time()
    hm = HostModel()
    sub_steps, iters = build_scene(hm, size, iters)
    types, bodies, params, _ = hm.constraints()
    off, ids = hm.groups()
    n = hm.num_particles(); ncons = len(types)
    x0 = hm.get("x0"); mass, _ = hm.masses()
    build_s = time.time() - t0
    eng = _capi.Engine(local)
    eng.set_particles(x0, mass)
    rb = hm.rigid_bodies()
    if len(rb):  # cfg4: the coupling rig (tests/scenes.py:coupling_rig)
        eng.set_rigid_bodies([0.0 if i % 3 == 0 else 1.0 for i in range(len(rb))], rb[:, :3], rb[:, 3:7],
                             [_sc.box_inertia(1.0, 0.5, 0.5, 0.5) if i % 3 == 0 else _sc.box_inertia(1.0, 0.4, 2.0, 0.4) for i in range(len(rb))])
    eng.add_flat(types, bodies, params)
    eng.set_groups(off, ids)
    eng.set_params(dt=0.005, sub_steps=sub_steps, max_iter=iters)
    hm.close()
    return eng, {"n": n, "ncons": ncons, "sub_steps": sub_steps, "iters": iters, "build_s": build_s, "proj_per_step": ncons * sub_steps * iters}


def timed_steps(eng, mode, steps, warmup, dist):
    """W untimed steps, then K steps between barrier + synchronize; device time from CUDA events on the engine's stream."""
    import torch
    eng.set_mode(mode)
    eng.step(warmup); eng.sync()
    l0 = eng.stats().kernel_launches
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    eng.step(steps); eng.sync()
    torch.cuda.synchronize()
    st = eng.stats()
    return st.last_step_ms, st.kernel_launches - l0


def pick_mode(eng, mode_arg, dist):
    """The execution mode: forced, or the faster of graph / resident on a short probe (both produce the same bits)."""
    from positionbaseddynamics_b200 import _capi
    modes = {"graph": _capi.MODE_GRAPH, "resident": _capi.MODE_RESIDENT, "launch": _capi.MODE_LAUNCH, "jacobi": _capi.MODE_JACOBI}
    if mode_arg != "auto":
        return mode_arg, modes[mode_arg], {}
    probe = {}
    for name in ("graph", "resident"):
        try:
            ms, _ = timed_steps(eng, modes[name], 3, 2, dist)
            probe[name] = ms / 3
        except Exception as ex:  # e.g. the scene does not fit the resident mode
            probe[name] = float("inf"); sys.stderr.write("mode %s not available: %s\n" % (name, ex))
    name = min(probe, key=probe.get)
    return name, modes[name], probe


def position_checksum(eng):
    """Checksum of the particle positions: CRC32 of the fp32 bytes + their float64 sum.  Execution is deterministic (no atomics on
    the data path, both modes bit-identical), so every replica and every run with the same K/W must print the same value."""
    import zlib
    import numpy as np
    from positionbaseddynamics_b200 import _capi
    x = np.ascontiguousarray(eng.get_attr(_capi.ATTR_X))
    return int(zlib.crc32(x.tobytes())), float(x.astype(np.float64).sum())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(eng, out_dir):
    """What a caller of the timed path receives after its last step: particle positions and velocities (and the rigid-body
    state of workloads that have rigid bodies), fp32.  Above DUMP_LIMIT_BYTES in all, the same seeded sample of particle rows
    is written for every array, so that two builds run with the same arguments can be compared file for file."""
    import numpy as np
    from positionbaseddynamics_b200 import _capi
    out = {"x": eng.get_attr(_capi.ATTR_X), "v": eng.get_attr(_capi.ATTR_V)}
    n = len(out["x"])
    per_row = sum(a[0].nbytes for a in out.values())
    if n * per_row > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // 2 // per_row, replace=False))
        out = {k: a[rows] for k, a in out.items()}
    if getattr(eng, "n_rb", 0):
        out["rigid_bodies"] = eng.get_rigid_bodies()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def l2_copy_bandwidth():
    """Measured L2-resident copy bandwidth (read + write bytes of a 2 x 24 MB working set that stays in the 126 MB L2), GB/s."""
    import torch
    a = torch.empty(6 * 1024 * 1024, dtype=torch.float32, device="cuda").normal_(); b = torch.empty_like(a)
    for _ in range(5):
        b.copy_(a)
    best = 0.0
    for _ in range(5):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            b.copy_(a)
        e1.record(); torch.cuda.synchronize()
        best = max(best, 10 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def run_b200(args):
    global WORKLOAD
    import numpy as np
    import torch
    from positionbaseddynamics_b200 import _capi

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != max(args.gpus, 1) and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    eng, info = make_engine(local, args.size, args.iters)
    args.iters = info["iters"]
    n, ncons, sub_steps, proj_per_step = info["n"], info["ncons"], info["sub_steps"], info["proj_per_step"]
    mode_name, mode, probe = pick_mode(eng, args.mode, dist)

    # ---- timed region: K steps, state resident in HBM ---------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed_steps(eng, mode, args.steps, max(args.warmup, 3), dist)
    clocks = sampler.stop() if rank == 0 else None
    crc, xsum = position_checksum(eng)
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    ms_t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    crc_t = torch.tensor([crc], device="cuda", dtype=torch.int64)
    if dist is not None:
        gathered = [torch.zeros_like(ms_t) for _ in range(world)]
        dist.all_gather(gathered, ms_t)
        ms_max = max(float(g.item()) for g in gathered)
        gc = [torch.zeros_like(crc_t) for _ in range(world)]
        dist.all_gather(gc, crc_t)
        crcs = [int(g.item()) for g in gc]
    else:
        ms_max = ms; crcs = [crc]
    value = world * proj_per_step * args.steps / (ms_max * 1e-3)

    # ---- e2e: pinned host buffers in and out every step ---------------------------------------------------------------
    xh = torch.empty((n, 3), dtype=torch.float32, pin_memory=True); vh = torch.empty((n, 3), dtype=torch.float32, pin_memory=True)
    xo = torch.empty((n, 3), dtype=torch.float32, pin_memory=True)
    xh.numpy()[:] = eng.get_attr(_capi.ATTR_X); vh.numpy()[:] = eng.get_attr(_capi.ATTR_V)
    e2e_steps = args.steps
    for _ in range(2):
        eng.step_host(1, xh.numpy(), vh.numpy(), xo.numpy())
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.step_host(1, xh.numpy(), vh.numpy(), xo.numpy())  # synchronises: result is in host memory on return
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if dist is not None:
        gathered = [torch.zeros_like(e2e_t) for _ in range(world)]
        dist.all_gather(gathered, e2e_t)
        e2e_max = max(float(g.item()) for g in gathered)
    else:
        e2e_max = e2e_s
    e2e_value = world * proj_per_step * e2e_steps / e2e_max
    x_blocking = xo.numpy().copy()
    # the same call with the device state authoritative (x_in = v_in = NULL: the host did not edit the state between steps, only the
    # result is downloaded) -- what integration/GpuTimeStepController.h does after setHostStateAuthoritative(false); reported beside e2e
    for _ in range(2):
        eng.step_host(1, None, None, xo.numpy())
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.step_host(1, None, None, xo.numpy())
    torch.cuda.synchronize()
    e2e_dev_s = time.perf_counter() - t0
    # pipelined form of the same call (pbd_step_host_async / pbd_step_host_wait): every step still uploads its x and v from pinned
    # host memory and downloads its result, but the copies of neighbouring steps overlap the projection kernels.  One call in flight
    # behind the host (lag 1); the region ends when the last result is in host memory.
    xin = [xh, xh.clone().pin_memory()]; vin = [vh, vh.clone().pin_memory()]
    xout = [xo, torch.empty((n, 3), dtype=torch.float32, pin_memory=True)]
    for k in range(3):
        eng.step_host_async(1, xin[k & 1].numpy(), vin[k & 1].numpy(), xout[k & 1].numpy())
    eng.step_host_wait(0)
    pipelined_equal = bool((xout[0].numpy() == x_blocking).all() and (xout[1].numpy() == x_blocking).all())
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        eng.step_host_async(1, xin[k & 1].numpy(), vin[k & 1].numpy(), xout[k & 1].numpy())
        eng.step_host_wait(1)
    eng.step_host_wait(0)
    torch.cuda.synchronize()
    e2e_pipe_s = time.perf_counter() - t0
    e2e_pt = torch.tensor([e2e_pipe_s], device="cuda", dtype=torch.float64)
    if dist is not None:
        gathered = [torch.zeros_like(e2e_pt) for _ in range(world)]
        dist.all_gather(gathered, e2e_pt)
        e2e_pipe_max = max(float(g.item()) for g in gathered)
    else:
        e2e_pipe_max = e2e_pipe_s
    e2e_pipe_value = world * proj_per_step * e2e_steps / e2e_pipe_max

    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- roofline (rank 0) -------------------------------------------------------------------------------------------------
    # Leading figure: the whole step, timed directly (CUDA events around the K steps): algorithmic bytes of a step / time per step.
    # Resident mode: the step IS the dominant kernel (one k_step_resident launch), so `achieved` is that same direct measurement.
    # Graph mode: the dominant bucket kernel's launches overlap (PDL), an isolated duration does not exist inside the pipeline; its
    # `achieved` is reported from serialized event timing (pbd_profile_step, PDL off) and marked as such.
    peak, peak_src = measured_peak()
    st = eng.stats()
    ms_step = ms_max / args.steps
    step_achieved = st.bytes_per_step / (ms_step * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    tdb = {}
    if os.path.exists(tpath):
        try:
            tdb = json.load(open(tpath)).get(WORKLOAD, {})
        except Exception:
            tdb = {}
    if mode_name == "jacobi":
        roof = {"kernel": "Jacobi comparison path (k_project_jacobi per type + k_jacobi_apply; not the reference's algorithm)", "bytes_per_launch": st.bytes_per_step,
                "ms_per_launch": ms_step, "launches_per_step": float(launches) / args.steps, "timing": "direct (whole step)"}
        achieved = step_achieved
    elif mode_name == "resident":
        roof = {"kernel": "k_step_resident (one launch = one step; CUDA events around the launches)", "bytes_per_launch": st.bytes_per_step,
                "ms_per_launch": ms_step, "launches_per_step": 1, "timing": "direct"}
        t = tdb.get("k_step_resident")
        if isinstance(t, dict):
            traffic = float(t["dram_bytes"])
            roof["l2_sector_bytes_per_launch"] = t.get("l2_sector_bytes")
            roof["executed_warp_instructions_per_launch"] = t.get("warp_instructions")
        achieved = step_achieved
    else:
        eng.set_mode(_capi.MODE_LAUNCH)
        eng.step(2); eng.sync()
        tms = np.zeros(_capi.NUM_TYPES); tl = np.zeros(_capi.NUM_TYPES); tmi = tmv = 0.0
        reps = 3
        for _ in range(reps):
            ms_t_, mi, mv, l_ = eng.profile_step()
            tms += ms_t_; tl += l_; tmi += mi; tmv += mv
        dom = int(np.argmax(tms))
        launches_per_step = tl[dom] / reps
        bytes_per_launch = float(st.constraints_per_type[dom] * PER_PROJ_NAMES.get(_capi.TYPE_NAMES[dom], 0.0) * args.iters * sub_steps / max(launches_per_step, 1))
        ser_ms = float(tms[dom] / max(tl[dom], 1))
        roof = {"kernel": "k_project<%s>" % _capi.TYPE_NAMES[dom], "bytes_per_launch": bytes_per_launch, "ms_per_launch": ser_ms,
                "launches_per_step": launches_per_step, "timing": "serialized launches (PDL off), CUDA events between consecutive launches",
                "share_of_serialized_step": float(tms[dom] / max(tms.sum() + tmi + tmv, 1e-9))}
        achieved = bytes_per_launch / (ser_ms * 1e-3) / 1e9
        t = tdb.get(roof["kernel"])
        if isinstance(t, dict):
            traffic = t["dram_bytes"] / t["constraints_in_launch"] * st.constraints_per_type[dom] * args.iters * sub_steps / max(launches_per_step, 1)
        eng.set_mode(mode)
    try:
        l2_gbs = l2_copy_bandwidth()
    except Exception:
        l2_gbs = None
    stream_bytes = None
    try:  # what has to come from DRAM every sweep: indices + per-constraint constants + multipliers (positions stay on chip)
        per = {"Distance": 12, "Distance_XPBD": 20, "Dihedral": 20, "IsometricBending": 32, "IsometricBending_XPBD": 40, "FEMTriangle": 32, "StrainTriangle": 28,
               "Volume": 20, "Volume_XPBD": 28, "FEMTet": 56, "FEMTet_XPBD": 64, "StrainTet": 52, "ShapeMatching": 112}
        stream_bytes = float(sum(st.constraints_per_type[t] * per.get(_capi.TYPE_NAMES[t], 0) for t in range(_capi.NUM_TYPES)) * args.iters * sub_steps)
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "step_bytes": st.bytes_per_step, "step_achieved": step_achieved, "step_frac": step_achieved / peak, **roof,
                "dram_stream_bytes_per_step": stream_bytes, "l2_copy_gbs_measured": l2_gbs,
                "note": "algorithmic bytes (DESIGN.md section 3) against the measured HBM copy bandwidth, as the contract defines it.  Most of those bytes are "
                        "particle float4s that never reach DRAM: resident mode keeps them in shared memory (DRAM carries the constraint stream only, `traffic`), "
                        "graph mode serves them from L2 (sector-throughput bound, profiles/README.md).  The fraction is therefore a distance to the "
                        "algorithmic-bytes roofline, not a DRAM utilisation."}

    # ---- side measurements: the latency-bound configs, so that the driver's record carries them too ---------------------------
    side = None
    if world == 1 and WORKLOAD == "cfg2" and not args.no_side:
        side = {}
        main = WORKLOAD
        eng.close()
        for w in ("cfg1", "cfg3", "cfg4", "cfg5"):
            try:
                WORKLOAD = w
                e2, inf = make_engine(local, args.size, 20)
                mn, md, pr = pick_mode(e2, args.mode if args.mode != "launch" else "auto", None)
                k = 10
                ms2, _ = timed_steps(e2, md, k, 3, None)
                side[w] = {"ms_per_step": ms2 / k, "value": inf["proj_per_step"] * k / (ms2 * 1e-3), "unit": UNIT, "mode": mn, "mode_probe_ms": pr,
                           "constraints": inf["ncons"], "particles": inf["n"], "sub_steps": inf["sub_steps"], "iterations": inf["iters"],
                           "checksum": {"crc32": position_checksum(e2)[0]}}
                e2.close()
            except Exception as ex:
                side[w] = {"error": str(ex)}
        WORKLOAD = main
        # the contact path (SURVEY f-4, static analytic colliders): cfg2 with a floor box, a sphere poking through the sheet and a torus
        try:
            e3, inf = make_engine(local, args.size, args.iters)
            mn, md, pr = pick_mode(e3, args.mode if args.mode != "launch" else "auto", None)
            k = 10
            ms_plain, _ = timed_steps(e3, md, k, 3, None)
            xc = e3.get_attr(_capi.ATTR_X)
            cx, cy, cz = [float(v) for v in xc.mean(axis=0)]
            ident = [1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0]
            def collider(shape, body, dim, centre, half):
                rc = _capi.RigidCollider(); rc.shape = shape; rc.body = body; rc.dim[:] = list(dim) + [0.0] * (3 - len(dim)); rc.thickness = 0.0; rc.invert_sdf = 0
                rc.restitution = 0.6; rc.friction = 0.2; rc.R[:] = ident; rc.v1[:] = [0.0, 0.0, 0.0]; rc.v2[:] = list(centre)
                rc.aabb_min[:] = [c - h - 0.05 for c, h in zip(centre, half)]; rc.aabb_max[:] = [c + h + 0.05 for c, h in zip(centre, half)]
                return rc
            centres = [(cx, cy - 3.0, cz), (cx, cy - 1.7, cz), (cx + 3.0, cy - 0.3, cz + 2.0)]
            e3.set_rigid_bodies([0.0, 0.0, 0.0], centres, [(1.0, 0.0, 0.0, 0.0)] * 3, [(1.0, 1.0, 1.0)] * 3)
            e3.set_colliders([_capi.ParticleCollider(0, inf["n"], 0.5, 0.1)],
                             [collider(_capi.SHAPE_BOX, 0, (50.0, 0.5, 50.0), centres[0], (50.0, 0.5, 50.0)),
                              collider(_capi.SHAPE_SPHERE, 1, (2.0,), centres[1], (2.0, 2.0, 2.0)),
                              collider(_capi.SHAPE_TORUS, 2, (1.5, 0.5), centres[2], (2.0, 0.5, 2.0))])
            e3.set_contact_params(tolerance=0.05, stiffness=100.0, max_iter_v=5)
            e3.record_contacts(1 << 20)
            ms_c, _ = timed_steps(e3, md, k, 3, None)
            _, found = e3.contacts(1)
            side["cfg2_contacts"] = {"ms_per_step": ms_c / k, "ms_per_step_without_colliders": ms_plain / k, "contact_kernel_ms": (ms_c - ms_plain) / k, "mode": mn,
                                     "contacts_in_last_step": int(found), "colliders": "static box + sphere + torus (analytic distance fields), 5 velocity iterations",
                                     "particles_tested_per_step": inf["n"], "value": inf["proj_per_step"] * k / (ms_c * 1e-3), "unit": UNIT}
            e3.close()
        except Exception as ex:
            side["cfg2_contacts"] = {"error": str(ex)}

    # ---- CPU baseline (rank 0, N=1 only, bounded sample) ----------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            r = cpu_arm(args.size, args.iters, args.cpu_steps, 1)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        except Exception as ex:
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": "failed: %s" % ex}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": dict(workload_config(args.size, args.iters, world), mode=mode_name, particles=n, constraints=ncons,
                                                 colour_groups=int(st.num_groups), buckets=int(st.num_buckets), scene_build_s=round(info["build_s"], 2)),
            "sim_steps_per_sec": world * args.steps / (ms_max * 1e-3),
            "e2e": {"value": e2e_pipe_value, "unit": UNIT, "h2d_bytes_per_step": 2 * n * 12, "d2h_bytes_per_step": n * 12,
                    "ms_per_step": 1e3 * e2e_pipe_max / e2e_steps,
                    "api": "pbd_step_host_async + pbd_step_host_wait(1) (C ABI, pinned host buffers; x and v uploaded and x downloaded EVERY step, "
                           "the copies of neighbouring steps overlap the kernels; region ends with the last result in host memory)",
                    "pipelined_equals_blocking": pipelined_equal,
                    "blocking": {"value": e2e_value, "ms_per_step": 1e3 * e2e_max / e2e_steps, "h2d_bytes_per_step": 2 * n * 12, "d2h_bytes_per_step": n * 12,
                                 "api": "pbd_step_host: upload, step, download, synchronise inside every call (what the TimeStep adapter does by default)"},
                    "download_only": {"ms_per_step": 1e3 * e2e_dev_s / e2e_steps, "value": proj_per_step * e2e_steps / e2e_dev_s, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": n * 12,
                                      "note": "rank 0; blocking call with x_in = v_in = NULL (device state authoritative between steps), result downloaded every step"}},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "mode_probe_ms": probe,
            "checksum": {"crc32": crcs[0], "x_sum": xsum, "per_rank_crc32": crcs, "after_steps": "mode probe + warmup + steps (deterministic for fixed K, W)"},
            "checksums_equal": all(c == crcs[0] for c in crcs), "side": side}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    WORKLOAD = a.workload
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
