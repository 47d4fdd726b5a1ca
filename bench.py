#!/usr/bin/env python
"""bench.py -- the headline measurement and every BASELINE configuration, one JSON line per run.

  python bench.py --gpus N --steps K --warmup W                  the B200 core (this repository), BASELINE config 2
  python bench.py --impl reference --gpus N ...                  the reference's own device programs compiled for the host
                                                                 (oracle/_ref, one process per core; oracle port if absent)
  python bench.py --config c1|c2|c4|c5|c3-<1M|10M|100M>-<coh|incoh>-<closest|any>
  python bench.py --scaling strong                               N > 1: a FIXED --spp-per-step per step, split over the ranks
  python bench.py ... --dump-outputs DIR                         also writes what the last timed step computed (dump_outputs)

Path-tracing configs (c1, c2, c4, c5).  A "step" renders `--spp-per-step` iterations (samples per pixel) of the frame:
[extend -> shade -> connect] x depth -> accumulate, one pass of the hot path over one batch of width*height*spp path samples.
  value     whole-job Msamples/s with the scene resident in HBM, device-timed with CUDA events on the launching stream,
            max over ranks.  N > 1: sample-range partition (every GPU renders its own iteration indices over the full frame)
            followed by ONE ncclReduce(mean) of the accumulation buffers over NVLink on the render stream, inside the timing.
  e2e       the same metric through the reference-facing classes (Application::render -> Raytracer -> Device -> librtcore)
            with the camera uploaded from pinned host memory and the float4 frame read back to host memory every step.
            --calling-pattern per-iteration issues the reference's own pattern: `unsigned int render()` once per iteration.
  roofline  the extend (closest-hit traversal) kernel: algorithmic bytes (ray 48 B + 80 B per node + 48 B per triangle + 64 B per
            instance record, counted by a second, untimed pass with the same seeds) / its device time, as fractions of the HBM
            peak (MEASURED_PEAKS.json), of the L2 gather bandwidth and the FP32 / issue peaks measured by probe kernels in this
            run (rtc_probe_*); `traffic` and the issue fraction come from an ncu child run of one step when ncu is usable.
  cpu_baseline  oracle/_ref (the reference's shader sources host-compiled, kind "reference"; traversal served by the oracle's
            intersector) on a bounded sample of the same workload, one process per host core, plus one single-threaded run.

  trace_schedule  which schedule of the triangle tests the timed steps ran with and the four warm-up batch times the library chose
            it from (include/rtc_core.h rtc_trace_schedule_get; needs >= 4 warm-up steps to be settled before the timed ones).

Ray configs (c3-*).  A step traces one set of rays against a synthetic triangle soup; value = Mrays/s.
"""
import argparse
import csv
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

S_RAY, S_NODE, S_TRI, S_INST = 48, 80, 48, 64          # algorithmic bytes: ray in + hit out, wide node, triangle record, instance record
F_NODE, F_TRI, F_INST = 192, 60, 36                    # algorithmic flops (SURVEY.md section 8d)
WORKLOADS = {
    "rtigo3_geometry": "rtigo3 geometry scene (planes/boxes/spheres/tori, 5 BSDFs, constant env + 4x4 parallelogram light), pathLengths 2 6",
    "rtigo3_cornell_box": "rtigo3 Cornell box (area light, mirror + glass spheres)",
    "rtigo3_instances": "instanced stress scene: instances of a 50 000-triangle torus (two-level BVH), constant environment",
    "rtigo3_textures": "rtigo3 geometry scene with albedo and cutout textures (ordered any-hit processing)",
}
# BASELINE.json configs -> (scene, resolution, spp per step); c3 is handled by run_rays()
CONFIGS = {
    "c1": ("rtigo3_cornell_box", "512 512", 16),       # the whole config is 16 spp: one step = the config
    "c2": ("rtigo3_geometry", "1920 1080", 32),        # 8 steps = the config's 256 spp
    "c4": ("rtigo3_instances", "1920 1080", 16),       # 4 steps = the config's 64 spp
    "c5": ("rtigo3_geometry", "3840 2160", 8),         # 128 steps = the config's 1024 spp
}


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=5)      # >= 4: the schedule tuner of the traversal kernels settles during the warm-up steps
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--spp-per-step", type=int, default=None)
    ap.add_argument("--resolution", default=None)
    ap.add_argument("--scene", default=None)
    ap.add_argument("--instances", type=int, default=10000)
    ap.add_argument("--rays", default="1e8")
    ap.add_argument("--calling-pattern", default="batched", choices=["batched", "per-iteration"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ncu", action="store_true")
    ap.add_argument("--no-probes", action="store_true")
    ap.add_argument("--ncu-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args(argv)
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if not args.config.startswith("c3"):
        if args.config not in CONFIGS:
            ap.error("unknown --config " + args.config)
        scene, res, spp = CONFIGS[args.config]
        args.scene = args.scene or scene
        args.resolution = args.resolution or res
        args.spp_per_step = args.spp_per_step or spp
    return args


def workload(args):
    return "%s, %s" % (WORKLOADS.get(args.scene, args.scene), args.resolution.replace(" ", "x"))


def metric_name(args):
    w, h = args.resolution.split()
    if args.scene == "rtigo3_geometry" and (w, h) == ("1920", "1080"):
        return "rtigo3_geometry_1080p_samples_per_s"            # BASELINE.json's headline metric
    return "%s_%sx%s_samples_per_s" % (args.scene, w, h)


def path_config(args, n):
    """The `config` object of a path-tracing line; identical for both arms (--impl b200 / reference), built from the flags only."""
    w, h = (int(v) for v in args.resolution.split())
    per_gpu = args.spp_per_step // n if args.scaling == "strong" else args.spp_per_step
    return {"workload": workload(args), "baseline_config": args.config, "spp_per_step": args.spp_per_step,
            "path_samples_per_step": w * h * args.spp_per_step * (1 if args.scaling == "strong" else n),
            "spp_per_step_per_gpu": per_gpu,
            "parallelism": ("sample-range x%d (%s scaling) + one NCCL reduce of the accumulation buffers" % (n, args.scaling)) if n > 1 else "single GPU",
            "l2": "wavefront state per step (%.0f MB per GPU) exceeds L2 (126 MB); no explicit flush" % (min(per_gpu * w * h, 64 << 20) * 320 / 1e6)}


class ClockSampler(threading.Thread):
    """Samples SM clocks, power and clock-event (throttle) reasons of ONE GPU while the timed region runs.

    In-process NVML (pynvml) on a handle looked up once by UUID: ~1 kHz capable, sampled every 5 ms, and it does not
    spawn a process per sample (nvidia-smi attaches to every GPU of the box on each call, which N ranks polling at once
    would feel).  Falls back to polling nvidia-smi where pynvml is missing."""

    def __init__(self, index, uuid=None):
        super().__init__(daemon=True)
        self.index = index
        self.uuid = uuid
        self.stop_flag = threading.Event()
        self.rows = []          # (sm_mhz, sm_max_mhz, power_w, reason_bits)
        self.source = "nvml"
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = (pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode()) if uuid
                           else pynvml.nvmlDeviceGetHandleByIndex(index))
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.source = "nvidia-smi"

    def _sample_nvml(self):
        nv = self.nvml
        sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
        try:
            bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        try:
            power = nv.nvmlDeviceGetPowerUsage(self.handle) / 1e3
        except Exception:
            power = None
        reasons = set()
        for name, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                          ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                          ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown)):
            if bits & bit:
                reasons.add(name)
        self.rows.append((sm, self.sm_max, power, reasons))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if not out:
            return
        r = [c.strip() for c in out.splitlines()[0].split(",")]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = {name for k, name in enumerate(names) if len(r) > 3 + k and r[3 + k].lower().startswith("active")}
        self.rows.append((float(r[0]), float(r[1]), float(r[2]) if r[2].replace(".", "").isdigit() else None, reasons))

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.005 if self.nvml is not None else 0.05)

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        power = [r[2] for r in self.rows if r[2] is not None]
        reasons = set()
        for r in self.rows:
            reasons |= r[3]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": max(r[1] for r in self.rows) if self.rows else None, "reasons": sorted(reasons),
                "power_w_max": max(power) if power else None, "samples": len(self.rows), "source": self.source}


DUMP_LIMIT = 64 * 10 ** 6          # bytes of array data that --dump-outputs writes at most


def dump_outputs(directory, outputs):
    """--dump-outputs: writes every array of `outputs` ({name: array}) as directory/<name>.npy, float32 arrays as they are and
    integer arrays as float64 (exact for 32-bit values), so that two builds run with the same arguments can be compared output
    for output.  When the arrays together exceed DUMP_LIMIT, each keeps the same fixed, seeded sample of its first-axis rows
    (frame rows, or rays), in order."""
    import numpy as np
    size = {name: a.size * (a.itemsize if a.dtype.kind == "f" else 8) for name, a in outputs.items()}
    total = sum(size.values())
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        if total > DUMP_LIMIT:
            keep = max(1, len(a) * DUMP_LIMIT // total)
            a = a[np.unique(np.random.default_rng(0).integers(0, len(a), keep))]
        if a.dtype.kind != "f":
            a = a.astype(np.float64)
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a))


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def system_file(tmp, args, device_ordinal):
    import helpers as H
    return H.write_system(tmp, args.scene, resolution=args.resolution, samplesSqrt=256, devicesMask=1 << device_ordinal, strategy=0)


def scene_file(tmp, args):
    """scenes/scene_<name>.txt; the instanced stress scene (config 4) is generated (tools/make_instances_scene.py)."""
    import helpers as H
    if args.scene == "rtigo3_instances":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import make_instances_scene
        path = os.path.join(tmp, "scene_rtigo3_instances.txt")
        if not os.path.exists(path):
            make_instances_scene.write_scene(path, count=args.instances)
        return path
    return H.scene_path(args.scene)


# ---- the CPU arms: the reference's own device programs compiled for the host (oracle/_ref/libref.so), or the oracle port ----
def cpu_sample(args, threads, iterations=2, row_step=16, first=0):
    """Oracle (kind "port") on rows y % row_step == 0 for `iterations` samples per pixel; returns (Msamples/s, seconds, description)."""
    import helpers as H
    from oracle import orc
    from tweeker_raytracer_b200 import host
    tmp = tempfile.mkdtemp()
    app = host.App(system_file(tmp, args, 0), scene_file(tmp, args), host_only=True)
    ref = H.oracle_scene(app)
    w, h = app.resolution
    st = orc.Stats()
    t0 = time.perf_counter()
    ref.render(H.oracle_sys(app), app.info.miss, w, h, iter_first=first, iter_count=iterations, row_step=row_step, row_offset=0, threads=threads, stats=st)
    dt = time.perf_counter() - t0
    desc = "rows y%%%d==0 of %dx%d, %d spp = %d path samples (%d radiance + %d shadow rays) in %.2f s, %d thread(s)" % (
        row_step, w, h, iterations, st.pathSamples, st.radianceRays, st.shadowRays, dt, threads)
    return st.pathSamples / dt / 1e6, dt, desc


_REF = {}


def _ref_init(system_path, scene_path):
    import helpers as H
    from oracle import orc
    from tweeker_raytracer_b200 import host
    app = host.App(system_path, scene_path, host_only=True)
    scene = H.oracle_scene(app, "libm")
    _REF.update(app=app, scene=scene, ref=orc.Reference(scene, app.info.miss), sysd=H.oracle_sys(app))


def _ref_rows(task):
    k, procs, first, iterations = task
    app = _REF["app"]
    w, h = app.resolution
    t0 = time.perf_counter()
    _REF["ref"].render(_REF["sysd"], w, h, iter_first=first, iter_count=iterations, row_step=procs, row_offset=k)
    return time.perf_counter() - t0


class ReferencePool:
    """The reference keeps its launch parameters in a global, so it is parallelised over processes: worker k renders the
    launch rows y % P == k.  Set-up (scene load, oracle BVH for optixTrace) happens once per worker, outside the timing."""

    def __init__(self, args, procs):
        import multiprocessing as mp
        tmp = tempfile.mkdtemp()
        self.system_path, self.scene_path = system_file(tmp, args, 0), scene_file(tmp, args)
        self.procs = procs
        self.pool = mp.get_context("fork").Pool(procs, initializer=_ref_init, initargs=(self.system_path, self.scene_path))
        self.pool.map(_ref_rows, [(k, 64 * procs, 0, 1) for k in range(procs)])       # touch every worker (set-up done)
        self.resolution = tuple(int(v) for v in args.resolution.split())

    def sample(self, iterations, first=0, stride=1):
        """`iterations` samples of the rows y % stride == 0 (stride 1: the full frame), split over the workers."""
        t0 = time.perf_counter()
        self.pool.map(_ref_rows, [(k * stride, self.procs * stride, first, iterations) for k in range(self.procs)], chunksize=1)
        dt = time.perf_counter() - t0
        w, h = self.resolution
        rows = len(range(0, h, stride))
        n = w * rows * iterations
        what = "full %dx%d frame" % (w, h) if stride == 1 else "rows y%%%d==0 of %dx%d" % (stride, w, h)
        return n / dt / 1e6, dt, "%s, %d spp = %d path samples in %.2f s, %d process(es)" % (what, iterations, n, dt, self.procs)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_reference(args, iterations, pool=None, procs=None, stride=1):
    """(value, seconds, description, cores, kind): oracle/_ref when it is built ("reference"), else the oracle port."""
    from oracle import orc
    cores = procs or orc.online_cores()
    if orc.reference_available():
        own = pool is None
        pool = pool or ReferencePool(args, cores)
        v, dt, desc = pool.sample(iterations, stride=stride)
        if own:
            pool.close()
        return v, dt, desc, cores, "reference"
    v, dt, desc = cpu_sample(args, cores, iterations=iterations, row_step=stride)
    return v, dt, desc, cores, "port"


def cpu_baseline_block(args, unit):
    """All host cores on ~100 spp of the full frame scaled to the config (10-30 s), then ONE thread on a 1/16 row subset."""
    w, h = (int(v) for v in args.resolution.split())
    iterations = max(2, min(96, int(200e6 / (w * h))))            # ~2e8 path samples for the all-core run
    v, dt, desc, cores, kind = cpu_reference(args, iterations)
    one_iter = max(1, min(8, int(4e6 / (w * h / 16.0))))          # ~4e6 path samples for the single-threaded run
    v1, dt1, desc1, _, kind1 = cpu_reference(args, one_iter, procs=1, stride=16)
    return {"value": v, "unit": unit, "cores": cores, "kind": kind, "sample": desc,
            "single_thread": {"value": v1, "unit": unit, "cores": 1, "kind": kind1, "sample": desc1}}


def run_reference(args, rank):
    """The reference arm: the reference's own device programs compiled for the host (oracle/_ref, kind "reference", one
    process per host core; falls back to the oracle port where libref.so does not exist), rank 0 only.  Each step renders the
    same `--spp-per-step` iterations of the same frame as the GPU arm when that stays within ~20 s per step; otherwise a row
    subset of the frame at the same spp (stated in cpu_baseline.sample)."""
    if rank != 0:
        return
    if args.config.startswith("c3"):
        run_rays_reference(args)
        return
    from oracle import orc
    cores = orc.online_cores()
    n = max(args.gpus, 1)
    w, h = (int(v) for v in args.resolution.split())
    spp = args.spp_per_step
    stride = 1
    while w * h * spp / stride > 30e6 * max(cores, 1):            # ~30 M path samples per core and step at most
        stride *= 2
    pool = ReferencePool(args, cores) if orc.reference_available() else None
    for _ in range(min(args.warmup, 1)):
        cpu_reference(args, 1, pool, stride=max(stride, 16))
    vals, secs, desc, kind = [], 0.0, "", "port"
    for _ in range(args.steps):
        v, dt, desc, cores, kind = cpu_reference(args, spp, pool, stride=stride)
        vals.append(v)
        secs += dt
    if pool:
        pool.close()
    value = sum(vals) / len(vals)
    unit = "Msamples/s"
    line = {"impl": "reference", "metric": metric_name(args), "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": path_config(args, n),
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "sample": "each step: " + desc},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---- ncu child: DRAM bytes and executed instructions of the traversal kernels of ONE step ---------------------------------
def ncu_child(args):
    """Runs under ncu (see ncu_measure): renders one warm-up iteration, then one step; no torch, no timing."""
    import helpers as H
    from tweeker_raytracer_b200 import core, host
    tmp = tempfile.mkdtemp()
    app = host.App(system_file(tmp, args, 0), scene_file(tmp, args))
    w, h = app.resolution
    ctx = app.context(0)
    app.render(1)
    app.synchronize()
    sysd = app.system_data(0)
    before = ctx.stats().kernelLaunches
    ctx.launch_ex(sysd, w, h, core.RAYGEN_FULL_FRAME, app.info.miss, 1, args.spp_per_step, 1, False)
    ctx.synchronize()
    print("NCU_CHILD step_launches %d" % (ctx.stats().kernelLaunches - before), flush=True)
    app.close()


def ncu_measure(args, schedule="group"):
    """{'extend': {...}, 'connect': {...}} per-launch averages of one step from an ncu child run, or (None, reason).
    schedule: the traversal schedule the timed steps ran with; the child is pinned to it (RTC_TRACE_SCHEDULE)."""
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    log = os.path.join(tempfile.mkdtemp(), "ncu_child.csv")
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,lts__t_bytes.sum,smsp__inst_executed.sum,smsp__thread_inst_executed.sum,gpu__time_duration.sum",
           "--clock-control", "none", "-k", "regex:k_trace|k_extend_primary", "--csv", "--log-file", log,
           sys.executable, os.path.abspath(__file__), "--ncu-child", "--config", args.config, "--scene", args.scene, "--resolution", args.resolution,
           "--spp-per-step", str(args.spp_per_step), "--instances", str(args.instances)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0"),
                                      RTC_TRACE_SCHEDULE={"one_tri": "onetri", "two_tri": "twotri"}.get(schedule, "group")))
    except Exception as e:
        return None, "ncu child failed: %r" % (e,)
    if out.returncode != 0 or not os.path.exists(log):
        return None, "ncu child exit %d: %s" % (out.returncode, (out.stderr or out.stdout)[-200:].replace("\n", " "))
    rows = [r for r in csv.reader(open(log)) if len(r) > 5]
    if not rows:
        return None, "empty ncu log"
    hdr = rows[0]
    try:
        iid, iname, imetric, ivalue = hdr.index("ID"), hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value")
    except ValueError:
        return None, "unexpected ncu csv header"
    launches = {}
    for r in rows[1:]:
        try:
            launches.setdefault(int(r[iid]), {"name": r[iname]})[r[imetric]] = float(r[ivalue].replace(",", ""))
        except Exception:
            pass
    ids = sorted(launches)
    step = [launches[i] for i in ids[len(ids) // 2:]]            # the second half: the step (the first is the warm-up iteration)
    res = {}
    for key, pred in (("extend", lambda nm: "k_extend_primary" in nm or "ExtendPaths" in nm), ("connect", lambda nm: "ConnectPaths" in nm)):
        sel = [l for l in step if pred(l["name"])]
        if sel:
            res[key] = {"launches": len(sel),
                        "dram_bytes_per_launch": sum(l.get("dram__bytes_read.sum", 0) + l.get("dram__bytes_write.sum", 0) for l in sel) / len(sel),
                        "l2_bytes_per_launch": sum(l.get("lts__t_bytes.sum", 0) for l in sel) / len(sel),
                        "warp_inst_per_launch": sum(l.get("smsp__inst_executed.sum", 0) for l in sel) / len(sel),
                        "thread_inst_per_warp_inst": sum(l.get("smsp__thread_inst_executed.sum", 0) for l in sel) / max(sum(l.get("smsp__inst_executed.sum", 0) for l in sel), 1)}
    return (res, "ncu child run of one step in this bench run (dram__bytes_read.sum + dram__bytes_write.sum, smsp__inst_executed.sum per launch)") if res else (None, "no traversal kernels in the ncu log")


def probes(ctx):
    """Roofline denominators measured now, on this GPU (csrc/probes.cu)."""
    return {"l2_gather_gbs": ctx.probe_gather(32 << 20), "hbm_gather_16B_gbs": ctx.probe_gather(8 << 30),
            "fp32_tflops": ctx.probe_pipes(0), "issue_gwarpinst_per_s": ctx.probe_pipes(1),
            "how": "rtc_probe_gather: random 16-byte LDG.128 gathers over a 32 MB (L2-resident) working set, and over 8 GB (every 16-byte gather costs a 32-byte sector and mostly a TLB miss: a floor, not a roofline); rtc_probe_pipes: independent FFMA chains, and FFMA + LOP3 alternating"}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.ncu_child:
        ncu_child(args)
        return
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.config.startswith("c3"):
        run_rays(args, rank, local_rank, world)
        return

    import numpy as np
    import torch
    import helpers as H
    from tweeker_raytracer_b200 import core, host

    if core.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: " + core.lib().rtc_last_error().decode())
    n = args.gpus
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(local_rank)
    if world != n and world > 1:
        n = world
    K, W = args.steps, args.warmup
    S_total = args.spp_per_step
    if args.scaling == "strong":
        if S_total % n != 0:
            raise SystemExit("--scaling strong needs --spp-per-step divisible by the number of GPUs")
        S = S_total // n                      # the step's samples are split over the ranks
    else:
        S = S_total                           # every rank renders the full step: total work grows with N

    tmp = tempfile.mkdtemp()
    app = host.App(system_file(tmp, args, local_rank), scene_file(tmp, args))
    w, h = app.resolution
    pixels = w * h
    ctx = app.context(0)
    app.render(1)                      # allocates the frame, warms the allocator
    app.synchronize()
    sysd = app.system_data(0)
    info = ctx.scene_info(sysd.topObject)

    # N > 1: the Application joins the process group of the host library (Raytracer::joinProcessGroup: sample-range partition,
    # its own NCCL communicator on the render stream); torch.distributed carries the 128-byte id and the barriers
    if dist is not None:
        ids = [host.process_group_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        app.join_group(rank, world, ids[0])
    # accumulation buffer of the device-timed arm, and the buffer the mean frame lands in on rank 0
    frame = torch.zeros(pixels * 4, dtype=torch.float32, device="cuda")
    combined = torch.zeros(pixels * 4, dtype=torch.float32, device="cuda") if rank == 0 else None
    sysd.outputBuffer = frame.data_ptr()

    def combine():
        # the one exchange step of the path: ncclReduce(mean) of the per-rank running averages over NVLink, on the render stream
        app.group_reduce_mean(frame.data_ptr(), combined.data_ptr() if rank == 0 else 0, pixels * 4)

    from tweeker_raytracer_b200 import partition

    def step(s, count_work=False):
        # sample-range partition: rank r of n renders iteration indices (s*n + r)*S .. +S as samples s*S.. of its own average
        first, count, accum = partition.bench_step_range(s, rank, n, S_total, args.scaling)
        ctx.launch_ex(sysd, w, h, core.RAYGEN_FULL_FRAME, app.info.miss, first, count, accum, count_work)

    def barrier():
        torch.cuda.synchronize()
        ctx.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(W):
        step(s)
    if dist is not None:       # warm the NCCL communicator up (connection set-up is not part of a render)
        combine()
    # NVML is initialised BEFORE the barrier: its start-up time differs from process to process, and anything between the
    # barrier and timer_start shows up as skew in the max-over-ranks time
    sampler = ClockSampler(local_rank, getattr(torch.cuda.get_device_properties(local_rank), "uuid", None))
    ctx.stats_reset()
    ctx.profile_enable(True)
    barrier()
    stamps = [time.time()]
    sampler.start()
    ctx.timer_start()
    stamps.append(time.time())
    for s in range(W, W + K):
        step(s)
    stamps.append(time.time())
    steps_ms = ctx.timer_stop()                 # synchronises the render stream
    stamps.append(time.time())
    reduce_ms = 0.0
    if dist is not None:
        ctx.timer_start()
        combine()
        reduce_ms = ctx.timer_stop()            # on each rank: waiting for the slowest rank + the transfer
    stamps.append(time.time())
    outputs = None
    if args.dump_outputs and rank == 0:         # the frame after the last timed step (in a group: the mean over the ranks)
        outputs = {"frame": (combined if dist is not None else frame).cpu().numpy().reshape(h, w, 4)}
    barrier()
    sampler.stop_flag.set()
    sampler.join()
    prof = ctx.profile()
    ctx.profile_enable(False)
    stats = ctx.stats()
    # which schedule of the triangle tests the timed steps ran with (the library times one warm-up batch with each and keeps the
    # faster: include/rtc_core.h rtc_trace_schedule_get); with fewer than 4 warm-up steps the measurement reaches into the timed steps
    try:
        schedule = ctx.trace_schedule()
    except Exception as e:          # reporting only
        schedule = {"schedule": "group", "error": repr(e)}
    total_ms = steps_ms + reduce_ms
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    rays = torch.tensor([float(stats.radianceRays + stats.shadowRays)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays, op=dist.ReduceOp.SUM)
    total_ms = float(t.item())
    per_rank = [[steps_ms, reduce_ms]]
    if dist is not None:        # diagnostics: each rank's own render time and its wait+reduce time
        g = [torch.zeros(2 + len(stamps), dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(g, torch.tensor([steps_ms, reduce_ms] + stamps, dtype=torch.float64, device="cuda"))
        t00 = min(float(x[2]) for x in g)
        # [render ms, reduce ms, then host wall-clock ms since the first rank left the barrier: barrier exit, timer started,
        #  steps enqueued, render finished, reduce finished]
        per_rank = [[round(float(x[0]), 3), round(float(x[1]), 3)] + [round((float(v) - t00) * 1e3, 3) for v in x[2:]] for x in g]
    value = n * K * S * pixels / (total_ms * 1e-3) / 1e6
    mrays = float(rays.item()) / (total_ms * 1e-3) / 1e6
    launches = int(stats.kernelLaunches)

    # ---- algorithmic bytes of the extend kernel: the same steps again, untimed, with work counters
    ctx.launch_counts_reset()
    for s in range(W, W + K):
        step(s, count_work=True)
    ext, con = ctx.launch_counts()
    ext_bytes = ext.rays * S_RAY + ext.nodes * S_NODE + ext.tris * S_TRI + ext.instances * S_INST
    con_bytes = con.rays * S_RAY + con.nodes * S_NODE + con.tris * S_TRI + con.instances * S_INST
    ext_flops = ext.nodes * F_NODE + ext.tris * F_TRI + ext.instances * F_INST
    ext_ms, ext_launches = prof["extend"]
    con_ms, con_launches = prof["connect"]
    peak, peak_src = measured_peak()
    achieved = ext_bytes / (ext_ms * 1e-3) / 1e9 if ext_ms > 0 else 0.0
    # Two kinds of fractions.  ALGORITHMIC: the bytes / flops the algorithm needs per second over a peak -- how the work compares
    # with what the memory system or the FP32 pipe could stream; above 1 against the L2 gather probe simply means that L1 serves
    # most node fetches.  PHYSICAL (from the ncu child run of one step): what the kernel really moved or issued over the
    # same peaks; `bound` is the largest physical fraction, i.e. the resource the kernel actually saturates.
    fractions = {"hbm_algorithmic": achieved / peak}
    peaks = {"hbm_gbs": peak}
    if not args.no_probes and rank == 0:
        pr = probes(ctx)
        peaks.update(pr)
        fractions["l2_algorithmic"] = achieved / pr["l2_gather_gbs"]
        fractions["fp32_algorithmic"] = (ext_flops / (ext_ms * 1e-3) / 1e12) / pr["fp32_tflops"] if ext_ms > 0 else 0.0
    traffic, traffic_src, ncu_res = None, "not measured (--no-ncu or N > 1)", None
    physical = {}
    if rank == 0 and n == 1 and not args.no_ncu:
        ncu_res, traffic_src = ncu_measure(args, schedule.get("schedule", "group"))
        if ncu_res and "extend" in ncu_res and ext_ms > 0:
            e = ncu_res["extend"]
            traffic = e["dram_bytes_per_launch"]
            step_s = ext_ms / K * 1e-3                # device time of one step's extend launches in THIS run (not under ncu)
            physical["dram"] = e["dram_bytes_per_launch"] * e["launches"] / step_s / 1e9 / peak
            if "l2_gather_gbs" in peaks:
                physical["l2"] = e["l2_bytes_per_launch"] * e["launches"] / step_s / 1e9 / peaks["l2_gather_gbs"]
            if "issue_gwarpinst_per_s" in peaks:
                physical["issue"] = e["warp_inst_per_launch"] * e["launches"] / step_s / 1e9 / peaks["issue_gwarpinst_per_s"]
            fractions.update(physical)
    bound = max(physical, key=physical.get) if physical else "hbm"
    roofline = {"bound": bound, "kernel": "k_trace<ANY=0, ExtendPaths> + k_extend_primary (closest-hit traversal of the radiance rays)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "fractions": fractions, "peaks": peaks,
                "fractions_note": "*_algorithmic: algorithmic bytes (or flops: 192 per node, 60 per triangle, 36 per instance) per second over the HBM copy peak / the L2 gather probe / the FFMA probe (`frac` is hbm_algorithmic, the contract's figure).  dram, l2, issue: PHYSICAL -- DRAM bytes, L2 bytes and executed warp instructions of the step's extend launches (ncu child) over the same peaks; `bound` is the largest of them.  The BVH lives in L2/L1, so real DRAM traffic is a small fraction of the algorithmic bytes: the kernel is bound by instruction issue at partial SIMD occupancy",
                "algorithmic_bytes_per_launch": ext_bytes / max(ext_launches, 1),
                "avg_launch_ms": ext_ms / max(ext_launches, 1), "launches": int(ext_launches),
                "per_ray": {"nodes": ext.nodes / max(ext.rays, 1), "tris": ext.tris / max(ext.rays, 1), "instances": ext.instances / max(ext.rays, 1),
                            "bytes": ext_bytes / max(ext.rays, 1), "flops": ext_flops / max(ext.rays, 1)},
                "extend_mrays_per_s": ext.rays / (ext_ms * 1e-3) / 1e6 if ext_ms > 0 else 0.0,
                "connect": {"achieved": con_bytes / (con_ms * 1e-3) / 1e9 if con_ms > 0 else 0.0,
                            "mrays_per_s": con.rays / (con_ms * 1e-3) / 1e6 if con_ms > 0 else 0.0,
                            "bytes_per_ray": con_bytes / max(con.rays, 1)},
                "kernel_share_of_step": {k: v[0] / max(sum(x[0] for x in prof.values()), 1e-9) for k, v in prof.items()},
                "ncu": ncu_res,
                "bvh_mb": (info.numNodes * 80 + info.numTris * 48) / 1e6}

    # ---- end to end through Application::render with host buffers.  N > 1: the Application joins the process group
    # (sample-range partition inside the host library, its own NCCL communicator), every rank renders its range and
    # fetching the frame is a collective: ncclReduce(mean) over NVLink to rank 0, which reads the combined frame back.
    app.restart()
    cam = app.camera()
    pinned = ctx.host_alloc(48)
    ctypes.memmove(pinned, cam.ctypes.data, 48)
    sys_host = app.system_data(0)
    per_iteration = args.calling_pattern == "per-iteration"

    def render_step():
        if per_iteration:
            app.render_calls(S)           # the reference's pattern: `unsigned int render()` once per iteration, coalesced by the Raytracer
        else:
            app.render(S)
    for _ in range(min(W, 3)):
        render_step()
        app.frame_view()
    barrier()
    t0 = time.perf_counter()
    checksum = 0.0
    for _ in range(K):
        ctx.upload_async(sys_host.cameraDefinitions, pinned, 48)      # this step's camera, from pinned host memory
        render_step()
        fr = app.frame_view()                                         # device -> host read of the step's result (rank 0 in a group)
        if fr is not None:
            checksum += float(fr[0, 0, 0])
    ctx.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n * K * S * pixels / float(te.item()) / 1e6
    ctx.host_free(pinned)

    # ---- N > 1: an untimed parity step.  Every rank renders ONE iteration of its range; rank 0 fetches the combined frame
    # (the collective) and compares rows y % 64 == 0 with the oracle's mean of the same iterations.
    parity = None
    if dist is not None:
        app.restart()
        app.render(1)
        fr = app.frame_view()
        if rank == 0:
            parity = parity_check(app, fr, world, app.spp // world)      # app.spp = samplesSqrt^2; a rank's share is spp / world

    line = None
    if rank == 0:
        cfg = path_config(args, n)
        scene_info = {"triangles": int(info.numTris), "bvh_nodes": int(info.numNodes), "instances": int(info.numInstances),
                      "distinct_gas": int(info.numGas), "gas_build_ms": info.gasBuildMs, "ias_build_ms": info.iasBuildMs}
        line = {"metric": metric_name(args), "value": value, "unit": "Msamples/s", "n_gpus": n, "steps": K, "warmup": W, "ms_per_step": total_ms / K,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg, "scene_info": scene_info,
                "mrays_per_s": mrays, "reduce_ms": reduce_ms, "per_rank_render_ms_and_reduce_ms": per_rank,
                "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": 48 + 192, "d2h_bytes_per_step": pixels * 16,
                        "calling_pattern": args.calling_pattern,
                        "path": ("Application::render(count)" if not per_iteration else "%d x unsigned int Raytracer::render() (coalesced)" % S)
                                + " + getOutputBufferHost per step" + (" (collective: ncclReduce mean to rank 0, then read back)" if n > 1 else "")},
                "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roofline, "trace_schedule": schedule}
        if parity is not None:
            line["parity_check"] = parity["result"]
            line["parity_detail"] = parity
        if n == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(args, "Msamples/s")
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    app.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def parity_check(app, frame, world, local):
    """Rank 0, untimed: the combined one-iteration-per-rank frame vs the oracle's mean of the same iterations on rows y % 64 == 0.
    The oracle is the checker here, nothing else.  Tolerance: the NCCL mean sums the ranks in an order of its own, so the
    comparison allows 4 ulp-ish relative error (|a-b| <= 1e-6 * max(1, |b|)); with one rank it would be bit-exact."""
    import numpy as np
    import helpers as H
    from tweeker_raytracer_b200 import host
    w, h = app.resolution
    ref = H.oracle_scene(app)
    sysd = H.oracle_sys(app)
    rows = np.arange(0, h, 64)                # local = a rank's share of the iteration indices (samplesSqrt^2 / world)
    xy = np.array([(x, y) for y in rows for x in range(w)], dtype=np.uint32)
    acc = np.zeros((len(xy), 3), dtype=np.float64)
    for r in range(world):
        # every rank's first iteration is sample 0 of ITS running average: the raw radiance of seed iteration r * local
        acc += ref.path_radiance(sysd, app.info.miss, w, xy, r * local)[:, :3]
    want = (acc / world).reshape(len(rows), w, 3)
    got = np.asarray(frame, dtype=np.float64).reshape(h, w, 4)[::64]
    ok = np.isfinite(want)                    # a NaN sample is dropped by the accumulate kernel (raygeneration.cu:220-228): not compared
    err = np.where(ok, np.abs(got[..., :3] - np.where(ok, want, 0.0)), 0.0)
    tol = 1e-6 * np.maximum(1.0, np.abs(np.where(ok, want, 0.0)))
    bad = int((err > tol).sum())
    return {"result": "pass" if bad == 0 else "fail", "rows": int(got.shape[0]), "pixels": int(got.shape[0] * w), "max_abs_err": float(err.max()),
            "tolerance": "1e-6 * max(1, |oracle|)", "mismatches": bad,
            "what": "combined frame of one iteration per rank (iteration indices r * %d) vs the oracle's mean, rows y %% 64 == 0" % local}


# ---- BASELINE config 3: rays against synthetic triangle soups ---------------------------------------------------------------
def c3_parse(name):
    parts = name.split("-")
    if len(parts) != 4 or parts[1] not in ("1M", "10M", "100M") or parts[2] not in ("coh", "incoh") or parts[3] not in ("closest", "any"):
        raise SystemExit("config 3 is spelt c3-<1M|10M|100M>-<coh|incoh>-<closest|any>")
    return {"1M": 10 ** 6, "10M": 10 ** 7, "100M": 10 ** 8}[parts[1]], parts[2], parts[3]


def soup_numpy(n, seed=0x1234567):
    """Triangle soup of SURVEY.md section 8d: centres uniform in the unit cube, edge ~ n^(-1/3); float32 [3n, 3], in chunks."""
    import numpy as np
    rng = np.random.default_rng(seed)
    edge = float(n) ** (-1.0 / 3.0)
    out = np.empty((3 * n, 3), dtype=np.float32)
    chunk = 1 << 22
    for a in range(0, n, chunk):
        m = min(chunk, n - a)
        c = rng.random((m, 1, 3), dtype=np.float32)
        v = c + (rng.random((m, 3, 3), dtype=np.float32) - 0.5) * (2.0 * edge)
        out[3 * a:3 * (a + m)] = v.reshape(-1, 3)
    return out


def rays_numpy(n, kind, mode, seed=0x89ABCDEF):
    import numpy as np
    from tweeker_raytracer_b200 import core
    rays = np.empty(n, dtype=core.RAY_DTYPE)
    if kind == "coh":
        side = int(n ** 0.5)
        m = side * side
        rays = rays[:m]
        ys, xs = np.divmod(np.arange(m, dtype=np.int64), side)
        dx = ((xs + 0.5) / side * 2 - 1).astype(np.float32) * np.float32(0.6)
        dy = ((ys + 0.5) / side * 2 - 1).astype(np.float32) * np.float32(0.6)
        inv = 1.0 / np.sqrt(dx * dx + dy * dy + 1.0)
        rays["ox"], rays["oy"], rays["oz"], rays["tmin"] = 0.5, 0.5, 2.2, 1e-5
        rays["dx"], rays["dy"], rays["dz"] = dx * inv, dy * inv, -inv
        rays["tmax"] = 1e27
    else:
        rng = np.random.default_rng(seed)
        chunk = 1 << 22
        for a in range(0, n, chunk):
            m = min(chunk, n - a)
            o = rng.random((m, 3), dtype=np.float32)
            d = rng.standard_normal((m, 3), dtype=np.float32)
            d /= np.linalg.norm(d, axis=1, keepdims=True)
            v = rays[a:a + m]
            v["ox"], v["oy"], v["oz"], v["tmin"] = o[:, 0], o[:, 1], o[:, 2], 1e-5
            v["dx"], v["dy"], v["dz"] = d[:, 0], d[:, 1], d[:, 2]
        rays["tmax"] = 1e27 if mode == "closest" else 0.5
    return rays


def c3_config(args, ntris, kind, mode, nrays):
    return {"workload": "ray microbenchmark: %d %s %s-hit rays against a soup of %d triangles (centres uniform in the unit cube, edge n^(-1/3))"
                        % (nrays, "coherent (pinhole)" if kind == "coh" else "incoherent (uniform origins and directions)", mode, ntris),
            "baseline_config": args.config, "rays_per_step": nrays, "triangles": ntris,
            "parallelism": "replicated soup, one rank per GPU, no collective",
            "l2": "triangles alone are %.0f MB (48 B each) and the ray set %.0f MB vs 126 MB L2; no explicit flush" % (ntris * 48 / 1e6, nrays * 32 / 1e6)}


def run_rays(args, rank, local_rank, world):
    """Config 3 on the GPU: one process per GPU, every rank traces the same ray set against its own copy of the soup (weak scaling,
    no data-path collective: rays shard without an exchange step)."""
    import numpy as np
    import torch
    from tweeker_raytracer_b200 import core
    ntris, kind, mode = c3_parse(args.config)
    nrays = int(float(args.rays))
    n = max(world, 1)
    dist = None
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = core.Context(local_rank)
    verts = soup_numpy(ntris)
    d_verts = ctx.malloc(verts.nbytes)
    ctx.upload(d_verts, verts)
    idx = np.arange(3 * ntris, dtype=np.uint32)
    d_idx = ctx.malloc(idx.nbytes)
    ctx.upload(d_idx, idx)
    ctx.synchronize()
    t0 = time.perf_counter()
    gas = ctx.gas_build(d_verts, 12, 3 * ntris, d_idx, ntris, core.BUILD_GPU_LBVH)
    ctx.synchronize()
    build_s = time.perf_counter() - t0
    inst = np.zeros(1, dtype=core.INSTANCE_DTYPE)
    inst[0]["transform"] = [1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0]
    inst[0]["gas"] = gas
    top = ctx.ias_build(inst)
    info = ctx.scene_info(top)
    del verts, idx
    rays = rays_numpy(nrays, kind, mode)
    nrays = rays.shape[0]
    d_rays = ctx.malloc(rays.nbytes)
    ctx.upload(d_rays, rays)
    out_bytes = nrays * (20 if mode == "closest" else 4)
    d_out = ctx.malloc(out_bytes)
    ctx.synchronize()

    def trace(ptr=None, count=None):
        if mode == "closest":
            ctx.trace_closest(top, ptr or d_rays, count or nrays, d_out)
        else:
            ctx.trace_any(top, ptr or d_rays, count or nrays, d_out)

    def barrier():
        ctx.synchronize()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    K, W = args.steps, args.warmup
    for _ in range(W):
        trace()
    # Schedule of the triangle tests (include/rtc_core.h rtc_trace_schedule_set).  The library measures it by itself only inside
    # rtc_launch; for the query interface the caller does what the library does there: one step with each schedule (group first
    # and last) after the warm-up, a capped schedule only if it beats the faster group step by 3 %.  Results are bit-identical.
    schedule = {"schedule": "group", "measured": False}
    if (os.environ.get("RTC_TRACE_SCHEDULE") or "auto")[0] not in "go01t2":
        try:
            times = []
            for name in ("group", "one_tri", "two_tri", "group"):
                ctx.set_trace_schedule(name)
                ctx.timer_start()
                trace()
                times.append(ctx.timer_stop())
            group = min(times[0], times[3])
            best = "group"
            if min(times[1], times[2]) < 0.97 * group:
                best = "one_tri" if times[1] <= times[2] else "two_tri"
            if dist is not None:        # one choice for the job: rank 0's
                pick = [best]
                dist.broadcast_object_list(pick, src=0)
                best = pick[0]
            ctx.set_trace_schedule(best)
            schedule = {"schedule": best, "measured": True, "group_ms": [times[0], times[3]], "one_tri_ms": times[1], "two_tri_ms": times[2]}
        except Exception as e:          # reporting only: fall back to the measured schedule
            ctx.set_trace_schedule("group")
            schedule = {"schedule": "group", "measured": False, "error": repr(e)}
    sampler = ClockSampler(local_rank, getattr(torch.cuda.get_device_properties(local_rank), "uuid", None))
    ctx.stats_reset()
    barrier()
    sampler.start()
    ctx.timer_start()
    for _ in range(K):
        trace()
    ms = ctx.timer_stop()
    barrier()
    outputs = None
    if args.dump_outputs and rank == 0:         # the hits (or occlusion flags) of the last timed step
        if mode == "closest":
            hits = ctx.download(d_out, core.HIT_DTYPE, nrays)
            outputs = {"hit_t": hits["t"], "hit_u": hits["u"], "hit_v": hits["v"], "hit_instance": hits["inst"], "hit_primitive": hits["prim"]}
        else:
            outputs = {"occluded": ctx.download(d_out, np.uint32, nrays)}
    sampler.stop_flag.set()
    sampler.join()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = n * K * nrays / (ms * 1e-3) / 1e6
    launches = int(ctx.stats().kernelLaunches)
    # algorithmic bytes on every 16th ray
    sub = np.ascontiguousarray(rays[::16])
    d_sub = ctx.malloc(sub.nbytes)
    ctx.upload(d_sub, sub)
    ctx.synchronize()
    counts = ctx.trace_count(top, d_sub, sub.shape[0], any_hit=(mode == "any"))
    per_ray = (S_RAY * counts.rays + S_NODE * counts.nodes + S_TRI * counts.tris + S_INST * counts.instances) / max(counts.rays, 1)
    flops_ray = (F_NODE * counts.nodes + F_TRI * counts.tris + F_INST * counts.instances) / max(counts.rays, 1)
    peak, peak_src = measured_peak()
    achieved = per_ray * nrays * K / (ms * 1e-3) / 1e9
    fractions, peaks = {"hbm_algorithmic": achieved / peak}, {"hbm_gbs": peak}
    if not args.no_probes and rank == 0:
        pr = probes(ctx)
        peaks.update(pr)
        fractions["l2_algorithmic"] = achieved / pr["l2_gather_gbs"]
        fractions["fp32_algorithmic"] = flops_ray * nrays * K / (ms * 1e-3) / 1e12 / pr["fp32_tflops"]
    bvh_mb = (info.numNodes * 80 + info.numTris * 48) / 1e6
    # end to end: rays from pinned host memory, hits back to host memory, every step (a bounded set of 2^24 rays)
    ne = min(nrays, 1 << 24)
    pin_in = ctx.host_alloc(ne * 32)
    pin_out = ctx.host_alloc(ne * (20 if mode == "closest" else 4))
    ctypes.memmove(pin_in, rays.ctypes.data, ne * 32)
    for _ in range(min(W, 2)):
        ctx.upload_async(d_rays, pin_in, ne * 32)
        trace(d_rays, ne)
        ctx.download_async(pin_out, d_out, ne * (20 if mode == "closest" else 4))
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        ctx.upload_async(d_rays, pin_in, ne * 32)
        trace(d_rays, ne)
        ctx.download_async(pin_out, d_out, ne * (20 if mode == "closest" else 4))
    ctx.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n * K * ne / float(te.item()) / 1e6
    if rank == 0:
        cfg = c3_config(args, ntris, kind, mode, nrays)
        scene_info = {"bvh_nodes": int(info.numNodes), "bvh_mb": bvh_mb, "gas_build_s": build_s}
        line = {"metric": "ray_microbenchmark_%s_mrays_per_s" % args.config.replace("-", "_"), "value": value, "unit": "Mrays/s", "n_gpus": n, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "scene_info": scene_info,
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": ne * 32, "d2h_bytes_per_step": ne * (20 if mode == "closest" else 4),
                        "path": "rtc_upload (pinned host rays) + rtc_trace_%s + rtc_download (hits) of %d rays per step" % (mode, ne)},
                "gpu_launches": launches, "clocks": sampler.summary(), "trace_schedule": schedule,
                "roofline": {"bound": "hbm" if bvh_mb > 126.0 else "l2", "kernel": "k_trace<ANY=%d, Query%s>" % (mode == "any", "Closest" if mode == "closest" else "Any"),
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                             "fractions": fractions, "peaks": peaks,
                             "per_ray": {"nodes": counts.nodes / max(counts.rays, 1), "tris": counts.tris / max(counts.rays, 1), "bytes": per_ray, "flops": flops_ray}}}
        if n == 1 and not args.no_cpu_baseline and ntris <= 10 ** 6:
            line["cpu_baseline"] = rays_cpu(args, ntris, kind, mode, rays)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def rays_cpu(args, ntris, kind, mode, rays, sample=400000, threads=0):
    """The oracle's intersector (kind "port": the reference has no traversal source, OptiX hides it) on a bounded ray sample."""
    import numpy as np
    from oracle import orc
    from tweeker_raytracer_b200 import host
    verts = soup_numpy(ntris)
    attrs = np.zeros(3 * ntris, dtype=host.ATTR_DTYPE)
    attrs["vertex"] = verts
    s = orc.Scene()
    s.add_geometry(attrs, np.arange(3 * ntris, dtype=np.uint32))
    s.add_instance(np.array([1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0], dtype=np.float32), 0, 0, -1)
    s.commit()
    sub = np.ascontiguousarray(rays[:: max(1, rays.shape[0] // sample)][:sample])
    t0 = time.perf_counter()
    if mode == "closest":
        s.trace_closest(sub)
    else:
        s.trace_any(sub)
    dt = time.perf_counter() - t0
    return {"value": sub.shape[0] / dt / 1e6, "unit": "Mrays/s", "cores": 1, "kind": "port", "seconds": dt,
            "sample": "%d rays (every %d-th of the set) in %.2f s, oracle binary BVH, one thread" % (sub.shape[0], max(1, rays.shape[0] // sample), dt)}


def run_rays_reference(args):
    ntris, kind, mode = c3_parse(args.config)
    if ntris > 10 ** 6:
        print(json.dumps({"impl": "reference", "unavailable": "the CPU oracle's BVH build over %d triangles does not fit the few-minute budget" % ntris}), flush=True)
        return
    nrays = int(float(args.rays))
    rays = rays_numpy(min(nrays, 1 << 22), kind, mode)
    vals, secs = [], 0.0
    base = None
    for _ in range(args.steps):
        base = rays_cpu(args, ntris, kind, mode, rays, sample=200000)
        vals.append(base["value"])
        secs += base["seconds"]
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": "ray_microbenchmark_%s_mrays_per_s" % args.config.replace("-", "_"), "value": v, "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": c3_config(args, ntris, kind, mode, nrays), "cpu_baseline": dict(base, value=v),
            "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
