#!/usr/bin/env python
"""bench.py -- Mrays/s (primary + secondary) of the path-tracing hot path on N B200s.

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torch.distributed.run)
  python bench.py --impl reference ...                   (the reference shader source / CPU oracle on the host cores, same config)
  python bench.py ... --dump-outputs DIR                 (also writes each workload's framebuffer after its last timed step)

Workloads (BASELINE.json configs; scenes of SURVEY.md 8d, ezrt_b200/scenes.py):
  N = 1  : configs[2] "C3" -- S-1M (201 Stanford bunnies + 4 spheres + floor = 999,860 triangles), 1920x1080, Disney BRDF +
           Sobol (mode disney_sobol_p5), 2 bounces; the north_star target (>= 1 Gray/s) is quoted on this scene.  After the
           headline the same invocation measures configs[1] "C2" (bunny 5,300 triangles, 1024x1024, diffuse) and
           configs[3] "C4" (C3 + HDR importance sampling + MIS) and appends them under "workloads".
  N > 1  : configs[4] "C5" -- the SAME scene and integrator on ONE fixed 3840x2160 image split by 16x16 tiles over the N
           GPUs (strong scaling; `--workload c4` selects the IS/MIS integrator), one NCCL framebuffer gather per render.
           --scaling weak keeps round 1's growing image (1920x1080 pixels per GPU).
One step = one pass of the hot path over one batch: `--spp-per-step` consecutive display() calls (default 16; the default
16 steps make up C3's 256 spp), accumulating into the same framebuffer with frameCounter advancing.

value     total rays of all ranks / max-over-ranks CUDA-event time of the K timed steps, scene and framebuffer resident in
          HBM (ezrt_render_device on the current stream; N > 1: plus the single gather, inside the timed region).
e2e       the same steps through host buffers: every step uploads lastFrame from pinned host memory and reads the new
          framebuffer back (N = 1: ezrt_render; N > 1: per-rank parts every step, the gathered image once per render).
parity    frame 0 of the workload (1 spp, the full image of all ranks) compared with the CPU reference render of the same
          frame: L-inf and the number of differing floats (0 expected: the arithmetic is bit-specified).
roofline / cpu_baseline: see DESIGN.md "Measurement".
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Mrays/s (primary+secondary)"
UNIT = "Mrays/s"
ENV_COLOR = (0.35, 0.45, 0.6)
WORKLOADS = {
    # name: (scene builder, width, height, mode, max_bounce, BASELINE config it stands for)
    "c3": ("s_1m_bunny", 1920, 1080, 2, 2, "configs[2]: 1M-tri merged Stanford scene, 1920x1080, Disney BRDF + Sobol"),
    "c2": ("s_p3_bunny", 1024, 1024, 0, 2, "configs[1]: bunny 5k tris, 1024x1024, diffuse-only BRDF"),
    "c4": ("s_1m_bunny", 1920, 1080, 3, 2, "configs[3]: C3 scene + HDR env-map importance sampling + MIS"),
    # round-1 stand-in scenes (procedural 'blob' mesh), kept as a second family
    "c3_blob": ("s_1m", 1920, 1080, 2, 2, "round-1 stand-in for configs[2] (procedural mesh)"),
    "c2_blob": ("s_bunny", 1024, 1024, 0, 2, "round-1 stand-in for configs[1] (procedural mesh)"),
    "c4_blob": ("s_1m", 1920, 1080, 3, 2, "round-1 stand-in for configs[3] (procedural mesh)"),
}
C5_IMAGE = (3840, 2160)   # configs[4]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ezrt", choices=["ezrt", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"])
    ap.add_argument("--image", default=None, help="WxH override of the whole image")
    ap.add_argument("--spp-per-step", type=int, default=16)
    ap.add_argument("--frames-per-batch", type=int, default=0)
    ap.add_argument("--traverse", default="accel", choices=["accel", "pruned", "reference"])
    ap.add_argument("--pipeline", default="wavefront", choices=["wavefront", "megakernel"])
    ap.add_argument("--extra-workloads", default=None, help="comma list measured after the headline (default at N=1: c2,c4; '' = none)")
    ap.add_argument("--extra-steps", type=int, default=4)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--cpu-reps", type=int, default=3, help="repetitions of the CPU sample (the fastest is reported, all are listed)")
    ap.add_argument("--cpu-sample", default=None, help="WxHxSPP of the CPU baseline sample (default: frame 0 of the whole image, 1 spp)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the framebuffer each measured workload holds after its last timed step as DIR/<workload>.npy (float32)")
    return ap.parse_args()


# ----------------------------------------------------------------------------------------------------------------------
# host resources
# ----------------------------------------------------------------------------------------------------------------------
def cpu_threads():
    """Threads the CPU legs may use: the scheduler affinity, capped by the cgroup CPU quota.  os.cpu_count() reports the
    host's cores even inside a container limited to a few, and torch.distributed.run sets OMP_NUM_THREADS=1 -- the CPU
    legs therefore always pass an explicit thread count to the renderers."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    n = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return n, {"affinity": aff, "cgroup_cpus": quota, "os_cpu_count": os.cpu_count(), "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 50 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------------------------
_SCENE_CACHE = {}


def find_reference_hdr():
    """The reference's own 2k environment map (P5/main.cpp:897) when an installed copy of the reference is readable."""
    p = os.path.join(ROOT, "baseline", "_ref", "part 5 -- Importance Sampling & Low Discrepancy Sequence", "source code", "HDR", "chinese_garden_2k.hdr")
    return p if os.path.exists(p) else None


def build_workload(name, device_cache=False):
    from ezrt_b200 import api, scenes
    builder, w, h, mode, bounces, what = WORKLOADS[name]
    t0 = time.time()
    if builder not in _SCENE_CACHE:
        _SCENE_CACHE[builder] = getattr(scenes, builder)()
    tris, nodes, eye, cam = _SCENE_CACHE[builder]
    hdr = cache = None
    env = "constant colour %s" % (ENV_COLOR,)
    if mode == 3:
        path = find_reference_hdr()
        if path is not None:
            hdr = api.hdr_load(path)
            env = "chinese_garden_2k.hdr (the reference's own map, P5/main.cpp:897)"
        else:
            hdr = scenes.synth_hdr(2048, 1024)
            env = "procedural 2048x1024 map (scenes.synth_hdr; the reference's chinese_garden_2k.hdr is not on this box)"
        # calculateHdrCache: on the GPU when there is one (bit-identical to the host restatement, tests/test_post.py)
        cache = api.hdr_cache_device(hdr)[0] if device_cache else api.hdr_cache(hdr)
    return dict(name=name, what=what, tris=tris, nodes=nodes, eye=eye, cam=cam, width=w, height=h, mode=mode, max_bounce=bounces, scene=builder,
                hdr=hdr, cache=cache, env=env, build_s=time.time() - t0)


def workload_config(args, wl, W, H, world, scaling):
    """The `config` object: identical in the ezrt arm and the reference arm of one invocation."""
    return {"workload": wl["name"], "baseline_config": wl["what"], "scene": wl["scene"], "triangles": int(wl["tris"].shape[0]),
            "bvh_nodes": int(wl["nodes"].shape[0]), "image": [W, H], "spp_per_step": args.spp_per_step, "mode": wl["mode"],
            "max_bounce": wl["max_bounce"], "environment": wl["env"], "first_frame": 0, "parallelism": "tiles%d" % world, "scaling": scaling,
            "l2": "inputs larger than L2: the wavefront state one step streams (%.0f MB: hit records, path queues, per-sample radiance of %d sample slots "
                  "per GPU) and, for the 1M-triangle scenes, the scene itself (%.0f MB of tree + triangle records) against 126 MB of L2; no flush needed"
                  % (W * H * args.spp_per_step / world * 72 / 1e6, W * H * args.spp_per_step // world, wl["tris"].shape[0] * (64 + 48 + 64 + 30) / 1e6)}


def image_for(args, wl, world):
    """(W, H, scaling label) of the whole image rendered by `world` GPUs."""
    if args.image:
        w, h = (int(x) for x in args.image.lower().split("x"))
        return w, h, ("strong" if args.scaling != "weak" else "weak")
    if world == 1:
        return wl["width"], wl["height"], "strong"
    if args.scaling == "weak":   # round 1: pixels per GPU fixed (2: 2WxH, 4: 2Wx2H, 8: 4Wx2H)
        a = b = 1
        k = world
        while k > 1:
            if a <= b:
                a *= 2
            else:
                b *= 2
            k //= 2
        if a * b != world:
            a, b = world, 1
        return wl["width"] * a, wl["height"] * b, "weak"
    return C5_IMAGE[0], C5_IMAGE[1], "strong"   # configs[4]: one fixed 3840x2160 image


# ----------------------------------------------------------------------------------------------------------------------
# CPU legs (the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_render(wl, W, H, spp, threads, want_counters=False):
    """Frame range [0, spp) of the workload on the host cores.  Uses the reference's own shader source compiled for the CPU
    (oracle/_ref/libezrt_refshader.so, kind "reference") when that library travelled here, else the oracle port.
    Returns dict(image, seconds, kind, counters or None)."""
    from ezrt_b200 import api
    from tests import oracle_binding as oracle
    from tests import refshader_binding as refshader
    cfg = api.RenderConfig(width=W, height=H, spp=spp, max_bounce=wl["max_bounce"], mode=wl["mode"], eye=tuple(wl["eye"]),
                           camera_rotate=tuple(wl["cam"]), env_color=ENV_COLOR, traverse=api.TRAVERSE_REFERENCE)
    counters = None
    if want_counters or not refshader.available():
        t0 = time.perf_counter()
        img, counters = oracle.render(wl["tris"], wl["nodes"], cfg, hdr=wl.get("hdr"), hdr_cache=wl.get("cache"), threads=threads)
        dt = time.perf_counter() - t0
        if not refshader.available():
            return dict(image=img, seconds=dt, kind="port", counters=counters)
    hdr, cache, linear = wl.get("hdr"), wl.get("cache"), True
    if hdr is None:  # a scene without an environment map gets a 1x1 map of the constant colour (GL_NEAREST): what env_color means to the shader
        hdr, cache, linear = np.array([[list(ENV_COLOR)]], np.float32), None, False
    t0 = time.perf_counter()
    img = refshader.render(wl["tris"], wl["nodes"], cfg, hdr, cache, hdr_linear=linear, threads=threads)
    dt = time.perf_counter() - t0
    return dict(image=img, seconds=dt, kind="reference", counters=counters)


def cpu_baseline_leg(args, wl, W, H, threads, thread_info):
    """cpu_baseline: a bounded sample of the workload (default frame 0 of the whole image) timed `--cpu-reps` times with an
    explicit thread count.  Also returns the frame for the parity check and the oracle's ray counters."""
    if args.cpu_sample:
        sw, sh, sspp = (int(x) for x in args.cpu_sample.lower().split("x"))
    else:
        sw, sh, sspp = W, H, 1
    first = cpu_render(wl, sw, sh, sspp, threads, want_counters=True)
    secs = [first["seconds"]]
    for _ in range(max(0, args.cpu_reps - 1)):
        secs.append(cpu_render(wl, sw, sh, sspp, threads)["seconds"])
    c = first["counters"]
    best = min(secs)
    what = "reference shader source (fshader.fsh of the mode transpiled to C++, oracle/_ref)" if first["kind"] == "reference" else "oracle port (oracle/ezrt_oracle.cpp)"
    base = {"value": c["rays"] / best / 1e6, "unit": UNIT, "cores": threads, "threads_used": threads, "kind": first["kind"],
            "sample": "%s renders frames [0,%d) of the %dx%d image of this workload, literal hitBVH traversal; best of %d runs (%s s)" %
                      (what, sspp, sw, sh, len(secs), ", ".join("%.2f" % s for s in secs)),
            "rays_in_sample": c["rays"], "host": thread_info}
    return base, first, (sw, sh, sspp)


def run_reference(args, rank, world):
    """--impl reference: the reference's own implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return
    wl = build_workload(args.workload)
    W, H, scaling = image_for(args, wl, world)
    threads, tinfo = cpu_threads()
    if args.cpu_sample:
        sw, sh, sspp = (int(x) for x in args.cpu_sample.lower().split("x"))
    else:
        sw, sh, sspp = W, H, 1
    first = cpu_render(wl, sw, sh, sspp, threads, want_counters=True)   # ray count of the sample + which implementation is available
    rays = first["counters"]["rays"]
    secs = []
    for i in range(args.warmup + args.steps):
        r = cpu_render(wl, sw, sh, sspp, threads)
        if i >= args.warmup:
            secs.append(r["seconds"])
    total_s = sum(secs)
    value = rays * len(secs) / total_s / 1e6
    what = "reference shader source (P3|P4|P5 fshader.fsh of the mode, transpiled to C++, oracle/_ref)" if first["kind"] == "reference" else "oracle port"
    sample = "%s renders frames [0,%d) of the %dx%d image per step (literal hitBVH traversal), %d threads" % (what, sspp, sw, sh, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_s / max(1, len(secs)), "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, wl, W, H, world, scaling),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "threads_used": threads, "kind": first["kind"], "sample": sample, "host": tinfo},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """Everything but the one JSON line goes to stderr: libraries (NCCL's version banner, the reference shaders' host
    code) must not share the stream the driver parses."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def load_json(path):
    try:
        return json.load(open(path))
    except Exception:
        return None


def gather_peak(record_bytes):
    """Measured ceiling for the traversal kernels' access pattern (tools/gather_bench.cu on this pool's B200, committed as
    profiles/gather_peak_r2.json): records/s of `record_bytes`-byte records read by divergent lanes with 256-bit loads from an
    L2-resident table."""
    data = load_json(os.path.join(ROOT, "profiles", "gather_peak_r2.json"))
    if not data:
        return None
    best = None
    for r in data.get("results", []):
        if r.get("record_bytes") == record_bytes and "ld256" in r.get("table", "") and r.get("table", "").startswith("global_16MB"):
            best = r["grecords_per_s"] * 1e9
    return best


# ----------------------------------------------------------------------------------------------------------------------
# one measured configuration on the GPUs
# ----------------------------------------------------------------------------------------------------------------------
class Runner:
    def __init__(self, args, wl, rank, world, local_rank, W, H):
        import torch
        from ezrt_b200 import api
        from ezrt_b200 import dist as ezdist
        self.torch, self.api = torch, api
        self.args, self.wl, self.rank, self.world, self.W, self.H = args, wl, rank, world, W, H
        t0 = time.perf_counter()
        self.scene = api.Scene(wl["tris"], wl["nodes"], wl.get("hdr"), wl.get("cache"), device=local_rank)
        self.upload_ms = 1e3 * (time.perf_counter() - t0)
        # the same call again (scene dropped at once): without the first call's one-off costs in this process (module load, first allocations)
        t0 = time.perf_counter()
        api.Scene(wl["tris"], wl["nodes"], wl.get("hdr"), wl.get("cache"), device=local_rank).close()
        self.upload_again_ms = 1e3 * (time.perf_counter() - t0)
        self.C = 3
        self.n_local = api.partition_pixels(W, H, rank, world)
        self.traverse = {"accel": api.TRAVERSE_ACCEL, "pruned": api.TRAVERSE_PRUNED, "reference": api.TRAVERSE_REFERENCE}[args.traverse]
        self.pipeline = api.PIPELINE_WAVEFRONT if args.pipeline == "wavefront" else api.PIPELINE_MEGAKERNEL
        self.stream = torch.cuda.current_stream()
        self.d_fb = torch.zeros(max(1, self.n_local) * self.C, dtype=torch.float32, device="cuda")
        self.gatherer = ezdist.FramebufferGather(W, H, self.C, rank, world, self.d_fb.device) if world > 1 else None

    def cfg(self, first_frame, spp, profile=0, accumulate=False):
        wl = self.wl
        return self.api.RenderConfig(width=self.W, height=self.H, spp=spp, first_frame=first_frame, max_bounce=wl["max_bounce"], mode=wl["mode"],
                                     eye=tuple(wl["eye"]), camera_rotate=tuple(wl["cam"]), env_color=ENV_COLOR, traverse=self.traverse,
                                     pipeline=self.pipeline, part_rank=self.rank, part_count=self.world,
                                     frames_per_batch=self.args.frames_per_batch, profile=profile, accumulate=accumulate)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()

    def step(self, s, profile=0, accumulate=False):
        spp = self.args.spp_per_step
        self.scene.render_device(self.cfg(s * spp, spp, profile, accumulate), self.d_fb, self.stream)

    def gather(self):
        """The single collective of a render: compact per-rank parts -> the row-major image on rank 0 (device tensor)."""
        if self.world == 1:
            return self.d_fb.reshape(self.H, self.W, self.C)
        return self.gatherer(self.d_fb)

    def frame0(self):
        """Frame 0 of the workload, 1 spp, as the whole image on rank 0 (host array) -- for the parity check."""
        self.scene.render_device(self.cfg(0, 1), self.d_fb, self.stream)
        full = self.gather()
        self.torch.cuda.synchronize()
        return None if full is None else full.detach().cpu().numpy().reshape(self.H, self.W, self.C)

    def allreduce(self, vals, op):
        import torch.distributed as dist
        t = self.torch.tensor(vals, dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return [float(x) for x in t]

    def measure(self, steps, warmup, do_e2e=True, sample_clocks=False):
        torch, args = self.torch, self.args
        # ---------------- value: device-resident inputs -----------------
        for s in range(warmup):
            self.step(s)
        if self.world > 1:
            self.gather()
        self.barrier()
        sampler = ClockSampler(torch.cuda.current_device()) if (sample_clocks and self.rank == 0) else None
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        ev0.record(self.stream)
        for s in range(steps):
            self.step(warmup + s, profile=1, accumulate=(s > 0))   # counters / kernel spans are read once, after the loop
            marks[s].record(self.stream)                           # per-step times for the stability record (no sync)
        last = self.gather()                                       # N > 1: the render's single NCCL gather
        ev1.record(self.stream)
        self.barrier()
        clocks = sampler.stop() if sampler else None
        # what the timed steps computed (rank 0: the whole image), copied before the legs below reuse the framebuffer
        self.last_step = last.detach().cpu().numpy().reshape(self.H, self.W, self.C) if (args.dump_outputs and last is not None) else None
        ms_local = ev0.elapsed_time(ev1)
        per_step = [(ev0 if s == 0 else marks[s - 1]).elapsed_time(marks[s]) for s in range(steps)]
        c = self.scene.counters()
        kt = self.scene.kernel_times()
        (ms,) = self.allreduce([ms_local], "max")
        rays, launches = self.allreduce([float(c.rays), float(c.kernel_launches)], "sum")
        rank_rays = self.allreduce([float(c.rays) if r == self.rank else 0.0 for r in range(self.world)], "sum")
        out = dict(value=rays / (ms * 1e-3) / 1e6, ms=ms, rays=rays, launches=launches, clocks=clocks, upload_ms=self.upload_ms, upload_again_ms=self.upload_again_ms,
                   kernel_ms={k: v[0] for k, v in kt.items()}, kernel_launches={k: v[1] for k, v in kt.items()},
                   deferred=float(c.deferred_rays), rank0_rays=float(c.rays), rank_rays=rank_rays, steps=steps,
                   step_ms={"min": min(per_step), "median": statistics.median(per_step), "max": max(per_step)},
                   samples=self.allreduce([float(c.samples)], "sum")[0])
        # ---------------- e2e: host buffers -----------------
        if do_e2e:
            host_fb = torch.zeros(max(1, self.n_local) * self.C, dtype=torch.float32).pin_memory()
            host_np = host_fb.numpy()
            full_host = torch.zeros(self.W * self.H * self.C, dtype=torch.float32).pin_memory() if (self.world > 1 and self.rank == 0) else None
            spp = args.spp_per_step

            def e2e_step(s, acc):
                # ezrt_render: H2D of this rank's lastFrame part (s > 0; it runs beside the tracing kernels), kernels, D2H of the part, sync
                self.scene.render(self.cfg(s * spp, spp, 0, acc), framebuffer=host_np)

            for s in range(warmup):
                e2e_step(s, False)
            self.barrier()
            t0 = time.perf_counter()
            for s in range(steps):
                e2e_step(warmup + s, s > 0)
            if self.world > 1:   # once per render: the parts go back to the devices, NCCL gather, the assembled image to the host on rank 0
                self.d_fb.copy_(host_fb, non_blocking=True)
                full = self.gather()
                if full is not None:
                    full_host.copy_(full.reshape(-1), non_blocking=True)
                torch.cuda.synchronize()
            self.barrier()
            e_ms_local = 1e3 * (time.perf_counter() - t0)
            (e_ms,) = self.allreduce([e_ms_local], "max")
            (e_rays,) = self.allreduce([float(self.scene.counters().rays)], "sum")
            part_bytes = self.n_local * self.C * 4
            out["e2e"] = {"value": e_rays / (e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": part_bytes, "d2h_bytes_per_step": part_bytes,
                          "d2h_bytes_once_per_render": (self.W * self.H * self.C * 4 if self.world > 1 else 0), "ms_per_step": e_ms / max(1, steps),
                          "what": "ezrt_render with pinned host framebuffers" if self.world == 1 else
                                  "per step: ezrt_render of this rank's part with pinned host buffers (H2D lastFrame part, kernels, D2H part) on every rank; "
                                  "once per render: H2D of the parts, NCCL gather, D2H of the whole image on rank 0"}
        return out

    def traversal_counts(self):
        """One step with the counting instantiation (params.profile = 2), outside every timed region: records the accel kernels
        fetch on their own layout."""
        spp = self.args.spp_per_step
        self.scene.render_device(self.cfg(self.args.warmup * spp, spp, profile=2), self.d_fb, self.stream)
        self.torch.cuda.synchronize()
        c = self.scene.counters()
        return dict(node_visits=int(c.node_visits), node_visits_96=int(c.node_visits_96), tri_tests=int(c.tri_tests), node_bytes=int(c.node_bytes),
                    tri_bytes=int(c.tri_bytes), rays=int(c.rays), primary=int(c.primary_rays), bounce=int(c.bounce_rays), shadow=int(c.shadow_rays))

    def close(self):
        self.scene.close()


def parity_of(gpu_img, cpu_img, what):
    if gpu_img is None or cpu_img is None:
        return None
    a, b = np.ascontiguousarray(gpu_img, np.float32), np.ascontiguousarray(cpu_img, np.float32)
    same_nan = np.isnan(a) == np.isnan(b)
    diff = np.abs(np.nan_to_num(a) - np.nan_to_num(b))
    differing = int((a.view(np.uint32) != b.view(np.uint32)).sum())
    return {"config": what, "linf": float(diff.max()), "differing": differing, "floats": int(a.size), "nan_positions_equal": bool(same_nan.all()),
            "tolerance": 1e-4}


def roofline_of(res, counts, wl_means, hbm_peak, peak_kind, kernel_name):
    """Roofline of the extend stage (accel kernels + their exact fallback passes, > 80 % of a step) on the kernel's OWN layout:
    achieved = bytes of node / triangle / ray records the traversal fetched per second; peak = the measured gather ceiling for
    that mix of record sizes (tools/gather_bench.cu).  HBM-side and reference-layout demand figures ride along."""
    ext_ms, ext_n = res["kernel_ms"]["extend"] + res["kernel_ms"]["shadow"], res["kernel_launches"]["extend"] + res["kernel_launches"]["shadow"]
    if not counts or ext_ms <= 0 or counts["node_visits"] == 0:
        return None
    steps = res["steps"]
    rays_step = counts["rays"]
    queue_rays = counts["bounce"] + counts["shadow"]
    n96, n128 = counts["node_visits_96"], counts["node_visits"] - counts["node_visits_96"]
    # per step (rank 0): node records + triangle records + 32-byte ray records read (queue rays) + 8-byte hit records written
    bytes_step = counts["node_bytes"] + counts["tri_bytes"] + queue_rays * 32 + rays_step * 8
    t_step = ext_ms * 1e-3 / steps
    achieved = bytes_step / t_step / 1e9
    p128, p96, p64 = gather_peak(128), gather_peak(96), gather_peak(64)
    out = {"bound": "hbm", "bound_detail": "memory system: L2 -> L1 gather of node / triangle records by divergent lanes (no dense contraction: tensor cores unused)",
           "kernel": kernel_name, "achieved": achieved, "unit": "GB/s",
           "algorithmic_bytes_per_launch": bytes_step * steps / max(1, ext_n), "launches": ext_n, "ms_per_launch": ext_ms / max(1, ext_n),
           "extend_share_of_step": ext_ms / res["ms"],
           "per_ray": {"node_records_128B": n128 / rays_step, "node_records_96B": n96 / rays_step, "triangle_records_64B": counts["tri_tests"] / rays_step,
                       "bytes": bytes_step / rays_step}}
    if p128 and p96 and p64:
        t_floor = n128 / p128 + n96 / p96 + counts["tri_tests"] / p64   # seconds per step at the measured gather ceilings
        peak = bytes_step / t_floor / 1e9 if t_floor > 0 else None
        out.update({"peak": peak, "frac": achieved / peak if peak else None,
                    "peak_source": "measured gather ceiling (profiles/gather_peak_r2.json: 128-byte records %.1f G/s, 96-byte %.1f G/s, 64-byte %.1f G/s; 256-bit loads, "
                                   "L2-resident table, this pool's B200), mixed by record counts" % (p128 / 1e9, p96 / 1e9, p64 / 1e9)})
    else:
        out.update({"peak": hbm_peak, "frac": achieved / hbm_peak, "peak_source": peak_kind + " (no gather_peak_r2.json)"})
    # HBM side: DRAM bytes of the extend kernels from the committed ncu capture of this command (tools/ncu_summaries.py dram)
    dram = load_json(os.path.join(ROOT, "profiles", "ncu_dram_r2.json"))
    traffic = None
    cls = (dram or {}).get(res.get("workload", ""), {})
    if "extend" in cls:   # mean over the accel launches of one step (extend + shadow passes)
        tot = sum(cls[k]["dram_bytes_per_launch"] * cls[k]["launches"] for k in ("extend", "shadow") if k in cls)
        cnt = sum(cls[k]["launches"] for k in ("extend", "shadow") if k in cls)
        traffic = tot / max(1, cnt)
    out["traffic"] = traffic
    out["traffic_source"] = "profiles/ncu_dram_r2.json (dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu capture of this command)" if traffic else None
    out["hbm"] = {"peak": hbm_peak, "peak_source": peak_kind, "achieved_gbs": (traffic / (ext_ms * 1e-3 / max(1, ext_n)) / 1e9) if traffic else None}
    if out["hbm"]["achieved_gbs"]:
        out["hbm"]["frac"] = out["hbm"]["achieved_gbs"] / hbm_peak
    if wl_means:   # SURVEY 8(d)'s demand figure on the REFERENCE layout and policy (48 N_node + 72 N_tri + 72 H + 24 per ray), for continuity
        demand = res["rank0_rays"] * wl_means["bytes_per_ray_reference"] / (ext_ms * 1e-3) / 1e9
        out["demand"] = {"gbs": demand, "frac_of_hbm_peak": demand / hbm_peak, "bytes_per_ray_reference_layout": wl_means["bytes_per_ray_reference"],
                         "ray_means": wl_means, "note": "demand bytes of the reference's layout and un-pruned traversal with no cross-ray reuse; "
                                                        "the kernels walk their own 4-wide tree (or the 8-wide one under EZRT_ACCEL=8), so this exceeds every physical peak by design"}
    return out


def b_ray(c):
    """Algorithmic bytes per ray on the reference layout (SURVEY.md 8d): 48 N_node + 72 N_tri + 72 H + 24."""
    return (48.0 * c["n_node"] + 72.0 * c["n_tri"] + 72.0 * c["hits"]) / c["rays"] + 24.0


def measure_workload(args, name, rank, world, local_rank, steps, warmup, headline):
    """Build, measure, check one workload.  Returns (result dict for the JSON line, Runner-independent extras)."""
    wl = build_workload(name, device_cache=True)
    W, H, scaling = image_for(args, wl, world)
    runner = Runner(args, wl, rank, world, local_rank, W, H)
    res = runner.measure(steps, warmup, do_e2e=not args.no_e2e, sample_clocks=headline)
    res["workload"] = name
    counts = runner.traversal_counts() if args.traverse == "accel" and args.pipeline == "wavefront" else None
    gpu0 = None if args.no_parity else runner.frame0()
    runner.close()
    out = {"config": workload_config(args, wl, W, H, world, scaling), "res": res, "counts": counts, "scaling": scaling, "wl": wl, "W": W, "H": H,
           "last_step": runner.last_step}
    if rank != 0:
        return out
    cpu_base = parity = means = None
    if not args.no_cpu_baseline:
        threads, tinfo = cpu_threads()
        cpu_base, first, (sw, sh, sspp) = cpu_baseline_leg(args, wl, W, H, threads, tinfo)
        c = first["counters"]
        means = {"n_node": c["n_node"] / c["rays"], "n_tri": c["n_tri"] / c["rays"], "hit_frac": c["hits"] / c["rays"], "bytes_per_ray_reference": b_ray(c)}
        if gpu0 is not None and (sw, sh, sspp) == (W, H, 1):
            parity = parity_of(gpu0, first["image"], "%s: frame 0 (1 spp) of the whole %dx%d image on %d GPU(s) vs the CPU %s render of the same frame" %
                               (name, W, H, world, "reference-shader" if first["kind"] == "reference" else "oracle"))
    out.update(cpu_baseline=cpu_base, parity=parity, means=means)
    return out


DUMP_BYTES = 64 * 10**6


def dump_outputs(directory, arrays):
    """--dump-outputs: every array as <directory>/<name>.npy in float32.  When they exceed 64 MB together, each is cut to the same
    fraction of its elements, chosen by a fixed seed, so that runs with the same arguments stay comparable element for element."""
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    frac = min(1.0, (DUMP_BYTES - 256 * len(arrays)) / max(1, sum(a.nbytes for a in arrays.values())))   # 256: room for each .npy header
    for name, a in arrays.items():
        if frac < 1.0:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, int(a.size * frac), replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def main():
    args = parse_args()
    quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload is None:
        args.workload = "c3"   # every N measures the same scene and integrator; `--workload c4` gives configs[4] with the IS/MIS integrator
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    head = measure_workload(args, args.workload, rank, world, local_rank, args.steps, args.warmup, headline=True)
    extras = {}
    names = args.extra_workloads
    if names is None:
        names = "c2,c4" if (world == 1 and args.workload == "c3") else ""
    for nm in [x for x in names.split(",") if x]:
        extras[nm] = measure_workload(args, nm, rank, world, local_rank, args.extra_steps, args.warmup, headline=False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_json(os.path.join(ROOT, "MEASURED_PEAKS.json")) or {}
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured copy bandwidth (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    kname = {"accel": "k_extend_accel (+ k_shadow_accel)", "pruned": "k_extend<PRUNE>", "reference": "k_extend"}[args.traverse]

    def pack(m):
        res = m["res"]
        d = {"value": res["value"], "unit": UNIT, "ms_per_step": res["ms"] / max(1, res["steps"]), "steps": res["steps"], "rays_per_step": res["rays"] / max(1, res["steps"]),
             "e2e": res.get("e2e"), "gpu_launches": int(res["launches"]), "kernel_ms": res["kernel_ms"], "step_ms_rank0": res["step_ms"], "deferred_ray_fraction": res["deferred"] / max(1.0, res["rank0_rays"]),
             "parity": m.get("parity"), "cpu_baseline": m.get("cpu_baseline"),
             "roofline": roofline_of(res, m["counts"], m.get("means"), hbm_peak, peak_kind, kname),
             "setup": {"scene_build_s": round(m["wl"]["build_s"], 2), "scene_upload_ms": round(res["upload_ms"], 1), "scene_upload_again_ms": round(res["upload_again_ms"], 1),
                       "what": "scene_build_s: synthetic scene + the reference's CPU BVH build (host, outside the product); scene_upload_ms: ezrt_scene_create "
                               "(upload, GPU build of the acceleration tree, repack) as first called in this process; _again: the same call repeated"}}
        if world > 1:
            rr = res["rank_rays"]
            d["rank_rays"] = {"per_rank": rr, "max_over_mean": max(rr) / (sum(rr) / len(rr)) if sum(rr) > 0 else None}
        return d

    h = pack(head)
    line = {
        "metric": METRIC, "value": h["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": head["scaling"], "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": head["config"],
        "rays_per_step": h["rays_per_step"], "e2e": h["e2e"], "gpu_launches": h["gpu_launches"], "clocks": head["res"]["clocks"],
        "kernel_ms": h["kernel_ms"], "step_ms_rank0": h["step_ms_rank0"], "parity": h["parity"], "roofline": h["roofline"], "cpu_baseline": h["cpu_baseline"],
        "deferred_ray_fraction": h["deferred_ray_fraction"], "setup": h["setup"],
        "run": {"traverse": args.traverse, "pipeline": args.pipeline,
                "gather": "none (1 GPU)" if world == 1 else "one NCCL gather of the compact per-rank framebuffers per render, after the K timed steps, inside the timed region"},
    }
    if world > 1:
        line["rank_rays"] = h["rank_rays"]
    if extras:
        line["workloads"] = {}
        for nm, m in extras.items():
            d = pack(m)
            d["config"] = m["config"]
            line["workloads"][nm] = d
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {m["res"]["workload"]: m["last_step"] for m in [head] + list(extras.values())})
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
