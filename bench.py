#!/usr/bin/env python
"""bench.py — Msamples/s of the VCM hot path on BASELINE.json's headline config (C3: the 1M-triangle spectral room at 1920x1080, the config the
north-star targets are quoted on; --workload C1|C2|C4|C5 select the other configs), one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W            # the CUDA module (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU VCM (oracle/_ref, all host threads), rank 0 only

A step = one VCM iteration (light pass + photon grid + camera pass + film update) over the whole frame of the workload:
W*H samples, one sample = one light subpath + one camera subpath with all connections and merges (SURVEY.md §8(d)).
metric value = W*H*K / device-time / 1e6 with the scene resident in HBM; e2e = the same through the public API (GPUVCM.update())
with the options pushed from the host and the float4 Result film read back to pinned host memory inside the timed region, every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Msamples/s (paths*spp/s) VCM"
UNIT = "Msamples/s"


def workload(args):
    from etx_tracer_b200 import scenes
    if args.workload == "C2":
        sd = scenes.cornell_box(args.res or 1024, args.res or 1024, samples=256, spectral=True, sphere=True)
        desc = "C2: Cornell box + dielectric sphere (20480 tris), spectral, %dx%d, full VCM (merging on)" % (sd.width, sd.height)
    elif args.workload == "C1":
        sd = scenes.cornell_box(args.res or 512, args.res or 512, samples=16, spectral=False)
        desc = "C1: Cornell box diffuse, RGB, %dx%d" % (sd.width, sd.height)
    elif args.workload == "C3":
        w, h = (args.res, args.res * 9 // 16) if args.res else (1920, 1080)
        sd = scenes.procedural_room(w, h, samples=1024, spectral=True)
        desc = "C3: %d-triangle procedural room (plastic/conductor/thin-film + env map), spectral, %dx%d, full VCM" % (sd.triangle_count, sd.width, sd.height)
    elif args.workload == "C4":
        sd = scenes.sss_dragon(args.res or 1024, args.res or 1024, samples=512, spectral=True)
        desc = "C4: %d-triangle displaced mesh, plastic + random-walk subsurface, 3 area emitters, spectral, %dx%d, full VCM" % (sd.triangle_count, sd.width, sd.height)
    elif args.workload == "C5":
        sd = scenes.cloud_box(args.res or 1024, args.res or 1024, samples=256, spectral=True, grid=256)
        desc = "C5: heterogeneous cloud (256^3 density grid) in a Boundary cube, sun + sky, spectral, %dx%d, VCM connect-only (volumetric BDPT)" % (sd.width, sd.height)
    else:
        raise SystemExit(f"unknown workload {args.workload}")
    return sd, desc


def workload_vcm_options(args):
    """Integrator options of the workload: the VCMOptions defaults (vcm_shared.cxx:6-28), C5 with merging off (= volumetric BDPT)."""
    from etx_tracer_b200 import structs as S
    opts = S.default_vcm_options()
    if args.workload == "C5":
        opts["options"] = S.VCM_CONNECT_ONLY
    return opts


def scene_factory(args, res):
    """The bench workload's scene at a reduced film size (CPU baseline samples)."""
    from etx_tracer_b200 import scenes
    if args.workload == "C2":
        return scenes.cornell_box(res, res, samples=256, spectral=True, sphere=True)
    if args.workload == "C3":
        return scenes.procedural_room(res, max(16, res * 9 // 16), samples=1024, spectral=True)
    if args.workload == "C4":
        return scenes.sss_dragon(res, res, samples=512, spectral=True)
    if args.workload == "C5":
        return scenes.cloud_box(res, res, samples=256, spectral=True, grid=256)
    return scenes.cornell_box(res, res, samples=16, spectral=False)


class ClockSampler:
    """SM clock + throttle reasons of this rank's GPU during the timed region (B200_PROFILING.md).  Read through NVML in-process (what nvidia-smi itself
    reads): the library is initialised when the sampler is CONSTRUCTED — before the warm-up, outside every timed region — and a sample is four cheap calls
    on one device; no child process starts inside a timed region that is only 0.3 s long at N = 8.  `nvidia-smi -lms 100` is the fallback."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index, self.handle, self.nvml, self.running = [], None, index, None, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)
            self.nvml, self.handle = pynvml, handle
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        try:
            reasons = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            try:
                reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            except Exception:
                reasons = 0
        flags = []
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            flags.append("Active" if (reasons & bit) else "Not Active")
        flags = [flags[0], flags[3], flags[2], flags[1]]  # the order of the nvidia-smi query below
        def safe(fn, default):
            try:
                return fn()
            except Exception:
                return default
        return [str(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)), str(safe(lambda: n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM), 0)),
                str(safe(lambda: n.nvmlDeviceGetPowerUsage(h) / 1000.0, 0.0))] + flags

    def _poll(self):
        while self.running:
            try:
                self.rows.append(self._sample_nvml())
            except Exception:
                pass
            time.sleep(0.025)

    def start(self):
        if self.nvml is not None:
            self.running = True
            threading.Thread(target=self._poll, daemon=True).start()
            return
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        self.running = False
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for r in list(self.rows):
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if (self.nvml is not None) and not sm:  # never leave the line without a clocks reading: one direct query after the region
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
                a, b = [float(x) for x in out.strip().split(",")[:2]]
                sm, mx = [a], b
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvml (in-process)" if self.nvml is not None else "nvidia-smi -lms 100"}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def oracle_built():
    from oracle import oracle_py
    return oracle_py.available("native") or oracle_py.available("parity")


DUMP_LIMIT = 64 << 20


def dump_outputs(directory, arrays):
    """Each array as float32 DIR/<name>.npy.  Past DUMP_LIMIT bytes in all, every s-th element of each (flattened) array is kept instead, the same
    elements on every run, so that two builds can still be compared output for output."""
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.asarray(v, np.float32) for k, v in arrays.items()}
    stride = -(-sum(a.nbytes for a in arrays.values()) // DUMP_LIMIT)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a if stride == 1 else np.ascontiguousarray(a.reshape(-1)[::stride]))


def bvh_bytes(nodes, tris):
    """SURVEY.md 8(d): 64 B per BVH node visited + 48 B per triangle tested."""
    return 64 * nodes + 48 * tris


def algorithmic_bytes(counters, n_pixels, steps):
    """SURVEY.md 8(d): device event counters x fixed byte costs (reference struct sizes), BVH node/triangle traffic excluded here (those
    counters exist only in the ETXB_COUNT_TRAVERSAL build, which main() runs for one extra pass: `roofline.bvh`).
    Returns (whole-step bytes, {kernel name: the bytes of ITS units})."""
    c = counters
    bl, bc, lv = c["bounces_light"], c["bounces_camera"], c["light_vertices"]
    merge = 128 * c["merge_queries"] + 12 * c["merge_candidates"] + 48 * c["merge_accepts"]
    per_kernel = {
        "trace_closest(light)": 48 * bl,                       # ray in (32 B) + hit record out (16 B)
        "trace_closest(camera)": 48 * bc,
        "light_bounce": (352 + 404) * bl + 112 * lv + 24 * c["splats"] + 48 * lv + 20 * n_pixels * steps,  # state RMW + hit geometry/material + vertex store + splat + its shadow ray
        "camera_shade": (352 + 404) * bc,                      # state RMW + hit geometry/material (connections and shadow rays are their own stages)
        "camera_connect": (112 + 404) * c["connections"],      # light vertex + its geometry/material per vertex connection
        "shadow_trace": 48 * max(c["rays_shadow"] - lv, 0),    # camera-side segments
        "camera_merge": merge,
        "camera_merge_generic": merge,
        "camera_continue": 352 * bc + 104 * n_pixels * steps,  # state RMW + film accumulate
        "lv_reorder": 2 * 112 * lv,
        "grid_build": (60 + 8) * lv,
    }
    total = (per_kernel["trace_closest(light)"] + per_kernel["trace_closest(camera)"] + per_kernel["light_bounce"] + per_kernel["camera_shade"] + per_kernel["camera_connect"]
             + per_kernel["shadow_trace"] + merge + per_kernel["camera_continue"] + per_kernel["lv_reorder"] + per_kernel["grid_build"])
    return total, per_kernel


def cpu_baseline_run(sd_factory, budget_s, threads, opts=None):
    """Times the reference's CPU VCM (oracle/_ref) on a bounded sample: same scene, resolution reduced until one iteration fits the budget."""
    from oracle import oracle_py
    flavor = "native"
    try:
        oracle_py.load(flavor)
    except OSError:
        flavor = "parity"
    probe = sd_factory(64)
    o = oracle_py.Oracle(probe, flavor)
    if opts is not None:
        o.set_options(opts)
    o.begin(0)
    t0 = time.time()
    o.run(1, threads=threads)
    rate = probe.width * probe.height / max(time.time() - t0, 1e-6)  # samples/s
    o.close()
    res = int(min(1024, max(64, (rate * budget_s * (probe.width / probe.height)) ** 0.5)) // 32 * 32)
    sd = sd_factory(res)
    o = oracle_py.Oracle(sd, flavor)
    if opts is not None:
        o.set_options(opts)
    o.begin(0)
    t0 = time.time()
    total = o.run(1, threads=threads)
    wall = time.time() - t0
    o.close()
    n = sd.width * sd.height
    return {"value": n / total / 1e6, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"1 VCM iteration of the same scene at {sd.width}x{sd.height} ({n} samples, {wall:.1f} s) by oracle/_ref/liboracle_{flavor}.so "
                      f"(reference headers compiled in place + our BVH instead of Embree)"}, flavor


def path_tracer_line(sd, device, iterations=8, cpu_iterations=1):
    """The second device integrator (SURVEY 8(f) N3: CPUPathTracing's algorithm) on the same workload, one iteration in flight, next to the reference's CPU
    path tracer (run_path_iteration compiled from the reference + the restated driver) on the host threads.  An extra key of the line, never its `value`."""
    from etx_tracer_b200 import structs as S
    from etx_tracer_b200.api import GPUPathTracing
    g = GPUPathTracing(sd, flavor="fast", device=device, profile=True)
    g.set_scene_settings(0.0, 0.0)  # no pixel converges: a sample = one pixel-iteration
    g.render(2)
    st = g.render(iterations, first_iteration=2)
    n = sd.width * sd.height
    out = {"metric": "Msamples/s (pixels*spp/s), unidirectional path tracer", "value": n * iterations / st["total_time"] / 1e6, "unit": UNIT, "iterations": iterations,
           "ms_per_iteration": 1e3 * st["total_time"] / iterations, "in_flight": 1,
           "kernel_ms_per_iteration (one in flight)": {k: round(v[0] / iterations, 3) for k, v in sorted(g.kernel_times().items(), key=lambda kv: -kv[1][0]) if v[1]},
           "rays_per_iteration": int((g.counters()["rays_closest"] + g.counters()["rays_shadow"]) / iterations)}
    g.close()
    # the throughput form, like the headline `value`: four iterations in flight (etxb_group lanes; adaptive sampling off)
    from etx_tracer_b200.api import GPUVCMGroup
    grp = GPUVCMGroup(sd, lanes=4, flavor="fast", device=device)
    grp.set_integrator(S.INTEGRATOR_PT)
    grp.render(4)
    grp.run(4)
    k = max(iterations, 12)
    grp.enqueue(k)
    grp.wait()
    st4 = grp.status()
    grp.close()
    out["one_in_flight"] = out["value"]
    out["value"] = n * k / st4["total_time"] / 1e6
    out["in_flight"] = 4
    out["ms_per_iteration"] = 1e3 * st4["total_time"] / k
    if cpu_iterations > 0:
        from oracle import oracle_py
        flavor = "native" if oracle_py.available("native") else "parity"
        o = oracle_py.Oracle(sd, flavor)
        o.set_integrator(S.INTEGRATOR_PT)
        o.pt_set_options(S.default_pt_options())
        o.set_scene_settings(0.0, 0.0)
        o.begin(2)
        threads = os.cpu_count() or 1
        t = o.run(cpu_iterations, threads=threads)
        o.close()
        out["cpu_baseline"] = {"value": n * cpu_iterations / t / 1e6, "unit": UNIT, "cores": threads, "kind": "reference",
                               "sample": f"{cpu_iterations} iteration(s) of the same scene and film ({t:.1f} s) by oracle/_ref/liboracle_{flavor}.so (run_path_iteration "
                                         f"compiled from the reference, our BVH instead of Embree)"}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from etx_tracer_b200 import scenes
    threads = os.cpu_count() or 1
    def factory(res):
        return scene_factory(args, res)
    from oracle import oracle_py
    flavor = "native"
    try:
        oracle_py.load(flavor)
    except OSError:
        flavor = "parity"
    opts = workload_vcm_options(args)
    probe = oracle_py.Oracle(factory(64), flavor)
    probe.set_options(opts)
    probe.begin(0)
    t0 = time.time()
    probe.run(1, threads=threads)
    rate = probe.width * probe.height / max(time.time() - t0, 1e-6)
    probe.close()
    # same film as the GPU arm when one iteration of it fits the per-step budget (the whole --steps/--warmup run must end within minutes),
    # else the largest film that does
    sd_full, _ = workload(args)
    per_step = max(2.0, min(20.0, 150.0 / max(args.steps + args.warmup, 1)))
    aspect = sd_full.height / sd_full.width
    res = int(min(sd_full.width, max(64, (rate * per_step / aspect) ** 0.5)) // 32 * 32)
    sd = sd_full if res >= sd_full.width // 32 * 32 else factory(res)
    res_n = sd.width * sd.height
    o = oracle_py.Oracle(sd, flavor)
    o.set_options(opts)
    o.begin(0)
    o.run(args.warmup, threads=threads)
    t0 = time.time()
    before = o.run(0, threads=threads)
    total = o.run(args.steps, threads=threads) - before
    wall = time.time() - t0
    value = res_n * args.steps / total / 1e6
    _, desc = workload(args)
    res = f"{sd.width}x{sd.height}"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "sample": f"each step = 1 VCM iteration of the same scene at {res} on {threads} host threads (pixel grains of 256 handed out dynamically, like the reference's task scheduler)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                             "sample": f"{args.steps} iterations at {res}, liboracle_{flavor}.so (reference headers + our BVH instead of Embree), wall {wall:.1f} s"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--res", type=int, default=0, help="override the film size (debug only; the default is the config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-split-leftover", action="store_true", help="iteration mode: deal the K %% N left-over iterations whole instead of splitting each by camera tile over N / (K %% N) ranks (A/B switch)")
    ap.add_argument("--no-path-tracer", action="store_true", help="skip the extra `path_tracer` key (the second device integrator on the same workload, N = 1 only)")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed path computed (the Result film after its last step) to DIR/<name>.npy")
    ap.add_argument("--lanes", type=int, default=4, help="iterations in flight per GPU (etxb_group); 1 = the plain one-context pump")
    ap.add_argument("--parallelism", default="both", choices=["both", "tile", "iteration"],
                    help="N > 1: how the job's K iterations are spread over the GPUs.  'tile' (the north star's mode) = every iteration split by pixel tile "
                         "inside the module (NCCL all-reduce / all-gather per iteration); 'iteration' = the K iterations dealt to the ranks (one NCCL "
                         "film reduce per frame); 'both' (default) measures the two on the same index set and reports the faster as `value`, both under `modes`")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from etx_tracer_b200 import structs as S
    from etx_tracer_b200.api import GPUVCM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the module has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    json_fd = None
    if world > 1:
        # stdout carries ONE JSON line.  NCCL prints its version banner on stdout (NCCL_DEBUG=VERSION|WARN ignore NCCL_DEBUG_FILE), so for the
        # whole multi-rank run file descriptor 1 points at stderr and rank 0 writes the JSON line to the saved descriptor
        sys.stdout.flush()
        json_fd = os.dup(1)
        os.dup2(2, 1)
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sd, desc = workload(args)
    n_pixels = sd.width * sd.height
    from etx_tracer_b200.api import GPUVCMGroup, comm_unique_ids
    lanes = max(1, min(args.lanes, 8))
    device = torch.device("cuda", local_rank)

    def sync_all():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def measure(mode):
        """One way of running the SAME job — the K whole-frame iterations with indices W .. W+K-1 — on `world` GPUs:
          single     one GPU, `lanes` iterations in flight
          tile       (north star) every iteration split by 32x32 pixel tile over the ranks INSIDE the module: per iteration ncclAllReduce of the light
                     image + all-gather of the photon records, per frame ncclReduce of the film (etxb_group_comm_init); `lanes` iterations in flight
          iteration  the K iterations dealt to the ranks (index j on rank j % world), no collective inside an iteration, one count-weighted
                     ncclReduce of the films per frame (etxb_group_comm_init_replicas)
        Strong scaling in every mode: a step = one whole-frame iteration of the job, value = W*H*K / time (max over ranks)."""
        from etx_tracer_b200.multigpu import distribute_comm_ids
        # tile mode: two iterations in flight per GPU (measured at N = 2: 30.7 Msamples/s with 2, 15.1 with 4 — every lane has two rendezvous with
        # its peers per iteration, and four lanes' collectives wait on each other across the ranks)
        mode_lanes = min(lanes, 2) if mode == "tile" else lanes
        # iteration mode: one more lane, reserved for camera-split iterations (the remainder when K is not a multiple of the GPUs).  Measured at N = 8,
        # K = 20 (profiles/r2o_*, r2p_*, r2q_*): the left-over 4 iterations dealt whole (3, 3, 3, 3, 2, 2, 2, 2) 158 / 156 Msamples/s (value / e2e); each of
        # them split over two ranks 174 end to end, but 150 in the `value` region of those runs — the region in which the split lane rendered its FIRST
        # iteration (it created its few thousand timing events there).  The events now exist from etxb_create, and the warm-up below exercises the split
        # lane on the same left-over geometry.  --no-split-leftover is the A/B switch.
        split = (mode == "iteration") and not args.no_split_leftover
        g = GPUVCMGroup(sd, lanes=mode_lanes + (1 if split else 0), flavor="fast", device=local_rank, profile=True)
        if mode == "tile":
            g.comm_init(world, rank, distribute_comm_ids(dist, rank, mode_lanes + 1, comm_unique_ids, device=device))
        elif mode == "iteration":
            g.comm_init_replicas(world, rank, distribute_comm_ids(dist, rank, 1, comm_unique_ids, device=device), split_lane=split)
        g.options[:] = workload_vcm_options(args)
        multi = mode != "single"
        warm = args.warmup * (world if mode == "iteration" else 1)  # every rank warms up on `warmup` iterations of its own
        if split:
            warm += args.steps % world  # ... and the camera-split lane on the left-over geometry it will render in the timed region

        def film_to_host(out):
            if multi:
                g.comm_reduce_film(S.FILM_RESULT, out=out)  # collective: ncclReduce to rank 0, then device -> host there
            else:
                g.film(S.FILM_RESULT, out=out)

        clocks = ClockSampler(local_rank) if rank == 0 else None  # NVML is initialised here, outside every timed region
        # ---- device-resident timing: warm-up on indices 0.., then the timed index set W .. W+K-1 from a cleared film
        g.run(0)
        g.enqueue(warm)
        g.wait()
        sync_all()
        g.run(args.warmup)
        c0, k0 = g.counters(), g.kernel_times()
        if rank == 0:
            clocks.start()
        g.enqueue(args.steps)
        g.wait()
        sync_all()
        clk = clocks.stop() if rank == 0 else None
        st1, c1, k1 = g.status(), g.counters(), g.kernel_times()
        # several iterations in flight: the streams overlap, so the module reports the span from the first enqueue (every lane idle and synchronised)
        # to the last lane's end-of-iteration synchronise; max over ranks
        elapsed = all_max(st1["total_time"])
        counters = {k: c1[k] - c0[k] for k in c1}
        if multi:  # every rank counted its own share
            keys = sorted(counters)
            t = torch.tensor([float(counters[k]) for k in keys], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            counters = {k: int(v) for k, v in zip(keys, t.tolist())}
        ktimes = {k: (k1[k][0] - k0[k][0], k1[k][1] - k0[k][1]) for k in k1}
        mine = max(1, sum(1 for j in range(args.steps) if (mode != "iteration") or (j % world == rank)))
        comm_ms = {k: round(v[0] / mine, 3) for k, v in ktimes.items() if k.startswith("nccl_")}

        # ---- end to end through the public API, host buffers inside the timed region: the K iterations are queued by the first step (the call a
        # user makes), every step pushes the options host -> module and brings the current frame (mean over the iterations finished so far) device ->
        # pinned host; the region ends when every queued iteration has finished and the final frame is on the host
        pinned = torch.empty((sd.height, sd.width, 4), dtype=torch.float32).pin_memory()
        host_film = pinned.numpy()
        g.run(0)
        g.enqueue(warm)
        g.wait()
        sync_all()
        g.run(args.warmup)
        film_to_host(host_film)  # untimed: the first collective on a communicator sets up its NVLink channels (hundreds of ms with 8 ranks)
        sync_all()
        t0 = time.time()
        film_reads = 0
        for step in range(args.steps):
            g.set_options()
            if step == 0:
                g.enqueue(args.steps)  # the call a user makes: render K iterations; the frame is then read once per step while they run
            film_to_host(host_film)
            film_reads += 1
        g.wait()
        film_to_host(host_film)
        film_reads += 1
        sync_all()
        e2e_s = all_max(time.time() - t0)
        finite = bool(np.isfinite(host_film).all()) if rank == 0 else True
        light_vertices = st1["light_vertices"]
        g.close()
        return {"mode": mode, "value": n_pixels * args.steps / elapsed / 1e6, "elapsed": elapsed, "counters": counters, "clocks": clk,
                "lanes": mode_lanes, "film": host_film.copy() if (args.dump_outputs and rank == 0) else None,
                "e2e": {"value": n_pixels * args.steps / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(g.options.nbytes) * mode_lanes,
                        "d2h_bytes_per_step": int(host_film.nbytes * film_reads / args.steps)},
                "collective_ms_per_iteration": comm_ms or None, "film_finite": finite, "light_vertices": light_vertices}

    if world == 1:
        results = [measure("single")]
    elif args.parallelism == "both":
        results = [measure("tile"), measure("iteration")]
    else:
        results = [measure(args.parallelism)]
    best = max(results, key=lambda r: r["value"])
    tile_mode = best["mode"] == "tile"
    value, elapsed, counters, e2e, clk = best["value"], best["elapsed"], best["counters"], best["e2e"], best["clocks"]
    st1 = {"light_vertices": best["light_vertices"]}

    if rank == 0:
        peaks = measured_peaks()
        peak = peaks["hbm_gbs"] if peaks else 6650.0
        total_bytes, _ = algorithmic_bytes(counters, n_pixels, args.steps)
        # per-kernel numbers come from a pass of their own: ONE iteration at a time on one context, so that the CUDA events around a launch
        # bracket that kernel alone (with several iterations in flight the streams overlap and every bracket also holds other lanes' work)
        kt_steps = max(2, min(args.steps, 6))
        single = GPUVCM(sd, flavor="fast", device=local_rank, profile=True)
        single.options[:] = workload_vcm_options(args)
        single.run(0)
        for _ in range(2):
            single.iterate()
        single._check(single.lib.etxb_wait(single.h))
        kc0, kk0 = single.counters(), single.kernel_times()
        for _ in range(kt_steps):
            single.iterate()
        single._check(single.lib.etxb_wait(single.h))
        kc1, kk1 = single.counters(), single.kernel_times()
        single.close()
        kcounters = {k: kc1[k] - kc0[k] for k in kc1}
        ktimes = {k: (kk1[k][0] - kk0[k][0], kk1[k][1] - kk0[k][1]) for k in kk1}
        _, kbytes = algorithmic_bytes(kcounters, n_pixels, kt_steps)
        if ktimes.get("camera_merge", (0, 0))[0] and ktimes.get("camera_merge_generic", (0, 0))[0]:
            # two gather kernels share the merge counters: split the bytes by their time
            tm, tg = ktimes["camera_merge"][0], ktimes["camera_merge_generic"][0]
            kbytes["camera_merge"], kbytes["camera_merge_generic"] = kbytes["camera_merge"] * tm / (tm + tg), kbytes["camera_merge_generic"] * tg / (tm + tg)
        # SURVEY 8(d) asks for the fractions with AND without the BVH term: one iteration (the first timed index) through the counting build
        bvh = None
        try:
            cnt = GPUVCM(sd, flavor="count", device=local_rank)
            cnt.options[:] = workload_vcm_options(args)
            cnt.run(args.warmup)
            cnt.iterate()
            cnt._check(cnt.lib.etxb_wait(cnt.h))
            cc = cnt.counters()
            cnt.close()
            it_bvh = bvh_bytes(cc["nodes_visited"], cc["tris_tested"])
            it_bvh_closest = bvh_bytes(cc["nodes_closest"], cc["tris_closest"])
            trace_ms = (ktimes.get("trace_closest(light)", (0, 0))[0] + ktimes.get("trace_closest(camera)", (0, 0))[0]) / kt_steps
            trace_bytes = (kbytes["trace_closest(light)"] + kbytes["trace_closest(camera)"]) / kt_steps
            bvh = {"n_node_per_iteration": int(cc["nodes_visited"]), "n_tri_per_iteration": int(cc["tris_tested"]),
                   "n_node_closest_hit_kernel": int(cc["nodes_closest"]), "n_tri_closest_hit_kernel": int(cc["tris_closest"]),
                   "rays_per_iteration": int(cc["rays_closest"] + cc["rays_shadow"]),
                   "nodes_per_ray": cc["nodes_visited"] / max(cc["rays_closest"] + cc["rays_shadow"], 1),
                   "tris_per_ray": cc["tris_tested"] / max(cc["rays_closest"] + cc["rays_shadow"], 1),
                   "bytes_per_iteration": int(it_bvh),
                   "step_algorithmic_GBps_without_bvh": total_bytes / elapsed / 1e9,
                   "step_algorithmic_GBps_with_bvh": (total_bytes + it_bvh * args.steps) / elapsed / 1e9,
                   "trace_closest_GBps_without_bvh": trace_bytes / max(trace_ms * 1e-3, 1e-12) / 1e9,
                   "trace_closest_GBps_with_bvh": (trace_bytes + it_bvh_closest) / max(trace_ms * 1e-3, 1e-12) / 1e9}
            # the traversal kernels' own algorithmic bytes include the nodes and triangles their rays touch (64 B / 48 B each); the ratio of the two
            # closest-hit kernels' ray counts splits the closest-hit term, the rest (shadow segments) goes to the shadow kernel
            rc_l, rc_c = kcounters["bounces_light"], kcounters["bounces_camera"]
            share_l = rc_l / max(rc_l + rc_c, 1)
            kbytes["trace_closest(light)"] += it_bvh_closest * kt_steps * share_l
            kbytes["trace_closest(camera)"] += it_bvh_closest * kt_steps * (1.0 - share_l)
            if ktimes.get("shadow_trace", (0, 0))[0] > 0:
                kbytes["shadow_trace"] += max(it_bvh - it_bvh_closest, 0) * kt_steps
            bvh["step_frac_without_bvh"] = bvh["step_algorithmic_GBps_without_bvh"] / peak
            bvh["step_frac_with_bvh"] = bvh["step_algorithmic_GBps_with_bvh"] / peak
            bvh["trace_closest_frac_with_bvh"] = bvh["trace_closest_GBps_with_bvh"] / peak
        except Exception as e:  # the counting build is an extra; the headline does not depend on it
            bvh = {"unavailable": str(e)[:200]}
        dominant = max(ktimes, key=lambda k: ktimes[k][0])
        dom_ms, dom_launches = ktimes[dominant]
        dom_bytes = kbytes.get(dominant, 0.0)
        achieved = dom_bytes / max(dom_ms * 1e-3, 1e-12) / 1e9
        # `traffic`: dram read + write of ONE head-of-pass launch of that kernel from the committed ncu --set full capture of this workload
        traffic, traffic_source = None, None
        try:
            summary = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get(args.workload, {})
            rec = summary.get(dominant) or summary.get(dominant.split("(")[0])
            if rec and (rec.get("dram_read_GB") is not None):
                traffic = (rec["dram_read_GB"] + rec["dram_write_GB"]) * 1e9
                traffic_source = f"profiles/{rec['file']} (head-of-pass launch, {rec['time_ms']:.3f} ms)"
        except Exception:
            traffic = None
        step_ms = sum(v[0] for v in ktimes.values())
        # the ceilings that actually bind (L2 bandwidth, issue slots, lanes per instruction) come from the committed ncu summaries
        ncu = None
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get(args.workload)
        except Exception:
            ncu = None
        roofline = {"bound": "hbm", "kernel": dominant, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s",
                    "bytes_per_launch": dom_bytes / max(dom_launches, 1), "launches": dom_launches, "avg_launch_ms": dom_ms / max(dom_launches, 1),
                    "kernel_share_of_step": dom_ms / max(step_ms, 1e-9),
                    "step_algorithmic_GBps": total_bytes / elapsed / 1e9,
                    "timing_pass": f"{kt_steps} iterations, one at a time on one context (events bracket single kernels); the headline value uses {lanes} iterations in flight",
                    "kernel_ms_per_iteration": {k: round(v[0] / kt_steps, 3) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0]) if v[1]},
                    "kernel_GBps": {k: round(kbytes[k] / max(ktimes[k][0] * 1e-3, 1e-12) / 1e9, 1) for k in kbytes if ktimes.get(k, (0, 0))[0] > 0},
                    "bvh": bvh, "ncu": ncu,
                    "note": "algorithmic bytes = device event counters x SURVEY.md 8(d) byte costs of the units THAT kernel processes, BVH node/triangle traffic excluded; "
                            "`traffic` = ncu dram read+write of one head-of-pass launch of the kernel (profiles/ncu_traffic.json).  The photon gather is served from L2 "
                            "(82 % hit rate) and the bounce kernels are latency / FP32 bound, so these fractions of the HBM copy peak are not DRAM utilisation"}
        cpu = None
        if not args.no_cpu_baseline and not oracle_built():
            cpu = {"unavailable": "oracle/_ref is not built (build() makes it where the reference sources exist)"}
        elif not args.no_cpu_baseline:
            from etx_tracer_b200 import scenes
            cpu, _ = cpu_baseline_run(lambda res: scene_factory(args, res), args.cpu_budget, os.cpu_count() or 1, workload_vcm_options(args))
        pt = None
        if (world == 1) and not args.no_path_tracer:
            try:
                pt = path_tracer_line(sd, local_rank, cpu_iterations=0 if (args.no_cpu_baseline or not oracle_built()) else 1)
            except Exception as e:  # an extra key must never cost the headline line
                pt = {"error": f"{type(e).__name__}: {e}"[:300]}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": desc,
                           "parallelism": {"single": f"one GPU, {lanes} iterations in flight",
                                           "tile": f"pixel tiles (32x32, round-robin) over {world} GPUs inside the module, {min(lanes, 2)} iterations in flight per GPU; per iteration "
                                                   f"ncclAllReduce of the light image + all-gather of the photon records, per frame ncclReduce of the film",
                                           "iteration": f"the job's iterations dealt to {world} GPUs (index j on rank j % {world}"
                                                        + ("; the K % N left over are split by camera tile, each part tracing the whole light pass itself" if not args.no_split_leftover else "")
                                                        + f"), {lanes} in flight per GPU; per frame one count-weighted ncclReduce of the films"}[best["mode"]],
                           "mode": best["mode"],
                           "collective": None if world == 1 else "NCCL (communicators created inside the module: etxb_group_comm_init / etxb_group_comm_init_replicas)",
                           "collective_ms_per_iteration": best["collective_ms_per_iteration"],
                           "timing": ("span from the first enqueue (all lanes idle, device synchronised) to the last lane's end-of-iteration stream synchronise, max over ranks"),
                           "l2": "inputs larger than L2 (path state + light-vertex pool + photon grid > 126 MB)",
                           "iterations": f"a fixed index set: {args.warmup} warm-up iterations (indices 0..{args.warmup - 1}), then the timed indices "
                                         f"{args.warmup}..{args.warmup + args.steps - 1} of the 1/(1 + i/256) merge-radius schedule (the most expensive end of a render)",
                           "light_vertices_per_iteration": st1["light_vertices"], "per_kernel_event_timing": True},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(counters["kernel_launches"]), "clocks": clk,
                "counters": counters, "path_tracer": pt,
                # every way of spreading the same K iterations that was measured in this run (N > 1, --parallelism both): `value` is the faster one
                "modes": {r["mode"]: {"value": r["value"], "ms_per_step": r["elapsed"] / args.steps * 1e3, "e2e": r["e2e"]["value"],
                                      "collective_ms_per_iteration": r["collective_ms_per_iteration"], "film_finite": r["film_finite"]} for r in results}}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"film_result": best["film"]})
        if json_fd is not None:
            sys.stdout.flush()
            os.write(json_fd, (json.dumps(line) + "\n").encode())
        else:
            print(json.dumps(line), flush=True)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
