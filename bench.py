#!/usr/bin/env python3
"""bench.py -- Mrays/s of the PathIntegrator hot path on N B200s (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload statue|cornell|conference|landscape|landscape-64|cornell-textured|cornell-direct|cornell-whitted|cornell-ao] [--impl reference]
    [--dump-outputs DIR]

A "step" is one full frame of the workload rendered through the wavefront kernels.  The default workload is
BASELINE.json configs[2] -- the Ganesha stand-in (4.31 M triangles, path integrator, 128 spp, 1024x1024), the largest
single-GPU configuration and the one whose BVH does not fit on chip, so that its roofline means something; configs[1]
(Cornell Box 1024x1024x256) rides along under `extra.cornell` for continuity with round 1.  For N > 1 the frame's 16x16
tiles are dealt to the ranks (scene replicated), each rank renders its tiles into a full-size device film and one NCCL
reduce(sum) merges the films on rank 0 -- total work is fixed, so scaling is "strong".
`value`   : rays (BVH traversals) of the whole frame / device time, scene and film resident in HBM.
`e2e`     : same metric through the plugin call with HOST buffers, every step: pbrt_gpu_scene_create (H2D of the
            scene) + pbrt_gpu_render into a host film (N = 1; for N > 1 the per-rank device films are reduced over
            NCCL and rank 0 copies the result to the host).
`roofline`: the dominant kernel (k_trace): algorithmic bytes (32 B/node visited + 48 B/triangle tested + 48 B/ray of
            queue traffic, DESIGN.md) / its CUDA-event time against MEASURED_PEAKS.json hbm_gbs, next to the DRAM
            traffic ncu measured for the same build, and what actually limits the kernel (`limiter`).
            `roofline_kernels` has the same for k_shade.
`cpu_baseline` / `--impl reference`: the oracle (C++ restatement of rs_pbrt's path; rs_pbrt itself cannot be
            built here: no Rust toolchain) on all host threads, on a bounded band of rows of the same frame.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

WORKLOADS = {
    # Variants of the Cornell workload for the rows of SURVEY.md section 8(f) that have not been measured yet (same frame, another
    # integrator / image textures): bench lines for them follow the same contract; the default stays BASELINE.json configs[1].
    "cornell-textured": dict(desc="Cornell Box with image textures (EWA, float textures, texture graph, bump maps), path integrator, sobol 256 spp, 1024x1024",
                             xres=1024, yres=1024, spp=256, cpu_rows=64, kw=dict(textures="ewa+float+graph+bump")),
    "cornell-direct": dict(desc="Cornell Box (glass / metal / plastic blocks), directlighting integrator strategy all, sobol 256 spp, 1024x1024",
                           xres=1024, yres=1024, spp=256, cpu_rows=64, kw=dict(integrator=("direct", "all"), materials="mixed")),
    "cornell-whitted": dict(desc="Cornell Box (glass / metal / plastic blocks), whitted integrator, sobol 256 spp, 1024x1024",
                            xres=1024, yres=1024, spp=256, cpu_rows=64, kw=dict(integrator="whitted", materials="mixed")),
    "cornell-ao": dict(desc="Cornell Box, ao integrator 16 samples, sobol 64 spp, 1024x1024", xres=1024, yres=1024, spp=64, cpu_rows=64,
                       kw=dict(integrator=("ao", 16, True))),
    # BASELINE.json configs[1]
    "cornell": dict(desc="Cornell Box, path integrator (maxdepth 5, spatial lights), sobol 256 spp, 1024x1024", xres=1024, yres=1024, spp=256,
                    cpu_rows=128),
    # BASELINE.json configs[2]
    "statue": dict(desc="Ganesha stand-in (4.31M triangles), path integrator, sobol 128 spp, 1024x1024", xres=1024, yres=1024, spp=128,
                   cpu_rows=128),
    # BASELINE.json configs[3] (quoted on 4 GPUs; fits one)
    "conference": dict(desc="Conference stand-in (0.3M triangles, 7 material kinds, 128 area lights), path integrator, sobol 512 spp, 1280x720",
                       xres=1280, yres=720, spp=512, cpu_rows=2),
    # BASELINE.json configs[4] (quoted on 8 GPUs) at its configured shape: ~3 k instances of 20 prototype plants on a terrain, distant + infinite
    # light, 1024 spp at 1920x1080 (SURVEY.md 8d item 4).  "landscape-64" is the same scene at 64 spp for quick single-GPU lines.
    "landscape": dict(desc="Landscape stand-in (131k-triangle terrain, 3000 instances of 20 plant prototypes, distant + infinite light, instancing=fixed), "
                           "path integrator, sobol 1024 spp, 1920x1080", xres=1920, yres=1080, spp=1024, cpu_rows=1),
    "landscape-64": dict(desc="Landscape stand-in (131k-triangle terrain, 3000 instances of 20 plant prototypes, distant + infinite light, instancing=fixed), "
                              "path integrator, sobol 64 spp, 1920x1080", xres=1920, yres=1080, spp=64, cpu_rows=16),
}



def host_cores():
    """Cores this process may actually use: the affinity mask, capped by the cgroup CPU quota (a container that reports 128
    logical CPUs may be allowed 16) -- so that `cores` in cpu_baseline is the parallelism really available, and the CPU leg
    is not oversubscribed."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            quota, period = open(path).read().split()[:2]
            if quota != "max":
                n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
        except (OSError, ValueError):
            pass
    try:  # cgroup v1
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and per > 0:
            n = min(n, max(1, int(q / per + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, n)

def make_scene(name, small=False):
    from rs_pbrt_b200 import scenes

    w = WORKLOADS[name]
    nthreads = host_cores()
    if name.startswith("cornell"):
        return scenes.cornell_box(xres=w["xres"], yres=w["yres"], spp=w["spp"], n_threads=nthreads, **w.get("kw", {}))
    if name == "conference":
        return scenes.conference(xres=w["xres"], yres=w["yres"], spp=w["spp"], n_chairs=40, detail=34 if not small else 6, n_light_quads=64, n_threads=nthreads)
    if name.startswith("landscape"):
        return scenes.landscape(xres=w["xres"], yres=w["yres"], spp=w["spp"], n_trees=3000 if not small else 50, n_prototypes=20 if not small else 3,
                                grid=256 if not small else 32, n_threads=nthreads)
    return scenes.statue(n_side=1468 if not small else 200, xres=w["xres"], yres=w["yres"], spp=w["spp"], n_threads=nthreads)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md), read through NVML in this process -- the numbers
    nvidia-smi prints, without forking a process five times a second: every nvidia-smi start takes driver-wide locks, and with them
    tens of milliseconds out of each end-to-end step (scene upload and film download are driver calls).  Falls back to nvidia-smi."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []  # (sm_mhz, sm_max_mhz, reasons bit mask)
        self.stop_flag = False
        self.source = "nvml"

    def _nvml(self):
        import pynvml as N

        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag:
            self.rows.append((float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)), float(mx), int(get_reasons(h))))
            time.sleep(0.1)

    def _smi(self):
        self.source = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [c.strip() for c in out.split(",")]
                mask = 0
                for (_, bit), v in zip(self.REASONS, r[2:6]):
                    if v.lower().startswith("active"):
                        mask |= bit
                self.rows.append((float(r[0]), float(r[1]), mask))
            except Exception:
                pass
            time.sleep(0.5)

    def run(self):
        try:
            self._nvml()
        except Exception:
            self._smi()

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        mx = max((r[1] for r in self.rows), default=0)
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": [n for n, bit in self.REASONS if mask & bit],
                "samples": len(sm), "source": self.source}


from rs_pbrt_b200.multigpu import band, reduce_film  # noqa: E402


def cpu_band(rect, rows):
    x0, y0, x1, y1 = rect
    mid = (y0 + y1) // 2
    a = max(y0, mid - rows // 2)
    return [x0, a, x1, min(y1, a + rows)]


def run_reference(args):
    """--impl reference: the CPU path on the host cores (oracle port; rs_pbrt cannot be built here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib

    w = WORKLOADS[args.workload]
    h = make_scene(args.workload, small=args.small)
    rp = h.params.contents
    rect = cpu_band(list(rp.sample_bounds), w["cpu_rows"])
    cores = host_cores()
    osc = oracle_lib.OracleScene(h.desc)
    for _ in range(args.warmup):
        osc.render(h.params, rect=cpu_band(list(rp.sample_bounds), 2), n_threads=cores)
    t0 = time.perf_counter()
    rays = 0
    for _ in range(args.steps):
        _, _, st = osc.render(h.params, rect=rect, n_threads=cores)
        rays += st["rays"]
    dt = time.perf_counter() - t0
    val = rays / dt / 1e6
    sample = "rows %d..%d of the %dx%d frame at %d spp (%d camera paths per step), oracle C++ port of rs_pbrt's path, %d threads" % (
        rect[1], rect[3], w["xres"], w["yres"], rp.spp, (rect[3] - rect[1]) * (rect[2] - rect[0]) * rp.spp, cores)
    line = {"impl": "reference", "metric": "Mrays/s", "value": val, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": w["desc"], "sample": sample},
            "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


RAY_COUNTERS = ("camera_rays", "rays", "closest_rays", "shadow_rays")


def measure(args, name, steps, warmup, dist, rank, world, local, want_cpu, dump_dir=None):
    """One workload through the contract: K device-resident steps, K end-to-end steps, the per-kernel pass.  Returns the JSON
    line (rank 0) or None.  `dump_dir`: rank 0 writes there what the last device-resident step handed its caller -- the
    frame's film (film.npy, float32 H x W x 4, reduced over the ranks) and the stats' ray counters (ray_counters.npy, float64,
    RAY_COUNTERS order, summed over the ranks)."""
    import numpy as np
    import torch

    from rs_pbrt_b200 import GpuScene, _abi, pin_description, unpin_description

    w = WORKLOADS[name]
    h = make_scene(name, small=args.small)
    rp = h.params.contents
    cb = list(rp.cropped_pixel_bounds)
    fh, fw = cb[3] - cb[1], cb[2] - cb[0]
    full = list(rp.sample_bounds)
    my_rect = full
    L = _abi.load()
    launches0 = L.pbrt_gpu_launch_count()
    gpu = GpuScene(h.desc, device=local)
    film = torch.zeros((fh, fw, 4), dtype=torch.float32, device="cuda")
    host_film = np.zeros((fh, fw, 4), np.float32)
    stream = torch.cuda.current_stream().cuda_stream

    def sync_all():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def render_share(g):
        """This rank's share: the whole frame at N = 1, else part `rank` of the frame's Morton-ordered 16x16 tiles (library side)."""
        if world == 1:
            return g.render_device(h.params, film.data_ptr(), rect=my_rect, stream=stream)
        return g.render_tiles_device(h.params, film.data_ptr(), rank, world, stream=stream)

    def step_resident():
        film.zero_()
        st = render_share(gpu)
        reduce_film(film, dist)
        return st

    def step_e2e():
        """The call a user of the plugin makes, host buffers in and out."""
        g2 = GpuScene(h.desc, device=local)  # pbrt_gpu_scene_create: H2D of the whole scene
        nbytes = g2.upload_bytes()
        if world == 1:
            host_film.fill(0.0)
            _, st = g2.render(h.params, rect=my_rect, film=host_film)  # pbrt_gpu_render: D2H of the film inside
        else:
            film.zero_()
            st = render_share(g2)
            reduce_film(film, dist)
            if rank == 0:
                host_film[...] = film.cpu().numpy()  # D2H of the reduced film
        g2.close()
        return st, nbytes

    for _ in range(warmup):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- timed: K steps, device-resident ---------------------------------------------------------
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rays = 0
    for _ in range(steps):
        st = step_resident()
        rays += st["rays"]
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    tot = torch.tensor([float(rays)], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_total = float(ms.item())
    rays_total = float(tot[0].item())
    outputs = None
    if dump_dir is not None:
        last = torch.tensor([float(st[k]) for k in RAY_COUNTERS], device="cuda", dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(last, op=dist.ReduceOp.SUM)
        outputs = {"film": film.cpu().numpy(), "ray_counters": last.cpu().numpy()}
    # ---- timed: K steps end to end (host buffers) ------------------------------------------------
    # The step's inputs live in pinned host memory, as the bench contract asks (the caller's scene arrays are page-locked once, here,
    # through pbrt_gpu_host_register; pbrt_gpu_scene_create then DMAs them where they lie).
    pinned = pin_description(h.desc)
    step_e2e()
    sync_all()
    t0 = time.perf_counter()
    rays_e2e = 0
    h2d = 0
    for _ in range(steps):
        st, h2d = step_e2e()
        rays_e2e += st["rays"]
    sync_all()
    t_e2e = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    r_e2e = torch.tensor([float(rays_e2e)], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        dist.all_reduce(r_e2e, op=dist.ReduceOp.SUM)
    unpin_description(pinned)
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    # ---- per-kernel pass: one untimed counting render gives the algorithmic bytes, one single-stream render the kernel times
    # (one batch in flight, so a co-resident kernel of the other batch does not inflate a kernel's duration; the throughput
    # numbers above use the default two-batch overlap)
    rp.flags = _abi.RENDER_COUNT_WORK | _abi.RENDER_SINGLE_STREAM
    film.zero_()
    stc = render_share(gpu)
    rp.flags = _abi.RENDER_SINGLE_STREAM
    film.zero_()
    sts = render_share(gpu)
    rp.flags = 0
    ser = torch.tensor([sts["ms_trace"], sts["ms_shade"], float(sts["trace_launches"]), sts["ms_total"]], device="cuda", dtype=torch.float64)
    cnt = torch.tensor([float(stc["nodes_visited"]), float(stc["tris_tested"]), float(stc["rays"]), float(stc["camera_rays"]),
                        float(stc.get("shade_slots", 0)), float(stc.get("shaded_vertices", 0))], device="cuda", dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(ser, op=dist.ReduceOp.SUM)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    launches = L.pbrt_gpu_launch_count() - launches0
    gpu.close()
    # ---- the one-process form of the same frame (what a single rs_pbrt process calls): pbrt_gpu_render_multi over all N devices from
    # rank 0, host film in and out; the other ranks wait at the barrier.  Reported under extra, never as `value`.
    inproc = None
    if world > 1 and args.inproc:
        sync_all()
        # the other ranks wait on the rendezvous store, on the CPU: an NCCL barrier would park a spinning kernel on their GPUs, which
        # rank 0's kernels would then have to time-slice with (measured: exactly half speed, profiles/r02_c5_*)
        store = dist.distributed_c10d._get_default_store()
        key = "inproc_done_%s" % name
        if rank == 0:
            from rs_pbrt_b200 import render_multi

            gs = [GpuScene(h.desc, device=d) for d in range(world)]
            render_multi(gs, h.params)
            t0 = time.perf_counter()
            r_mp = 0
            for _ in range(steps):
                host_film.fill(0.0)
                _, stm = render_multi(gs, h.params, film=host_film)
                r_mp += stm["rays"]
            dt = time.perf_counter() - t0
            inproc = {"call": "pbrt_gpu_render_multi (one process, %d devices, host film)" % world, "value": r_mp / dt / 1e6, "unit": "Mrays/s",
                      "ms_per_step": dt / max(steps, 1) * 1e3, "device_ms_last": stm["ms_total"]}
            for g in gs:
                g.close()
            store.set(key, "1")
        else:
            store.wait([key])
        sync_all()
    if rank != 0:
        return None
    if outputs is not None:
        assert sum(a.nbytes for a in outputs.values()) <= 64 << 20  # every workload's film is at most 1920 x 1080 x 4 floats
        os.makedirs(dump_dir, exist_ok=True)
        for k, a in outputs.items():
            np.save(os.path.join(dump_dir, k + ".npy"), a)
    nodes_v, tris_t, rays_frame, cam_frame, slots_frame, verts_frame = (float(x) for x in cnt.tolist())
    trace_ms = float(ser[0].item()) / world  # mean over ranks of one frame's k_trace time (single-stream pass)
    shade_ms = float(ser[1].item()) / world
    n_launch = max(float(ser[2].item()) / world, 1.0)  # per rank; k_shade is launched once per k_trace launch
    serial_ms = float(ser[3].item()) / world
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if peaks_path.exists():
        try:
            peak = float(json.loads(peaks_path.read_text())["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json hbm_gbs"
        except Exception:
            pass

    def ncu_record(kernel):
        """DRAM traffic, SIMT efficiency and stall picture of `kernel` on this workload from the committed ncu summary of the
        same sources (profiles/ncu_<kernel>_<workload>.json, tools/ncu_summary.py; ncu replays kernels, so it is never run
        inside the timed bench)."""
        prof = ROOT / "profiles" / ("ncu_%s_%s.json" % (kernel, name))
        if not prof.exists():
            return {}
        try:
            d = json.loads(prof.read_text())
            return {"traffic": d.get("dram_bytes_per_launch"), "ncu_launches": d.get("launches"), "ncu_ns_per_launch": d.get("ns_per_launch"),
                    "ncu_dram_gbs": d.get("dram_gbs"), "active_lanes_per_inst": d.get("active_lanes_per_inst"),
                    "issue_active_pct": d.get("issue_active_pct"), "warps_active_pct": d.get("warps_active_pct"), "limiter": d.get("limiter"),
                    "ncu_source": "profiles/" + prof.name}
        except Exception:
            return {}

    def roof(kernel, alg_bytes_frame, ms_frame, note):
        achieved = alg_bytes_frame / world / (ms_frame * 1e-3) / 1e9 if ms_frame > 0 else None
        r = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
             "frac": (achieved / peak) if achieved else None, "traffic": None,
             "algorithmic_bytes_per_launch": alg_bytes_frame / world / n_launch, "ms_per_launch": ms_frame / n_launch,
             "share_of_step": ms_frame / serial_ms if serial_ms > 0 else None, "algorithmic_bytes": note}
        r.update(ncu_record(kernel))
        if r.get("traffic") and r.get("ncu_launches") and world == 1:
            # the ncu record covers one whole frame; this line's "launch" is one wavefront iteration (n_launch per frame, several
            # k_shade instantiations count as one), so the measured bytes are re-expressed per iteration of THIS run
            r["traffic"] = r["traffic"] * r["ncu_launches"] / n_launch
        elif r.get("traffic"):
            r["traffic"] = None  # a rank's share of the frame is not the frame the record was taken on
        if r.get("traffic") and r["ms_per_launch"] > 0:
            # the measured-DRAM fraction: what the HBM roof really sees of this kernel (ncu bytes / live CUDA-event time)
            r["dram_frac"] = r["traffic"] / (r["ms_per_launch"] * 1e-3) / 1e9 / peak
        return r

    alg_trace = 32.0 * nodes_v + 48.0 * tris_t + 48.0 * rays_frame
    # k_shade moves, per slot of its queue, the path state in and out (ray direction 16 B, hit 16 B, beta 16 B, L + flags 16 B,
    # sampler index / dimension 12 B read; L, beta, direction, dimension 52 B written) and 32 B per ray it emits
    alg_shade = 128.0 * slots_frame + 32.0 * max(rays_frame - cam_frame, 0.0)
    r_trace = roof("k_trace", alg_trace, trace_ms, "32 B x nodes visited + 48 B x triangles tested + 48 B x rays (record in, hit out)")
    r_shade = roof("k_shade", alg_shade, shade_ms, "128 B x queue slots (path state in + out) + 32 B x rays emitted")
    dominant = r_trace if trace_ms >= shade_ms else r_shade
    value = rays_total / (ms_total * 1e-3) / 1e6
    e2e_val = float(r_e2e.item()) / float(t_e2e.item()) / 1e6
    line = {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_total / max(steps, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": w["desc"], "parallelism": "16x16 tiles in Morton order dealt round robin to %d rank(s) (pbrt_gpu_render_tiles_device), scene replicated, 1 ncclReduce(sum) of the film" % world,
                   "n_tris": int(h.desc.contents.n_tris), "n_bvh_nodes": int(h.desc.contents.n_nodes), "rays_per_frame": rays_frame,
                   "l2": "inputs larger than L2: %.0f MB of BVH nodes + triangles and >= 1 GiB of wavefront state per batch; no explicit flush"
                         % ((32.0 * h.desc.contents.n_nodes + 48.0 * h.desc.contents.n_tris) / 1e6)},
        "e2e": {"value": e2e_val, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(fh * fw * 16),
                "inputs": "scene arrays in pinned host memory (pbrt_gpu_host_register, once)",
                "call": "pbrt_gpu_scene_create + pbrt_gpu_render (host film)" if world == 1 else "pbrt_gpu_scene_create + pbrt_gpu_render_tiles_device + ncclReduce + D2H on rank 0"},
        "gpu_launches": int(launches),
        "roofline": dominant,
        "roofline_kernels": [r_trace, r_shade],
        "kernel_ms_per_step": {"note": "single-stream pass (no overlap of batches)", "frame": serial_ms, "k_trace": trace_ms, "k_shade": shade_ms,
                               "other (raygen, sort, light grid, resolve)": serial_ms - trace_ms - shade_ms},
        "clocks": sampler.summary(),
    }
    if inproc:
        line["extra_inproc"] = inproc
    # ---- CPU baseline: the oracle on the host cores, bounded sample (rank 0, N = 1 only) ----------
    if world == 1 and want_cpu:
        import oracle_lib

        cores = host_cores()
        rect = cpu_band(full, w["cpu_rows"])
        osc = oracle_lib.OracleScene(h.desc)
        t0 = time.perf_counter()
        _, _, ost = osc.render(h.params, rect=rect, n_threads=cores)
        dt = time.perf_counter() - t0
        r1 = cpu_band(full, max(2, w["cpu_rows"] // 16))
        t1 = time.perf_counter()
        _, _, ost1 = osc.render(h.params, rect=r1, n_threads=1)
        dt1 = time.perf_counter() - t1
        line["cpu_baseline"] = {"value": ost["rays"] / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                                "single_thread_value": ost1["rays"] / dt1 / 1e6,
                                "sample": "rows %d..%d of the frame, %d camera paths, %.1f s, oracle C++ port (rs_pbrt needs a Rust toolchain); 1 thread: rows %d..%d, %.1f s" % (
                                    rect[1], rect[3], (rect[3] - rect[1]) * (rect[2] - rect[0]) * rp.spp, dt, r1[1], r1[3], dt1)}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="statue", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the short Cornell (configs[1]) measurement reported under extra.cornell")
    ap.add_argument("--small", action="store_true", help="debug: smaller statue mesh")
    ap.add_argument("--no-inproc", dest="inproc", action="store_false", help="N > 1: skip the pbrt_gpu_render_multi (one process, N devices) leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the film and ray counters of the last timed step of --workload as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.steps < 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs --steps >= 1 and --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    line = measure(args, args.workload, args.steps, args.warmup, dist, rank, world, local, want_cpu=not args.no_cpu, dump_dir=args.dump_outputs)
    if args.workload == "statue" and not args.no_extra:
        # BASELINE.json configs[1] (round 1's default) in short form, so that the driver's records keep a Cornell number
        ex = measure(args, "cornell", min(args.steps, 3), 3, dist, rank, world, local, want_cpu=False)
        if line is not None and ex is not None:
            line["extra"] = {"cornell": {k: ex[k] for k in ("value", "unit", "ms_per_step", "steps", "e2e", "kernel_ms_per_step", "roofline_kernels", "config") if k in ex}}
            if "extra_inproc" in ex:
                line["extra"]["cornell"]["render_multi"] = ex["extra_inproc"]
    if line is not None and "extra_inproc" in line:
        line.setdefault("extra", {})["render_multi"] = line.pop("extra_inproc")
    if line is not None:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
