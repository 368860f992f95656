#!/usr/bin/env python
"""bench.py - headline benchmark of the terrain hot path (BASELINE.json: "height cells/s @8192^2 8-octave").

A step = one pass of the hot path over one 8192x8192 tile: tw_heightgen_2d (8-octave domain-warped simplex fBm, glaciate + hmap sine bias,
fused min/max), BASELINE.json configs[1]. `value` is measured with the output resident in HBM (CUDA events on the library's own stream);
`e2e` is the same call with a pinned HOST output buffer, i.e. including the device->host copy of the 268 MB grid and the host->device
copy of the parameter blocks, through the public C ABI. N>1 (torchrun): every rank generates its own 8192^2 tile of one larger terrain
(tiles are pure functions of global coordinates: no data-path collective; one 2-float min/max all-reduce per step) => weak scaling.

--impl reference times the reference's own CPU implementation (the unmodified reference objects in oracle/_ref when present, else the
plain-C oracle port) on the host cores, on a bounded sample of the same workload.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned to its caller (rank 0's tile): DIR/height_rows.npy
= DUMP_ROWS whole rows of the 8192^2 grid drawn with DUMP_SEED (dump_rows(); 16 MB of the 256 MB grid), DIR/minmax.npy = the step's
(zmin, zmax). The inputs are fixed, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HM_CFG = dict(sine_mag=5.0, sine_freq=0.001, sine_bias=-4.0)   # scene_config/config.txt:76
N_TILE = 8192
WORKLOAD = "heightgen 8192x8192 tile, mesh_gen_mode 4 (domain-warped simplex), 8 octaves (mesh_freq_filter 1), fp32, glaciate + hmap sine"
FLOP_PER_CELL = 5200.0    # fp32 pipe operations per cell (FMUL/FADD/FFMA each counted once, floor included): 40 simplex evaluations x ~128 (SASS count of
                          # the scalar kernel's loop) + epilogue; SURVEY.md section 8(d) estimated ~6.8 k with FMA counted twice
FLOP_EXEC_PER_CELL = 2968.5   # fallback only: fp32 FMUL/FADD/FFMA lane operations the shipped kernel executes per cell. bench.py takes the number from
                          # profiles/roofline_r02.json (ncu per-opcode executed counts of the SASS view, written by tools/ncu_summary.py --opcodes); this
                          # constant is the round-1 capture's value (profiles/ncu_noise_grid2_l3_kernel_r01.json re-read with the same script)
BYTES_PER_CELL = 4.0      # one fp32 store per cell, no reads
DUMP_ROWS, DUMP_SEED = 512, 0


def dump_rows():
    """The grid rows that --dump-outputs writes, ascending: the same for every run and every build."""
    return np.sort(np.random.default_rng(DUMP_SEED).choice(N_TILE, DUMP_ROWS, replace=False))


def dump_outputs(path, height_rows, zrange):
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "height_rows.npy"), np.asarray(height_rows, np.float32))
    np.save(os.path.join(path, "minmax.npy"), np.array(zrange, np.float32))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


class ClockSampler:
    """nvidia-smi -lms 20 in the background during the timed region (the profiling recipe's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.lines = []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.perf_counter(), ln))

    def wait_ready(self, timeout=8.0):
        """Blocks until nvidia-smi has printed its first sample (its start-up can take longer than the whole warm-up + timed region on a fresh box)."""
        t_end = time.perf_counter() + timeout
        while self.proc is not None and not self.lines and time.perf_counter() < t_end and self.proc.poll() is None:
            time.sleep(0.01)
        return bool(self.lines)

    def mark(self):
        self.t0 = time.perf_counter()

    def in_window(self):
        return sum(1 for (t, _) in self.lines if t >= getattr(self, "t0", 0.0))

    def summary(self):
        t1 = time.perf_counter()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [[x.strip() for x in ln.split(",")] for (t, ln) in self.lines if self.t0 <= t <= t1 + 0.12]
        rows = [r for r in rows if len(r) >= 7]
        if not rows:
            rows = [[x.strip() for x in ln.split(",")] for (t, ln) in self.lines][-3:]
            rows = [r for r in rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows), "reasons": reasons, "samples": len(rows)}


def host_cpu_info():
    """Threads the CPU legs may really use (scheduler affinity capped by the cgroup CPU quota - NOT os.cpu_count(), which is the host's total
    even when this process is confined to a slice of it), plus CPU model and physical core count (BASELINE.md section 3)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
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
    threads = max(1, min(aff, int(quota + 0.999)) if quota else aff)
    model, phys, logical = "unknown", set(), 0
    try:
        pid = cid = None
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name") and model == "unknown":
                model = ln.split(":", 1)[1].strip()
            elif ln.startswith("processor"):
                logical += 1
            elif ln.startswith("physical id"):
                pid = ln.split(":", 1)[1].strip()
            elif ln.startswith("core id"):
                cid = ln.split(":", 1)[1].strip()
                phys.add((pid, cid))
    except Exception:
        pass
    return {"threads_used": threads, "affinity_cpus": aff, "cgroup_quota_cpus": quota, "logical_cpus": logical or (os.cpu_count() or 1),
            "physical_cores": len(phys) or None, "cpu_model": model}


def cpu_runner(cores, nx, ny):
    """The reference's own CPU path for the workload on an nx x ny window (build_arrays + enable_glaciate + eval_index over the grid):
    the unmodified reference objects (oracle/_ref) when the prebuilt library is present, else the plain-C oracle port."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import refapi as R
        if R.available():
            R.lib().ref_set_threads(cores)
            R.setup(mode=4, freq_filter=1, seed=1, zmax_est=2.3, hmap=HM_CFG)
            dx, dy = R.lib().ref_get_dx(), R.lib().ref_get_dy()
            return "reference", (lambda rows=ny: R.heightgen(-N_TILE / 2, -N_TILE / 2, dx, dy, nx, rows, cache_values=0, glaciate=1))
    except Exception:
        pass
    import oracle as O
    hp = O.HeightParams()
    hp.gen_mode, hp.gen_shape, hp.start_eval_sin, hp.glaciate = 4, 0, 10, 1
    hp.mesh_scale = hp.mesh_scale_z_inv = hp.mesh_height_scale = 1.0
    hp.dx_val_inv = hp.dy_val_inv = 16.0
    hp.mesh_height, hp.zmax_est = 0.4, 2.3
    hp.rx, hp.ry = O.gen_rx_ry(1, 0, 4)
    hp.hmap = O.hmap_params(**HM_CFG)
    return "port", (lambda rows=ny: O.heightgen_2d(O.Grid2D(-N_TILE / 2, -N_TILE / 2, 0.0625, 0.0625, nx, rows), hp, None, 1, 0, cores))


def reference_arm(args):
    """bench.py --impl reference: the reference's CPU implementation of the path on all host cores, bounded sample per step."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    hc = host_cpu_info()
    cores = hc["threads_used"]
    nx, ny = 1024, 1024                     # bounded sample: 1 M cells of the same grid (rows/cols 0..1023 of the 8192^2 tile): 8 rows per thread on a
                                            # 128-thread host, ~0.1 s per step there - long enough for the OpenMP team to reach a steady rate
    kind, run = cpu_runner(cores, nx, ny)
    for _ in range(args.warmup):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = time.perf_counter() - t0
    value = nx * ny * args.steps / dt
    sample = ("%dx%d-cell window (rows/cols 0..%d) of the 8192^2 grid per step, %d OpenMP threads on %s (%s physical cores, %d logical, affinity %d); "
              "a per-cell RATE on a bounded sample of the same grid, not the whole 8192^2 step" % (nx, ny, nx - 1, cores, hc["cpu_model"], hc["physical_cores"], hc["logical_cpus"], hc["affinity_cpus"]))
    print(json.dumps({
        "impl": "reference", "metric": "height cells/s @8192^2 8-octave domain-warp", "value": value, "unit": "cells/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "cells_per_step": nx * ny, "same_grid_bounded_sample": True},
        "cpu_baseline": dict({"value": value, "unit": "cells/s", "cores": cores, "kind": kind, "sample": sample}, **{k: hc[k] for k in ("cpu_model", "physical_cores", "logical_cpus", "affinity_cpus", "cgroup_quota_cpus")}),
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_leg(gpu_map_8192=None):
    """Bounded CPU samples of the same workloads (rank 0, N=1), the unmodified reference objects (oracle/_ref) when present, on the threads this
    process may really use: the headline (config 2) plus configs 3, 4 and 5 AT THE SAME CONFIGURATION as the GPU rows (gpu_map_8192 = the GPU's
    8192^2 simplex map, bit-identical to what the reference would generate, so the erosion input is the same)."""
    hc = host_cpu_info()
    cores = hc["threads_used"]
    nx, ny = 1024, 1024
    kind, run = cpu_runner(cores, nx, ny)
    run(128)
    t0 = time.perf_counter()
    run()
    dt = time.perf_counter() - t0
    what = "unmodified reference objects (oracle/_ref)" if kind == "reference" else "plain-C oracle port"
    res = {"value": nx * ny / dt, "unit": "cells/s", "cores": cores, "kind": kind,
           "sample": "%s, %dx%d-cell window of the 8192^2 grid, OpenMP %d threads" % (what, nx, ny, cores)}
    res.update({k: hc[k] for k in ("cpu_model", "physical_cores", "logical_cpus", "affinity_cpus", "cgroup_quota_cpus")})
    if kind != "reference":
        return res
    try:
        import refapi as R
        RL = R.lib()
        # ---- config 3: apply_erosion on the 8192^2 map, 1000 / 1e5 (/ 1e6) droplets; 1 thread = the deterministic order the GPU reproduces bit for bit,
        #      all threads = the reference's shipped OpenMP loop (racy, order-dependent output: a speed number only)
        R.setup(mode=1, freq_filter=1, seed=1, zmax_est=2.3, hmap=HM_CFG)
        if gpu_map_8192 is not None:
            z = gpu_map_8192
        else:
            z = R.heightgen(-N_TILE / 2, -N_TILE / 2, RL.ref_get_dx(), RL.ref_get_dy(), N_TILE, N_TILE, 0, 1)
        scene = importlib.import_module("3dworld_b200.scene")
        ep = scene.SceneConfig(mesh_gen_mode=1, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3).erosion_params()
        zmin = float(z.min())
        c3 = {"config": "apply_erosion on the 8192^2 8-octave simplex map (BASELINE config 3), same input and parameters as the GPU rows"}
        for label, thr, counts in (("1_thread", 1, (1000, 100000)), ("openmp_%d_threads" % cores, cores, (1000, 100000, 1000000))):
            RL.ref_set_threads(thr)
            for n in counts:
                t0 = time.perf_counter()
                R.apply_erosion(z, zmin, n, erode_amount=ep.erode_amount, water_plane_z=ep.water_plane_z, half_dxy=ep.half_dxy, zmin=ep.zmin, zmax=ep.zmax,
                                relh_adj_tex=ep.relh_adj_tex, clip_hd1=ep.clip_hd1)
                c3["droplets_per_s_%s_%d_droplets" % (label, n)] = n / (time.perf_counter() - t0)
        RL.ref_set_threads(cores)
        res["config3_erosion_8192"] = c3
        del z
        # ---- config 4: 512^3 sine voxel density (noise_gen_3d + the create_procedural loop), all threads
        vcfg = scene.SceneConfig(scene_size=(16.0, 16.0, 4.0), mesh_size=(128, 128, 64))
        vp = scene.voxel_landscape_params(vcfg, 512, 512, 512)
        nyv = 128                                # bounded: a 512 x 128 x 512 slab of the same grid (the loop is uniform in y)
        t0 = time.perf_counter()
        R.voxel_fill(512, nyv, 512, list(vp.lo_pos), list(vp.vsz), list(vp.offset), vp.mag, vp.freq, vp.normalize_to_1, vp.rseed1, vp.rseed2, 0, vp.zscale)
        res["config4_voxels_512"] = {"voxels_per_s": 512 * nyv * 512 / (time.perf_counter() - t0), "sample": "512x%dx512 slab of the 512^3 grid, sine mode, %d threads" % (nyv, cores)}
        # ---- config 5: per tile = 258^2 8-octave domain-warp generation + 1000 droplets (tile_t::create_zvals semantics); a sample of tiles spread over the 65536
        R.setup(mode=4, freq_filter=1, seed=1, zmax_est=2.3, hmap=HM_CFG, mesh=(256, 256, 1))
        cfg5 = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3, mesh_size=(256, 256, 1))
        ep5 = cfg5.erosion_params()
        sample_tiles = [(tx * 256, ty * 256) for ty in range(4, 256, 36) for tx in range(7, 256, 62)]
        dx, dy = RL.ref_get_dx(), RL.ref_get_dy()
        t0 = time.perf_counter()
        for x1, y1 in sample_tiles:
            tz = R.heightgen(float(x1 - 128), float(y1 - 128), dx, dy, 258, 258, 0, 1)
            R.apply_erosion(tz, ep5.zmin, 1000, erode_amount=ep5.erode_amount, water_plane_z=ep5.water_plane_z, half_dxy=ep5.half_dxy, zmin=ep5.zmin, zmax=ep5.zmax,
                            relh_adj_tex=ep5.relh_adj_tex, clip_hd1=ep5.clip_hd1)
        dt5 = time.perf_counter() - t0
        res["config5_tiled_terrain"] = {"tiles_per_s": len(sample_tiles) / dt5, "cells_per_s": len(sample_tiles) * 258 * 258 / dt5, "droplets_per_s": len(sample_tiles) * 1000 / dt5,
                                        "seconds_extrapolated_65536_tiles": 65536 * dt5 / len(sample_tiles),
                                        "sample": "%d of the 65536 tiles (every 36th tile row, every 62nd column), generation + erosion per tile, %d threads" % (len(sample_tiles), cores)}
    except Exception as e:   # noqa: BLE001 - secondary numbers only
        res["secondary_note"] = "reference secondary timing failed: %s: %s" % (type(e).__name__, e)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements (sine / erosion / voxel)")
    ap.add_argument("--kernel-only", action="store_true", help="only the device-resident timed loop (for ncu runs): no e2e, cpu_baseline, extra")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference times a bounded CPU sample of a different shape")
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    tw = importlib.import_module("3dworld_b200")
    scene = importlib.import_module("3dworld_b200.scene")
    numa_bound = tw.bind_thread_to_device(local)   # pinned host buffers allocated below land on the GPU's own NUMA node (GPU0-3 / GPU4-7 hang off different sockets)
    ctx = tw.Context(local)
    if world > 1:   # the library's own communicator: the z-range reduction of the path is an ncclAllReduce inside lib3dworld_b200.so, not a torch call
        uid = [tw.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.dist_init(world, rank, uid[0])
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))   # time on the stream the kernels are launched on

    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
    hp = cfg.height_params()
    g = cfg.heightmap_grid(N_TILE, N_TILE)
    g.y0 = g.y0 + rank * N_TILE             # rank r owns tile row r of one larger terrain
    cells = N_TILE * N_TILE
    d_out = torch.empty((N_TILE, N_TILE), dtype=torch.float32, device="cuda")
    mm = tw.MinMax()
    zrange = [0.0, 0.0]

    def step_device():
        ctx.heightgen_2d_launch(g, hp, 1, 0, d_out, mm)
        ctx.heightgen_2d_poll(wait=True)
        if world > 1:                       # global z-range (get_heightmap_z_range over all tiles): the only collective of the path
            zrange[0], zrange[1] = ctx.dist_allreduce_minmax(mm.zmin, mm.zmax)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dump_idx = torch.from_numpy(dump_rows()).cuda() if (args.dump_outputs and rank == 0) else None
    sampler = ClockSampler(local)           # started before the warm-up so that nvidia-smi is already streaming when the timed region begins
    sampler.wait_ready()
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler.mark()
    launches0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count - launches0
    if dump_idx is not None:                # the last timed step's outputs, before the replay / e2e steps below rewrite them
        dumped = (d_out[dump_idx].cpu().numpy(), list(zrange) if world > 1 else [mm.zmin, mm.zmax])
    replayed = False
    if sampler.in_window() < 3:             # a 70 ms timed region can fall between two 20 ms samples of a slow nvidia-smi: replay the SAME steps (untimed) under the sampler
        replayed = True
        t_end = time.perf_counter() + 0.5
        while time.perf_counter() < t_end:      # the kernels of the step only: no collective in a time-bounded loop (ranks would disagree on the count)
            ctx.heightgen_2d_launch(g, hp, 1, 0, d_out, mm)
            ctx.heightgen_2d_poll(wait=True)
            torch.cuda.synchronize()
    clocks = sampler.summary()
    if dump_idx is not None:
        dump_outputs(args.dump_outputs, *dumped)
    if replayed:
        clocks["sampled_during"] = "timed region + an untimed 0.5 s replay of the same kernels right after it (fewer than 3 samples fell inside the timed region)"
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * cells * args.steps / (ms * 1e-3)

    if args.kernel_only:
        if rank == 0:
            print(json.dumps({"metric": "height cells/s @8192^2 8-octave domain-warp", "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps,
                              "ms_per_step": ms / args.steps, "gpu_launches": launches, "clocks": clocks, "note": "kernel-only run (profiling aid)"}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end to end: pinned HOST output buffer through the same C-ABI call (D2H of the grid inside the timed region) ----
    h_out = torch.empty((N_TILE, N_TILE), dtype=torch.float32).pin_memory()

    def step_e2e():
        ctx.heightgen_2d_launch(g, hp, 1, 0, h_out, mm)
        ctx.heightgen_2d_poll(wait=True)
        return mm.zmin

    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * cells * e2e_steps / float(dt.item())
    h2d = C.sizeof(tw.Grid2D) + C.sizeof(tw.HeightParams)
    d2h = cells * 4 + 8

    def run_config5():                      # BASELINE config 5 (strong scaling over the ranks); never allowed to take the headline down
        try:
            return config5_strong(tw, scene, ctx, torch, dist, rank, world, barrier)
        except Exception as e:              # noqa: BLE001
            return {"error": "%s: %s" % (type(e).__name__, e)}

    cfg5 = run_config5() if (world > 1 and not args.no_extra) else None   # at N = 1 it runs after the secondary rows below

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, peak_kind, sm_max_mhz = peaks()
    kernel_ms = ms / args.steps            # one dominant kernel (noise_grid_kernel) per step
    achieved_gbs = BYTES_PER_CELL * cells / (kernel_ms * 1e-3) / 1e9
    traffic, exec_ops, prof_src = None, FLOP_EXEC_PER_CELL, None
    for prof in ("roofline_r02.json", "roofline_r01.json"):   # per-launch numbers of the dominant kernel from the committed ncu --set full capture (tools/ncu_summary.py)
        pp = os.path.join(ROOT, "profiles", prof)
        if os.path.exists(pp):
            pj = json.load(open(pp))
            k = pj.get("noise_grid2_kernel", pj.get("noise_grid_kernel", {}))
            traffic = k.get("dram_bytes_per_launch")
            exec_ops = k.get("fp32_mul_add_fma_lane_ops_per_unit", exec_ops)
            prof_src = "profiles/" + prof
            break
    sm_mhz = clocks.get("sm_mhz") or sm_max_mhz
    alu_peak = 148 * 128 * sm_mhz * 1e6   # fp32 lane-instructions/s at the clock observed during the run
    out = {
        "metric": "height cells/s @8192^2 8-octave domain-warp", "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "cells_per_step_per_gpu": cells, "parallelism": "tile-row per rank, no data-path collective; z range = ncclAllReduce inside the library (%d rank%s)" % (world, "s" if world > 1 else ""),
                   "host_numa_bound": bool(numa_bound),
                   "l2": "output 268 MB per step > 126 MB L2; the kernel reads no input arrays", "bit_exact_vs_reference": True},
        "gpu_launches": launches,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "cells/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "path": "tw_heightgen_2d_launch/poll with a pinned host output buffer"},
        "roofline": {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak, "traffic": traffic,
                     "peak_kind": peak_kind, "traffic_source": prof_src, "kernel": "noise_grid2_kernel<simplex,warp> (two cells per thread, packed fp32x2, hash/gradient table in shared memory)", "algorithmic_bytes_per_cell": BYTES_PER_CELL,
                     "note": "the kernel is FP32-pipe bound by construction (4 B/cell vs ~5.2 k fp32 operations/cell; SURVEY.md 8d): see 'alu' and profiles/",
                     "alu": {"achieved_fp32_ops_per_s": FLOP_PER_CELL * cells / (kernel_ms * 1e-3), "peak_fp32_lane_instr_per_s": alu_peak,
                             "frac": FLOP_PER_CELL * cells / (kernel_ms * 1e-3) / alu_peak, "flop_per_cell": FLOP_PER_CELL,
                             "executed_fp32_ops_per_cell": exec_ops, "frac_executed": exec_ops * cells / (kernel_ms * 1e-3) / alu_peak, "executed_ops_source": prof_src,
                             "note": "flop_per_cell = the reference algorithm's fp32 operations (what the CPU path executes); the kernel tabulates part of "
                                     "them, so frac (algorithmic) can exceed 1 while the FMA pipe itself is ~80 % busy (frac_executed, profiles/)"}},
    }
    gpu_map = None
    if world == 1:
        if not args.no_extra:   # before the CPU leg, while the GPU clocks are still up
            try:
                out["extra"] = extra_measurements(tw, scene, ctx, stream, torch)
                gpu_map = out["extra"].pop("_map_8192", None)
            except Exception as e:          # noqa: BLE001 - secondary rows must not take the headline line down
                out["extra"] = {"error": "%s: %s" % (type(e).__name__, e)}
            cfg5 = run_config5()
        out["cpu_baseline"] = cpu_baseline_leg(gpu_map)
    if cfg5 is not None:
        out["config5_tiled_terrain"] = cfg5
    # ---- the other two thirds of BASELINE.json's metric as first-class top-level scalars (the driver's record keeps only scalars of this level) ----
    out["hbm_roofline_frac"] = achieved_gbs / hbm_peak
    ex = out.get("extra") or {}
    if "single_map_8192_serial_1000_droplets_per_s" in ex:
        out["erosion_iters_per_s"] = ex["single_map_8192_serial_1000_droplets_per_s"]                 # config 3: 8192^2 map, 1000 droplets, the reference's serial order (bit-exact; speculative parallel walks committed in order)
        out["erosion_iters_per_s_one_warp_walk"] = ex.get("single_map_8192_one_warp_walk_1000_droplets_per_s")   # the same order walked droplet after droplet by one warp (round 1's path)
        out["erosion_iters_per_s_1e5_droplets"] = ex.get("single_map_8192_serial_100000_droplets_per_s")
        out["erosion_iters_per_s_openmp_mode_1e6_droplets"] = ex.get("single_map_8192_openmp_mode_1e6_droplets_per_s")
        out["erosion_us_per_move"] = ex.get("single_map_8192_serial_100000_droplets_us_per_move")
    if "voxel_sine_512_voxels_per_s" in ex:
        out["voxels_per_s"] = ex["voxel_sine_512_voxels_per_s"]                                         # config 4
    if cfg5 and "seconds" in cfg5:
        out["config5_seconds"] = cfg5["seconds"]                                                        # config 5: 65536 tiles of 258^2, generation + 1000 droplets per tile
        out["config5_cells_per_s"] = cfg5["cells_per_s"]
        out["config5_erosion_iters_per_s"] = cfg5["droplets_per_s"]
        if "strong_scaling_efficiency" in cfg5:
            out["strong_scaling_speedup"] = cfg5["strong_scaling_speedup"]
            out["strong_scaling_efficiency"] = cfg5["strong_scaling_efficiency"]
    cb = out.get("cpu_baseline") or {}
    c3 = cb.get("config3_erosion_8192") or {}
    if c3 and out.get("erosion_iters_per_s"):
        out["cpu_erosion_iters_per_s_1_thread"] = c3.get("droplets_per_s_1_thread_1000_droplets")
        out["cpu_erosion_iters_per_s_1e5_droplets_1_thread"] = c3.get("droplets_per_s_1_thread_100000_droplets")
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def config5_strong(tw, scene, ctx, torch, dist, rank, world, barrier, device="cuda", side=256, iters=1000):
    """BASELINE config 5: the 65536^2 tiled terrain = 256 x 256 tiles of 258^2 cells (S = 256), 8-octave domain-warped generation at each tile's
    global origin + 1000 droplets per tile (the reference's per-tile semantics, src/tiled_mesh.cpp:515), through the fused C-ABI call.
    STRONG scaling: the 65536 tiles are split evenly over the ranks (contiguous tile rows, no communication); time = max over ranks."""
    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3, mesh_size=(256, 256, 1))
    hp, ep = cfg.height_params(), cfg.erosion_params()
    zv, total = 258, side * side
    t0, t1 = total * rank // world, total * (rank + 1) // world
    origins = [((t % side) * 256, (t // side) * 256) for t in range(t0, t1)]
    dxv, dyv = float(cfg.dx_val), float(cfg.dy_val)
    # every rank always reaches every collective: local failures are caught and reported through the reductions, never by skipping one
    local = [0.0, 0.0, 1.0]                 # seconds of the timed pass, droplet moves, ok flag
    err = None
    tiles = None
    t_single = None
    if world > 1:                            # the N = 1 denominator of the strong-scaling efficiency, measured in THIS run: rank 0 does all tiles alone
        if rank == 0:
            try:
                all_org = [((t % side) * 256, (t // side) * 256) for t in range(total)]
                full = torch.empty((total, zv, zv), dtype=torch.float32, device=device)
                ctx.create_zvals_batch(all_org, cfg.mesh_size, dxv, dyv, zv, hp, iters, ep, ep.zmin, out=full)   # warm-up (scratch allocation)
                s0 = time.perf_counter()
                ctx.create_zvals_batch(all_org, cfg.mesh_size, dxv, dyv, zv, hp, iters, ep, ep.zmin, out=full)
                t_single = time.perf_counter() - s0
                del full, all_org
            except Exception as e:          # noqa: BLE001
                t_single = None
        barrier()
    try:
        tiles = torch.empty((t1 - t0, zv, zv), dtype=torch.float32, device=device)
        ctx.create_zvals_batch(origins, cfg.mesh_size, dxv, dyv, zv, hp, iters, ep, ep.zmin, out=tiles)   # warm-up pass (scratch allocation)
    except Exception as e:                  # noqa: BLE001
        local[2], err = 0.0, "%s: %s" % (type(e).__name__, e)
    barrier()                               # aligned start of the timed pass
    if err is None:
        try:
            s0 = time.perf_counter()
            ctx.create_zvals_batch(origins, cfg.mesh_size, dxv, dyv, zv, hp, iters, ep, ep.zmin, out=tiles)   # synchronises before it returns
            local[0], local[1] = time.perf_counter() - s0, float(ctx.last_erosion_steps)
        except Exception as e:              # noqa: BLE001
            local[2], err = 0.0, "%s: %s" % (type(e).__name__, e)
    red = torch.tensor(local, dtype=torch.float64, device=device)
    if world > 1:
        tmax, tsum, tmin = red[:1].clone(), red[1:2].clone(), red[2:].clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        secs, steps, ok = float(tmax.item()), float(tsum.item()), float(tmin.item())
    else:
        secs, steps, ok = local
    del tiles
    if ok < 1.0 or secs <= 0.0:
        return {"error": err or "a rank failed", "scaling": "strong"}
    res = {"workload": "%d tiles of 258^2 (65536^2 terrain), mode 4 8-octave + %d droplets per tile, fused tw_create_zvals_batch" % (total, iters),
           "scaling": "strong", "tiles_per_rank": t1 - t0, "seconds": secs, "cells_per_s": total * zv * zv / secs,
           "droplets_per_s": total * iters / secs, "droplet_moves_per_s": steps / secs}
    if t_single:
        res.update({"seconds_1_gpu_same_run": t_single, "strong_scaling_speedup": t_single / secs, "strong_scaling_efficiency": t_single / secs / world})
    return res


def extra_measurements(tw, scene, ctx, stream, torch):
    """Secondary numbers for the other rows of the path (not the headline): sine-table grid, voxel fill, tiled erosion."""
    res = {}

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    d_out = torch.empty((N_TILE, N_TILE), dtype=torch.float32, device="cuda")
    for name, mode in (("simplex_8oct", 1), ("perlin_8oct", 2), ("sine_8band", 0)):
        cfg = scene.SceneConfig(mesh_gen_mode=mode, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
        hp, g = cfg.height_params(), cfg.heightmap_grid(N_TILE, N_TILE)
        if mode == 0:
            ctx.set_sine_params(cfg.sine_params())
        ms = timed(lambda: ctx.heightgen_2d(g, hp, out=d_out), 5)
        res["heightgen_%s_cells_per_s" % name] = N_TILE * N_TILE / (ms * 1e-3)
    # voxels: 512^3 sine density (BASELINE config 4)
    vcfg = scene.SceneConfig(scene_size=(16.0, 16.0, 4.0), mesh_size=(128, 128, 64))
    vp = scene.voxel_landscape_params(vcfg, 512, 512, 512)
    d_vox = torch.empty((512, 512, 512), dtype=torch.float32, device="cuda")
    ms = timed(lambda: ctx.voxel_fill(vp, out=d_vox), 3)
    res["voxel_sine_512_voxels_per_s"] = 512 ** 3 / (ms * 1e-3)
    res["voxel_sine_512_store_GBps"] = 4 * 512 ** 3 / (ms * 1e-3) / 1e9
    # config 4 "also mode 1/2": GLM 3-D simplex / Perlin fBm, 5 octaves (mesh_freq_filter 0)
    vcfg0 = scene.SceneConfig(scene_size=(16.0, 16.0, 4.0), mesh_size=(128, 128, 64), mesh_freq_filter=0, mesh_seed=1)
    for name, mode in (("simplex3", 1), ("perlin3", 2)):
        vpn = scene.voxel_landscape_params(vcfg0, 512, 512, 512, gen_mode=mode)
        ms = timed(lambda: ctx.voxel_fill(vpn, out=d_vox), 2)
        res["voxel_%s_5oct_512_voxels_per_s" % name] = 512 ** 3 / (ms * 1e-3)
    del d_vox
    # tiled terrain + erosion (BASELINE config 5 shape): 16384 tiles of 258^2 (a quarter of the 65536^2 grid), 1000 droplets per tile,
    # reference per-tile semantics; tw_create_zvals_batch = chunked multi-stream pipeline (generation overlaps the droplet walks)
    cfg = scene.SceneConfig(mesh_gen_mode=4, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3, mesh_size=(256, 256, 1))
    hp, ep = cfg.height_params(), cfg.erosion_params()
    nt, zv = 16384, 258
    origins = [((t % 128) * 256, (t // 128) * 256) for t in range(nt)]
    tiles = torch.empty((nt, zv, zv), dtype=torch.float32, device="cuda")
    dxv, dyv = float(cfg.dx_val), float(cfg.dy_val)
    for rep in range(2):   # first pass = warm-up (the 4.6 GB padded scratch is allocated on first use)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.heightgen_tiles(origins, cfg.mesh_size, dxv, dyv, zv, hp, out=tiles)
        t_gen = time.perf_counter() - t0
        t0 = time.perf_counter()
        ctx.erode_tiles(tiles, 1000, ep, min_zval_all=ep.zmin)
        t_ero = time.perf_counter() - t0
        steps = ctx.last_erosion_steps
        t0 = time.perf_counter()
        ctx.create_zvals_batch(origins, cfg.mesh_size, dxv, dyv, zv, hp, 1000, ep, ep.zmin, out=tiles)
        t_fused = time.perf_counter() - t0
    res["tiles_258_config"] = "%d tiles x 258^2, mode 4 8-octave + 1000 droplets/tile, %.1f moves/droplet" % (nt, steps / (nt * 1000.0))
    res["tiles_heightgen_cells_per_s"] = nt * zv * zv / t_gen
    res["tiles_erosion_droplets_per_s"] = nt * 1000 / t_ero
    res["tiles_erosion_moves_per_s"] = steps / t_ero
    res["tiles_fused_pipeline_s"] = t_fused
    res["tiles_separate_calls_s"] = t_gen + t_ero
    res["tiles_fused_cells_per_s"] = nt * zv * zv / t_fused
    res["tiles_fused_droplets_per_s"] = nt * 1000 / t_fused
    del tiles
    # one big heightmap (BASELINE config 3 shape, 8192^2 simplex): the serial droplet order (bit-exact, one warp) and the reference's
    # OpenMP mode (tw_erode_parallel: droplets in flight like `#pragma omp parallel for schedule(dynamic,1)`, order-dependent like the reference)
    cfg = scene.SceneConfig(mesh_gen_mode=1, mesh_freq_filter=1, mesh_seed=1, hmap=HM_CFG, zmax_est=2.3)
    ep = cfg.erosion_params()
    base = torch.empty((N_TILE, N_TILE), dtype=torch.float32, device="cuda")
    _, (zmin, _zmax) = ctx.heightgen_2d(cfg.heightmap_grid(N_TILE, N_TILE), cfg.height_params(), out=base, want_minmax=True)
    work = torch.empty_like(base)
    res["_map_8192"] = base.cpu().numpy()    # the CPU leg erodes the same map (popped by main(), never printed)
    def one_warp(w, n):       # the plain serial walk (one warp, droplet after droplet): what round 1 shipped, kept as the comparison
        os.environ["TW_EROSION_MODE"] = "global"
        try:
            ctx.erode(w, zmin, n, ep)
        finally:
            os.environ.pop("TW_EROSION_MODE", None)
    # "serial" = the reference's serial droplet ORDER, bit for bit; the default path walks the droplets speculatively in parallel and commits them in that order (M_SPEC)
    for name, iters, fn in (("single_map_8192_serial_1000_droplets", 1000, lambda w, n: ctx.erode(w, zmin, n, ep)),
                            ("single_map_8192_serial_100000_droplets", 100000, lambda w, n: ctx.erode(w, zmin, n, ep)),
                            ("single_map_8192_one_warp_walk_1000_droplets", 1000, one_warp),
                            ("single_map_8192_openmp_mode_1e6_droplets", 1000000, lambda w, n: ctx.erode_parallel(w, zmin, n, ep, 0))):
        for rep in range(2):
            work.copy_(base)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn(work, iters)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        res[name + "_s"] = dt
        res[name + "_per_s"] = iters / dt
        res[name + "_moves_per_s"] = ctx.last_erosion_steps / dt
        res[name + "_us_per_move"] = 1e6 * dt / max(1, ctx.last_erosion_steps)
    return res


if __name__ == "__main__":
    main()
