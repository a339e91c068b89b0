#!/usr/bin/env python
"""
bench.py -- headline measurement: fp64 ray*surfaces/s of the fused trace on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]              # this framework (one rank per GPU under torchrun)
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]   # the reference algorithm on the host cores
    python bench.py ... --dump-outputs DIR      # also save what the last timed step computed (see dump_outputs)

Workload (BASELINE.json config 5 / north star): the 10-surface achromat relay of
scripts/2022_08_24_relay_astigmatism.py (8 spherical + 2 flat surfaces, 6 Sellmeier + 3 constant media, 0.785 um),
a Cartesian bundle of collimated rays sharded by contiguous index range over the ranks (weak scaling:
--rays-per-gpu rays on every GPU, 1.25e8 by default = 1e9 rays on 8 GPUs).

One step = one pass of the hot path over this rank's rays, resident in HBM as the reference's (N, 8) float64 array:
read 64 B/ray, trace 10 surfaces in registers, write the final (N, 8) slab, and -- fused in the same kernel -- the
spot statistics and the 2048^2 pupil-grid accumulation (sum cos phi, sum sin phi, count); at N > 1 the grid and the
statistics are all-reduced over NCCL (the only communication).  Timed with CUDA events on the launching stream,
barrier + synchronize on both sides, max over ranks.

`value` is device-resident throughput; `e2e` is the same trace through the host-buffer C-ABI call
(rtb_trace_host: pinned host rays in, final slab out, copies inside the timed region).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

# SURVEY.md 8d: algorithmic FP64-pipe instructions and bytes for the 10-surface relay
I_ALG_PER_RAY = 2900.0      # 1268 add/mul + 8*(130 div + 74 sqrt)
F_ALG_PER_RAY = 1472.0      # plain flop count (div = sqrt = 1)
N_SURFACES = 10
BYTES_PER_RAY = 128.0       # 64 B in + 64 B out (final-slab mode)
WAVELENGTH = 0.785
GRID_N = 2048


def relay_system():
    import systems
    import ray_trace_pb_b200.materials as rtm
    import ray_trace_pb_b200.raytrace as rt
    system = systems.relay10_system(rt, rtm)
    materials = [rtm.Vacuum()] + list(system.materials) + [rtm.Vacuum()]
    return system, materials


def beam_source(n_rays_total: int):
    """The whole job's bundle: an on-axis Cartesian grid of collimated rays, half-width 12 mm; ranks take
    contiguous index ranges of it (ray_trace_pb_b200.sharding.shard_range)."""
    from ray_trace_pb_b200.device import RaySource
    side = int(np.ceil(np.sqrt(n_rays_total)))
    return RaySource.grid([0, 0, 0], 12.0, side, WAVELENGTH, n_v=side), side


def link_probe(torch, device: int, nbytes: int = 1 << 28):
    """Host<->device copy rates of THIS box (pinned memory, GB/s): the ceiling of the host-buffer path.  The boxes
    of the pool differ by almost 2x here (virtualised PCIe), so `e2e` is only meaningful next to this."""
    h_in = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d_a = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{device}")
    d_b = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{device}")
    s1, s2 = torch.cuda.Stream(device), torch.cuda.Stream(device)

    def h2d():
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)

    def d2h():
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)

    def best(fn, moved):
        t = 1e30
        for _ in range(3):
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize(device)
            t = min(t, time.perf_counter() - t0)
        return moved / t / 1e9

    out = {"h2d_gbps": best(h2d, nbytes), "d2h_gbps": best(d2h, nbytes),
           "both_gbps": best(lambda: (h2d(), d2h()), 2 * nbytes)}
    out["_both"] = lambda: (h2d(), d2h())          # (for the all-ranks-at-once measurement; removed by the caller)
    out["_bytes"] = 2 * nbytes
    return out


def link_probe_concurrent(torch, dist, probe, world: int, device: int):
    """Every rank copies both ways AT THE SAME TIME (barrier, 3 back-to-back rounds, barrier): the box's aggregate
    host<->device ceiling, which is what the N-GPU host-buffer path competes for."""
    fn, moved = probe.pop("_both"), probe.pop("_bytes")
    if world == 1:
        probe["aggregate_gbps"] = probe["both_gbps"]
        return probe
    rounds = 3
    fn()
    torch.cuda.synchronize(device)
    dist.barrier()
    t0 = time.perf_counter()
    for _ in range(rounds):
        fn()
    torch.cuda.synchronize(device)
    mine = rounds * moved / (time.perf_counter() - t0) / 1e9
    t = torch.tensor([mine], dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    probe["aggregate_gbps"] = float(t[0])
    probe["concurrent_gbps_this_rank"] = mine
    return probe


# SURVEY.md 8d: algorithmic FP64-pipe instructions per surface kind (+ one dispersion evaluation of the new medium)
I_ALG_KIND = {"SphericalSurface": 268.0, "FlatSurface": 210.0, "PlaneMirror": 185.0, "PerfectLens": 330.0}
I_ALG_DISPERSION = 42.0


def algorithmic_instr_per_ray(system, final_material):
    """I_alg of SURVEY.md 8d for any system: per-kind step costs plus 42 per surface whose new medium is dispersive."""
    total = 0.0
    media = list(system.materials) + [final_material]
    for surf, medium in zip(system.surfaces, media):
        kind = next(k.__name__ for k in type(surf).__mro__ if k.__name__ in I_ALG_KIND)
        total += I_ALG_KIND[kind]
        if type(medium).__name__ not in ("Vacuum", "Constant"):
            total += I_ALG_DISPERSION
    return total


def config_block(torch, dfma_rate: float):
    """BASELINE.json configs 1-5 at full size on this GPU, device part only, timed with CUDA events (best of 3 after a
    warm-up): the systems of the reference's scripts with their own bundles, through the same public calls as
    examples/run_configs.py.  `frac` = FP64-pipe instructions the config's kernels execute (ncu) x rays/s / the measured DFMA
    rate; `algorithmic` = the same with that system's own I_alg (SURVEY.md 8d)."""
    import systems
    import ray_trace_pb_b200.materials as rtm
    import ray_trace_pb_b200.raytrace as rt
    from ray_trace_pb_b200 import analysis, device as dev

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return best

    vac = rtm.Vacuum()
    out = {}

    # FP64-pipe instructions each config's kernels EXECUTE per ray (ncu, tools/config_counts.sh): `frac` is the share of
    # the pipe's issue slots in use, like the headline's; the algorithmic form of SURVEY.md 8d rides along
    try:
        counts = json.loads((ROOT / "profiles" / "r02_config_counts.json").read_text())
    except Exception:
        counts = {}

    def entry(name, workload, system, m_out, n_rays, ms):
        i_alg = algorithmic_instr_per_ray(system, m_out)
        n_surf = len(system.surfaces)
        rays_per_s = n_rays / (ms * 1e-3)
        executed = counts.get(name, {}).get("fp64_pipe_instr_per_ray")
        roof = {"bound": "fp64", "peak": dfma_rate / 1e9, "unit": "G FP64-pipe instr/s",
                "algorithmic": {"instr_per_ray": i_alg, "achieved": i_alg * rays_per_s / 1e9,
                                "frac": i_alg * rays_per_s / dfma_rate}}
        if executed is not None:
            roof.update({"executed_fp64_instr_per_ray": executed, "achieved": executed * rays_per_s / 1e9,
                         "frac": executed * rays_per_s / dfma_rate,
                         "note": "kernel_ms spans the whole call (probe launch, reduction reset, host gaps), so this "
                                 "is a lower bound of the trace kernel's own pipe utilisation"})
        else:
            roof.update({"achieved": i_alg * rays_per_s / 1e9, "frac": i_alg * rays_per_s / dfma_rate,
                         "note": "algorithmic count (no ncu count for this config)"})
        out[name] = {"workload": workload, "rays": int(n_rays), "surfaces": n_surf, "kernel_ms": ms,
                     "value": rays_per_s * n_surf, "unit": "ray*surfaces/s", "roofline": roof}

    # config 1: scripts/2022_10_27_plano_convex_lens.py scaled up (1001 x 1000 collimated rays), final slab
    system, m_in, m_out, _ = systems.plano_convex(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    src = dev.RaySource.collimated([0, 0, -5], 25.4, 1001, 0.5, nphis=1000)
    ms = timed(lambda: dev.trace_source(system.surfaces, mats, src, keep="last"))
    entry("config1", "plano-convex lens, 1001 x 1000 collimated rays generated on the device, final slab", system, m_out,
          src.n_rays, ms)
    # config 2: scripts/2022_08_04_ACT508-100-B.py:58-72, 3 wavelengths x 4096^2 grid, spot statistics at the d-line focus
    doublet = rt.Doublet(rtm.Nlak22(), rtm.Nsf6ht(), radius_crown=65.8, radius_flint=-280.6, radius_interface=-56,
                         thickness_crown=13.0, thickness_flint=2.0, aperture_radius=25.4, names="AC508-100-B")
    wls = (0.7065, 0.855, 1.015)
    focus_z = float(doublet.get_cardinal_points(0.855, vac, vac)[1][2])
    system = rt.System([rt.FlatSurface([0, 0, -5.0], [0, 0, 1], 25.4)], []).concatenate(doublet, vac)
    system = system.concatenate(rt.FlatSurface([0, 0, focus_z], [0, 0, 1], 25.4), vac)
    sources = [dev.RaySource.grid([0, 0, -10.0], 10.0, 4096, w) for w in wls]
    ms = timed(lambda: analysis.spot_statistics(system, vac, vac, sources, slab=-2))
    entry("config2", "AC508-100-B doublet + 2 flats, 3 wavelengths x 4096^2 grid in one sweep launch, fused spot "
          "statistics at the focal plane (includes the statistics' device->host read)", system, vac, 3 * sources[0].n_rays, ms)
    # config 3: scripts/2022_08_24_relay_astigmatism.py, 32 field bundles x 2048^2
    system = systems.relay10_system(rt, rtm)
    thetas = np.linspace(0, np.pi / 180, 32)
    sources = [dev.RaySource.grid([0, 0, 0], 12.0, 2048, WAVELENGTH, normal=(np.sin(t), 0, np.cos(t))) for t in thetas]
    ms = timed(lambda: analysis.spot_statistics(system, vac, vac, sources, slab=-2))
    entry("config3", "10-surface relay, 32 field bundles x 2048^2 rays in one sweep launch, fused spot statistics per "
          "field (includes the statistics' device->host read)", system, vac, 32 * sources[0].n_rays, ms)
    # config 4: scripts/2022_01_25_ray_trace_ideal_opm.py, 16001 x 16000 fan -> O3 pupil grid
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    src = dev.RaySource.fan([1e-3, 1e-3, 1e-3 * np.tan(theta)], alpha1, 16001, 532e-6, nphis=16000)
    o3n = system.surfaces[8].normal
    e2 = np.array([0.0, 1.0, 0.0])
    e1 = np.cross(e2, o3n)
    chief = system.ray_trace(rt.get_ray_fan([1e-3, 1e-3, 1e-3 * np.tan(theta)], 0.0, 1, 532e-6), m_in, m_out)
    ms = timed(lambda: analysis.pupil_grid(system, m_in, m_out, src, slab=-5, origin=system.surfaces[8].center, e1=e1,
                                           e2=e2, grid_n=GRID_N, half_width=3.2, phase_ref=float(chief[-5, 0, 6])), reps=2)
    entry("config4", "ideal OPM (6 perfect lenses + 5 flats, one tilted), 16001 x 16000 ray fan generated on the device "
          "-> 2048^2 pupil grid at O3", system, m_out, src.n_rays, ms)
    # config 5 on the script's own system: scripts/2024_08_08_achromat_imaging.py, one GPU's share of 1e9 rays
    system = systems.achromat_imaging_system(rt, rtm)
    src = dev.RaySource.fan([2.0, 0, 0], 4 * np.pi / 180, 11181, 0.635, nphis=11180)
    pupil = system.surfaces[4]
    ms = timed(lambda: analysis.pupil_grid(system, vac, vac, src, slab=2 * 4 + 2, origin=pupil.center, e1=(1, 0, 0),
                                           e2=(0, 1, 0), grid_n=GRID_N, half_width=8.0))
    entry("config5_achromat", "9-surface achromat imaging system (two AC508-075-A-ML, Ebaf11 / Nsf11 tabulated on the "
          "host), 1.25e8-ray fan generated on the device -> 2048^2 pupil grid at the stop", system, vac, src.n_rays, ms)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.t_mark = 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def mark(self):
        """the timed region starts now: only samples that arrive from here on are reported"""
        self.t_mark = time.monotonic()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for t_line, line in self.lines:
            if t_line < self.t_mark:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline_run(n_threads: int, target_seconds: float = 12.0):
    """The oracle port (oracle/rt_oracle.c, OpenMP) on a bounded sample of the same workload, all host cores."""
    import systems
    import ray_trace_pb_b200.materials as rtm
    import ray_trace_pb_b200.raytrace as rt
    from oracle import oracle
    system = systems.relay10_system(rt, rtm)
    materials = [rtm.Vacuum()] + list(system.materials) + [rtm.Vacuum()]

    def run(n_side):
        rays = systems.lattice_rays(n_side, 12.0, 0.0, WAVELENGTH)
        go = oracle.prepared_trace(system.surfaces, materials, rays, keep_all=False, n_threads=n_threads)
        t0 = time.perf_counter()
        go()
        return rays.shape[0], time.perf_counter() - t0

    n, dt = run(512)                                           # calibration: 262,144 rays
    rate = n * N_SURFACES / dt
    side = int(min(4096, max(512, np.sqrt(rate * target_seconds / N_SURFACES))))
    best = None
    for _ in range(2):
        n, dt = run(side)
        r = n * N_SURFACES / dt
        best = r if best is None else max(best, r)
    return best, f"{side}x{side} = {side * side} rays x {N_SURFACES} surfaces, final slab only, best of 2"


def dump_outputs(path: Path, out, reducer, n_rows: int = 1 << 18, n_cells: int = 1 << 20):
    """What the timed step hands its caller, as finite float64 .npy files (42 MB at most) for comparing two builds
    output for output.  A fixed seeded sample of the final slab's rays (in index order) is split in two, since the
    trace marks a ray that leaves the system (outside an aperture, total internal reflection) with NaN:
    final_slab_alive.npy, 1 or 0 per sampled ray for whether its whole row is finite, and final_slab.npy, the rows of
    the sampled rays that came through.  spot_stats.npy holds the spot statistics; pupil_grid.npy, a fixed seeded
    sample of the pupil grid's cells, (3 planes, cells)."""
    import torch
    path.mkdir(parents=True, exist_ok=True)
    n = out.shape[1]
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, n_rows), replace=False))
    slab = out[0, torch.as_tensor(rows, device=out.device)].cpu().numpy()
    alive = np.isfinite(slab).all(axis=1)
    np.save(path / "final_slab_alive.npy", alive.astype(np.float64))
    np.save(path / "final_slab.npy", slab[alive])
    if reducer is not None and reducer.stats_t is not None:
        np.save(path / "spot_stats.npy", reducer.stats_t.cpu().numpy())
    if reducer is not None and reducer.grid_t is not None:
        grid = reducer.grid_t.reshape(3, -1)
        cells = np.sort(np.random.default_rng(1).choice(grid.shape[1], size=min(grid.shape[1], n_cells), replace=False))
        np.save(path / "pupil_grid.npy", grid[:, torch.as_tensor(cells, device=out.device)].cpu().numpy())


WORKLOAD = ("relay10 (BASELINE config 5 system): 10-surface achromat relay, 0.785 um, collimated Cartesian bundle, "
            "final slab + fused pupil reduction")


def numpy_leg(procs: int, reps: int, budget_s: float, rays: int = 1_000_000):
    """The UNMODIFIED reference's NumPy path (baseline/_ref, installed by baseline/install_ref.sh) on the host cores:
    SURVEY.md 8d "CPU baseline timing".  Runs in fresh interpreters (baseline/numpy_leg.py): nothing of this
    framework is imported there."""
    script = ROOT / "baseline" / "numpy_leg.py"
    try:
        r = subprocess.run([sys.executable, str(script), "--rays", str(rays), "--procs", str(procs), "--reps", str(reps),
                            "--budget-s", str(budget_s)], capture_output=True, text=True, timeout=900)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as exc:                                    # reported, never fatal: it is a baseline
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


def run_reference(args):
    """--impl reference: the reference's algorithm on all host cores.  `value` is the C restatement (oracle/rt_oracle.c,
    OpenMP) -- some 40x faster per core than the reference's own NumPy code, i.e. the harder baseline; the unmodified
    NumPy path on the same cores is reported next to it (cpu_baseline.numpy_allcores)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import systems
    import ray_trace_pb_b200.materials as rtm
    import ray_trace_pb_b200.raytrace as rt
    from oracle import oracle
    oracle.build()
    cores = os.cpu_count() or 1
    system = systems.relay10_system(rt, rtm)
    materials = [rtm.Vacuum()] + list(system.materials) + [rtm.Vacuum()]
    side = 2048                                                 # 4.2M rays per step: a bounded sample
    rays = systems.lattice_rays(side, 12.0, 0.0, WAVELENGTH)
    go = oracle.prepared_trace(system.surfaces, materials, rays, keep_all=False, n_threads=cores)
    warm = oracle.prepared_trace(system.surfaces, materials, rays[:200_000], keep_all=False, n_threads=cores)
    for _ in range(args.warmup):
        warm()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        go()
    dt = time.perf_counter() - t0
    value = rays.shape[0] * N_SURFACES * args.steps / dt
    sample = (f"a bounded sample of the same bundle per step: {side}x{side} = {rays.shape[0]} rays x {N_SURFACES} surfaces "
              f"(same system, same wavelength, same 12 mm half-width; the final slab is produced, the pupil reduction -- "
              f"3 atomics per ray on the GPU -- is not part of the CPU arm)")
    line = {"impl": "reference", "metric": "ray_surfaces_per_s_fp64", "value": value, "unit": "ray*surfaces/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": value, "unit": "ray*surfaces/s", "cores": cores, "kind": "port", "sample": sample,
                             "numpy_allcores": numpy_leg(cores, 2, 15.0)},
            "e2e": {"value": value, "unit": "ray*surfaces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rays-per-gpu", type=float, default=1.25e8)
    ap.add_argument("--e2e-rays", type=float, default=float(1 << 24))
    ap.add_argument("--reduce", default="grid", choices=["none", "stats", "grid"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config block (BASELINE configs 1-5, N = 1)")
    ap.add_argument("--no-bind", action="store_true", help="do not pin each rank to its GPU's local CPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from ray_trace_pb_b200 import _ffi, device as dev, engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # one process per GPU: sit on the CPUs next to that GPU before any page-locked buffer is allocated
    from ray_trace_pb_b200.sharding import bind_to_device_cpus
    all_cpus = os.sched_getaffinity(0)
    bound = None if args.no_bind else bind_to_device_cpus(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    L = _ffi.lib()
    _ffi.require_device()

    system, materials = relay_system()
    from ray_trace_pb_b200.sharding import shard_range
    source, side = beam_source(int(args.rays_per_gpu) * world)
    first, n_rays = shard_range(source.n_rays, rank, world)

    # ---- resident inputs / outputs ---------------------------------------------------------------------
    rays = source.generate(first=first, count=n_rays, device=local)         # this rank's (N, 8) shard in HBM
    out = torch.empty((1, n_rays, 8), dtype=torch.float64, device=f"cuda:{local}")
    # Two reducers, used alternately: step i's grid / statistics are exchanged (NCCL, on a side stream) while step
    # i+1 traces into the other one -- the exchange is the only communication of the job and nothing waits for it
    # except the reset of the same reducer two steps later and the end of the timed region.
    reducers = []
    if args.reduce != "none":
        # sample just after the second doublet (slab 12), where the relay's beam is collimated: the pupil
        reducers = [dev.Reducer(12, origin=(8.0, 0, 0), grid_n=GRID_N if args.reduce == "grid" else 0,
                                half_width=8.0, device=local) for _ in range(2 if world > 1 else 1)]
    reducer = reducers[0] if reducers else None
    comm = None
    if world > 1 and reducers:
        from ray_trace_pb_b200.sharding import Comm
        comm = Comm.from_torch_distributed(local)          # the library's own communicator (rtb_comm_*, C ABI)
    comm_stream = torch.cuda.Stream(local) if comm is not None else None
    ev_traced = [torch.cuda.Event() for _ in reducers]
    ev_reduced = [torch.cuda.Event() for _ in reducers]

    def step(i, k0=None, k1=None):
        red = reducers[i % len(reducers)] if reducers else None
        slot = i % len(reducers) if reducers else 0
        if red is not None:
            if comm is not None:
                torch.cuda.current_stream().wait_event(ev_reduced[slot])     # its last exchange has to be over
            red.reset()
        if k0 is not None:
            k0.record()
        dev.trace_tensor(system.surfaces, materials, rays, keep="last", wavelengths=[WAVELENGTH], reducer=red, out=out)
        if k1 is not None:
            k1.record()
        if comm is not None:
            ev_traced[slot].record()
            with torch.cuda.stream(comm_stream):
                comm_stream.wait_event(ev_traced[slot])
                red.allreduce(comm=comm)
                ev_reduced[slot].record(comm_stream)

    def join_exchange():
        if comm_stream is not None:
            torch.cuda.current_stream().wait_stream(comm_stream)

    # ---- roofline denominators measured live --------------------------------------------------------------
    dfma = ctypes.c_double()
    ms_probe = ctypes.c_double()
    _ffi.check(L.rtb_measure_dfma_rate(local, ctypes.byref(dfma), ctypes.byref(ms_probe)))
    # the same pipe fed by latency-bound warps (one dependent chain each, the trace kernels' occupancy): DESIGN.md 4a
    dfma_chain = ctypes.c_double()
    _ffi.check(L.rtb_measure_dfma_chain_rate(local, 1, ctypes.byref(dfma_chain), ctypes.byref(ms_probe)))
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    # what the dominant kernel executes per ray, from its ncu capture (profiles/r02_traffic.json: opcode counts and DRAM
    # bytes of trace_lean_kernel on this workload)
    prof = {}
    try:
        tj = json.loads((ROOT / "profiles" / "r02_traffic.json").read_text())
        prof = tj if args.reduce != "none" else tj["fast_kernel"]
    except Exception:
        pass
    traffic_per_ray = prof.get("dram_bytes_per_ray")
    EXEC_FP64_PER_RAY = prof.get("fp64_pipe_instr_per_ray")
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "MEASURED_PEAKS.json (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"

    # nvidia-smi takes a few hundred ms to deliver its first sample: it is started before the warm-up so that samples
    # are already flowing (every 20 ms) when the timed region begins; only those taken inside the region are reported
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for w in range(max(args.warmup, 3)):
        step(w)
        if w == 0:
            # the first launch of a system feeds the library's verdict cache (its probe counts are read back
            # asynchronously); waiting for it here puts the remaining warm-up steps in the steady state -- the pure
            # lean kernels -- instead of leaving their first launch to the timed region
            join_exchange()
            torch.cuda.synchronize()
    join_exchange()
    torch.cuda.synchronize()
    if rank == 0:
        deadline = time.monotonic() + 2.0
        while not sampler.lines and sampler.proc is not None and time.monotonic() < deadline:
            # (still warm-up, this rank only -- no collective) keep the GPU under load until the first sample is in
            dev.trace_tensor(system.surfaces, materials, rays, keep="last", wavelengths=[WAVELENGTH], reducer=reducer,
                             out=out)
            torch.cuda.synchronize()

    # ---- timed region -----------------------------------------------------------------------------------------
    if rank == 0:
        sampler.mark()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = L.rtb_launch_count()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev0.record()
    for i in range(args.steps):
        step(i, k0[i], k1[i])
    join_exchange()
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = L.rtb_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev0.elapsed_time(ev1)
    kernel_ms = [a.elapsed_time(b) for a, b in zip(k0, k1)]
    t = torch.tensor([elapsed_ms, statistics.mean(kernel_ms)], dtype=torch.float64, device=f"cuda:{local}")
    per_rank = [t.clone() for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, kernel_ms_mean = float(t[0]), float(t[1])
    kernel_ms_per_rank = [float(x[1]) for x in per_rank]
    total_ray_surfaces = float(source.n_rays) * N_SURFACES * args.steps
    value = total_ray_surfaces / (elapsed_ms * 1e-3)

    # sanity: the trace did real work (valid rays came out)
    n_valid = int(torch.isfinite(out[0, :, 0]).sum())
    last = reducers[(args.steps - 1) % len(reducers)] if reducers else None
    stats = last.stats() if (last is not None and last.stats_t is not None) else None
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), out, last)

    # ---- the reference's own output mode (full (2S+1, N, 8) history), device resident: the HBM-bound regime ------
    full_history = None
    if rank == 0:
        n_fh = min(n_rays, 4_000_000)
        fh_out = torch.empty((2 * N_SURFACES + 1, n_fh, 8), dtype=torch.float64, device=f"cuda:{local}")
        fh_in = rays[:n_fh]
        for _ in range(2):
            dev.trace_tensor(system.surfaces, materials, fh_in, keep="all", wavelengths=[WAVELENGTH], out=fh_out)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(5):
            dev.trace_tensor(system.surfaces, materials, fh_in, keep="all", wavelengths=[WAVELENGTH], out=fh_out)
        f1.record()
        torch.cuda.synchronize()
        fh_ms = f0.elapsed_time(f1) / 5
        fh_bytes = n_fh * 64.0 * (2 * N_SURFACES + 2)                # 64 B in + 21 x 64 B out per ray
        full_history = {"bound": "hbm", "achieved": fh_bytes / (fh_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": fh_bytes / (fh_ms * 1e-3) / 1e9 / hbm_peak, "rays": n_fh, "kernel_ms": fh_ms,
                        "ray_surfaces_per_s": n_fh * N_SURFACES / (fh_ms * 1e-3),
                        "algorithmic_bytes_per_ray": 64.0 * (2 * N_SURFACES + 2), "peak_source": hbm_src}
        del fh_out

    # ---- the other arithmetic modes on the same resident rays (final slab only): the north star's fp32 mode with its
    # stated tolerance, and the FMA fp64 mode (tests/test_gpu_parity.py::test_fast_modes_tolerance holds both to them) ----
    other_modes = None
    if rank == 0:
        other_modes = {}
        n_m = min(n_rays, 40_000_000)
        m_in = rays[:n_m]
        m_out = torch.empty((1, n_m, 8), dtype=torch.float64, device=f"cuda:{local}")
        for mode, note in (("f64", "bit-exact (the headline's arithmetic), final slab only, no reduction"),
                           ("f64_fast", "fp64 with FMA and the direct Snell form: positions 1e-11 L, directions / phase 1e-12"),
                           ("f32", "fp32 geometry, fp64 positions / sphere quadratic / phase: positions and directions 2e-6")):
            for _ in range(2):
                dev.trace_tensor(system.surfaces, materials, m_in, keep="last", wavelengths=[WAVELENGTH], out=m_out,
                                 precision=mode)
                torch.cuda.synchronize()
            best = None
            for _ in range(3):
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                dev.trace_tensor(system.surfaces, materials, m_in, keep="last", wavelengths=[WAVELENGTH], out=m_out,
                                 precision=mode)
                f1.record()
                torch.cuda.synchronize()
                ms = f0.elapsed_time(f1)
                best = ms if best is None else min(best, ms)
            other_modes[mode] = {"value": n_m * N_SURFACES / (best * 1e-3), "unit": "ray*surfaces/s", "rays": n_m,
                                 "kernel_ms": best, "tolerance": note}
        del m_out

    # ---- end-to-end through the host-buffer C ABI ---------------------------------------------------------------
    n_e2e = int(args.e2e_rays)
    e2e_side = int(np.sqrt(n_e2e))
    n_e2e = e2e_side * e2e_side
    e2e_src, _ = beam_source(n_e2e * world)
    e2e_first, n_e2e = shard_range(e2e_src.n_rays, rank, world)
    host_in = _ffi.pinned_empty((n_e2e, 8))
    host_in[:] = e2e_src.generate(first=e2e_first, count=n_e2e, device=local).cpu().numpy()
    host_out = _ffi.pinned_empty((1, n_e2e, 8))
    for _ in range(2):
        engine.trace_host(system.surfaces, materials, host_in, keep="last", device=local, out=host_out)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        engine.trace_host(system.surfaces, materials, host_in, keep="last", device=local, out=host_out)
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = float(e2e_src.n_rays) * N_SURFACES * e2e_steps / float(te[0])
    assert np.isfinite(host_out[0, n_e2e // 2, 0])
    link = link_probe_concurrent(torch, dist, link_probe(torch, local), world, local)

    # the unmodified reference call: System.ray_trace(numpy rays) -> full (2S+1, N, 8) history in host memory
    dropin = None
    if rank == 0:
        import systems
        probe = systems.lattice_rays(1000, 12.0, 0.0, WAVELENGTH)               # 1e6 rays, pageable NumPy
        vac = materials[0]
        best = None
        for _ in range(4):
            t0 = time.perf_counter()
            hist = system.ray_trace(probe, vac, vac)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        dropin = {"value": probe.shape[0] * N_SURFACES / best, "unit": "ray*surfaces/s", "rays": int(probe.shape[0]),
                  "api": "System.ray_trace(numpy (N,8)) -> numpy (21, N, 8), the reference's own call",
                  "d2h_bytes": int(hist.nbytes), "h2d_bytes": int(probe.nbytes)}
        del hist

    # ---- BASELINE configs 1-5 on one GPU (the headline above is config 5's size on the relay) -----------------------
    configs = None
    if rank == 0 and world == 1 and not args.no_configs:
        del rays, out
        torch.cuda.empty_cache()
        try:
            configs = config_block(torch, dfma.value)
        except Exception as exc:                               # reported, not fatal: the headline stands on its own
            configs = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        rays_per_s_gpu = float(n_rays) / (kernel_ms_mean * 1e-3)
        achieved_inst = I_ALG_PER_RAY * rays_per_s_gpu
        line = {
            "metric": "ray_surfaces_per_s_fp64", "value": value, "unit": "ray*surfaces/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "rays_total": source.n_rays, "rays_rank0": n_rays, "surfaces": N_SURFACES, "keep": "last", "reduce": args.reduce,
                       "grid": GRID_N if args.reduce == "grid" else 0,
                       "l2": "inputs (8 GB/GPU at the default size) are larger than L2; no flush needed",
                       "valid_rays_rank0": n_valid, "parity": "fp64 bit-exact mode"},
            # frac = FP64-pipe instructions the kernel EXECUTES per second / the measured DFMA rate: the share of the FP64
            # pipe's issue slots in use, which is what ncu's sm__pipe_fp64_cycles_active reports for the same kernel
            # (profiles/r02_bench_step_ncu_summary.txt).  The algorithmic form of SURVEY.md 8d (2900 instr/ray: every
            # division and square root counted as its own 8-instruction sequence, no shared reciprocals) is kept below.
            "roofline": {"bound": "fp64",
                         "achieved": None if EXEC_FP64_PER_RAY is None else EXEC_FP64_PER_RAY * rays_per_s_gpu / 1e9,
                         "peak": dfma.value / 1e9, "unit": "G FP64-pipe instr/s",
                         "frac": None if EXEC_FP64_PER_RAY is None else EXEC_FP64_PER_RAY * rays_per_s_gpu / dfma.value,
                         "traffic": None if traffic_per_ray is None else traffic_per_ray * n_rays,
                         "traffic_note": "DRAM bytes per launch = ncu dram__bytes_read+write per ray (profiles/r02_traffic.json) "
                                         "x rays of this launch; algorithmic = 128 B/ray",
                         "peak_source": "DFMA register micro-benchmark run in this process (rtb_measure_dfma_rate)",
                         "kernel": "trace_lean_kernel (csrc/trace_lean.cu)", "kernel_ms": kernel_ms_mean,
                         "kernel_ms_per_rank": kernel_ms_per_rank,
                         "executed": {"fp64_instr_per_ray": EXEC_FP64_PER_RAY,
                                      "other_instr_per_ray": prof.get("other_instr_per_ray"),
                                      "ncu_fp64_pipe_active_pct": prof.get("fp64_pipe_active_pct"),
                                      "note": "per-ray counts from ncu opcode statistics; the kernel is bound by the "
                                              "sub-partition's operand-read port, which every pipe shares: cycles per "
                                              "ray ~ 2 x FP64 + 1 per DFMA with three register operands + 1 per other "
                                              "instruction (DESIGN.md 4a, tools/ubench/rf_bandwidth.cu)"},
                         "algorithmic": {"instr_per_ray": I_ALG_PER_RAY, "achieved": achieved_inst / 1e9,
                                         "frac": achieved_inst / dfma.value,
                                         "dependent_dfma_chain_rate": dfma_chain.value / 1e9},
                         "flops_form": {"achieved_tflops": F_ALG_PER_RAY * rays_per_s_gpu / 1e12,
                                        "peak_tflops_fma2": 2 * dfma.value / 1e12},
                         "hbm": {"achieved": BYTES_PER_RAY * rays_per_s_gpu / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": BYTES_PER_RAY * rays_per_s_gpu / 1e9 / hbm_peak, "peak_source": hbm_src}},
            "e2e": {"value": e2e_value, "unit": "ray*surfaces/s", "h2d_bytes_per_step": n_e2e * 64,
                    "d2h_bytes_per_step": n_e2e * 64, "rays_per_gpu_per_step": n_e2e, "steps": e2e_steps,
                    "api": "rtb_trace_host via engine.trace_host (pinned host buffers, keep='last')",
                    "link": link, "cpus_bound_rank0": (len(bound) if bound else None),
                    # bytes the job moves per second over the host links, against what all ranks' links deliver at once
                    "link_frac": (e2e_value / N_SURFACES * 128 / 1e9) / link["aggregate_gbps"],
                    "link_frac_note": "e2e bytes/s (64 B in + 64 B out per ray, all ranks) / link.aggregate_gbps, the "
                                      "rate measured with every rank copying both ways at the same time"},
            "roofline_full_history": full_history, "other_modes": other_modes,
            "configs": configs,
            "dropin_full_history": dropin,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if stats is not None:
            line["config"]["reduce_count"] = stats["count"]
        if not args.no_cpu_baseline and world == 1:        # the CPU baseline is reported at N = 1 only
            os.sched_setaffinity(0, all_cpus)               # the CPU baseline gets every core of the box again
            cores = len(all_cpus)
            v, sample = cpu_baseline_run(cores)
            line["cpu_baseline"] = {"value": v, "unit": "ray*surfaces/s", "cores": cores, "kind": "port", "sample": sample,
                                    # the reference's own NumPy code (unmodified, baseline/_ref), 1 core and all cores
                                    "numpy_1core": numpy_leg(1, 2, 20.0),
                                    "numpy_allcores": numpy_leg(cores, 3, 20.0)}
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
