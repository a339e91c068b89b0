"""Where |c|^2 lands in the lean refracting steps, per surface, for a system and a bundle (CPU only).

The lean sphere and flat steps (csrc/lean_steps.cuh) build the Snell basis b^ = (d x n) / |d x n|, c = n x b^, and divide
c by |c|.  They read sqrt(|c|^2) and its reciprocal from a table of the 256 doubles s = bits(1.0) + k, k in [-128, 127]
(csrc/exact_math.cuh, xm::near_one); a ray whose |c|^2 falls outside is re-traced by the careful path (trace_lean.cu:
redo_ray), which costs time and no bit.  This tool is the evidence for the table's size: it prints, per surface with a
lean step, the range of k = bits(|c|^2) - bits(1.0) and the ray-surfaces outside the table.

The point on each surface and the incoming direction come from the CPU oracle's history (the "at" slab), which has the
reference's bits, as the lean steps do; n, b^ and c are then formed with the lean steps' own operations (IEEE products and
quotients, the same left-associated sums).  A workload's sources are sampled by whole lines of their index space (one
azimuth of a fan, one row of a grid), evenly spaced, so every sampled ray is a ray of the full-size bundle.

    python tools/near_unit_histogram.py [--rays 1e6] [workload ...]      (workloads: bench config2 ... config5 tests)
"""
from __future__ import annotations

import argparse
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

TABLE_LO, TABLE_HI = -128, 127
ONE_BITS = np.float64(1.0).view(np.int64)


def _workloads(rt, rtm, systems):
    """name -> (description, system, materials, sources); a source is the argument tuple of oracle.source_rays
    (kind, n_a, n_b, a_max, pt, axis, wavelength, b_max): the same index spaces as bench.py's device sources"""
    vac = rtm.Vacuum()
    out = {}
    relay = systems.relay10_system(rt, rtm)
    relay_mats = [vac] + list(relay.materials) + [vac]
    side = 11181                                   # bench.py: ceil(sqrt(1.25e8))
    out["bench"] = ("relay, the bench step's 11181^2 collimated grid (half-width 12 mm, 0.785 um)", relay, relay_mats,
                    [("grid", side, side, 12.0, (0, 0, 0), (0, 0, 1), 0.785, 12.0)])
    doublet = rt.Doublet(rtm.Nlak22(), rtm.Nsf6ht(), radius_crown=65.8, radius_flint=-280.6, radius_interface=-56,
                         thickness_crown=13.0, thickness_flint=2.0, aperture_radius=25.4, names="AC508-100-B")
    focus_z = float(doublet.get_cardinal_points(0.855, vac, vac)[1][2])
    system = rt.System([rt.FlatSurface([0, 0, -5.0], [0, 0, 1], 25.4)], []).concatenate(doublet, vac)
    system = system.concatenate(rt.FlatSurface([0, 0, focus_z], [0, 0, 1], 25.4), vac)
    out["config2"] = ("AC508-100-B doublet + 2 flats, 3 wavelengths x 4096^2 grid", system,
                      [vac] + list(system.materials) + [vac],
                      [("grid", 4096, 4096, 10.0, (0, 0, -10.0), (0, 0, 1), w, 10.0) for w in (0.7065, 0.855, 1.015)])
    thetas = np.linspace(0, np.pi / 180, 32)
    out["config3"] = ("relay, 32 field bundles x 2048^2 grid", relay, relay_mats,
                      [("grid", 2048, 2048, 12.0, (0, 0, 0), (np.sin(t), 0, np.cos(t)), 0.785, 12.0) for t in thetas])
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    out["config4"] = ("ideal OPM, 16001 x 16000 fan", system, [m_in] + list(system.materials) + [m_out],
                      [("fan", 16001, 16000, alpha1, (1e-3, 1e-3, 1e-3 * np.tan(theta)), (0, 0, 1), 532e-6, 0.0)])
    system = systems.achromat_imaging_system(rt, rtm)
    out["config5"] = ("achromat imaging, 11181 x 11180 fan", system, [vac] + list(system.materials) + [vac],
                      [("fan", 11181, 11180, 4 * np.pi / 180, (2.0, 0, 0), (0, 0, 1), 0.635, 0.0)])
    # the relay under the collimated lattice of tests/test_gpu_lean.py's probe test, which expects no failure at all
    out["tests"] = ("relay, tests' 300^2 collimated lattice (half-width 12 mm)", relay, relay_mats, "lattice")
    return out


def _sample(oracle, systems, sources, n_rays):
    if sources == "lattice":
        yield systems.lattice_rays(300, 12.0, 0.0, 0.785)
        return
    per_source = max(1, int(n_rays) // len(sources))
    for kind, n_a, n_b, a_max, pt, axis, wl, b_max in sources:
        n_lines = min(n_b, max(1, -(-per_source // n_a)))
        for line in np.unique(np.linspace(0, n_b - 1, n_lines).round().astype(np.int64)):
            yield oracle.source_rays(kind, n_a, n_b, a_max, pt, axis, wl, b_max=b_max, first=int(line) * n_a, count=n_a)


def _c_norm_sq(at, nrm):
    """|c|^2 with c = n x ((d x n) / |d x n|), the lean steps' operations; at: (N, 8) rows at the surface"""
    d = at[:, 3:6]
    b = np.stack([d[:, 1] * nrm[:, 2] - d[:, 2] * nrm[:, 1],
                  d[:, 2] * nrm[:, 0] - d[:, 0] * nrm[:, 2],
                  d[:, 0] * nrm[:, 1] - d[:, 1] * nrm[:, 0]], axis=1)
    b = b / np.sqrt((b[:, 0] * b[:, 0] + b[:, 1] * b[:, 1]) + b[:, 2] * b[:, 2])[:, None]
    c = np.stack([nrm[:, 1] * b[:, 2] - nrm[:, 2] * b[:, 1],
                  nrm[:, 2] * b[:, 0] - nrm[:, 0] * b[:, 2],
                  nrm[:, 0] * b[:, 1] - nrm[:, 1] * b[:, 0]], axis=1)
    return (c[:, 0] * c[:, 0] + c[:, 1] * c[:, 1]) + c[:, 2] * c[:, 2]


def histogram(rt, oracle, system, materials, batches):
    """surface index -> (int64 array of k = bits(|c|^2) - bits(1.0) over the rays that reach it, the number of those
    with d x n = 0: a beam along a flat's normal, which the zero-tolerant flat step takes without c)"""
    lean = {}
    for j, s in enumerate(system.surfaces):
        axis = np.asarray(s.input_axis, dtype=float).reshape(-1)
        if isinstance(s, rt.FlatSurface) or (isinstance(s, rt.SphericalSurface) and axis[0] == 0 and axis[1] == 0):
            lean[j] = ([], [0])
    threads = os.cpu_count() or 1
    for rays in batches:
        for lo in range(0, len(rays), 1 << 16):
            hist = oracle.trace(system.surfaces, materials, rays[lo:lo + (1 << 16)], keep_all=True, n_threads=threads)
            for j in lean:
                s = system.surfaces[j]
                at = hist[2 * j + 1]
                at = at[np.isfinite(at[:, :6]).all(axis=1)]
                with np.errstate(all="ignore"):
                    if isinstance(s, rt.SphericalSurface):
                        nrm = (at[:, 0:3] - np.asarray(s.center, dtype=float)[None, :]) / s.radius
                    else:
                        nrm = np.broadcast_to(np.asarray(s.normal, dtype=float).reshape(1, 3), (len(at), 3))
                    sq = _c_norm_sq(at, nrm)
                lean[j][1][0] += int((~np.isfinite(sq)).sum())
                lean[j][0].append(sq[np.isfinite(sq)].view(np.int64) - ONE_BITS)
    return {j: (np.concatenate(k) if k else np.zeros(0, np.int64), along[0]) for j, (k, along) in lean.items()}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("workloads", nargs="*", default=["bench", "config2", "config3", "config4", "config5"])
    ap.add_argument("--rays", type=float, default=1e6, help="rays sampled per workload (whole source lines)")
    args = ap.parse_args()
    import systems
    import ray_trace_pb_b200.materials as rtm
    import ray_trace_pb_b200.raytrace as rt
    from oracle import oracle
    table = _workloads(rt, rtm, systems)
    print(f"k = bits(|c|^2) - bits(1.0); the table holds k in [{TABLE_LO}, {TABLE_HI}]")
    for name in args.workloads:
        what, system, materials, sources = table[name]
        ks = histogram(rt, oracle, system, materials, _sample(oracle, systems, sources, args.rays))
        total = sum(len(k) for k, _ in ks.values())
        outside = sum(int(((k < TABLE_LO) | (k > TABLE_HI)).sum()) for k, _ in ks.values())
        print(f"\n{name}: {what}")
        print(f"  {total} ray-surfaces with a c to normalise at {len(ks)} surfaces with a lean step, {outside} outside "
              f"the table ({outside / max(total, 1):.2e})")
        print("  surface  kind        rays  k min  k max  distinct k  outside  d along n")
        for j, (k, along) in ks.items():
            kind = "sphere" if isinstance(system.surfaces[j], rt.SphericalSurface) else "flat"
            if len(k) == 0:
                print(f"  {j:7d}  {kind:6s}  {0:8d}  {'':5s}  {'':5s}  {'':10s}  {'':7s}  {along:9d}")
                continue
            out = int(((k < TABLE_LO) | (k > TABLE_HI)).sum())
            print(f"  {j:7d}  {kind:6s}  {len(k):8d}  {k.min():5d}  {k.max():5d}  {len(np.unique(k)):10d}  {out:7d}"
                  f"  {along:9d}")

if __name__ == "__main__":
    main()
