"""
The two fast trace modes (precision "f32" and "f64_fast", csrc/trace_fast.cu) against the fp64 reference on every kernel
route (`-m gpu`).  The reference is the CPU oracle's history or, where the oracle would be too slow, the exact mode on
the device, which is bit-identical to it (tests/test_gpu_parity.py).  Every comparison goes through
tests/fast_tolerance.py: values within the stated tolerance until a ray's first departure, and every first departure
explained by a knife edge of the reference.  Each route prints its largest error per column as a multiple of the
tolerance and its explained rays per reason (run with -s to see them).

Which test reaches which instantiation trace_fast_kernel<T, USE_TABLE, FROM_SOURCE, SWEEP, LAST> (for T = float and
T = double alike: every test runs in both modes; test_every_instantiation_is_launched checks the list with the
profiler):

    USE_TABLE FROM_SOURCE SWEEP  LAST  reached by
    true      false       false  0     test_device_rays (keep all / list, rows and planes), test_systems, test_host_paths,
                                       test_intersect_only, test_reductions (keep=[slab], reduction at slab 0)
    true      false       false  1     test_device_rays (keep "last"), test_bench_workload
    true      false       false  2     test_reductions (keep "last" / "none" + reduction behind the launch rays)
    false     false       false  0     test_device_rays (wavelengths=None, keep all)
    false     false       false  1     test_device_rays (wavelengths=None, keep "last")
    false     false       false  2     test_reductions (wavelengths=None)
    true      true        false  0     test_sources (keep all, first / count slice)
    true      true        false  1     test_sources (keep "last")
    true      true        false  2     test_sources (keep "last" + reduction)
    false     true        false  0/1/2 test_sources (system packed without a table: in-kernel Sellmeier)
    true      true        true   0/1/2 test_sweeps (keep list / "last" / "none" + reduction)
    false     true        true   0/1/2 test_sweeps (more than 8 wavelengths through closed-formula media)

A sampled host table with unlisted wavelengths runs in the USE_TABLE = true kernels (test_device_rays, test_host_paths).
"""
import re

import numpy as np
import pytest

import fast_tolerance as ft
import systems

pytestmark = pytest.mark.gpu

MODES = ["f32", "f64_fast"]


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    return torch


@pytest.fixture(scope="module")
def dev():
    import ray_trace_pb_b200.device as dev
    return dev


def _check(what, got, want_hist, slabs, mode, surfaces, mats, hard=False, minority=0.01):
    rep = ft.compare(got, want_hist, slabs, mode, hard, surfaces, mats)
    print(rep.summary(what))
    if minority is not None and hard is not True:          # explained rays are capped outside the hard class
        ft.assert_minority(rep, minority, what)
    return rep


def _np(t):
    return t.cpu().numpy()


def _mats(system, m_in, m_out):
    return [m_in] + list(system.materials) + [m_out]


# ------------------------------------------------------------------------------------------------ device rays
@pytest.mark.parametrize("mode", MODES)
def test_device_rays(mode, rt, rtm, oracle, torch, dev):
    """rows / planes, keep all / list / "last", host table / in-kernel Sellmeier / a sampled table with unlisted rays"""
    system, m_in, m_out, rays = systems.relay10(rt, rtm, n_disps=41, nphis=36, n_fields=4)
    rays[::7, 7] = 0.6328
    mats = _mats(system, m_in, m_out)
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    S = want.shape[0]
    d = torch.from_numpy(rays).cuda()
    planes = d.t().contiguous()
    for wavelengths in ("auto", None, [0.785]):          # [0.785]: the 0.6328 rays are not in the table
        tag = f"wavelengths={wavelengths}"
        got = dev.trace_tensor(system.surfaces, mats, d, keep="all", precision=mode, wavelengths=wavelengths)
        _check(f"relay rows keep all {tag}", _np(got), want, range(S), mode, system.surfaces, mats)
        last = dev.trace_tensor(system.surfaces, mats, d, keep="last", precision=mode, wavelengths=wavelengths)
        _check(f"relay rows keep last {tag}", _np(last), want, [S - 1], mode, system.surfaces, mats)
    keep = [0, 3, 8, 13, S - 1]
    got = dev.trace_tensor(system.surfaces, mats, planes, keep=keep, precision=mode, layout="planes",
                           wavelengths=[0.785, 0.6328])
    _check("relay planes keep list", _np(got.permute(0, 2, 1)), want, keep, mode, system.surfaces, mats)
    got = dev.trace_tensor(system.surfaces, mats, planes, keep="last", precision=mode, layout="planes",
                           wavelengths=None)
    _check("relay planes keep last Sellmeier", _np(got.permute(0, 2, 1)), want, [S - 1], mode, system.surfaces, mats)


# ------------------------------------------------------------------------------------------------ systems
def _bundle_cases(rt, rtm):
    for seed in range(systems.N_RANDOM_SYSTEMS):
        system, m_in, m_out, rays = systems.random_system(rt, rtm, seed)
        yield f"random {seed}", system, m_in, m_out, rays, "random_system"
    for which in range(5):
        system, m_in, m_out, rays = systems.launched_on_plane(rt, rtm, which, n=4000, seed=1234)
        yield f"launched on plane {which}", system, m_in, m_out, rays, "launched_on_plane"
    system, m_in, m_out, rays = systems.retro_mirror(rt, rtm)
    yield "retro mirror", system, m_in, m_out, np.concatenate(
        (rays, rt.get_collimated_rays([0, 0, -5], 12.0, 60, 0.6, nphis=40))), "retro_mirror"
    system, m_in, m_out, rays = systems.perfect_imaging_in_focus(rt, rtm, n_thetas=61, nphis=40)
    yield "perfect imaging in focus", system, m_in, m_out, rays, "perfect_imaging"
    system, m_in, m_out, rays = systems.perfect_imaging(rt, rtm, n_thetas=61, nphis=40)
    yield "perfect imaging", system, m_in, m_out, rays, "perfect_imaging"
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    rays = rt.get_ray_fan([1e-3, -2e-3, 5e-4], 1.05 * alpha1, 201, 532e-6, nphis=60)
    yield "opm", system, m_in, m_out, rays, "opm"
    system = systems.relay10_system(rt, rtm)
    skew = []
    for k, (tx, ty) in enumerate(((0.012, 0.0), (0.0, -0.015), (0.009, 0.011), (-0.02, 0.004))):
        skew.append(systems.lattice_rays(61, 13.0, 0.0, (0.785, 0.6328, 0.9, 0.785)[k], tilt=(tx, ty)))
    yield "relay skew", system, rtm.Vacuum(), rtm.Vacuum(), np.concatenate(skew), "relay10"


# Open f32 findings, each limited to one named bundle and a numeric ceiling: the bundle must still pass its class
# scaled by the ceiling, every other bundle and every other failure still fails, and the test then reports an
# expected failure naming them.  Neither is localized to a kernel operation yet:
#   opm: 4 of 12 060 rays leave the O3 objective (f = 2 mm) with a direction error of up to 4x the hard class;
#   launched on plane 4: behind a perfect lens at the launch plane the phase, a small sum of ~5e2 rad terms of both
#   signs, exceeds even the PHASE_F32 class.
OPEN_F32 = {"opm": (1.0, 5.0, 1.0), "launched on plane 4": (1.0, 1.0, 10.0)}


@pytest.mark.parametrize("mode", MODES)
def test_systems(mode, rt, rtm, oracle, torch, dev):
    """40 random systems (f32: phase class PHASE_F32), the exact-zero bundles, perfect imaging at NA 0.3, the ideal OPM fan (hard), the relay under
    skew bundles: full history of device rays against the oracle"""
    totals, failures, open_f32 = {}, [], []
    for name, system, m_in, m_out, rays, family in _bundle_cases(rt, rtm):
        mats = _mats(system, m_in, m_out)
        hard = ft.class_tolerance(family, mode)
        # a bundle launched on its first plane puts every ray at t = +-0 there: all of them are knife edges by
        # construction, so the share of explained rays is not capped
        minority = None if family == "launched_on_plane" or ft.is_hard(family) else 0.01
        want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
        got = dev.trace_tensor(system.surfaces, mats, torch.from_numpy(rays).cuda(), keep="all", precision=mode)
        try:
            rep = _check(name, _np(got), want, range(want.shape[0]), mode, system.surfaces, mats, hard=hard,
                         minority=minority)
        except AssertionError as e:               # every system is reported, not just the first that fails
            if mode == "f32" and name in OPEN_F32:
                kp, kd, kph = OPEN_F32[name]
                t = ft.class_tolerance(family, mode)
                try:
                    ft.compare(_np(got), want, range(want.shape[0]), mode,
                               ft.Tolerance(t.pos * kp, t.dir * kd, t.phase * kph), system.surfaces, mats)
                    open_f32.append(name)
                    continue
                except AssertionError as e2:
                    e = e2
            failures.append(f"{name}: {e}")
            continue
        for why, n in rep.counts().items():
            totals[why] = totals.get(why, 0) + n
    print(f"test_systems [{mode}] explained per reason: {totals}")
    assert not failures, "\n".join(failures)
    if open_f32:
        pytest.xfail(f"open f32 findings within their ceilings: {open_f32}")


# ------------------------------------------------------------------------------------------------ sources and sweeps
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kind", ["fan", "collimated", "grid"])
def test_sources(kind, mode, rt, rtm, oracle, torch, dev):
    """fused generate + trace against the oracle on src.generate() (the same rays in every mode)"""
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    nrm = np.array([np.sin(0.01), 0, np.cos(0.01)])
    nrm /= np.linalg.norm(nrm)
    if kind == "fan":
        src = dev.RaySource.fan([0.3, -0.2, -150.0], 0.09, 201, 0.785, nphis=64)
    elif kind == "collimated":
        src = dev.RaySource.collimated([0, 0, 0], 25.6, 151, 0.785, nphis=90, phi_start=0.1, normal=nrm)
    else:
        src = dev.RaySource.grid([0, 0, 0], 25.6, 130, 0.785, half_width_v=9.0, n_v=110, normal=nrm)
    rays = _np(src.generate())
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    S = want.shape[0]
    sys_ = system.surfaces
    for packed, tag in ((None, "table"), (dev.prepare(sys_, mats, None), "Sellmeier")):
        got = dev.trace_source(sys_, mats, src, keep="all", precision=mode, packed=packed)
        _check(f"{kind} source keep all ({tag})", _np(got), want, range(S), mode, sys_, mats)
        got = dev.trace_source(sys_, mats, src, keep="last", precision=mode, packed=packed)
        _check(f"{kind} source keep last ({tag})", _np(got), want, [S - 1], mode, sys_, mats)
        part = dev.trace_source(sys_, mats, src, first=1000, count=777, keep=[0, 9, S - 1], precision=mode,
                                packed=packed)
        _check(f"{kind} source slice ({tag})", _np(part), want[:, 1000:1777], [0, 9, S - 1], mode, sys_, mats,
               minority=None)
        for slab in (9, 14):
            red = dev.Reducer(slab, origin=(5.0, 0, 0), grid_n=32, half_width=26.0)
            last = dev.trace_source(sys_, mats, src, keep="last", precision=mode, packed=packed, reducer=red)
            _check(f"{kind} source keep last + reduction ({tag})", _np(last), want, [S - 1], mode, sys_, mats)
            samples = dev.trace_source(sys_, mats, src, keep=[slab], precision=mode, packed=packed)
            _check_reduction(red, _np(samples[0]), (5.0, 0, 0), (1, 0, 0), (0, 1, 0), 32, 26.0,
                             f"{kind} source slab {slab} ({tag})")


@pytest.fixture(params=["one_launch", "launch_per_source"])
def sweep_form(request):
    from ray_trace_pb_b200 import _ffi
    L = _ffi.lib()
    _ffi.check(L.rtb_tune(b"sweep_split_rays", 0 if request.param == "launch_per_source" else -1))
    yield request.param
    _ffi.check(L.rtb_tune(b"sweep_split_rays", 1 << 24))


@pytest.mark.parametrize("mode", MODES)
def test_sweeps(mode, sweep_form, rt, rtm, oracle, torch, dev):
    """rtb_trace_sources in both forms: field x wavelength sweeps with a host table (<= 8 wavelengths) and with the
    in-kernel Sellmeier (> 8 wavelengths through closed-formula media), keep list / "last" / "none" + reduction"""
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    sys_ = system.surfaces
    slab = 12
    for n_wl in (3, 10):
        wls = np.linspace(0.6, 1.0, n_wl)
        sources = []
        for k in range(n_wl):
            th = 0.004 * k
            nrm = np.array([np.sin(th), 0.0, np.cos(th)])
            sources.append(dev.RaySource.grid([0, 0, 0], 25.6, 41, float(wls[k]), normal=nrm / np.linalg.norm(nrm)))
        n = sources[0].n_rays
        rays = np.concatenate([_np(s.generate()) for s in sources])
        want = oracle.trace(sys_, mats, rays, keep_all=True, n_threads=8)
        S = want.shape[0]
        tag = f"{n_wl} wavelengths, {sweep_form}"
        red = dev.Reducer(slab, origin=(8.0, 0, 0), grid_n=32, half_width=26.0, buckets=n_wl)
        out = dev.trace_sources(sys_, mats, sources, keep=[0, slab, S - 1], precision=mode, reducer=red)
        _check(f"sweep keep list ({tag})", _np(out), want, [0, slab, S - 1], mode, sys_, mats)
        for k in range(n_wl):
            _check_reduction(red, _np(out[1, k * n:(k + 1) * n]), (8.0, 0, 0), (1, 0, 0), (0, 1, 0), 32, 26.0,
                             f"sweep bucket {k} keep list ({tag})", bucket=k)
        last = dev.trace_sources(sys_, mats, sources, keep="last", precision=mode)
        _check(f"sweep keep last ({tag})", _np(last), want, [S - 1], mode, sys_, mats)
        red2 = dev.Reducer(slab, origin=(8.0, 0, 0), grid_n=32, half_width=26.0, buckets=n_wl)
        assert dev.trace_sources(sys_, mats, sources, keep="none", precision=mode, reducer=red2) is None
        for k in range(n_wl):
            _check_reduction(red2, _np(out[1, k * n:(k + 1) * n]), (8.0, 0, 0), (1, 0, 0), (0, 1, 0), 32, 26.0,
                             f"sweep bucket {k} keep none ({tag})", bucket=k)


# ------------------------------------------------------------------------------------------------ reductions
def _check_reduction(red, samples, origin, e1, e2, grid_n, half_width, what, bucket=None, phase_ref=0.0):
    """
    (b) of the reduction check: the fused reduction equals the plain NumPy definition (oracle.reduce_stats /
    reduce_grid) applied to the fast mode's OWN samples of that slab.  trace_fast.cu is compiled with FMA contraction,
    so its u, v projections may differ from NumPy's in the last bits: extrema within a few ulps, and the count plane
    exact except in the cells next to samples that lie within a few ulps of a cell edge.
    """
    from oracle import oracle
    stats = _np(red.stats_t)
    grid = _np(red.grid_t) if red.grid_t is not None else None
    if bucket is not None:
        stats, grid = stats[bucket], (grid[bucket] if grid is not None else None)
    want = oracle.reduce_stats(samples, origin, e1, e2, phase_ref)
    assert stats[0] == want[0], f"{what}: count {stats[0]} != {want[0]}"
    if want[0] == 0:
        return
    np.testing.assert_allclose(stats[1:8], want[1:8], rtol=1e-10, atol=1e-9, err_msg=what)
    ext = np.abs(want[8:]).max()
    np.testing.assert_allclose(stats[8:], want[8:], rtol=0, atol=8 * np.finfo(float).eps * max(ext, 1.0), err_msg=what)
    if grid is None:
        return
    want_grid = oracle.reduce_grid(samples, origin, e1, e2, grid_n, half_width, phase_ref)
    p = samples[:, 0:3] - np.asarray(origin, dtype=float)
    mask = np.zeros((grid_n, grid_n), bool)
    with np.errstate(invalid="ignore"):
        xu = (p @ np.asarray(e1, float) + half_width) * (grid_n / (2 * half_width))
        xv = (p @ np.asarray(e2, float) + half_width) * (grid_n / (2 * half_width))
        near = (np.abs(xu - np.round(xu)) <= 8 * np.finfo(float).eps * np.maximum(np.abs(xu), 1.0)) | \
               (np.abs(xv - np.round(xv)) <= 8 * np.finfo(float).eps * np.maximum(np.abs(xv), 1.0))
    for u, v in zip(xu[near & np.isfinite(xu) & np.isfinite(xv)], xv[near & np.isfinite(xu) & np.isfinite(xv)]):
        iu, iv = int(np.floor(u)), int(np.floor(v))
        mask[max(iv - 1, 0):min(iv + 2, grid_n), max(iu - 1, 0):min(iu + 2, grid_n)] = True
    n_edge = int(near.sum())
    assert np.array_equal(grid[2][~mask], want_grid[2][~mask]), f"{what}: count plane ({n_edge} samples on edges)"
    assert abs(grid[2].sum() - want_grid[2].sum()) <= n_edge
    np.testing.assert_allclose(grid[:2][:, ~mask], want_grid[:2][:, ~mask], rtol=0,
                               atol=1e-9 * max(1.0, want_grid[2].max()), err_msg=what)


@pytest.mark.parametrize("mode", MODES)
def test_reductions(mode, rt, rtm, oracle, torch, dev):
    """(a) keep=[slab] samples against the oracle; (b) the LAST = 2 and LAST = 0 reductions against the NumPy
    definition on those samples; at an after-slab, an at-slab and slab 0, host table and in-kernel Sellmeier"""
    system, m_in, m_out, _ = systems.edge_mix(rt, rtm)
    mats = _mats(system, m_in, m_out)
    from test_gpu_parity import _fuzz_rays
    rays = _fuzz_rays(30_000, seed=11)
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    S = want.shape[0]
    d = torch.from_numpy(rays).cuda()
    origin = (0.5, -0.25, 0.0)
    for slab in (4, 7, 0, S - 1):                        # after surface 1, at surface 3, the launch rays, the last
        for wavelengths in ("auto", None):
            tag = f"slab {slab}, wavelengths={wavelengths}"
            samples = dev.trace_tensor(system.surfaces, mats, d, keep=[slab], precision=mode, wavelengths=wavelengths)
            _check(f"edge mix samples {tag}", _np(samples), want, [slab], mode, system.surfaces, mats, hard=True)
            for keep in ("last", "none", [0, S - 1]):    # LAST = 2 (slab >= 1) / LAST = 0
                red = dev.Reducer(slab, origin=origin, grid_n=48, half_width=6.0)
                out = dev.trace_tensor(system.surfaces, mats, d, keep=keep, precision=mode, wavelengths=wavelengths,
                                       reducer=red)
                if keep == "last":
                    _check(f"edge mix last + reduction {tag}", _np(out), want, [S - 1], mode, system.surfaces, mats,
                           hard=True)
                _check_reduction(red, _np(samples[0]), origin, (1, 0, 0), (0, 1, 0), 48, 6.0, f"{tag}, keep={keep}")


# ------------------------------------------------------------------------------------------------ host paths
@pytest.mark.parametrize("mode", MODES)
def test_host_paths(mode, rt, rtm, oracle, monkeypatch):
    """the drop-in call over several staging chunks, 37 wavelengths in groups of 8, 70 surfaces in two segments"""
    monkeypatch.setenv("RTB_HOST_CHUNK_MIB", "1")        # 16384-ray chunks
    system, m_in, m_out, _ = systems.plano_convex(rt, rtm)
    rays = systems.lattice_rays(260, 26.0, -5.0, 0.5, tilt=(0.01, 0.0))
    rays[::5, 7] = 0.6328                                # not in the sampled table
    mats = _mats(system, m_in, m_out)
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    got = system.ray_trace(rays, m_in, m_out, precision=mode)
    _check("drop-in, 5 chunks", got, want, range(want.shape[0]), mode, system.surfaces, mats)
    last = system.ray_trace(rays, m_in, m_out, precision=mode, keep="last")
    _check("drop-in, 5 chunks, keep last", last, want, [want.shape[0] - 1], mode, system.surfaces, mats)
    monkeypatch.delenv("RTB_HOST_CHUNK_MIB")

    system, m_in, m_out, _ = systems.cauchy_singlet(rt, rtm)
    rays = systems.lattice_rays(150, 15.0, -5.0, 0.5)
    rays[:, 7] = np.random.default_rng(0).choice(np.linspace(0.4, 0.7, 37), size=rays.shape[0])
    rays[11, 7] = np.nan
    mats = _mats(system, m_in, m_out)
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    got = system.ray_trace(rays, m_in, m_out, precision=mode)
    _check("37 wavelengths in groups", got, want, range(want.shape[0]), mode, system.surfaces, mats)

    system = systems.long_train_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + system.materials + [vac]
    rays = systems.lattice_rays(60, 15.5, 0.0, 0.5876, tilt=(0.002, -0.001))
    rays[::7, 7] = 0.4861
    want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    got = system.ray_trace(rays, vac, vac, precision=mode)
    hard = ft.class_tolerance("long_train", mode)
    _check("70 surfaces in segments", got, want, range(want.shape[0]), mode, system.surfaces, mats, hard=hard)
    keep = [0, 5, 127, 128, 129, 140]
    got = system.ray_trace(rays, vac, vac, precision=mode, keep=keep)
    _check("70 surfaces in segments, keep list", got, want, keep, mode, system.surfaces, mats, hard=hard)


@pytest.mark.parametrize("mode", MODES)
def test_intersect_only(mode, rt, rtm, torch, dev):
    """FLAG_INTERSECT_ONLY through trace_tensor: against the exact mode under the same flag"""
    from ray_trace_pb_b200 import _ffi
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    rays = torch.from_numpy(systems.lattice_rays(120, 13.0, 0.0, 0.785, tilt=(0.005, 0.002))).cuda()
    want = _np(dev.trace_tensor(system.surfaces, mats, rays, keep="all", flags=_ffi.FLAG_INTERSECT_ONLY))
    got = _np(dev.trace_tensor(system.surfaces, mats, rays, keep="all", precision=mode, flags=_ffi.FLAG_INTERSECT_ONLY))
    _check("intersect only", got, want, range(want.shape[0]), mode, system.surfaces, mats)


# ------------------------------------------------------------------------------------------------ the bench workload
@pytest.mark.parametrize("mode", MODES)
def test_bench_workload(mode, rt, rtm, oracle, torch, dev):
    """bench.py's fast-mode leg: the relay, the first 4e7 rays of its grid bundle, keep="last" -- ordinary class, as
    bench prints it.  Compared on the device with the exact mode's final slab; departing rays are classified from an
    oracle history of just those rays."""
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    n = 40_000_000
    # bench.beam_source at bench's default 1.25e8 rays per GPU (--gpus 1): the fast-mode leg traces the first 4e7 rays
    # of that grid (its first ~3577 rows)
    side = int(np.ceil(np.sqrt(int(1.25e8))))
    src = dev.RaySource.grid([0, 0, 0], 12.0, side, 0.785, n_v=side)
    rays = src.generate(count=n)
    ref = dev.trace_tensor(system.surfaces, mats, rays, keep="last", wavelengths=[0.785])[0]
    got = dev.trace_tensor(system.surfaces, mats, rays, keep="last", wavelengths=[0.785], precision=mode)[0]
    tol = ft.tolerance(mode)
    gn, wn = torch.isnan(got), torch.isnan(ref)
    err = torch.where(gn | wn, torch.zeros_like(got), (got - ref).abs())
    lim = torch.tensor([tol.pos] * 3 + [tol.dir] * 3 + [tol.phase, 0.0], dtype=torch.float64, device="cuda")
    lim = lim.expand_as(err).clone()
    lim[:, 6] *= torch.clamp(torch.nan_to_num(ref[:, 6], nan=1.0).abs(), min=1.0)
    mult = err[:, :7] / lim[:, :7]
    wl_bad = (~gn[:, 7] & ~wn[:, 7]) & (got[:, 7].view(torch.int64) != ref[:, 7].view(torch.int64))
    departs = (gn != wn).any(dim=1) | (mult > 1).any(dim=1) | wl_bad
    dep = torch.nonzero(departs).flatten()
    keep = ~departs
    worst = {name: float(mult[keep][:, sl].max()) for name, sl in
             (("position", slice(0, 3)), ("direction", slice(3, 6)), ("phase", slice(6, 7)))}
    print(f"bench workload [{mode}] {n} rays: max error {worst}; departing {dep.numel()}")
    assert all(v <= 1.0 for v in worst.values())
    assert int(torch.isfinite(ref[:, 0]).sum()) > 0.9 * n
    if dep.numel():
        assert dep.numel() <= 0.001 * n
        launch = _np(rays[dep])
        hist = oracle.trace(system.surfaces, mats, launch, keep_all=True, n_threads=8)
        assert np.array_equal(ft_bits(hist[-1]), ft_bits(_np(ref[dep]))), "exact mode vs oracle on departing rays"
        _check("bench workload departing rays", _np(got[dep])[None], hist, [hist.shape[0] - 1], mode,
               system.surfaces, mats, minority=None)


def ft_bits(a):
    import parity
    return parity.canonical(a)


# ------------------------------------------------------------------------------------------------ coverage
_KERNEL = re.compile(r"trace_fast_kernel<(float|double), (true|false), (true|false), (true|false), (\d)>")


def test_every_instantiation_is_launched(rt, rtm, torch, dev):
    """every trace_fast_kernel instantiation that launch_trace_fast can reach, launched by the routes above (one
    small call per route, recorded by the profiler)"""
    from torch.profiler import ProfilerActivity, profile
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    sys_ = system.surfaces
    rays = torch.from_numpy(systems.lattice_rays(20, 10.0, 0.0, 0.785)).cuda()
    src = dev.RaySource.grid([0, 0, 0], 10.0, 20, 0.785)
    sweep8 = [dev.RaySource.grid([0, 0, 0], 10.0, 20, w) for w in (0.7, 0.8)]
    sweep10 = [dev.RaySource.grid([0, 0, 0], 10.0, 20, w) for w in np.linspace(0.6, 1.0, 10)]
    bare = dev.prepare(sys_, mats, None)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for mode in MODES:
            for wl in ("auto", None):
                dev.trace_tensor(sys_, mats, rays, keep="all", precision=mode, wavelengths=wl)
                dev.trace_tensor(sys_, mats, rays, keep="last", precision=mode, wavelengths=wl)
                dev.trace_tensor(sys_, mats, rays, keep="last", precision=mode, wavelengths=wl,
                                 reducer=dev.Reducer(5))
            for packed in (None, bare):
                dev.trace_source(sys_, mats, src, keep="all", precision=mode, packed=packed)
                dev.trace_source(sys_, mats, src, keep="last", precision=mode, packed=packed)
                dev.trace_source(sys_, mats, src, keep="none", precision=mode, packed=packed, reducer=dev.Reducer(5))
            for sw in (sweep8, sweep10):
                dev.trace_sources(sys_, mats, sw, keep="all", precision=mode)
                dev.trace_sources(sys_, mats, sw, keep="last", precision=mode)
                dev.trace_sources(sys_, mats, sw, keep="none", precision=mode,
                                  reducer=dev.Reducer(5, buckets=len(sw)))
        torch.cuda.synchronize()
    seen = {m.groups() for e in prof.events() for m in [_KERNEL.search(e.name)] if m}
    want = {(t, tab, srcf, sw, last) for t in ("float", "double") for tab in ("true", "false")
            for srcf, sw in (("false", "false"), ("true", "false"), ("true", "true")) for last in "012"}
    assert want <= seen, f"not launched: {sorted(want - seen)}"
    assert seen <= want, f"unexpected: {sorted(seen - want)}"
