"""
GPU parity tests (`-m gpu`): the CUDA path, called through the drop-in API and the C ABI, against
  (1) the golden vectors written from the reference itself (bit for bit),
  (2) the CPU oracle on larger seeded batches (bit for bit),
  (3) sha256 pins of reference outputs at 1e5 rays,
and the project's own reductions / sources against their NumPy definitions (1e-10 relative: atomics reorder sums).

Bar: fp64 mode is BIT-EXACT for positions, directions, phase, wavelength and NaN masks (north star asks 1e-10).
"""
import numpy as np
import pytest

import parity
import systems
from conftest import load_golden
from test_oracle_golden import BIG, _tables_match

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    return torch


@pytest.fixture(scope="module")
def dev():
    import ray_trace_pb_b200.device as dev
    return dev


# ------------------------------------------------------------------------------------------------ golden vectors
@pytest.mark.parametrize("name", sorted(systems.CASES))
def test_golden_history(name, rt, rtm):
    g = load_golden(name)
    system, m_in, m_out = systems.rebuild_system(g["system"], rt, rtm)
    got = system.ray_trace(g["rays_in"], m_in, m_out)
    materials = [m_in] + system.materials + [m_out]
    if name in systems.POWER_DEPENDENT and not _tables_match(g, materials):
        parity.assert_close_same_mask(got, g["history"], rtol=1e-10, what=name)
    else:
        parity.assert_bit_identical(got, g["history"], name)


@pytest.mark.parametrize("name", ["relay10", "opm", "edge_mix", "doublet_nlak22", "mirrors"])
def test_reference_side_stub(name, rt, rtm):
    """INTEGRATION.md section 2: the bare ctypes stub against the C ABI reproduces the reference's history"""
    import reference_stub
    g = load_golden(name)
    system, m_in, m_out = systems.rebuild_system(g["system"], rt, rtm)
    got = reference_stub.ray_trace(system, g["rays_in"], m_in, m_out)
    parity.assert_bit_identical(got, g["history"], name)


def test_input_shapes(rt, rtm):
    g = load_golden("input_shapes")
    system, m_in, m_out = systems.rebuild_system(g["system"], rt, rtm)
    parity.assert_bit_identical(system.ray_trace(g["rays"][3], m_in, m_out), g["single"], "(8,) input")
    parity.assert_bit_identical(system.ray_trace(g["pre"], m_in, m_out), g["ext"], "(K,N,8) input")
    empty = system.ray_trace(np.zeros((0, 8)), m_in, m_out)
    assert empty.shape == (7, 0, 8)


@pytest.mark.parametrize("name", sorted(BIG))
def test_big_batch_checksum(name, rt, rtm, checksums):
    ref = checksums["big"][name]
    system, m_in, m_out = systems.rebuild_system(ref["system"], rt, rtm)
    hist = system.ray_trace(BIG[name](), m_in, m_out)
    assert int(np.isnan(hist[-1, :, 0]).sum()) == ref["nan_rays_at_end"]
    assert parity.digest(hist) == ref["sha256_history"]
    last = system.ray_trace(BIG[name](), m_in, m_out, keep="last")
    assert parity.digest(last[0]) == ref["sha256_last"]


@pytest.mark.parametrize("seed", range(systems.N_RANDOM_SYSTEMS))
def test_random_systems_checksum(seed, rt, rtm, checksums):
    """40 random systems: the GPU history hashes to the sha256 recorded from the reference itself"""
    system, m_in, m_out, rays = systems.random_system(rt, rtm, seed)
    ref = checksums["random"][str(seed)]
    hist = system.ray_trace(rays, m_in, m_out)
    assert int(np.isfinite(hist[-1, :, 0]).sum()) == ref["alive_at_end"]
    assert parity.digest(hist) == ref["sha256_history"]


# ------------------------------------------------------------------------------------------------ vs the oracle
def _fuzz_rays(n, seed, zlo=-8.0, spread=0.35):
    rng = np.random.default_rng(seed)
    rays = np.zeros((n, 8))
    rays[:, 0:2] = rng.uniform(-14, 14, (n, 2))
    rays[:, 2] = rng.uniform(zlo, zlo + 6, n)
    d = rng.standard_normal((n, 3)) * np.array([spread, spread, 0.1]) + np.array([0, 0, 1.0])
    rays[:, 3:6] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays[:, 6] = rng.uniform(0, 100, n)
    rays[:, 7] = rng.choice(np.array([0.405, 0.532, 0.785, 1.064]), size=n)
    rays[rng.integers(0, n, n // 200)] = np.nan
    rays[rng.integers(0, n, n // 200), 7] = np.nan
    return rays


def test_fuzz_edge_mix_vs_oracle(rt, rtm, oracle):
    system, m_in, m_out, _ = systems.edge_mix(rt, rtm)
    rays = _fuzz_rays(200_000, seed=3)
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "edge_mix fuzz")
    # a healthy mix of outcomes
    dead = np.isnan(want[-1, :, 0]).mean()
    assert 0.05 < dead < 0.98


def test_partially_invalid_input_rays_vs_oracle(rt, rtm, oracle):
    """inf / NaN in single columns of the launch rays (the reference never produces these itself, users can)"""
    rng = np.random.default_rng(21)
    for builder in (systems.edge_mix, systems.plano_convex, systems.mirrors, systems.perfect_lens_phase):
        system, m_in, m_out, _ = builder(rt, rtm)
        rays = _fuzz_rays(4000, seed=5, zlo=-6.0, spread=0.2)
        rays[:, 0:2] *= 0.3
        for col in range(8):
            rows = rng.integers(0, rays.shape[0], 60)
            rays[rows[:30], col] = np.nan
            rays[rows[30:45], col] = np.inf
            rays[rows[45:], col] = -np.inf
        got = system.ray_trace(rays, m_in, m_out)
        want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
        parity.assert_bit_identical(got, want, builder.__name__)


def test_rays_launched_on_a_plane_vs_oracle(rt, rtm, oracle):
    """t = +-0 at the first surface (the reference's scripts put the source on a flat at z = 0); signs of zeros count"""
    for which in range(5):
        system, m_in, m_out, rays = systems.launched_on_plane(rt, rtm, which, n=30_000, seed=1234)
        got = system.ray_trace(rays, m_in, m_out)
        want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
        parity.assert_bit_identical(got, want, f"launched on plane {which}")
        assert np.isfinite(want[-1, :, 0]).mean() > 0.5


def test_degenerate_bundles_stay_on_the_fast_path_and_match(rt, rtm, oracle, torch, dev):
    """beams along the axis / sources at the focus: exactly normal incidence on planes, exactly zero transverse
    direction and focal-plane height in perfect lenses -- whole bundles of them, at a size where a slow path shows"""
    wl = 0.6
    system, m_in, m_out, _ = systems.retro_mirror(rt, rtm)
    rays = rt.get_collimated_rays([0, 0, -5], 12.0, 300, wl, nphis=200)
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "retro mirror")
    assert np.isfinite(want[-1]).all()
    system, m_in, m_out, _ = systems.perfect_imaging_in_focus(rt, rtm)
    rays = rt.get_ray_fan([0.0, 0.0, 0.0], 0.25, 300, 0.532e-3, nphis=200)
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "perfect imaging, source at the focus")
    assert np.isfinite(want[-1]).all()


def test_degenerate_first_surface_hint_never_changes_a_result(rt, rtm, oracle, torch, dev):
    """RTB_HINT_DEGENERATE selects the kernels whose hot loop handles exact zeros at a marked flat in line: the same
    bits with the hint on or off, on bundles that are degenerate there, on bundles that are not, and on mixtures."""
    from ray_trace_pb_b200 import engine
    system, m_in, m_out = systems.rebuild_system(load_golden("doublet_nlak22")["system"], rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    assert isinstance(system.surfaces[0], rt.FlatSurface)
    z0 = float(system.surfaces[0].center[2])
    on_plane = systems.lattice_rays(120, 9.0, z0, 0.855, tilt=(0.01, -0.02))            # t = +-0 at the first flat
    along = systems.lattice_rays(120, 9.0, z0 - 7.0, 0.855)                             # d x n = 0 there
    ordinary = systems.lattice_rays(120, 9.0, z0 - 7.0, 0.855, tilt=(0.01, -0.02))
    mixed = np.concatenate((on_plane[::3], along[1::3], ordinary[2::3]))
    mixed[5, 0] = np.inf
    for name, rays, expect in (("on plane", on_plane, True), ("along normal", along, True),
                               ("ordinary", ordinary, False), ("mixed", mixed, False)):
        assert engine.degenerate_first_surface(system.surfaces, rays=rays[::97]) == expect, name
        want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
        d_rays = torch.from_numpy(rays).cuda()
        for hint in (None, False, True, "auto"):
            for keep in ("all", "last"):
                got = dev.trace_tensor(system.surfaces, mats, d_rays, keep=keep, degenerate_first=hint)
                parity.assert_bit_identical(got.cpu().numpy(), want if keep == "all" else want[[-1]],
                                            f"{name}, hint={hint}, keep={keep}")
        parity.assert_bit_identical(system.ray_trace(rays, m_in, m_out), want, f"{name}, drop-in call (sampled hint)")
    # on-device sources decide from their own description
    src = dev.RaySource.grid([0, 0, z0], 8.0, 201, 0.855)
    assert src.degenerate_at_first(system.surfaces)
    assert not dev.RaySource.grid([0, 0, z0 - 1.0], 8.0, 201, 0.855, normal=(0, np.sin(0.1), np.cos(0.1))
                                  ).degenerate_at_first(system.surfaces)
    fan_on = dev.RaySource.fan([0.5, 0, z0], 0.1, 101, 0.855, nphis=50)
    assert fan_on.degenerate_at_first(system.surfaces)
    for source in (src, fan_on):
        rays = source.generate().cpu().numpy()
        want = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
        got = dev.trace_source(system.surfaces, mats, source, keep="all")
        parity.assert_bit_identical(got.cpu().numpy(), want, "fused source with the hint")
    with pytest.raises(ValueError):
        dev.trace_tensor(system.surfaces, mats, d_rays, degenerate_first="maybe")


def test_fuzz_opm_vs_oracle(rt, rtm, oracle):
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    rays = rt.get_ray_fan([1e-3, -2e-3, 5e-4], 1.05 * alpha1, 301, 532e-6, nphis=97)
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "opm fan")


def test_fuzz_mirrors_vs_oracle(rt, rtm, oracle):
    system, m_in, m_out, _ = systems.mirrors(rt, rtm)
    rays = _fuzz_rays(50_000, seed=9, zlo=-3.0, spread=0.25)
    rays[:, 0:2] *= 0.2
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "mirror fuzz")


def test_keep_modes(rt, rtm, oracle):
    system, m_in, m_out, rays = systems.relay10(rt, rtm)
    full = oracle.ray_trace(system, rays, m_in, m_out)
    parity.assert_bit_identical(system.ray_trace(rays, m_in, m_out, keep="last")[0], full[-1], "keep=last")
    sel = system.ray_trace(rays, m_in, m_out, keep=[0, 9, -2, -1])
    parity.assert_bit_identical(sel, full[[0, 9, 19, 20]], "keep=list")
    with pytest.raises(ValueError):
        system.ray_trace(rays, m_in, m_out, keep=[5, 4])
    with pytest.raises(ValueError):
        system.ray_trace(rays, m_in, m_out, keep=[99])


def test_host_pipeline_many_chunks(rt, rtm, oracle):
    """more rays than one staging chunk, pageable and pinned buffers, full history"""
    from ray_trace_pb_b200 import _ffi, engine
    system, m_in, m_out, _ = systems.plano_convex(rt, rtm)
    rays = systems.lattice_rays(900, 26.0, -5.0, 0.5)            # 810,000 rays x 7 slabs: 3 chunks
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    got = system.ray_trace(rays, m_in, m_out)
    parity.assert_bit_identical(got, want, "pageable")
    pin_in = _ffi.pinned_empty(rays.shape)
    pin_in[:] = rays
    pin_out = _ffi.pinned_empty(want.shape)
    materials = [m_in] + system.materials + [m_out]
    engine.trace_host(system.surfaces, materials, pin_in, keep="all", out=pin_out)
    parity.assert_bit_identical(pin_out, want, "pinned")
    last = engine.trace_host(system.surfaces, materials, pin_in, keep="last")
    parity.assert_bit_identical(last[0], want[-1], "pinned in, pageable out, last")


def test_surface_propagate_operator(rt, rtm, oracle):
    """Surface.propagate is the per-surface operator of the reference API (raytrace.py:1092)"""
    system, m_in, m_out, rays = systems.edge_mix(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    cur = rays
    for k, s in enumerate(system.surfaces):
        cur = s.propagate(cur, mats[k], mats[k + 1])
    want = oracle.ray_trace(system, rays, m_in, m_out)
    parity.assert_bit_identical(cur, want, "chained propagate")


# ------------------------------------------------------------------------------------------------ full-size properties
def test_full_size_config2_sampled_oracle_and_invariances(rt, rtm, oracle, torch, dev):
    """
    BASELINE config 2 at full size: AC508-100-B doublet, 4096 x 4096 pupil grid (16.8 M rays) per wavelength, three
    wavelengths.  Too big for the oracle as a whole, so: (1) a random 60k-ray sample of each batch is checked bit for
    bit against the oracle, (2) permuting the rays permutes the result (no cross-ray coupling, no index-dependent
    arithmetic), (3) two half-launches equal one launch, (4) the fused reduction counts exactly the finite rays.
    """
    g = load_golden("doublet_nlak22")
    system, m_in, m_out = systems.rebuild_system(g["system"], rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    rng = np.random.default_rng(42)
    for wl in (0.7065, 0.855, 1.015):
        src = dev.RaySource.grid([0, 0, -10.0], 10.0, 4096, wl)
        rays = src.generate()
        n = rays.shape[0]
        assert n == 4096 * 4096
        red = dev.Reducer(2 * 4 + 1, origin=system.surfaces[4].center)            # at the focal-plane flat
        last = dev.trace_tensor(system.surfaces, mats, rays, keep="last", wavelengths=[wl], reducer=red)[0]
        assert int(red.stats()["count"]) == int(torch.isfinite(last[:, 0]).sum()) > 0.99 * n
        pick = torch.from_numpy(rng.choice(n, size=60_000, replace=False)).cuda()
        sample_in = rays[pick].cpu().numpy()
        want = oracle.trace(system.surfaces, mats, sample_in, keep_all=False, n_threads=8)
        parity.assert_bit_identical(last[pick].cpu().numpy(), want, f"sampled oracle parity, {wl} um")
        if wl == 0.855:
            perm = torch.randperm(n, device="cuda")
            shuffled = dev.trace_tensor(system.surfaces, mats, rays[perm].contiguous(), keep="last", wavelengths=[wl])[0]
            assert torch.equal(shuffled.view(torch.int64), last[perm].view(torch.int64)), "permutation invariance"
            half = n // 2 + 77
            a = dev.trace_tensor(system.surfaces, mats, rays[:half].contiguous(), keep="last", wavelengths=[wl])[0]
            b = dev.trace_tensor(system.surfaces, mats, rays[half:].contiguous(), keep="last", wavelengths=[wl])[0]
            assert torch.equal(torch.cat((a, b)).view(torch.int64), last.view(torch.int64)), "launch splitting"
            fused = dev.trace_source(system.surfaces, mats, src, keep="last")[0]
            assert torch.equal(fused.view(torch.int64), last.view(torch.int64)), "fused source == materialised rays"


def test_full_size_opm_fan_sampled_oracle(rt, rtm, oracle, torch, dev):
    """BASELINE config 4 shape (ideal OPM, perfect lenses, ray fan generated on the device) at 16 M rays: sampled
    bit-exact parity with the oracle run on the device-generated rays, plus pupil-grid mass conservation."""
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    src = dev.RaySource.fan([1e-3, 1e-3, 1e-3 * np.tan(theta)], alpha1, 4001, 532e-6, nphis=4000)
    slab = 2 * 8 + 2
    o3n = system.surfaces[8].normal
    e2 = np.array([0.0, 1.0, 0.0])
    red = dev.Reducer(slab, origin=system.surfaces[8].center, e1=np.cross(e2, o3n), e2=e2, grid_n=512, half_width=3.2)
    rays = src.generate()
    last = dev.trace_tensor(system.surfaces, mats, rays, keep="last", wavelengths=[532e-6], reducer=red)[0]
    pick = torch.from_numpy(np.random.default_rng(1).choice(rays.shape[0], size=50_000, replace=False)).cuda()
    want = oracle.trace(system.surfaces, mats, rays[pick].cpu().numpy(), keep_all=False, n_threads=8)
    parity.assert_bit_identical(last[pick].cpu().numpy(), want, "sampled oracle parity, OPM fan")
    stats = red.stats()
    assert float(red.grid[2].sum()) == stats["count"] > 0.5 * rays.shape[0]     # every counted ray landed in the grid


# ------------------------------------------------------------------------------------------------ refractive indices
def test_formula_mode_equals_table_mode(rt, rtm, torch, dev):
    system = systems.relay10_system(rt, rtm)
    mats = [rtm.Vacuum()] + system.materials + [rtm.Vacuum()]
    rays = torch.from_numpy(systems.lattice_rays(300, 14.0, 0.0, 0.785, tilt=(0.003, 0.001))).cuda()
    a = dev.trace_tensor(system.surfaces, mats, rays, keep="all", wavelengths="auto")
    b = dev.trace_tensor(system.surfaces, mats, rays, keep="all", wavelengths=[0.785])
    c = dev.trace_tensor(system.surfaces, mats, rays, keep="all", wavelengths=None)   # in-kernel Sellmeier
    parity.assert_bit_identical(a.cpu().numpy(), b.cpu().numpy(), "auto vs given")
    parity.assert_bit_identical(c.cpu().numpy(), b.cpu().numpy(), "in-kernel Sellmeier vs host table")


def test_continuous_spectrum_uses_in_kernel_sellmeier(rt, rtm, oracle):
    """one wavelength per ray (> RTB_MAX_WAVELENGTHS distinct values)"""
    system = systems.relay10_system(rt, rtm)
    rays = systems.lattice_rays(150, 12.0, 0.0, 0.785)
    rays[:, 7] = np.linspace(0.45, 1.1, rays.shape[0])
    rays[5, 7] = np.nan
    got = system.ray_trace(rays, rtm.Vacuum(), rtm.Bk7())
    want = oracle.ray_trace(system, rays, rtm.Vacuum(), rtm.Bk7(), n_threads=8)
    parity.assert_bit_identical(got, want, "continuous spectrum")
    # a medium that only exists as Python code cannot follow: loud refusal, no CPU fallback
    cauchy = systems.make_cauchy(rtm)(1.5, 0.004)
    with pytest.raises(NotImplementedError):
        system.ray_trace(rays, rtm.Vacuum(), cauchy)


def test_sampled_table_with_unlisted_wavelengths(rt, rtm, oracle):
    """host batches of Sellmeier media tabulate a 64-ray sample; rays the sample missed are evaluated in the kernel"""
    from ray_trace_pb_b200 import engine
    system = systems.relay10_system(rt, rtm)
    rays = systems.lattice_rays(200, 12.0, 0.0, 0.785)
    rays[12345, 7] = 0.6328
    rays[12346:12400, 7] = 1.064
    rays[777, 7] = np.nan
    mats = [rtm.Vacuum()] + system.materials + [rtm.Vacuum()]
    assert engine.choose_wavelength_table(mats, rays).tolist() == [0.785]
    got = system.ray_trace(rays, rtm.Vacuum(), rtm.Vacuum())
    want = oracle.ray_trace(system, rays, rtm.Vacuum(), rtm.Vacuum(), n_threads=8)
    parity.assert_bit_identical(got, want, "unlisted wavelengths")


def test_table_only_medium_gets_a_complete_scan(rt, rtm, oracle):
    """a medium that only exists as Python code needs every distinct wavelength of the batch in the host table"""
    from ray_trace_pb_b200 import engine
    system, m_in, m_out, _ = systems.cauchy_singlet(rt, rtm)
    rays = systems.lattice_rays(150, 15.0, -5.0, 0.5)
    rays[4321, 7] = 0.45
    rays[9999:10050, 7] = 0.65
    mats = [m_in] + system.materials + [m_out]
    assert engine.choose_wavelength_table(mats, rays).tolist() == [0.45, 0.5, 0.65]
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "complete scan")
    # more distinct wavelengths than one table holds: traced in wavelength groups, still exact
    rays[:, 7] = np.random.default_rng(0).choice(np.linspace(0.4, 0.7, 37), size=rays.shape[0])
    rays[11, 7] = np.nan
    got = system.ray_trace(rays, m_in, m_out)
    want = oracle.ray_trace(system, rays, m_in, m_out, n_threads=8)
    parity.assert_bit_identical(got, want, "37 wavelengths in groups of 8")
    parity.assert_bit_identical(system.ray_trace(rays, m_in, m_out, keep="last")[0], want[-1], "grouped, keep=last")
    rays[:, 7] = np.linspace(0.4, 0.7, rays.shape[0])
    with pytest.raises(NotImplementedError):
        system.ray_trace(rays, m_in, m_out)


def test_distinct_wavelengths_on_device(torch, dev):
    rays = torch.zeros((100_000, 8), dtype=torch.float64, device="cuda")
    wl = np.random.default_rng(0).choice([0.4, 0.5, 0.6, 0.7, np.nan], size=100_000)
    rays[:, 7] = torch.from_numpy(wl).cuda()
    assert dev.distinct_wavelengths_tensor(rays).tolist() == [0.4, 0.5, 0.6, 0.7]
    rays[:, 7] = torch.arange(100_000, dtype=torch.float64, device="cuda")
    assert dev.distinct_wavelengths_tensor(rays) is None
    rays[:, 7] = float("nan")
    assert dev.distinct_wavelengths_tensor(rays).size == 0


# ------------------------------------------------------------------------------------------------ device API, sources
def test_tensor_api_matches_host_api(rt, rtm, torch, dev):
    system, m_in, m_out, rays = systems.opm(rt, rtm)
    host = system.ray_trace(rays, m_in, m_out)
    t = system.ray_trace(torch.from_numpy(rays).cuda(), m_in, m_out)
    assert t.is_cuda and tuple(t.shape) == host.shape
    parity.assert_bit_identical(t.cpu().numpy(), host, "tensor api")
    with pytest.raises(TypeError):
        dev.trace_tensor(system.surfaces, [m_in] + system.materials + [m_out], torch.zeros((4, 8), device="cuda"))


def test_plane_layout_equals_row_layout(rt, rtm, torch, dev):
    """structure-of-arrays I/O ((8, N) in, (n_slabs, 8, N) out) carries the same bits as the (N, 8) rows"""
    system, m_in, m_out, rays = systems.edge_mix(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    rows = torch.from_numpy(rays).cuda()
    planes = rows.t().contiguous()
    for keep in ("all", "last", [0, 3, 8]):
        a = dev.trace_tensor(system.surfaces, mats, rows, keep=keep)
        b = dev.trace_tensor(system.surfaces, mats, planes, keep=keep, layout="planes")
        assert tuple(b.shape) == (a.shape[0], 8, a.shape[1])
        parity.assert_bit_identical(b.permute(0, 2, 1).contiguous().cpu().numpy(), a.cpu().numpy(), f"planes, keep={keep}")
    c = dev.trace_tensor(system.surfaces, mats, planes, keep="last", layout="planes", precision="f32")
    d = dev.trace_tensor(system.surfaces, mats, rows, keep="last", precision="f32")
    parity.assert_bit_identical(c.permute(0, 2, 1).contiguous().cpu().numpy(), d.cpu().numpy(), "planes, f32")
    with pytest.raises(ValueError):
        dev.trace_tensor(system.surfaces, mats, rows, layout="planes")


@pytest.mark.parametrize("kind", ["fan", "collimated", "grid"])
def test_sources_generate_and_fused_trace(kind, rt, rtm, oracle, dev):
    system = systems.relay10_system(rt, rtm)
    mats = [rtm.Vacuum()] + system.materials + [rtm.Vacuum()]
    nrm = np.array([np.sin(0.01), 0, np.cos(0.01)])
    nrm = nrm / np.linalg.norm(nrm)
    if kind == "fan":
        src = dev.RaySource.fan([0.3, -0.2, -150.0], 0.05, 201, 0.785, nphis=64)
        ref = oracle.source_rays("fan", 201, 64, 0.05, [0.3, -0.2, -150.0], (0, 0, 1), 0.785)
    elif kind == "collimated":
        src = dev.RaySource.collimated([0, 0, 0], 12.0, 151, 0.785, nphis=90, phi_start=0.1, normal=nrm)
        ref = oracle.source_rays("collimated", 151, 90, 12.0, [0, 0, 0], nrm, 0.785, b_start=0.1)
    else:
        src = dev.RaySource.grid([0, 0, 0], 12.0, 130, 0.785, half_width_v=9.0, n_v=110, normal=nrm)
        ref = oracle.source_rays("grid", 130, 110, 12.0, [0, 0, 0], nrm, 0.785, b_max=9.0)
    rays = src.generate()
    got = rays.cpu().numpy()
    assert got.shape == ref.shape
    if kind == "grid":
        parity.assert_bit_identical(got, ref, "grid source is libm-free, so exact")
    else:
        np.testing.assert_allclose(got, ref, rtol=0, atol=5e-16 * max(1.0, np.abs(ref[:, :6]).max()))
    # slices of the index space
    part = src.generate(first=1000, count=777).cpu().numpy()
    parity.assert_bit_identical(part, got[1000:1777], "slice of the source")
    # fused generate+trace == trace of the generated rays == oracle on those exact rays
    fused = dev.trace_source(system.surfaces, mats, src, keep="all").cpu().numpy()
    want = oracle.trace(system.surfaces, mats, got, keep_all=True, n_threads=8)
    parity.assert_bit_identical(fused, want, "fused source trace vs oracle")
    fused_part = dev.trace_source(system.surfaces, mats, src, first=1000, count=777, keep="last").cpu().numpy()
    parity.assert_bit_identical(fused_part[0], want[-1, 1000:1777], "fused source slice")


# ------------------------------------------------------------------------------------------------ reductions
@pytest.fixture(params=["one_launch", "launch_per_source"])
def sweep_form(request):
    """rtb_trace_sources' two forms: one launch whose grid y is the source (small sources), one launch per source with
    its source and bucket in the kernel parameters (rtb_tune "sweep_split_rays": sources of 2^24 rays and more)"""
    from ray_trace_pb_b200 import _ffi
    L = _ffi.lib()
    _ffi.check(L.rtb_tune(b"sweep_split_rays", 0 if request.param == "launch_per_source" else -1))
    yield request.param
    _ffi.check(L.rtb_tune(b"sweep_split_rays", 1 << 24))


def test_sweep_in_one_launch_equals_per_source_launches(rt, rtm, oracle, dev, torch, sweep_form):
    """rtb_trace_sources: field x wavelength sweep, grid y = source; rows, statistics and grids per source"""
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    sources = []
    for k, (th, wl) in enumerate([(0.0, 0.785), (0.004, 0.785), (0.009, 0.65), (0.013, 0.9), (0.017, 0.785)]):
        nrm = np.array([np.sin(th), 0.0, np.cos(th)])
        sources.append(dev.RaySource.grid([0, 0, 0], 12.0, 61, wl, normal=nrm / np.linalg.norm(nrm)))
    n = sources[0].n_rays
    slab = 12
    for precision in ("f64", "f64_fast", "f32"):
        red = dev.Reducer(slab, origin=(8.0, 0, 0), grid_n=64, half_width=8.0, buckets=len(sources))
        out = dev.trace_sources(system.surfaces, mats, sources, keep=[0, slab, -1], precision=precision, reducer=red)
        assert out.shape == (3, len(sources) * n, 8)
        stats = red.stats()
        for k, src in enumerate(sources):
            one = dev.Reducer(slab, origin=(8.0, 0, 0), grid_n=64, half_width=8.0)
            ref = dev.trace_source(system.surfaces, mats, src, keep=[0, slab, -1], precision=precision, reducer=one)
            got = out[:, k * n:(k + 1) * n]
            parity.assert_bit_identical(got.cpu().numpy(), ref.cpu().numpy(), f"sweep rows of source {k} ({precision})")
            a, b = stats[k]["raw"], one.stats()["raw"]
            assert a[0] == b[0] and a[0] > 0
            np.testing.assert_allclose(a, b, rtol=1e-11, atol=1e-9)
            np.testing.assert_allclose(red.grid[k].cpu().numpy(), one.grid.cpu().numpy(), rtol=0, atol=1e-9)
            assert red.grid[k][2].sum().item() == one.grid[2].sum().item()
        # the same sweep keeping only the final slab / nothing: other kernel instantiations (the fast modes' final-slab
        # + reduction kernels, the exact mode's lean kernels), the same rows and the same reductions
        for keep in ("last", "none"):
            red2 = dev.Reducer(slab, origin=(8.0, 0, 0), grid_n=64, half_width=8.0, buckets=len(sources))
            out2 = dev.trace_sources(system.surfaces, mats, sources, keep=keep, precision=precision, reducer=red2)
            if keep == "last":
                parity.assert_bit_identical(out2[0].cpu().numpy(), out[2].cpu().numpy(), f"final slab, keep='last' ({precision})")
            a, b = red2.stats_t.cpu().numpy(), red.stats_t.cpu().numpy()
            assert (a[:, 0] == b[:, 0]).all()
            np.testing.assert_array_equal(a[:, 8:], b[:, 8:])
            np.testing.assert_allclose(a[:, 1:8], b[:, 1:8], rtol=1e-11, atol=1e-9)
            np.testing.assert_array_equal(red2.grid[:, 2].cpu().numpy(), red.grid[:, 2].cpu().numpy())
            np.testing.assert_allclose(red2.grid.cpu().numpy(), red.grid.cpu().numpy(), rtol=0, atol=1e-9)
        if precision == "f64":       # and against the oracle on the generated rays
            rays = out[0].cpu().numpy()
            want = oracle.ray_trace(system, rays, vac, vac, n_threads=8)
            parity.assert_bit_identical(out[2].cpu().numpy(), want[-1], "sweep final slab vs oracle")
    # a reducer with the wrong number of buckets, sources of different sizes
    with pytest.raises(ValueError):
        dev.trace_sources(system.surfaces, mats, sources, reducer=dev.Reducer(slab))
    with pytest.raises(ValueError):
        dev.trace_sources(system.surfaces, mats, sources[:1] + [dev.RaySource.grid([0, 0, 0], 12.0, 9, 0.785)])
    # analysis.spot_statistics takes the single-launch route for equal-size sources: same numbers as one by one
    from ray_trace_pb_b200 import analysis
    many = analysis.spot_statistics(system, vac, vac, sources, slab=-2)
    for k, src in enumerate(sources):
        single = analysis.spot_statistics(system, vac, vac, src, slab=-2)
        assert many[k]["count"] == single["count"]
        np.testing.assert_allclose(many[k]["raw"], single["raw"], rtol=1e-11, atol=1e-9)


def test_final_slab_plus_reduction_mode(rt, rtm, oracle, dev, torch):
    """keep="last" with a reduction on the launch rays or an "after" slab (the headline configuration): same final
    slab as the plain trace, same reduction as with other slab selections, rays dying before / at / after the sampled
    surface included"""
    system, m_in, m_out, _ = systems.edge_mix(rt, rtm)
    mats = [m_in] + list(system.materials) + [m_out]
    rays_np = _fuzz_rays(60_000, seed=11)
    rays = torch.from_numpy(rays_np).cuda()
    n_slabs = 2 * len(system.surfaces) + 1
    want_hist = oracle.ray_trace(system, rays_np, m_in, m_out, n_threads=8)
    for slab in (0, 2, 4, n_slabs - 1):
        fast = dev.Reducer(slab, origin=(0.5, -0.25, 0.0), grid_n=48, half_width=6.0)
        last = dev.trace_tensor(system.surfaces, mats, rays, keep="last", reducer=fast)
        parity.assert_bit_identical(last.cpu().numpy()[0], want_hist[-1], f"final slab with reduction at slab {slab}")
        general = dev.Reducer(slab, origin=(0.5, -0.25, 0.0), grid_n=48, half_width=6.0)
        dev.trace_tensor(system.surfaces, mats, rays, keep=[1, n_slabs - 1], reducer=general)     # general kernel
        a, b = fast.stats()["raw"], general.stats()["raw"]
        assert a[0] == b[0] and a[0] == np.isfinite(want_hist[slab][:, [0, 1, 2, 6]]).all(axis=1).sum()
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-9)
        assert torch.equal(fast.grid[2], general.grid[2])
        np.testing.assert_allclose(fast.grid.cpu().numpy(), general.grid.cpu().numpy(), rtol=0, atol=1e-9)
    # from a source as well
    src = dev.RaySource.fan([0.1, 0.0, -20.0], 0.2, 300, 0.532, nphis=64)
    fast = dev.Reducer(4)
    last = dev.trace_source(system.surfaces, mats, src, keep="last", reducer=fast)
    general = dev.Reducer(4)
    both = dev.trace_source(system.surfaces, mats, src, keep=[0, n_slabs - 1], reducer=general)
    parity.assert_bit_identical(last.cpu().numpy()[0], both.cpu().numpy()[1], "source, final slab")
    np.testing.assert_allclose(fast.stats()["raw"], general.stats()["raw"], rtol=1e-12, atol=1e-9)


def test_final_slab_plus_reduction_on_an_axial_system(rt, rtm, oracle, dev, torch):
    """the same shape on a system whose every axis is +-z (the bench's relay): this is what the dedicated kernel
    (MODE 4: the final-slab loop in two legs around the sample) runs; rays die before, at and after the sampled surface"""
    system = systems.relay10_system(rt, rtm)
    m_in = m_out = rtm.Vacuum()
    mats = [m_in] + list(system.materials) + [m_out]
    rays_np = systems.lattice_rays(220, 22.0, 0.0, 0.785, tilt=(0.03, 0.0))      # walks off: rays die at surfaces 0, 3, 4, 5
    rays_np[::5, 7] = 0.6328                      # a second wavelength; every 11th ray arrives dead
    rays_np[::11, 0] = np.nan
    rays = torch.from_numpy(rays_np).cuda()
    n_slabs = 2 * len(system.surfaces) + 1
    want_hist = oracle.ray_trace(system, rays_np, m_in, m_out, n_threads=8)
    dead = [int(np.isnan(want_hist[j, :, 0]).sum()) for j in (0, 2, 8, 10, 12)]
    assert 0 < dead[0] < dead[1] < dead[2] < dead[3] < dead[4] < rays_np.shape[0], dead
    for slab in (2, 10, n_slabs - 1):
        for keep in ("last", "none"):
            for wavelengths in ("auto", None):                               # host table / in-kernel Sellmeier
                fast = dev.Reducer(slab, origin=(5.0, 0.0, 0.0), grid_n=64, half_width=30.0)
                last = dev.trace_tensor(system.surfaces, mats, rays, keep=keep, reducer=fast, wavelengths=wavelengths)
                if keep == "last":
                    parity.assert_bit_identical(last.cpu().numpy()[0], want_hist[-1], f"final slab, reduction at {slab}")
                else:
                    assert last is None
                want = oracle.reduce_stats(want_hist[slab], (5.0, 0.0, 0.0), (1, 0, 0), (0, 1, 0))
                got = fast.stats_t.cpu().numpy()
                assert got[0] == want[0] > 1000
                np.testing.assert_allclose(got[1:8], want[1:8], rtol=1e-10, atol=1e-6)
                np.testing.assert_allclose(got[8:], want[8:], rtol=1e-13)
                assert np.array_equal(fast.grid.cpu().numpy()[2],
                                      oracle.reduce_grid(want_hist[slab], (5.0, 0.0, 0.0), (1, 0, 0), (0, 1, 0), 64, 30.0)[2])
    # generated rays
    src = dev.RaySource.grid([5.0, 0, 0.0], 26.0, 301, 0.785)
    s_hist = oracle.trace(system.surfaces, mats, src.generate().cpu().numpy(), keep_all=True, n_threads=8)
    fast = dev.Reducer(10, origin=(5.0, 0.0, 0.0))
    last = dev.trace_source(system.surfaces, mats, src, keep="last", reducer=fast)
    parity.assert_bit_identical(last.cpu().numpy()[0], s_hist[-1], "source, final slab")
    want = oracle.reduce_stats(s_hist[10], (5.0, 0.0, 0.0), (1, 0, 0), (0, 1, 0))
    assert fast.stats_t.cpu().numpy()[0] == want[0]
    np.testing.assert_allclose(fast.stats_t.cpu().numpy()[1:8], want[1:8], rtol=1e-10, atol=1e-6)


def test_fused_reductions(rt, rtm, oracle, dev, torch):
    system, m_in, m_out, alpha1, theta = systems.opm_system(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    rays = rt.get_ray_fan([1e-3, 1e-3, 1e-3 * np.tan(theta)], alpha1, 401, 532e-6, nphis=200)
    hist = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    slab = 2 * 8 + 2                                   # just after the O3 pupil flat
    o3n = system.surfaces[8].normal
    e2 = np.array([0.0, 1.0, 0.0])
    e1 = np.cross(e2, o3n)
    origin = system.surfaces[8].center
    ok = ~np.isnan(hist[slab, :, 6])
    phase_ref = float(np.mean(hist[slab, ok, 6]))
    red = dev.Reducer(slab, origin=origin, e1=e1, e2=e2, grid_n=64, half_width=3.2, phase_ref=phase_ref)
    out = dev.trace_tensor(system.surfaces, mats, torch.from_numpy(rays).cuda(), keep="last", reducer=red)
    parity.assert_bit_identical(out[0].cpu().numpy(), hist[-1], "trace output unaffected by the reduction")
    want_stats = oracle.reduce_stats(hist[slab], origin, e1, e2, phase_ref)
    got_stats = red.stats_t.cpu().numpy()
    assert got_stats[0] == want_stats[0] > 1000
    np.testing.assert_allclose(got_stats[1:8], want_stats[1:8], rtol=1e-10, atol=1e-9)
    np.testing.assert_allclose(got_stats[8:], want_stats[8:], rtol=1e-13)
    want_grid = oracle.reduce_grid(hist[slab], origin, e1, e2, 64, 3.2, phase_ref)
    got_grid = red.grid.cpu().numpy()
    assert np.array_equal(got_grid[2], want_grid[2])
    np.testing.assert_allclose(got_grid[:2], want_grid[:2], rtol=0, atol=1e-9 * max(1.0, want_grid[2].max()))
    s = red.stats()
    assert s["count"] == int(want_stats[0]) and s["rms_radius"] > 0
    # accumulate across calls, keep="none" (reduction-only launch), then reset
    dev.trace_tensor(system.surfaces, mats, torch.from_numpy(rays).cuda(), keep="none", reducer=red)
    assert red.stats_t.cpu().numpy()[0] == 2 * want_stats[0]
    red.reset()
    assert red.stats_t.cpu().numpy()[0] == 0 and float(red.grid.abs().sum()) == 0.0


def test_system_longer_than_one_launch(rt, rtm, oracle, dev, torch):
    """70 surfaces (> RTB_MAX_SURFACES): two chained segments must give the reference loop's history, in every mode.
    (The full history and keep="last" are also pinned by the sha256 of the reference's output: long_train_lattice.)"""
    system = systems.long_train_system(rt, rtm)
    m_in = m_out = rtm.Vacuum()
    mats = [m_in] + system.materials + [m_out]
    rays = systems.lattice_rays(40, 15.5, 0.0, 0.5876, tilt=(0.002, -0.001))
    rays[::7, 7] = 0.4861                                   # a second wavelength
    hist = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    n_slabs = 2 * 70 + 1
    assert hist.shape[0] == n_slabs
    dead_at = np.array([np.isnan(hist[j, :, 0]).sum() for j in (0, 128, 140)])
    assert dead_at[0] == 0 and dead_at[1] < dead_at[2] < rays.shape[0], dead_at   # rays also die in the second segment
    parity.assert_bit_identical(system.ray_trace(rays, m_in, m_out), hist, "drop-in call, full history")
    for keep in ([0, 5, 127, 128, 129, 140], [128], [129, 130], [3], "last", [0]):
        got = system.ray_trace(rays, m_in, m_out, keep=keep)
        want = hist[[-1]] if keep == "last" else hist[keep]
        parity.assert_bit_identical(got, want, f"long system, keep={keep}")
    # device tensors, both layouts; the fused source path falls back to generate + chain
    d_rays = torch.from_numpy(rays).cuda()
    got = dev.trace_tensor(system.surfaces, mats, d_rays, keep=[1, 128, 139, 140])
    parity.assert_bit_identical(got.cpu().numpy(), hist[[1, 128, 139, 140]], "long system, tensor API")
    got = dev.trace_tensor(system.surfaces, mats, d_rays.t().contiguous(), keep=[64, 130], layout="planes")
    parity.assert_bit_identical(got.permute(0, 2, 1).contiguous().cpu().numpy(), hist[[64, 130]], "long system, planes")
    src = dev.RaySource.grid([0, 0, 0.0], 12.0, 33, 0.5876)
    s_rays = src.generate().cpu().numpy()
    s_hist = oracle.trace(system.surfaces, mats, s_rays, keep_all=True, n_threads=8)
    got = dev.trace_source(system.surfaces, mats, src, keep=[100, 140])
    parity.assert_bit_identical(got.cpu().numpy(), s_hist[[100, 140]], "long system, fused source")
    # fused reductions at a slab of the first and of the second segment (negative index included)
    for slab in (100, 130, -1):
        red = dev.Reducer(slab, origin=(0, 0, 0), grid_n=32, half_width=16.0)
        out = dev.trace_tensor(system.surfaces, mats, d_rays, keep="last", reducer=red)
        parity.assert_bit_identical(out[0].cpu().numpy(), hist[-1], "long system, keep last + reduction")
        want = oracle.reduce_stats(hist[slab], (0, 0, 0), (1, 0, 0), (0, 1, 0))
        got_stats = red.stats_t.cpu().numpy()
        assert got_stats[0] == want[0] > 100
        np.testing.assert_allclose(got_stats[1:8], want[1:8], rtol=1e-10, atol=1e-6)
        assert np.array_equal(red.grid.cpu().numpy()[2],
                              oracle.reduce_grid(hist[slab], (0, 0, 0), (1, 0, 0), (0, 1, 0), 32, 16.0)[2])
    # structural errors are the reference's
    with pytest.raises(ValueError):
        system.ray_trace(rays, m_in, m_out, keep=[141])


def test_reduction_at_input_and_with_source(rt, rtm, oracle, dev):
    system, m_in, m_out, _ = systems.plano_convex(rt, rtm)
    mats = [m_in] + system.materials + [m_out]
    src = dev.RaySource.grid([0, 0, -5.0], 20.0, 257, 0.5)
    rays = src.generate().cpu().numpy()
    hist = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
    for slab in (0, 3, 6):
        red = dev.Reducer(slab, origin=(0, 0, 0), grid_n=32, half_width=21.0)
        dev.trace_source(system.surfaces, mats, src, keep="none", reducer=red)
        want = oracle.reduce_stats(hist[slab], (0, 0, 0), (1, 0, 0), (0, 1, 0))
        got = red.stats_t.cpu().numpy()
        assert got[0] == want[0]
        np.testing.assert_allclose(got[1:8], want[1:8], rtol=1e-10, atol=1e-6)
        assert np.array_equal(red.grid.cpu().numpy()[2], oracle.reduce_grid(hist[slab], (0, 0, 0), (1, 0, 0), (0, 1, 0), 32, 21.0)[2])


# ------------------------------------------------------------------------------------------------ pupil grid -> PSF
def _dft_matrix(m, g, df, half):
    cell = 2 * half / g
    f = (np.arange(m) - 0.5 * (m - 1)) * df
    x = (np.arange(g) + 0.5) * cell - half
    return np.exp(-2j * np.pi * np.outer(f, x))


def test_psf_contraction_matches_numpy(dev, torch):
    """E = A P B^T against NumPy with the same definition, and against fftshift(fft2(ifftshift(P))) for odd sizes"""
    rng = np.random.default_rng(3)
    for g, m, df_scale in ((95, 95, 1.0), (128, 33, 0.37), (200, 70, 2.1)):
        half = 1.7
        red = dev.Reducer(0, grid_n=g, half_width=half)
        grid = rng.standard_normal((3, g, g))
        grid[2] = rng.integers(0, 4, (g, g))
        red.grid[...] = torch.from_numpy(grid).cuda()
        df = df_scale / (2 * half)
        psf, field = red.psf(m, df, field=True)
        d = _dft_matrix(m, g, df, half)
        want = d @ (grid[0] + 1j * grid[1]) @ d.T
        scale = np.abs(want).max()
        np.testing.assert_allclose(field.cpu().numpy(), want, rtol=0, atol=2e-12 * scale)
        np.testing.assert_allclose(psf.cpu().numpy(), np.abs(want) ** 2, rtol=0, atol=4e-12 * scale**2)
        with np.errstate(all="ignore"):
            pn = np.where(grid[2] > 0, (grid[0] + 1j * grid[1]) / grid[2], 0)
        got_n = red.psf(m, df, normalize_by_count=True).cpu().numpy()
        np.testing.assert_allclose(got_n, np.abs(d @ pn @ d.T) ** 2, rtol=0, atol=4e-12 * np.abs(d @ pn @ d.T).max() ** 2)
        if g == m and g % 2 == 1 and df_scale == 1.0:
            p = grid[0] + 1j * grid[1]
            fft = np.fft.fftshift(np.fft.fft2(np.fft.ifftshift(p)))
            np.testing.assert_allclose(field.cpu().numpy(), fft, rtol=0, atol=2e-12 * scale)


def test_psf_airy_known_answer(rt, rtm, dev, torch):
    """
    The reference's PSF known answer (scripts/2022_02_06_perfect_imaging_system_psf.py:168-171): an NA-limited
    perfect imaging system images an on-axis point to the Airy pattern |2 J1(v)/v|^2.  Here: device fan -> fused trace
    -> pupil grid at the pupil flat -> zoomed-DFT PSF.
    """
    from scipy.special import j1
    wavelength, na, f1, f2 = 0.532e-3, 0.3, 3.0, 30.0
    alpha = np.arcsin(na)
    system = rt.System([rt.PerfectLens(f1, [0, 0, f1], [0, 0, 1], alpha),
                        rt.FlatSurface([0, 0, 2 * f1], [0, 0, 1], 3 * f1),
                        rt.PerfectLens(f2, [0, 0, 2 * f1 + f2], [0, 0, 1], alpha),
                        rt.FlatSurface([0, 0, 2 * f1 + 2 * f2], [0, 0, 1], 10.)],
                       [rtm.Vacuum(), rtm.Vacuum(), rtm.Vacuum()])
    mats = [rtm.Vacuum()] * 5
    chief = system.ray_trace(np.array([0, 0, 0, 0, 0, 1.0, 0, wavelength]), rtm.Vacuum(), rtm.Vacuum())
    phase_ref = float(chief[4, 0, 6])                                   # slab 4 = just after the pupil flat
    src = dev.RaySource.fan([0, 0, 0], alpha * (1 - 1e-9), 2001, wavelength, nphis=2000)
    r_pupil = f1 * na
    red = dev.Reducer(4, origin=(0, 0, 2 * f1), grid_n=256, half_width=1.0, phase_ref=phase_ref)
    dev.trace_source(system.surfaces, mats, src, keep="none", reducer=red)
    grid = red.grid.cpu().numpy()
    filled = grid[2] > 0
    # constant phase across the pupil: every filled cell's mean phasor is 1
    phasor = (grid[0] + 1j * grid[1])[filled] / grid[2][filled]
    assert np.abs(phasor - 1).max() < 1e-5
    # filled cells = the disk of radius f1 * NA
    c = (np.arange(256) + 0.5) * (2.0 / 256) - 1.0
    rr = np.hypot(*np.meshgrid(c, c))
    assert filled[rr < r_pupil - 0.02].all() and not filled[rr > r_pupil + 0.02].any()
    m, df = 65, 0.05
    psf = red.psf(m, df, normalize_by_count=True).cpu().numpy()
    psf /= psf[m // 2, m // 2]
    f = (np.arange(m) - (m - 1) / 2) * df
    v = 2 * np.pi * np.hypot(*np.meshgrid(f, f)) * r_pupil
    with np.errstate(all="ignore"):
        airy = np.where(v > 0, (2 * j1(v) / v) ** 2, 1.0)
    assert np.abs(psf - airy).max() < 0.01
    row = psf[m // 2, m // 2:]
    first_min = f[m // 2:][np.argmax(np.diff(row) > 0)]
    assert abs(first_min - 3.8317 / (2 * np.pi * r_pupil)) <= df


# ------------------------------------------------------------------------------------------------ workload helpers
def test_analysis_spot_statistics_and_axial_crossing(rt, rtm, oracle, dev):
    """analysis.spot_statistics (fused source -> trace -> statistics) against NumPy on the oracle's trace"""
    from ray_trace_pb_b200 import analysis
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + system.materials + [vac]
    sources = []
    for th in (0.0, 0.01):
        nrm = np.array([np.sin(th), 0, np.cos(th)])
        sources.append(dev.RaySource.grid([0, 0, 0], 12.0, 181, 0.785, normal=nrm / np.linalg.norm(nrm)))
    got = analysis.spot_statistics(system, vac, vac, sources, slab=-2, chunk=10_000)      # several launches per source
    for src, g in zip(sources, got):
        rays = src.generate().cpu().numpy()
        hist = oracle.trace(system.surfaces, mats, rays, keep_all=True, n_threads=8)
        want = oracle.reduce_stats(hist[-2], system.surfaces[-1].center, (1, 0, 0), (0, 1, 0))
        assert g["count"] == int(want[0]) > 30_000
        np.testing.assert_allclose(g["raw"][1:8], want[1:8], rtol=1e-10, atol=1e-7)
        p = hist[-2][np.isfinite(hist[-2][:, 0]), 0:2] - system.surfaces[-1].center[0:2]
        np.testing.assert_allclose(g["centroid"], p.mean(axis=0), rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(g["rms_radius"], np.sqrt(((p - p.mean(axis=0)) ** 2).sum(axis=1).mean()), rtol=1e-7)
    # paraxial focus of a doublet from the crossing of two meridional rays = the cardinal-point back focal point
    doublet = rt.Doublet(rtm.Nlak22(), rtm.Nsf6ht(), radius_crown=65.8, radius_flint=-280.6, radius_interface=-56,
                         thickness_crown=13.0, thickness_flint=2.0, aperture_radius=25.4)
    z = analysis.axial_crossing(doublet, vac, vac, 0.855, 1e-3, pt=(0, 0, -10.0))[2]
    assert abs(z - doublet.get_cardinal_points(0.855, vac, vac)[1][2]) < 1e-4


# ------------------------------------------------------------------------------------------------ helpers
def test_intersect_rays(rt, torch):
    g = load_golden("intersect_rays")
    parity.assert_bit_identical(rt.intersect_rays(g["r1"], g["r2"]), g["pts"], "pairs")
    parity.assert_bit_identical(rt.intersect_rays(g["axis_ray"], g["others"]), g["pts_axis"], "broadcast")
    parity.assert_bit_identical(rt.intersect_rays(g["a"], g["b"]), g["pts_deg"], "degenerate")
    t = rt.intersect_rays(torch.from_numpy(g["r1"]).cuda(), torch.from_numpy(g["r2"]).cuda())
    assert t.is_cuda
    parity.assert_bit_identical(t.cpu().numpy(), g["pts"], "tensor in, tensor out")
    with pytest.raises(ValueError):
        rt.intersect_rays(g["r1"][:3], g["r2"][:4])


def test_propagate_ray2plane_and_friends(rt, rtm, host_api):
    g = load_golden("ray2plane")
    out, ts = rt.propagate_ray2plane(g["rays"], np.array([0, 0.6, 0.8]), np.array([0, 0, 5.]), rtm.Bk7())
    parity.assert_bit_identical(out, g["out"], "ray2plane rays")
    parity.assert_bit_identical(ts, g["ts"], "ray2plane ts")
    dists, near = rt.dist_pt2plane(np.array([[1., 2, 3], [0, 0, -1]]), np.array([0, 0.6, 0.8]), np.array([0, 0, 1.]))
    np.testing.assert_allclose(dists, host_api["dist_pt2plane"]["dists"], rtol=1e-15)
    np.testing.assert_allclose(near, host_api["dist_pt2plane"]["nearest"], rtol=1e-15, atol=1e-16)
    # backward exclusion and per-ray centres
    rays = g["rays"].copy()
    centers = np.tile(np.array([0, 0, 5.0]), (len(rays), 1))
    centers[::2, 2] = -5.0
    out2, ts2 = rt.propagate_ray2plane(rays, np.array([0, 0, 1.0]), centers, rtm.Vacuum(), exclude_backward_propagation=True)
    assert np.all(np.isnan(out2[::2])) and not np.any(np.isnan(out2[1::2])) and np.all(ts2[::2] < 0)


def test_get_intersect_operator(rt, rtm, oracle):
    system, m_in, m_out, rays = systems.edge_mix(rt, rtm)
    # for forward-travelling rays get_intersect equals the at-surface slab of propagate
    fwd = rays[np.nan_to_num(rays[:, 5]) > 0.2]
    for s, m in ((system.surfaces[0], m_in), (system.surfaces[1], system.materials[0])):
        at = s.get_intersect(fwd, m)
        want = oracle.trace([s], [m, m], fwd, keep_all=True)[1]
        parity.assert_bit_identical(at, want, type(s).__name__)
    # a backwards ray is NOT culled by get_intersect of a sphere (only propagate applies the front-side test)
    back = np.array([[0, 0, 40.0, 0, 0, -1.0, 0, 0.5]])
    at = system.surfaces[1].get_intersect(back, m_in)
    assert np.isfinite(at[0, 2]) and np.isnan(oracle.trace([system.surfaces[1]], [m_in, m_in], back)[1, 0, 2])


def test_auto_focus_ray_modes(rt, rtm, host_api):
    d = rt.Doublet(rtm.Nsk11(), rtm.Nsf19(), radius_crown=64.1, radius_flint=-183.685, radius_interface=-43.249,
                   thickness_crown=3.5, thickness_flint=1.5, aperture_radius=10.)
    for mode in ("ray-fan", "collimated"):
        got = np.asarray(d.auto_focus(0.5876, rtm.Vacuum(), rtm.Vacuum(), mode=mode), dtype=float)
        want = np.asarray(host_api["kidger_autofocus"][mode], dtype=float)
        assert np.array_equal(np.isnan(got), np.isnan(want))
        np.testing.assert_allclose(got[~np.isnan(got)], want[~np.isnan(want)], rtol=1e-9)


@pytest.mark.parametrize("precision", ["f32", "f64_fast"])
@pytest.mark.parametrize("name", ["relay10_script", "doublet_nlak22", "opm", "mirrors", "edge_mix", "plano_convex_3d"])
def test_fast_modes_tolerance(name, precision, rt, rtm):
    """
    The two fast modes against the reference history, at the tolerances stated in csrc/trace_fast.cu (the contract is
    tests/fast_tolerance.py):
      f32       positions 2e-6 * L (L = 1000 mm), directions 2e-6, phase 2e-6 relative
      f64_fast  positions 1e-11 * L, directions 1e-12, phase 1e-12 relative
    (10x / 100x looser for the high-NA perfect-lens system and the deliberately extreme edge-mix rays, where the
    direction error is amplified by 1/cos(theta)).  Every ray is within tolerance up to its first departure, and every
    departure is explained by a knife edge of the reference at that surface: an aperture edge, a grazing or missing
    intersection, a root or a flat at t ~ 0, the front-side cull, the critical angle, a perfect lens's NA, or the
    reference's absolute 1e-12 on-surface test.  tests/test_gpu_fast_modes.py covers the other kernel routes.
    """
    import fast_tolerance
    g = load_golden(name)
    system, m_in, m_out = systems.rebuild_system(g["system"], rt, rtm)
    mats = [m_in] + list(system.materials) + [m_out]
    want = g["history"]
    got = system.ray_trace(g["rays_in"], m_in, m_out, precision=precision)
    assert got.shape == want.shape
    rep = fast_tolerance.compare(got, want, range(want.shape[0]), precision, fast_tolerance.is_hard(name),
                                 system.surfaces, mats)
    print(rep.summary(name))
    if not fast_tolerance.is_hard(name):
        fast_tolerance.assert_minority(rep, 0.01, name)
    # the final-slab-only instantiations of the fast kernels (no per-surface slab bookkeeping, dead rays leave the loop)
    # perform the same arithmetic: same bits as the last slab of the full history
    last = system.ray_trace(g["rays_in"], m_in, m_out, precision=precision, keep="last")
    parity.assert_bit_identical(last[0], got[-1], f"{name} {precision}: keep='last' vs the history's last slab")


def test_exact_math_selftest():
    """csrc/exact_math.cuh (factored IEEE division / sqrt) against the built-in operators: no bit may differ"""
    import ctypes
    from ray_trace_pb_b200 import _ffi
    bad = (ctypes.c_uint64 * 3)()
    for seed in (1, 0xDEADBEEF):
        _ffi.check(_ffi.lib().rtb_selftest_exact_math(0, seed, 200_000_000, bad))
        assert list(bad) == [0, 0, 0], f"mismatches (div, div3, sqrt) = {list(bad)} for seed {seed}"


def test_launch_counter_and_probes():
    import ctypes
    from ray_trace_pb_b200 import _ffi
    L = _ffi.lib()
    before = L.rtb_launch_count()
    rate = ctypes.c_double()
    ms = ctypes.c_double()
    _ffi.check(L.rtb_measure_dfma_rate(0, ctypes.byref(rate), ctypes.byref(ms)))
    assert 1e12 < rate.value < 1e14, rate.value          # B200: ~1.9e13 DFMA/s nominal
    # latency-bound issue rate: one chain per warp runs at about 2/3 of the eight-chain rate (DESIGN.md 4a)
    one, eight = ctypes.c_double(), ctypes.c_double()
    _ffi.check(L.rtb_measure_dfma_chain_rate(0, 1, ctypes.byref(one), ctypes.byref(ms)))
    _ffi.check(L.rtb_measure_dfma_chain_rate(0, 8, ctypes.byref(eight), ctypes.byref(ms)))
    assert 0.55 < one.value / eight.value < 0.85, (one.value, eight.value)
    assert 0.8 < eight.value / rate.value < 1.1, (eight.value, rate.value)
    bw = ctypes.c_double()
    _ffi.check(L.rtb_measure_copy_bandwidth(0, 1 << 30, ctypes.byref(bw)))
    assert 1e12 < bw.value < 1.2e13, bw.value
    assert L.rtb_launch_count() >= before
