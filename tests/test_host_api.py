"""
CPU tests (no GPU) of the host side of the drop-in API: packaging, the C-ABI library's exports, error behaviour,
and the O(S) paraxial helpers against values recorded from the reference (tests/golden/host_api.json).
"""
import ctypes
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import parity
import systems
from conftest import load_golden

ROOT = Path(__file__).resolve().parent.parent


# ------------------------------------------------------------------------------------------------ C ABI
def test_library_loads_and_exports_every_declared_symbol():
    from ray_trace_pb_b200 import _ffi
    L = _ffi.lib()
    header = (ROOT / "include" / "rtb.h").read_text()
    declared = set(re.findall(r"\b(rtb_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found in include/rtb.h"
    assert declared == set(_ffi.EXPORTS), declared ^ set(_ffi.EXPORTS)
    for name in declared:
        assert hasattr(L, name), f"librtb.so does not export {name}"
    assert L.rtb_abi_version() == _ffi.RTB_ABI_VERSION


def test_struct_layouts_match_the_header(tmp_path):
    """sizes the C compiler gives the header's structs == ctypes' sizes"""
    from ray_trace_pb_b200 import _ffi
    src = ('#include <stdio.h>\n#include "rtb.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(rtb_surface),'
           'sizeof(rtb_material), sizeof(rtb_system), sizeof(rtb_reduce), sizeof(rtb_trace_opts), sizeof(rtb_source));}')
    exe = tmp_path / "rtb_sizes"
    subprocess.run(["gcc", "-x", "c", "-", "-I", str(ROOT / "include"), "-o", str(exe)], input=src.encode(), check=True)
    sizes = [int(v) for v in subprocess.run([str(exe)], capture_output=True, check=True).stdout.split()]
    want = [ctypes.sizeof(c) for c in (_ffi.RtbSurface, _ffi.RtbMaterial, _ffi.RtbSystem, _ffi.RtbReduce,
                                       _ffi.RtbTraceOpts, _ffi.RtbSource)]
    assert sizes == want


def test_no_cpu_fallback_without_a_device(rt, rtm):
    """On a box without a GPU the hot path must fail loudly, not compute on the CPU."""
    from ray_trace_pb_b200 import _ffi
    if _ffi.lib().rtb_device_count() > 0:
        pytest.skip("a GPU is visible")
    system, m_in, m_out, rays = systems.plano_convex(rt, rtm, n_disps=5)
    with pytest.raises(_ffi.RtbError, match="no CPU fallback"):
        system.ray_trace(rays, m_in, m_out)
    with pytest.raises(_ffi.RtbError):
        rt.intersect_rays(rays[0], rays[1])


def test_product_never_imports_the_oracle():
    for path in list((ROOT / "ray_trace_pb_b200").rglob("*.py")) + list((ROOT / "raytrace").rglob("*.py")) + \
            list((ROOT / "examples").rglob("*.py")):
        text = path.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle", text, re.M), path
        assert "rt_oracle" not in text and "librt_oracle" not in text, path
    for path in (ROOT / "ray_trace_pb_b200" / "csrc").glob("*"):
        if path.is_file():
            assert "rt_oracle" not in path.read_text(errors="ignore"), path


# ------------------------------------------------------------------------------------------------ structural errors
def test_structural_errors(rt, rtm):
    flat = rt.FlatSurface([0, 0, 0], [0, 0, 1], 1.0)
    with pytest.raises(ValueError):
        rt.System([flat, flat, flat], [rtm.Vacuum(), rtm.Vacuum(), rtm.Vacuum()])
    with pytest.raises(ValueError):
        rt.System([flat], [], surfaces_by_name=[0, 1])
    with pytest.raises(ValueError, match="length of materials"):
        rt.System([flat, flat], []).ray_trace(np.zeros((1, 8)), rtm.Vacuum(), rtm.Vacuum())
    with pytest.raises(ValueError):
        rt.get_ray_fan([0, 0, 0], 0.1, 3, 0.5, center_ray=(0, 0, 2))
    with pytest.raises(ValueError):
        rt.get_collimated_rays([0, 0, 0], 1.0, 3, 0.5, normal=(0, 0, 1.1))
    with pytest.raises(TypeError):
        rt.System([flat], []).concatenate("not a surface", rtm.Vacuum())
    with pytest.raises(ValueError):
        rt.System([flat], []).seidel_third_order(0.5, rtm.Vacuum(), rtm.Vacuum())
    with pytest.raises(ValueError):
        rt.System([flat], []).auto_focus(0.5, rtm.Vacuum(), rtm.Vacuum(), mode="bogus")
    # System([s], []) is legal (reference raytrace.py:378)
    assert len(rt.System([flat], []).surfaces) == 1


def test_packing_rejects_unknown_objects(rt, rtm):
    from ray_trace_pb_b200 import engine

    class Weird(rt.Surface):
        pass

    w = Weird([0, 0, 1], [0, 0, 1], [0, 0, 0], [0, 0, 0], 1.0)
    with pytest.raises(NotImplementedError):
        engine.pack_system([w], [rtm.Vacuum(), rtm.Vacuum()])

    class BentFlat(rt.FlatSurface):          # re-defines the geometry: must be refused, not silently ignored
        def get_normal(self, pts):
            return super().get_normal(pts) * 0.5

    class TaggedFlat(rt.FlatSurface):        # adds bookkeeping only: fine
        label = "stop"

    with pytest.raises(NotImplementedError, match="overrides get_normal"):
        engine.pack_system([BentFlat([0, 0, 0], [0, 0, 1], 1.0)], [rtm.Vacuum(), rtm.Vacuum()])
    assert engine.pack_system([TaggedFlat([0, 0, 0], [0, 0, 1], 1.0)], [rtm.Vacuum(), rtm.Vacuum()]).n_surfaces == 1
    with pytest.raises(ValueError):
        engine.pack_system([], [rtm.Vacuum(), rtm.Vacuum()])
    # user media with their own n() need the host table
    cauchy = systems.make_cauchy(rtm)(1.5, 0.004)
    flat = rt.FlatSurface([0, 0, 0], [0, 0, 1], 1.0)
    with pytest.raises(NotImplementedError):
        engine.pack_system([flat], [cauchy, rtm.Vacuum()], wavelengths=None)
    packed = engine.pack_system([flat], [cauchy, rtm.Vacuum()], wavelengths=[0.5, 0.6])
    assert packed.sys.n_wavelengths == 2
    table = np.ctypeslib.as_array(packed.sys.n_table, shape=(3, 2))
    assert table[0, 0] == 1.5 + 0.004 / 0.5**2 and table[1, 1] == 1.0 and np.isnan(table[2, 0])


def test_device_records_use_the_reference_expressions(rt):
    s = rt.SphericalSurface(-56.3, [1, 2, 3], 12.0)
    r = s.device_record()
    assert r["radius_sq"] == (-56.3) ** 2 and r["abs_radius"] == 56.3
    pl = rt.PerfectLens(3.7, [0, 0, 1], np.array([0.6, 0, 0.8]), 0.4)
    r = pl.device_record()
    assert np.array_equal(r["normal_f"], np.array([0.6, 0, 0.8]) * 3.7) and r["sin_alpha"] == np.sin(0.4)
    rev = rt.System([rt.FlatSurface([0, 0, 0], [0, 0, 1], 1.0)], []).reverse().surfaces[0]
    r = rev.device_record()
    assert list(r["normal"]) == [0, 0, 1] and list(r["input_axis"]) == [0, 0, -1]


def test_distinct_wavelengths():
    from ray_trace_pb_b200 import engine
    wl = np.array([0.5, 0.6, np.nan, 0.5, 0.7, 0.6, np.nan])
    assert engine.distinct_wavelengths(wl, 16).tolist() == [0.5, 0.6, 0.7]
    assert engine.distinct_wavelengths(np.arange(1, 40, dtype=float), 16) is None
    assert engine.distinct_wavelengths(np.array([np.nan]), 16).size == 0


def test_host_wavelength_scan_and_table_choice(rt, rtm):
    """threaded C scan (complete list, for media that only exist as Python code) and the 64-ray sample otherwise"""
    from ray_trace_pb_b200 import engine
    rays = np.zeros((300_000, 8))
    rays[:, 7] = 0.5
    rays[123_456, 7] = 0.61
    rays[200_000:200_100, 7] = 0.42
    rays[17, 7] = np.nan
    assert engine.distinct_wavelengths_scan(rays).tolist() == [0.42, 0.5, 0.61]
    rays2 = rays.copy()
    rays2[:, 7] = np.arange(rays.shape[0])
    assert engine.distinct_wavelengths_scan(rays2) is None
    assert engine.distinct_wavelengths_scan(np.full((5, 8), np.nan)).size == 0
    sellmeier = [rtm.Vacuum(), rtm.Bk7()]
    assert engine.choose_wavelength_table(sellmeier, rays).tolist() == [0.5]          # sample: kernel covers the rest
    assert engine.choose_wavelength_table(sellmeier, rays2) is None                   # continuous spectrum
    custom = [rtm.Vacuum(), rtm.Ebaf11()]
    assert engine.choose_wavelength_table(custom, rays).tolist() == [0.42, 0.5, 0.61]  # complete
    assert engine.choose_wavelength_table(custom, rays2) is None
    assert engine.choose_wavelength_table(custom, np.full((5, 8), np.nan)).tolist() == [1.0]


def test_resolve_keep():
    from ray_trace_pb_b200 import _ffi, engine
    assert engine.resolve_keep("all", 7)[::2] == (_ffi.KEEP_ALL, 7)
    assert engine.resolve_keep("last", 7)[::2] == (_ffi.KEEP_LAST, 1)
    mode, idx, n = engine.resolve_keep([0, -2, -1], 7)
    assert mode == _ffi.KEEP_LIST and idx.tolist() == [0, 5, 6] and n == 3
    with pytest.raises(ValueError):
        engine.resolve_keep([3, 2], 7)
    with pytest.raises(ValueError):
        engine.resolve_keep([9], 7)


# ------------------------------------------------------------------------------------------------ materials
def test_materials_match_reference(rtm, host_api):
    wls = np.array(host_api["wavelengths"])
    for name, ref in host_api["materials_n"].items():
        m = getattr(rtm, name)()
        got = np.asarray(m.n(wls), dtype=float)
        if name == "Ebaf11":
            np.testing.assert_allclose(got, ref["n"], rtol=4e-16)
        else:
            parity.assert_bit_identical(got, np.array(ref["n"]), name)
        if ref["vd"] is None:
            assert m.vd is None
        elif np.isnan(ref["vd"]):
            assert np.isnan(m.vd)
        else:
            assert m.vd == ref["vd"]
    c = rtm.Constant(1.33)
    assert c.n(0.5) == 1.33 and c.n(np.array([0.4, np.nan])).tolist() == [1.33, 1.33]
    assert rtm.Material.wd == 0.5876 and rtm.Material.wf == 0.4861 and rtm.Material.wc == 0.6563


# ------------------------------------------------------------------------------------------------ generators
def test_generators_match_reference(rt):
    g = load_golden("generators")
    fan = rt.get_ray_fan([0.1, 0.2, 0.3], 0.7, 11, 0.6, nphis=7, center_ray=(0, 0, 1))
    col = rt.get_collimated_rays([1, 2, 3], 4.0, 9, 0.5, nphis=5, phi_start=0.25, normal=g["normal"])
    coly = rt.get_collimated_rays([0, 0, 0], 2.0, 4, 0.5, nphis=3, normal=(0, 1, 0))
    for got, want in ((fan, g["fan"]), (col, g["collimated"]), (coly, g["collimated_y"])):
        assert got.shape == want.shape
        np.testing.assert_allclose(got, want, rtol=0, atol=4e-16 * max(1.0, np.abs(want).max()))
    # per-ray wavelengths are accepted (reference raytrace.py:115)
    w = np.linspace(0.4, 0.7, 9 * 5)
    assert np.array_equal(rt.get_collimated_rays([0, 0, 0], 1.0, 9, w, nphis=5)[:, 7], w)


# ------------------------------------------------------------------------------------------------ paraxial helpers
def _kidger(rt, rtm):
    d = rt.Doublet(rtm.Nsk11(), rtm.Nsf19(), radius_crown=64.1, radius_flint=-183.685, radius_interface=-43.249,
                   thickness_crown=3.5, thickness_flint=1.5, aperture_radius=10.)
    d.set_aperture_stop(0)
    return d


def test_seidel_sums_kidger_doublet(rt, rtm, host_api):
    """the reference's only unit test (tests/rt_unittest.py:12-46): Kidger section 8.2.2 table, atol 1e-5"""
    d = _kidger(rt, rtm)
    ab = d.seidel_third_order(0.5876, rtm.Vacuum(), rtm.Vacuum(), object_distance=np.inf, object_angle=0.01746)
    np.testing.assert_allclose(ab.sum(axis=0), [0.001889, -0.000088, 0.000295, 0.000210, 0.000002], atol=1e-5)
    np.testing.assert_allclose(ab, host_api["kidger_seidel"], rtol=1e-11, atol=1e-18)
    ab2 = d.seidel_third_order(0.5876, rtm.Vacuum(), rtm.Vacuum(), object_distance=120.0, object_height=2.0)
    np.testing.assert_allclose(ab2, host_api["kidger_seidel_finite"], rtol=1e-11, atol=1e-18)


def test_abcd_cardinal_points_gaussian(rt, rtm, host_api):
    d = _kidger(rt, rtm)
    np.testing.assert_allclose(d.get_ray_transfer_matrix(0.5876, rtm.Vacuum(), rtm.Vacuum()), host_api["kidger_abcd"],
                               rtol=1e-13, atol=1e-15)
    cps = d.get_cardinal_points(0.5876, rtm.Constant(1.1), rtm.Constant(1.333))
    for got, want in zip(cps, host_api["kidger_cardinal"]):
        np.testing.assert_allclose(np.asarray(got, dtype=float), want, rtol=1e-12, atol=1e-12)
    qs = d.gaussian_paraxial(1j * 50.0, 0.5876, rtm.Vacuum(), rtm.Vacuum())
    np.testing.assert_allclose(np.stack((qs.real, qs.imag), axis=1), host_api["kidger_gaussian_q"], rtol=1e-12)
    for mode in ("paraxial-focused", "paraxial-collimated"):
        got = d.auto_focus(0.5876, rtm.Vacuum(), rtm.Vacuum(), mode=mode)
        np.testing.assert_allclose(np.asarray(got, dtype=float), host_api["kidger_autofocus"][mode], rtol=1e-12)


def test_concatenate_builds_the_reference_prescription(rt, rtm, host_api):
    """config 5's system is assembled with Doublet / concatenate / get_cardinal_points: every number must agree"""
    system = systems.achromat_imaging_system(rt, rtm)
    got = systems.describe_system(system, rtm.Vacuum(), rtm.Vacuum())
    want = host_api["achromat_system"]
    assert [s["type"] for s in got["surfaces"]] == [s["type"] for s in want["surfaces"]]
    assert got["materials"] == want["materials"]
    for a, b in zip(got["surfaces"], want["surfaces"]):
        for key in b:
            if key == "type":
                continue
            np.testing.assert_allclose(a[key], b[key], rtol=1e-12, atol=1e-11, err_msg=key)
    assert system.aperture_stop == host_api["achromat_aperture_stop"]
    assert system.surfaces_by_name.tolist() == host_api["achromat_surfaces_by_name"]
    assert system.names == host_api["achromat_names"]
    ab = system.seidel_third_order(0.635, rtm.Vacuum(), rtm.Vacuum(), object_height=5)
    np.testing.assert_allclose(ab, host_api["achromat_seidel"], rtol=1e-8, atol=1e-14)


def test_reverse_and_small_helpers(rt, rtm, host_api):
    d = _kidger(rt, rtm)
    r = d.reverse()
    assert [type(s).__name__ for s in r.surfaces] == ["SphericalSurface"] * 3
    assert r.surfaces[0].radius == d.surfaces[2].radius and r.surfaces[0].input_axis.tolist() == [0, 0, -1]
    assert np.array_equal(r.surfaces[0].center, d.surfaces[2].center) and r.names == [""]
    assert [type(m).__name__ for m in r.materials] == ["Nsf19", "Nsk11"]
    assert np.array_equal(rt.get_free_space_abcd(3.0, 1.5), np.array([[1, 2.0], [0, 1]]))
    g = load_golden("generators")
    angles, na = rt.ray_angle_about_axis(g["fan"][:5], np.array([0, 0, 1.0]))
    np.testing.assert_allclose(angles, host_api["ray_angle_about_axis"]["angles"], rtol=1e-13)
    np.testing.assert_allclose(na, host_api["ray_angle_about_axis"]["na"], rtol=1e-13, atol=1e-16)
    s = rt.SphericalSurface.get_on_axis(50.0, 2.0, 10.0)
    assert s.center.tolist() == [0, 0, 52.0] and s.paraxial_center.tolist() == [0, 0, 2.0]
    np.testing.assert_allclose(s.solve_img_eqn(-1e13, 1.0, 1.5), [150.0])
    np.testing.assert_allclose(s.get_ray_transfer_matrix(1.0, 1.5), [[1, 0], [-0.01, 1]])
    pl = rt.PerfectLens(4.0, [0, 0, 0], [0, 0, 1], 0.5)
    assert pl.aperture_rad == 4.0 * np.sin(0.5)
    on = s.is_pt_on_surface(np.array([[0, 0, 2.0], [0, 0, 2.1], [np.nan, 0, 0]]))
    assert on.tolist() == [True, False, False]
    assert np.array_equal(s.get_normal(np.array([[0, 0, 2.0]])), [[0, 0, -1.0]])


def test_doublet_orientations(rt, rtm):
    kw = dict(radius_crown=50.8, radius_flint=-247.7, radius_interface=-41.7, thickness_crown=20.,
              thickness_flint=3., aperture_radius=25.4)
    fwd = rt.Doublet(rtm.Ebaf11(), rtm.Nsf11(), input_collimated=True, **kw)
    bwd = rt.Doublet(rtm.Ebaf11(), rtm.Nsf11(), input_collimated=False, **kw)
    assert [s.radius for s in fwd.surfaces] == [50.8, -41.7, -247.7]
    assert [s.radius for s in bwd.surfaces] == [247.7, 41.7, -50.8]
    assert [s.paraxial_center[2] for s in bwd.surfaces] == [0, 3.0, 23.0]
    assert [type(m).__name__ for m in bwd.materials] == ["Nsf11", "Ebaf11"]
    flat_back = rt.Doublet(rtm.Nlak22(), rtm.Nsf6(), radius_crown=167.7, radius_flint=np.inf, radius_interface=-285.8,
                           thickness_crown=9.0, thickness_flint=4.0)
    assert type(flat_back.surfaces[2]).__name__ == "FlatSurface" and flat_back.radius_flint == np.inf


def test_raytrace_shim_package(rt):
    import raytrace.materials as shim_m
    import raytrace.raytrace as shim
    assert shim.System is rt.System and shim.get_ray_fan is rt.get_ray_fan
    assert shim_m.Nsf11 is not None


def test_plan_segments_covers_every_slab_once():
    """systems longer than one launch: the segment plan returns each requested slab exactly once, in order, and
    chains through the last slab of every segment but the final one"""
    from ray_trace_pb_b200 import engine
    for S, width in ((70, 64), (130, 64), (64, 64), (5, 2), (1, 64)):
        n_slabs = 2 * S + 1
        for kept in (list(range(n_slabs)), [n_slabs - 1], [], [0], [2 * min(S, width)], [1, 2 * min(S, width) + 1],
                     list(range(0, n_slabs, 3))):
            kept = sorted({k for k in kept if k < n_slabs})
            plan = engine.plan_segments(S, kept, reduce_slab=None, width=width)
            assert [a for a, *_ in plan] == list(range(0, S, width))
            seen = []
            for a, b, local, chain, red in plan:
                assert b - a <= width and chain == (b < S) and red is None
                slabs = [l for l, _ in local]
                assert slabs == sorted(set(slabs)) and all(0 <= l <= 2 * (b - a) for l in slabs)
                if chain:
                    assert slabs[-1] == 2 * (b - a)
                seen += [(2 * a + l, pos) for l, pos in local if pos >= 0]
            assert [g for g, _ in seen] == kept and [p for _, p in seen] == list(range(len(kept)))
        # a reduction lands in exactly one segment, at the right local slab
        for g in (0, 1, 2 * min(S, width), min(2 * min(S, width) + 1, n_slabs - 1), n_slabs - 1):
            hits = [(a, red) for a, b, local, chain, red in engine.plan_segments(S, [], g, width) if red is not None]
            assert len(hits) == 1 and 2 * hits[0][0] + hits[0][1] == g
    kept, n_out = engine.global_keep_list("last", 141)
    assert kept == [140] and n_out == 1
    assert engine.global_keep_list("all", 5) == ([0, 1, 2, 3, 4], 5)
    assert engine.global_keep_list([-1, ], 141)[0] == [140]


def test_degenerate_first_surface_detection(rt, rtm):
    """the speed hint for bundles that meet a flat first surface with exact zeros (engine.degenerate_first_surface)"""
    from ray_trace_pb_b200 import engine
    flat = rt.FlatSurface([0, 0, 2.0], [0, 0, 1], 10.0)
    tilted = rt.FlatSurface([0, 0, 2.0], [0, np.sin(0.25), np.cos(0.25)], 10.0)
    sphere = rt.SphericalSurface.get_on_axis(50.0, 2.0, 10.0)
    rays = np.zeros((5, 8))
    rays[:, 0] = np.linspace(-1, 1, 5)
    rays[:, 5] = 1.0
    rays[:, 7] = 0.5
    assert engine.degenerate_first_surface([flat], rays=rays)                     # along the normal
    assert not engine.degenerate_first_surface([tilted], rays=rays)
    assert not engine.degenerate_first_surface([sphere], rays=rays)
    assert not engine.degenerate_first_surface([], rays=rays)
    skew = rays.copy()
    skew[:, 3], skew[:, 5] = 0.6, 0.8
    assert not engine.degenerate_first_surface([flat], rays=skew)
    skew[:, 2] = 2.0
    assert engine.degenerate_first_surface([flat], rays=skew)                     # launched on the plane
    skew[2, 2] = 2.5
    assert not engine.degenerate_first_surface([flat], rays=skew)                 # ... but not all of them
    skew[2, :3] = np.nan
    assert engine.degenerate_first_surface([flat], rays=skew)                     # invalid rows do not vote
    assert not engine.degenerate_first_surface([flat], rays=np.full((3, 8), np.nan))
    assert engine.degenerate_first_surface([flat], origin=[3, 4, 2.0]) and not engine.degenerate_first_surface(
        [flat], origin=[3, 4, 2.1])
    assert engine.degenerate_first_surface([flat], direction=[0, 0, -1]) and not engine.degenerate_first_surface(
        [flat], direction=[0, 0.6, 0.8])
    packed = engine.pack_system([flat, sphere], [rtm.Vacuum(), rtm.Bk7(), rtm.Vacuum()], None)
    assert packed.sys.surfaces[0].hints == 0
    engine.set_first_surface_hint(packed, True)
    assert packed.sys.surfaces[0].hints == 1 and packed.sys.surfaces[1].hints == 0
    engine.set_first_surface_hint(packed, False)
    assert packed.sys.surfaces[0].hints == 0



def test_pack_memo_is_keyed_by_value(rt, rtm):
    """engine.pack_system_memo: the same prescription comes out of the memo, a changed attribute is a different key (the
    surface objects stay mutable, as in the reference), media that only exist as Python code are packed afresh"""
    from ray_trace_pb_b200 import engine
    system = systems.relay10_system(rt, rtm)
    vac = rtm.Vacuum()
    mats = [vac] + list(system.materials) + [vac]
    a = engine.pack_system_memo(system.surfaces, mats, [0.785])
    assert engine.pack_system_memo(system.surfaces, mats, [0.785]) is a
    assert engine.pack_system_memo(system.surfaces, mats, [0.532]) is not a
    assert engine.pack_system_memo(system.surfaces, mats, None) is not a
    rebuilt = systems.relay10_system(rt, rtm)                          # other objects, same values
    assert engine.pack_system_memo(rebuilt.surfaces, [vac] + list(rebuilt.materials) + [vac], [0.785]) is a
    system.surfaces[3].center = system.surfaces[3].center + np.array([0.0, 0.0, 1e-9])
    b = engine.pack_system_memo(system.surfaces, mats, [0.785])
    assert b is not a and b.sys.surfaces[3].center[2] != a.sys.surfaces[3].center[2]
    system.surfaces[0].aperture_rad = 20.0
    c = engine.pack_system_memo(system.surfaces, mats, [0.785])
    assert c is not b and c.sys.surfaces[0].aperture_rad == 20.0
    mats[2] = rtm.Constant(1.7)
    d = engine.pack_system_memo(system.surfaces, mats, [0.785])
    assert d is not c and d.sys.materials[2].n_const == 1.7
    # byte for byte what the plain packer produces
    plain = engine.pack_system(system.surfaces, mats, [0.785])
    for k in range(len(system.surfaces)):
        assert bytes(d.sys.surfaces[k]) == bytes(plain.sys.surfaces[k])

    class Cauchy:                                                       # a medium that is only Python code
        def n(self, wl):
            return 1.5 + 0.004 / np.asarray(wl, dtype=float) ** 2

    flat = rt.FlatSurface([0, 0, 0], [0, 0, 1], 5.0)
    x = engine.pack_system_memo([flat], [Cauchy(), vac], [0.5])
    assert engine.pack_system_memo([flat], [Cauchy(), vac], [0.5]) is not x

    class BentFlat(rt.FlatSurface):
        def propagate(self, rays, n1, n2):
            return rays

    with pytest.raises(NotImplementedError):
        engine.pack_system_memo([BentFlat([0, 0, 0], [0, 0, 1], 1.0)], [vac, vac], [0.5])
