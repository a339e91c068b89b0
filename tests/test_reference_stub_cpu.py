"""
CPU test (no GPU): the ctypes stub of INTEGRATION.md section 2 (tests/reference_stub.py) run against the REAL reference
objects -- as recorded in the golden cases by tests/golden/make_golden.py: every attribute the stub reads from the
reference's surfaces (the case's `system` prescription) and the reference media's n() at the case's wavelengths
(`n_table`) -- up to, and not including, the device call: every struct the stub packs from them must equal, byte for
byte, what this framework's host layer packs from its mirror of the same system, and the refractive-index tables must
be the same bits.
"""
import ctypes
import json
from types import SimpleNamespace

import numpy as np
import pytest

import systems
from conftest import load_golden


class RecordedMedium:
    """One of the reference's media, answering n() with the values recorded from it.  The stub also asks for n(NaN);
    where a case did not record that column, the reference's rule applies, as edge_mix's table records it: a Constant
    gives its index, every Sellmeier medium (Vacuum included) NaN."""

    def __init__(self, desc, wavelengths, values):
        self.known = dict(zip(wavelengths.tolist(), values.tolist()))
        recorded = [v for w, v in self.known.items() if np.isnan(w)]
        self.at_nan = recorded[0] if recorded else (desc["n"] if desc["type"] == "Constant" else np.nan)

    def n(self, wavelength):
        return np.array([self.at_nan if np.isnan(w) else self.known[w] for w in np.asarray(wavelength).reshape(-1)])


def recorded_reference(name):
    """(system, m_in, m_out, rays) of a golden case, standing in for the reference's own objects"""
    g = load_golden(name)
    desc = json.loads(str(g["system"]))
    surfaces = []
    for d in desc["surfaces"]:
        s = type(d["type"], (), {})()                  # the stub dispatches on the class name
        s.__dict__.update({k: np.array(v) if isinstance(v, list) else v for k, v in d.items() if k != "type"})
        surfaces.append(s)
    media = [desc["initial_material"]] + desc["materials"] + [desc["final_material"]]
    media = [RecordedMedium(m, g["unique_wavelengths"], g["n_table"][:, k]) for k, m in enumerate(media)]
    return SimpleNamespace(surfaces=surfaces, materials=media[1:-1]), media[0], media[-1], g["rays_in"], desc


@pytest.mark.parametrize("builder", ["relay10", "opm", "edge_mix", "doublet_nlak22", "mirrors", "reversed_doublet"])
def test_stub_packs_the_real_reference_classes(builder, rt, rtm):
    import reference_stub
    from ray_trace_pb_b200 import engine
    system, m_in, m_out, rays, desc = recorded_reference(builder)                    # the reference's own values
    sysd, packed_rays, _keep = reference_stub.pack(system, rays, m_in, m_out)
    assert sysd.n_surfaces == len(system.surfaces) and packed_rays.shape == (len(rays), 8)

    mirror, mm_in, mm_out = systems.rebuild_system(desc, rt, rtm)
    wl = np.unique(rays[~np.isnan(rays[:, 7]), 7])
    ours = engine.pack_system(mirror.surfaces, [mm_in] + mirror.materials + [mm_out], wl)
    assert ours.sys.n_surfaces == sysd.n_surfaces and ours.sys.n_wavelengths == sysd.n_wavelengths
    for k in range(sysd.n_surfaces):
        a, b = sysd.surfaces[k], ours.sys.surfaces[k]
        b.hints = 0                                          # (speed hints are this framework's own business)
        assert bytes(a) == bytes(b), f"surface {k} of {builder}"
    n_tab = (sysd.n_wavelengths + 1) * (sysd.n_surfaces + 1)
    ta = np.ctypeslib.as_array(sysd.n_table, shape=(n_tab,))
    tb = np.ctypeslib.as_array(ours.sys.n_table, shape=(n_tab,))
    assert np.array_equal(ta.view(np.uint64), tb.view(np.uint64)), "refractive-index table"
    assert ctypes.sizeof(reference_stub.RtbSurface) == ctypes.sizeof(type(ours.sys.surfaces[0]))
