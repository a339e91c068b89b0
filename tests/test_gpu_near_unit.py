"""
GPU test (`-m gpu`) of the lean steps' near-one table (csrc/exact_math.cuh, xm::near_one): the second Snell basis vector
c = n x b^ is divided by sqrt(|c|^2) read from a table of the 256 doubles next to 1.0, and a ray whose |c|^2 falls outside
the table fails its lean step and is re-traced by the careful path.  A sphere far from the origin with a small radius
puts |c|^2 hundreds of ulps from 1.0 for most rays (the position on the sphere carries the rounding error of z ~ 1e4, the
normal divides it by R ~ 5); the lean kernel must still give the oracle's bits, with the probe counting those failures.
"""
import numpy as np
import pytest

import parity
import systems
from test_gpu_lean import lean  # noqa: F401  (fixture: lean kernel forced on, probe-driven or pure)

pytestmark = pytest.mark.gpu


def _far_sphere(rt, rtm):
    sphere = rt.SphericalSurface.get_on_axis(5.0, 1e4 - 5.0, 4.5)          # centre at z = 1e4
    flat = rt.FlatSurface([0, 0, 1e4 + 20.0], [0, 0, 1], 50.0)
    return rt.System([sphere, flat], [rtm.Constant(1.5)])


def test_far_sphere_outside_the_near_one_table(rt, rtm, oracle, lean):  # noqa: F811
    system = _far_sphere(rt, rtm)
    vac = rtm.Vacuum()
    rays = systems.lattice_rays(200, 4.0, 1e4 - 30.0, 0.785, tilt=(0.003, -0.002))
    got = system.ray_trace(rays, vac, vac, keep="last")
    want = oracle.ray_trace(system, rays, vac, vac, n_threads=8)[-1:]
    parity.assert_bit_identical(got, want, "sphere at z = 1e4, R = 5")
    assert np.isfinite(want[0, :, 0]).sum() > 30_000                       # the bundle gets through
    counts = lean.probe_counts(len(system.surfaces))
    # about nine in ten probe rays fail the sphere's lean step (|c|^2 outside the table: k from -3252 to 1642 in
    # tools/near_unit_histogram.py's mirror of the step); the flat behind it stays lean
    assert counts[0, 0] > 1500 and counts[0, 1] * 2 > counts[0, 0], counts
    assert counts[1, 1] == 0, counts
