"""
GPU test (`-m gpu`) of the sign and zero tests of the lean on-axis steps (csrc/lean_steps.cuh): the front-side cull
dz az < 0, the flat's t < 0 and the products by nz = +-1 are taken from sign bits there, and a dz whose high word is that
of a zero fails the lean flag.  So a ray with dz = +-0 or a subnormal dz, a back-facing ray, and surfaces whose normal
or input axis is -z must still give the oracle's bits.

One lens train traced along +z and its mirror image traced along -z (spheres with input axis -z, flats with normal
-z).  Each train has a flat whose input axis is opposite to its normal and whose normal has a -0 component.  The bundle
mixes ordinary skew rays, rays that travel sideways (dx = 1, dz = +-0 or a subnormal of either sign) into the side of
the first sphere's cap, rays that meet the first sphere from behind, and rays that start beyond the first flat of a
second train (t < 0 there) or run backwards into it.
"""
import numpy as np
import pytest

import parity
from test_gpu_lean import lean  # noqa: F401  (fixture: lean kernel forced on, probe-driven or pure)

pytestmark = pytest.mark.gpu

SIDEWAYS_DZ = np.array([0.0, -0.0, 5e-324, -5e-324, 1e-310, -1e-310])


def _train(rt, rtm, s, flat_first):
    """s = +1: along +z; s = -1: the mirror image z -> -z"""
    def sphere(radius, vertex_z, ap):
        return rt.SphericalSurface(radius, [0, 0, s * (vertex_z + radius)], ap, input_axis=(0, 0, s))

    flipped = rt.FlatSurface([0, 0, s * 26.0], [-0.0, 0.0, -s * 1.0], 45.0)
    flipped.input_axis = -flipped.input_axis                    # normal against the light, input axis along it
    surfaces = [sphere(30.0, 5.0, 25.0), rt.FlatSurface([0, 0, s * 20.0], [0, 0, s * 1.0], 45.0), flipped,
                sphere(-80.0, 32.0, 45.0)]
    # (indices rising along the train: the steep sideways rays are not totally reflected)
    media = [rtm.Constant(1.5), rtm.Constant(1.6), rtm.Constant(1.65)]
    if flat_first:
        surfaces.insert(0, rt.FlatSurface([0, 0, 0.0], [0, 0, s * 1.0], 30.0))
        media.insert(0, rtm.Vacuum())
    return rt.System(surfaces, media)


def _bundle(s, n=24_000, seed=5):
    rng = np.random.default_rng(seed + (s > 0))
    rays = np.zeros((n, 8))
    rays[:, 0:2] = rng.uniform(-14, 14, (n, 2))
    rays[:, 2] = -5.0
    d = rng.standard_normal((n, 3)) * np.array([0.05, 0.05, 0.0]) + np.array([0, 0, 1.0])
    rays[:, 3:6] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rays[:, 6] = rng.uniform(0, 20, n)
    rays[:, 7] = 0.6328
    q = n // 8
    groups = {}
    # sideways into the side of the first sphere's cap (z = 8 between its vertex at 5 and its rim)
    side = slice(0, q)
    rays[side, 0] = -40.0
    rays[side, 1] = rng.uniform(-5, 5, q)
    rays[side, 2] = 8.0
    rays[side, 3:6] = 0.0
    rays[side, 3] = 1.0
    rays[side, 5] = rng.choice(SIDEWAYS_DZ, q)
    groups["sideways"] = side
    # from behind the first sphere, travelling back towards it: culled there (dz az < 0)
    back = slice(q, 2 * q)
    rays[back, 2] = 9.0
    rays[back, 5] *= -1
    groups["back"] = back
    # beyond the first flat of the flat-first train, forwards (t < 0 there) or backwards (dz az < 0)
    beyond = slice(2 * q, 3 * q)
    rays[beyond, 2] = 3.0
    rays[2 * q: 3 * q: 2, 5] *= -1
    groups["beyond"] = beyond
    rays[:, 2] *= s
    rays[:, 5] *= s
    return rays, groups


@pytest.mark.parametrize("s", [1, -1], ids=["plus_z", "minus_z"])
@pytest.mark.parametrize("flat_first", [False, True], ids=["sphere_first", "flat_first"])
def test_lean_signs_and_zeros_vs_oracle(s, flat_first, rt, rtm, oracle, lean):  # noqa: F811
    system = _train(rt, rtm, s, flat_first)
    rays, groups = _bundle(s)
    vac, out = rtm.Vacuum(), rtm.Constant(1.7)
    got = system.ray_trace(rays, vac, out, keep="last")
    want = oracle.ray_trace(system, rays, vac, out, n_threads=8)[-1:]
    parity.assert_bit_identical(got, want, f"signs and zeros, s = {s}, flat first = {flat_first}")
    assert np.isfinite(want[0, :, 0]).sum() > len(rays) // 4                       # the ordinary rays get through
    if not flat_first:
        assert np.isfinite(want[0, groups["sideways"], 0]).any()                  # some sideways rays too
