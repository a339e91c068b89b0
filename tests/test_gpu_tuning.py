"""
`-m gpu`: the environment variables of the tuning knobs (include/rtb.h) set initial values only.  They are read when
the library is loaded, so an rtb_tune call made before the first trace wins over them.
"""
import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

# (a fresh process: the environment is read once per process)
_CHILD = f"""
import sys
sys.path[:0] = [{str(ROOT)!r}, {str(ROOT / "tests")!r}]
import ray_trace_pb_b200.materials as rtm
import ray_trace_pb_b200.raytrace as rt
import systems
from ray_trace_pb_b200 import _ffi

L = _ffi.lib()
_ffi.check(L.rtb_tune(b"lean_min_rays", 0))
system = systems.relay10_system(rt, rtm)
vac = rtm.Vacuum()
rays = systems.lattice_rays(64, 12.0, 0.0, 0.785)
before = L.rtb_launch_count()
system.ray_trace(rays, vac, vac, keep="last")
print("launches", L.rtb_launch_count() - before)
"""


def test_rtb_tune_before_the_first_trace_wins_over_the_environment():
    """RTB_LEAN_MIN_RAYS=-1 would keep every launch off the lean kernel; rtb_tune("lean_min_rays", 0) before the first
    trace puts 4096 rays of the relay on it: probe + lean trace (2 kernels), not trace_f64 (1)"""
    env = dict(os.environ, RTB_LEAN_MIN_RAYS="-1")
    r = subprocess.run([sys.executable, "-c", _CHILD], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    launches = [line.split()[1] for line in r.stdout.splitlines() if line.startswith("launches ")]
    assert launches == ["2"], r.stdout[-3000:]
