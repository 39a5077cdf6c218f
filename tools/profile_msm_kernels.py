#!/usr/bin/env python3
"""Device time per kernel of one G1 MSM (all window tables, random scalars) under torch.profiler, for the one-pass
counting sort (msm_scatter = 0) and the two-level sort (msm_scatter = 2); mean of 3 calls after 2 warm-up calls.
Usage: profile_msm_kernels.py [log_n]"""
import collections
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
import playsnark_b200 as ps  # noqa: E402
from playsnark_b200 import _lib as L  # noqa: E402

log_n = int(sys.argv[1]) if len(sys.argv) > 1 else 24
be = ps.Backend(0)
rng = np.random.default_rng(5)


def rand_scalars(n):
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 0] &= 0x3F  # big-endian rows: below r
    return a.tobytes()


n = 1 << log_n
bases = be.bases_from_scalars(L.PS_G1, rand_scalars(n), 0, -1)
sc = rand_scalars(n)
CALLS = 3
for mode in (0, 2):
    be.set_option("msm_scatter", mode)
    be.msm(bases, sc)
    be.msm(bases, sc)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(CALLS):
            be.msm(bases, sc)
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0, 0.0])
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            a = agg[e.name[:100]]
            a[0] += 1
            a[1] += e.device_time / 1000.0
    print("2^%d points, msm_scatter = %d, phases of the last call:" % (log_n, mode), be.msm_timing())
    for k, (c, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        if t / CALLS > 0.005:
            print("  %8.3f ms/call  x%-3d %s" % (t / CALLS, c // CALLS, k))
be.set_option("msm_scatter", 1)
bases.close()
