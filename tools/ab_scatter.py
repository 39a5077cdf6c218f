#!/usr/bin/env python3
"""A/B of the MSM's bucket sort: the one-pass counting sort (msm_scatter = 0) vs the two-level sort (msm_scatter = 2).
Usage: ab_scatter.py [g1_logs] [ones_logs] [rounds] [json_path]
  g1_logs: sizes with random scalars (default 20,22,24); ones_logs: sizes with every scalar 1 (default 22), which
  puts every entry into one bucket.  Each configuration runs both modes alternately, `rounds` times (default 5),
  and reports the median and the range of every phase; the tool asserts identical result bytes.  The rows and the
  card's name, power limit and maximum SM clock are also written as JSON to json_path when it is given."""
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import playsnark_b200 as ps  # noqa: E402
from playsnark_b200 import _lib as L  # noqa: E402


def _logs(i, default):
    return [int(x) for x in (sys.argv[i] if len(sys.argv) > i else default).split(",") if x]


rand_logs, ones_logs = _logs(1, "20,22,24"), _logs(2, "22")
rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 5
json_path = sys.argv[4] if len(sys.argv) > 4 else None
be = ps.Backend(0)
rng = np.random.default_rng(5)
PHASES = ("sort_ms", "accumulate_ms", "combine_ms", "reduce_ms", "total_ms")


def rand_scalars(n):
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 0] &= 0x3F  # big-endian rows: below r
    return a.tobytes()


def ones_scalars(n):
    a = np.zeros((n, 32), dtype=np.uint8)
    a[:, 31] = 1
    return a.tobytes()


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


rows = []
for log_n, kind in [(k, "rand") for k in rand_logs] + [(k, "ones") for k in ones_logs]:
    n = 1 << log_n
    bases = be.bases_from_scalars(L.PS_G1, rand_scalars(n), 0, -1)
    info = (ctypes.c_int * 4)()
    be.lib.ps_bases_info(bases.handle, info)
    sc = rand_scalars(n) if kind == "rand" else ones_scalars(n)
    outs, runs = {}, {0: [], 2: []}
    for mode in (0, 2):  # warm-up of both paths (arena growth, first launches)
        be.set_option("msm_scatter", mode)
        outs[mode] = be.msm(bases, sc)
    for _ in range(rounds):
        for mode in (0, 2):
            be.set_option("msm_scatter", mode)
            be.msm(bases, sc)
            runs[mode].append(be.msm_timing())
    for mode in (0, 2):
        row = dict(group="G1", log_n=log_n, scalars=kind, scatter=mode, c=info[0], W=info[1], rounds=rounds)
        for k in PHASES:
            v = [t[k] for t in runs[mode]]
            row[k] = round(statistics.median(v), 3)
            row[k + "_range"] = [round(min(v), 3), round(max(v), 3)]
        rows.append(row)
        print(row, flush=True)
    assert outs[0] == outs[2], "one-pass and two-level sort disagree"
    bases.close()
be.set_option("msm_scatter", 1)
gpu = gpu_info()
print("gpu:", gpu, flush=True)
if json_path:
    with open(json_path, "w") as f:
        json.dump({"gpu": gpu, "rows": rows}, f, indent=1)
