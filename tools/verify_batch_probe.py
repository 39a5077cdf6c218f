#!/usr/bin/env python3
"""Measurement of the batch Groth16 verifier (ps_g16_verify_batch) on proofs of the 2^10 squaring chain.

Checks the decisions first, then times the call (host clock around the call, which ends in a device synchronise) at
N = 1, 64, 1024, 4096, 16384 with pre-marshalled inputs (io values pinned in a HostBuffer), with the device phases of
ps_last_verify_batch_timing; then a failed batch's bisection with 1 and 8 invalid proofs, and ps_g16_verify one proof per
call for comparison.  Prints the card's name and power limit with the numbers.
Usage: verify_batch_probe.py [--out FILE.md] [--sizes 1,64,...] [--reps K]"""
import argparse
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import playsnark_b200 as ps  # noqa: E402
from playsnark_b200 import api  # noqa: E402
from tests import verify_batch_cases as V  # noqa: E402

PHASES = ("upload", "decode+subgroup", "weighting", "io upload+convert", "Miller loops", "tree", "root check", "bisection")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown (nvidia-smi unavailable)"


def timed(fn, reps):
    fn()                                   # warm-up of this shape
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts)


def phases(be):
    import ctypes as C
    t = (C.c_float * 9)()
    be._check(be.lib.ps_last_verify_batch_timing(be.ctx, t))
    return [t[i] for i in range(9)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--sizes", default="1,64,1024,4096,16384")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    lines = []

    def out(s=""):
        print(s, flush=True)
        lines.append(s)

    be = ps.Backend(0)
    out("# Batch Groth16 verification (ps_g16_verify_batch), 2^10 squaring chain")
    out()
    out("Card (name, power limit, max SM clock): %s" % card())
    t0 = time.time()
    pool = V.Pool(be, n=1 << 10, count=64, seed=3)
    n_io = len(pool.tr.IoLP)
    out("Key: 2^10 gates, %d public inputs per proof; pool of 64 distinct device proofs, cycled (%.1f s to make)."
        % (n_io, time.time() - t0))
    blobs = [api._fr_bytes(v) for v in pool.ios]

    def batch(N):
        return [pool.proofs[i % 64] for i in range(N)], api.HostBuffer(be, b"".join(blobs[i % 64] for i in range(N)))

    out()
    out("| N | call (ms, median of %d) | proofs/s | %s | device total (ms) |" % (a.reps, " | ".join(PHASES[:7])))
    out("|---|---|---|%s---|" % ("---|" * 7))
    for N in [int(x) for x in a.sizes.split(",")]:
        proofs, hb = batch(N)
        assert pool.verify(proofs, hb) is True, N                      # decisions before timing
        bad, _ = V.mutate(proofs, [[0]] * N, N // 2, "C+G")
        assert pool.verify(bad, hb) is False, N
        dt = timed(lambda: pool.verify(proofs, hb), a.reps)
        ph = phases(be)
        out("| %d | %.2f | %.0f | %s | %.2f |" % (N, dt * 1e3, N / dt, " | ".join("%.2f" % x for x in ph[:7]), ph[8]))
        hb.close()
    out()
    out("Failed batch, N = 4096, per-proof verdicts (bisection over the proof tree):")
    out()
    out("| invalid | call with per_proof (ms) | bisection phase (ms) | call without per_proof (ms) |")
    out("|---|---|---|---|")
    N = 4096
    for k in (1, 8):
        proofs, hb = batch(N)
        pos = sorted(random.Random(k).sample(range(N), k))
        for t, i in enumerate(pos):
            proofs, _ = V.mutate(proofs, [[0]] * N, i, ("A+G", "B+H", "C+G")[t % 3])
        assert pool.verify(proofs, hb, per_proof=True) == [i not in pos for i in range(N)]
        dt = timed(lambda: pool.verify(proofs, hb, per_proof=True), a.reps)
        ph = phases(be)
        dn = timed(lambda: pool.verify(proofs, hb), a.reps)
        out("| %d | %.2f | %.2f | %.2f |" % (k, dt * 1e3, ph[7], dn * 1e3))
        hb.close()
    out()
    p0, io0 = pool.proofs[0], pool.ios[0]
    assert api.Groth16Verify(pool.tr, pool.q, p0, io0, backend=be)
    dv = timed(lambda: api.Groth16Verify(pool.tr, pool.q, p0, io0, backend=be), a.reps)
    out("ps_g16_verify, one proof per call: %.2f ms (%.1f proofs/s)." % (dv * 1e3, 1 / dv))
    pool.close()
    be.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
