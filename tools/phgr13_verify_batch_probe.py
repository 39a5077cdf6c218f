#!/usr/bin/env python3
"""Measurement of the batch PHGR13 verifier (ps_phgr13_verify_batch) on proofs of the 2^10 squaring chain, and of the
row-batched MSM (ps_msm_rows) it is built on.

Checks the decisions first, then times the call (host clock around the call, which ends in a device synchronise) at
N = 1, 64, 1024, 4096 with pre-marshalled inputs (io values pinned in a HostBuffer), with the device phases of
ps_last_verify_batch_timing; then a failed batch's bisection with 1 and 8 invalid proofs; ps_phgr13_verify one proof per
call; and ps_msm_rows over 4096 rows of 1023 points in G1 and G2, in one call and as calls of 12 rows each.  Prints the
card's name and power limit with the numbers.
Usage: phgr13_verify_batch_probe.py [--out FILE.md] [--sizes 1,64,...] [--reps K]"""
import argparse
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import playsnark_b200 as ps  # noqa: E402
from oracle import ps_oracle as O  # noqa: E402
from playsnark_b200 import _lib as L, api  # noqa: E402
from tests import phgr13_verify_batch_cases as V  # noqa: E402
from tools.verify_batch_probe import PHASES, card, phases, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--sizes", default="1,64,1024,4096")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    lines = []

    def out(s=""):
        print(s, flush=True)
        lines.append(s)

    be = ps.Backend(0)
    out("# Batch PHGR13 verification (ps_phgr13_verify_batch), 2^10 squaring chain")
    out()
    out("Card (name, power limit, max SM clock): %s" % card())
    t0 = time.time()
    pool = V.Pool(be, n=1 << 10, count=64, seed=3)
    out("Key: 2^10 gates, %d public values per proof; pool of 64 distinct device proofs, cycled (%.1f s to make)."
        % (pool.diff, time.time() - t0))
    blobs = [api._fr_bytes(v) for v in pool.ios]

    def batch(N):
        return [pool.proofs[i % 64] for i in range(N)], api.HostBuffer(be, b"".join(blobs[i % 64] for i in range(N)))

    out()
    out("Phase [3] is the io upload and conversion plus both per-proof io MSMs (msm_rows in G1 and in G2).")
    out()
    out("| N | call (ms, median of %d) | proofs/s | %s | device total (ms) |" % (a.reps, " | ".join(PHASES[:7])))
    out("|---|---|---|%s---|" % ("---|" * 7))
    for N in [int(x) for x in a.sizes.split(",")]:
        proofs, hb = batch(N)
        assert pool.verify(proofs, hb) is True, N                      # decisions before timing
        bad, _ = V.mutate(proofs, [[0]] * N, N // 2, "gz")
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
            proofs, _ = V.mutate(proofs, [[0]] * N, i, ("hs", "wss", "gz")[t % 3])
        assert pool.verify(proofs, hb, per_proof=True) == [i not in pos for i in range(N)]
        dt = timed(lambda: pool.verify(proofs, hb, per_proof=True), a.reps)
        ph = phases(be)
        dn = timed(lambda: pool.verify(proofs, hb), a.reps)
        out("| %d | %.2f | %.2f | %.2f |" % (k, dt * 1e3, ph[7], dn * 1e3))
        hb.close()
    out()
    p0, io0 = pool.proofs[0], pool.ios[0]
    assert pool.verify_one(p0, io0)
    dv = timed(lambda: pool.verify_one(p0, io0), a.reps)
    out("ps_phgr13_verify, one proof per call: %.2f ms (%.1f proofs/s)." % (dv * 1e3, 1 / dv))
    pool.close()

    out()
    out("ps_msm_rows, 4096 rows x 1023 points (uniform scalars; bases with all window tables at c = 10, the window the")
    out("verifier picks for this shape), host clock around calls that end in a device synchronise, scalar upload included:")
    out()
    out("| group | one call, 4096 rows (ms) | 342 calls of 12 rows (ms) | ratio |")
    out("|---|---|---|---|")
    rows, n = 4096, 1023
    raw = np.random.default_rng(1).integers(0, 256, size=(rows * n, 32), dtype=np.uint8)
    raw[:, 0] &= 0x3F
    buf = raw.tobytes()
    rng = random.Random(2)
    for group in (L.PS_G1, L.PS_G2):
        bases = be.bases_from_scalars(group, [rng.randrange(1, O.R) for _ in range(n)], 10, -1)
        whole = be.msm_rows(bases, buf, rows)
        step = 12 * n * 32
        parts = [p for r0 in range(0, rows, 12) for p in be.msm_rows(bases, buf[r0 * n * 32:r0 * n * 32 + step], min(12, rows - r0))]
        assert parts == whole
        t1 = timed(lambda: be.msm_rows(bases, buf, rows), a.reps)
        t12 = timed(lambda: [be.msm_rows(bases, buf[r0 * n * 32:r0 * n * 32 + step], min(12, rows - r0))
                             for r0 in range(0, rows, 12)], max(1, a.reps // 2))
        out("| G%d | %.2f | %.2f | %.1f |" % (group, t1 * 1e3, t12 * 1e3, t12 / t1))
        bases.close()
    be.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
