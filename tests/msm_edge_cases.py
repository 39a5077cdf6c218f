"""Degenerate MSM inputs, shared by the GPU suite (test_gpu_msm_edges.py) and the host emulation (test_emu_msm_edges.py).

Ordinary MSM tests draw every base as k_i G with k_i uniform, so no two entries of a bucket are ever equal or opposite
and the exceptional branches of the group law (doubling, cancellation to infinity, restart from infinity) never run
inside the MSM kernels.  The base families below make them run: in the bucket accumulation, in the merge of boundary
partials and in the bucket reduction, on both the team and the one-thread tails.  Bases are still k_i G, so the
expectation is (sum k_i s_i mod r) G from one scalar multiplication of the oracle."""
from __future__ import annotations

import random

from oracle import ps_oracle as O
from tests import parity_cases as PC

# same: one point everywhere; pm: P, -P alternating with pairwise equal scalars; fold: equal bases with s and r - s
# (the signed-digit fold puts P and -P into one bucket); inf-*: the point at infinity everywhere, on every other
# entry, or first and last; few: k_i in {1, 2, 3, r-1, r-2}; zero-sum: the last scalar makes the sum vanish
FAMILIES = ("same", "pm", "fold", "inf-all", "inf-alt", "inf-ends", "few", "zero-sum")
DEFAULTS = {"msm_team": 1, "msm_wave_floor": 1, "msm_scatter": 1}


def edge_inputs(family, kind, n, rng):
    """(base exponents k_i, scalars s_i) of one family"""
    sc = PC.scalars_of(kind, n, rng)
    k = rng.randrange(1, O.R)
    if family == "same":
        ks = [k] * n
    elif family == "pm":
        ks = [k if i % 2 == 0 else O.R - k for i in range(n)]
        sc = [sc[i - i % 2] for i in range(n)]
    elif family == "fold":
        ks = [0] * n
        for i in range(0, n, 2):
            ks[i] = rng.randrange(1, O.R)
            if i + 1 < n:
                ks[i + 1] = ks[i]
                sc[i + 1] = (O.R - sc[i]) % O.R
    elif family == "inf-all":
        ks = [0] * n
    elif family == "inf-alt":
        ks = [0 if i % 2 == 0 else rng.randrange(1, O.R) for i in range(n)]
    elif family == "inf-ends":
        ks = [rng.randrange(1, O.R) for _ in range(n)]
        ks[0] = ks[-1] = 0
    elif family == "few":
        ks = [rng.choice((1, 2, 3, O.R - 1, O.R - 2)) for _ in range(n)]
    elif family == "zero-sum":
        ks = [rng.choice((1, 2, 3, O.R - 1, rng.randrange(1, O.R))) for _ in range(n)]
        if not any(sc[:-1]):
            sc[0] = 1
        part = sum(a * b for a, b in zip(ks[:-1], sc[:-1])) % O.R
        sc[-1] = -part * pow(ks[-1], -1, O.R) % O.R
    else:
        raise ValueError(family)
    return ks, sc


def msm_edge_check(be, group, n, family, kind="rand", window_bits=0, tables=1, seed=0, team=None, wave_floor=None, scatter=None):
    """MSM of one base family through ps_msm against the oracle (and against the reference's term-by-term sum for
    n <= 64), with the MSM options set for the call and restored afterwards"""
    F, gen, comp, dec = PC._grp(group)
    rng = random.Random("%s/%s/%d/%d/%d" % (family, kind, n, seed, group))
    ks, sc = edge_inputs(family, kind, n, rng)
    opts = {"msm_team": team, "msm_wave_floor": wave_floor, "msm_scatter": scatter}
    bases = None
    try:
        for name, v in opts.items():
            if v is not None:
                be.set_option(name, v)
        bases = be.bases_from_scalars(group, ks, window_bits, tables)
        got = be.msm(bases, sc)
        total = sum(k * s for k, s in zip(ks, sc)) % O.R
        want = comp(O.pt_mul(F, total, gen))
        label = ("G%d" % group, n, family, kind, window_bits, tables, opts)
        assert got == want, label
        if family == "zero-sum":
            assert got == comp(None), label
        if n <= 64:
            pts = [dec(p) for p in bases.export()]
            assert got == comp(O.msm_naive(F, sc, pts)), label
    finally:
        if bases is not None:
            bases.close()
        for name, v in opts.items():
            if v is not None:
                be.set_option(name, DEFAULTS[name])
