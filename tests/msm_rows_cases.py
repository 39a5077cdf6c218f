"""Row-batched MSM (ps_msm_rows / Backend.msm_rows): many scalar rows against one base set in one call, shared by the
host-emulation suite (test_emu_msm_rows.py) and the GPU suite (test_gpu_msm_rows.py).

Every row must equal what ps_msm gives for that row alone, byte for byte, and (at small sizes) the oracle's
(sum_i k_i s_i) G for bases k_i G.  The rows mix the degenerate cases the row mode must keep apart: all-zero rows
(infinity), identical rows (the same digits landing in different rows' buckets), rows of r - 1 (every digit negated)
and the base families of msm_edge_cases."""
from __future__ import annotations

import random

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L
from tests import msm_edge_cases as E
from tests import parity_cases as PC

DEFAULTS = E.DEFAULTS


def mixed_rows(n, rows, rng):
    """row k: 0 -> all zero, 1 and 2 -> the same random row, 3 -> all r - 1, otherwise random"""
    same = [rng.randrange(O.R) for _ in range(n)]
    out = []
    for k in range(rows):
        kind = k % 5
        if kind == 0:
            out.append([0] * n)
        elif kind in (1, 2):
            out.append(list(same))
        elif kind == 3:
            out.append([O.R - 1] * n)
        else:
            out.append([rng.randrange(O.R) for _ in range(n)])
    return out


def _with_options(be, opts, fn):
    try:
        for name, v in opts.items():
            if v is not None:
                be.set_option(name, v)
        return fn()
    finally:
        for name, v in opts.items():
            if v is not None:
                be.set_option(name, DEFAULTS[name])


def rows_check(be, group, n, rows, window_bits=0, tables=1, seed=0, team=None, scatter=None, oracle=True, family=None,
               spot=None):
    """ps_msm_rows over `rows` rows of n scalars against per-row ps_msm (all rows, or the indices in `spot`) and, with
    oracle=True, against the oracle.  family: bases and rows from msm_edge_cases.edge_inputs instead of mixed_rows."""
    F, gen, comp, _ = PC._grp(group)
    rng = random.Random("rows/%d/%d/%d/%s/%d" % (group, n, rows, family, seed))
    if family is None:
        ks = [rng.randrange(1, O.R) for _ in range(n)]
        sc = mixed_rows(n, rows, rng)
    else:
        ks, first = E.edge_inputs(family, "rand", n, rng)
        sc = [first] + [E.edge_inputs(family, "rand", n, random.Random("%s/%d/%d" % (family, seed, k)))[1] for k in range(1, rows)]

    def run():
        bases = be.bases_from_scalars(group, ks, window_bits, tables)
        try:
            got = be.msm_rows(bases, [v for row in sc for v in row], rows)
            assert len(got) == rows
            label = ("G%d" % group, n, rows, window_bits, tables, team, scatter, family)
            for k in (range(rows) if spot is None else spot):
                assert got[k] == be.msm(bases, sc[k]), label + (k,)
                if oracle:
                    assert got[k] == comp(O.pt_mul(F, sum(a * b for a, b in zip(ks, sc[k])) % O.R, gen)), label + (k,)
            if family is None:
                for k in range(rows):
                    if k % 5 == 0:
                        assert got[k] == comp(None), label + (k,)
                    if k % 5 == 2:
                        assert got[k] == got[k - 1], label + (k,)
            return got
        finally:
            bases.close()

    return _with_options(be, {"msm_team": team, "msm_scatter": scatter}, run)


def bad_arguments(be):
    """a row length other than the base set's -> ValueError (PS_ERR_LENGTH); zero rows -> []; a scalar >= r ->
    PS_ERR_ENCODING"""
    import pytest
    from playsnark_b200._lib import PlaysnarkError
    bases = be.bases_from_scalars(L.PS_G1, [3, 5, 7])
    try:
        with pytest.raises(ValueError):
            be.msm_rows(bases, [1] * 8, 2)
        assert be.msm_rows(bases, [], 0) == []
        bad = b"".join(int(v).to_bytes(32, "big") for v in (1, 2, 3, 4, O.R, 6))
        with pytest.raises(PlaysnarkError) as e:
            be.msm_rows(bases, bad, 2)
        assert e.value.status == L.PS_ERR_ENCODING
    finally:
        bases.close()
