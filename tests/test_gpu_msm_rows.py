"""Row-batched MSM (tests/msm_rows_cases.py) on the product library: the host-emulation cases at full size, 4096 rows
of 1023 points in G1 and G2 (spot-checked against ps_msm), and a call whose rows x n x W passes 2^31 entries, which
runs as several pipelines."""
import random

import numpy as np
import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api
from tests import msm_edge_cases as E
from tests import msm_rows_cases as M

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    b = api.Backend(0)
    yield b
    b.close()


@pytest.mark.parametrize("group", [L.PS_G1, L.PS_G2])
@pytest.mark.parametrize("rows", [1, 12, 13, 100])
@pytest.mark.parametrize("n", [1, 1023])
def test_rows(be, group, rows, n):
    M.rows_check(be, group, n, rows, oracle=(n == 1 or rows <= 13))


@pytest.mark.parametrize("group", [L.PS_G1, L.PS_G2])
@pytest.mark.parametrize("team", [0, 1])
@pytest.mark.parametrize("scatter", [0, 2])
def test_rows_modes(be, group, team, scatter):
    M.rows_check(be, group, 1023, 13, window_bits=16, tables=-1, team=team, scatter=scatter, oracle=False)
    M.rows_check(be, group, 1023, 100, window_bits=10, tables=-1, team=team, scatter=scatter, oracle=False)


@pytest.mark.parametrize("family", E.FAMILIES)
def test_rows_edge_families(be, family):
    M.rows_check(be, L.PS_G1, 1023, 13, family=family, team=0)
    M.rows_check(be, L.PS_G2, 64, 13, family=family, team=1)


def test_rows_bad_arguments(be):
    M.bad_arguments(be)


def _random_rows(rows, n, seed):
    """rows x n uniform scalars below 2^254 < r as wire bytes"""
    raw = np.random.default_rng(seed).integers(0, 256, size=(rows * n, 32), dtype=np.uint8)
    raw[:, 0] &= 0x3F
    return raw.tobytes()


@pytest.mark.parametrize("group", [L.PS_G1, L.PS_G2])
def test_rows_4096x1023(be, group):
    """4096 rows of 1023 points with all window tables at the batch window: spot rows equal ps_msm"""
    rng = random.Random(group)
    bases = be.bases_from_scalars(group, [rng.randrange(1, O.R) for _ in range(1023)], 10, -1)
    try:
        buf = _random_rows(4096, 1023, group)
        got = be.msm_rows(bases, buf, 4096)
        for k in (0, 1, 2047, 4094, 4095):
            assert got[k] == be.msm(bases, buf[k * 1023 * 32:(k + 1) * 1023 * 32]), k
    finally:
        bases.close()


def test_rows_pipeline_split(be):
    """window 2 (W = 128), 2^14 points, 1100 rows: 2.3 * 10^9 entries, more than one pipeline takes (2^31); rows on both
    sides of the split equal ps_msm"""
    rng = random.Random(11)
    n, rows = 1 << 14, 1100
    bases = be.bases_from_scalars(L.PS_G1, [rng.randrange(1, O.R) for _ in range(n)], 2, 1)
    try:
        buf = _random_rows(rows, n, 11)
        got = be.msm_rows(bases, buf, rows)
        cap = (2 ** 31 - 1) // (n * 128)
        for k in (0, cap - 1, cap, rows - 1):
            assert got[k] == be.msm(bases, buf[k * n * 32:(k + 1) * n * 32]), k
    finally:
        bases.close()
