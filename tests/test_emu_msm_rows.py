"""Row-batched MSM (tests/msm_rows_cases.py) through the host emulation of the C ABI (-DPS_HOST_EMU) at small sizes;
test_gpu_msm_rows.py runs the same cases on the device, up to 4096 rows of 1023 points."""
import os

import pytest

from playsnark_b200 import _lib as L, api, build as B
from tests import msm_edge_cases as E
from tests import msm_rows_cases as M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def be():
    so = B.build_host_emulation(os.path.join(ROOT, "tests", "_build"))
    lib = L.bind(so)
    assert b"HOST EMULATION" in lib.ps_version()
    b = api.Backend(0, lib=lib)
    yield b
    b.close()


@pytest.mark.parametrize("group", [L.PS_G1, L.PS_G2])
@pytest.mark.parametrize("rows", [1, 12, 13, 100])
@pytest.mark.parametrize("n", [1, 33])
def test_rows_small(be, group, rows, n):
    M.rows_check(be, group, n, rows)


@pytest.mark.parametrize("group", [L.PS_G1, L.PS_G2])
@pytest.mark.parametrize("rows", [1, 13])
def test_rows_1023(be, group, rows):
    M.rows_check(be, group, 1023, rows, oracle=(group == L.PS_G1))


@pytest.mark.parametrize("team", [0, 1])
@pytest.mark.parametrize("scatter", [0, 2])
def test_rows_modes(be, team, scatter):
    """both tail paths and both scatters; window 16 with all its tables keeps W <= 16, so scatter 2 stages the row mode
    through the two-pass scatter"""
    M.rows_check(be, L.PS_G1, 20, 13, window_bits=16, tables=-1, team=team, scatter=scatter)
    M.rows_check(be, L.PS_G1, 33, 12, window_bits=5, tables=1, team=team, scatter=scatter)
    M.rows_check(be, L.PS_G2, 9, 13, window_bits=16, tables=-1, team=team, scatter=scatter)


@pytest.mark.parametrize("family", E.FAMILIES)
def test_rows_edge_families(be, family):
    M.rows_check(be, L.PS_G1, 24, 5, family=family, team=0)
    M.rows_check(be, L.PS_G2, 6, 3, family=family, team=1)


def test_rows_bad_arguments(be):
    M.bad_arguments(be)
