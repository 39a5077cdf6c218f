"""Degenerate MSM inputs (tests/msm_edge_cases.py) through the host emulation of the C ABI (-DPS_HOST_EMU) at small
sizes; test_gpu_msm_edges.py runs the same families on the device."""
import os

import pytest

from playsnark_b200 import _lib as L, api, build as B
from tests import msm_edge_cases as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def be():
    so = B.build_host_emulation(os.path.join(ROOT, "tests", "_build"))
    lib = L.bind(so)
    assert b"HOST EMULATION" in lib.ps_version()
    b = api.Backend(0, lib=lib)
    yield b
    b.close()


@pytest.mark.parametrize("family", E.FAMILIES)
def test_msm_edge_families(be, family):
    """degenerate bases (equal, opposite, infinity, small multiples, a vanishing sum) on both tail paths"""
    E.msm_edge_check(be, L.PS_G1, 40, family, "rand", 5, 3, team=0, scatter=2)
    E.msm_edge_check(be, L.PS_G1, 33, family, "ones", 4, 1, team=1, wave_floor=0)
    E.msm_edge_check(be, L.PS_G2, 9, family, "small", 0, 1, team=0)
    E.msm_edge_check(be, L.PS_G2, 6, family, "edge", 6, 4, team=1)


@pytest.mark.parametrize("kind", ["neg", "edge"])
def test_msm_edge_two_points(be, kind):
    for family in ("same", "pm", "fold", "zero-sum"):
        E.msm_edge_check(be, L.PS_G1, 2, family, kind, 13, 1)
