"""Batch PHGR13 verification (tests/phgr13_verify_batch_cases.py) through the host emulation of the C ABI (-DPS_HOST_EMU)
at N <= 5; test_gpu_phgr13_verify_batch.py runs the same cases on the device."""
import os

import pytest

from playsnark_b200 import _lib as L, api, build as B
from tests import phgr13_verify_batch_cases as V

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pool():
    so = B.build_host_emulation(os.path.join(ROOT, "tests", "_build"))
    lib = L.bind(so)
    assert b"HOST EMULATION" in lib.ps_version()
    be = api.Backend(0, lib=lib)
    p = V.Pool(be, n=8, count=5)
    yield p
    p.close()
    be.close()


@pytest.mark.parametrize("N", [1, 2, 5])
def test_honest(pool, N): V.honest(pool, N)


@pytest.mark.parametrize("kind", V.MUTATIONS)
@pytest.mark.parametrize("pos", [0, 2, 4])
def test_one_invalid(pool, kind, pos): V.one_invalid(pool, 5, pos, kind)


def test_two_invalid(pool): V.several_invalid(pool, 5, [1, 3])
def test_all_invalid(pool): V.several_invalid(pool, 5, list(range(5)))
def test_weights_independent(pool): V.weights_independent(pool)
def test_matches_oracle(pool): V.matches_oracle(pool)
def test_no_io(pool): V.no_io(pool.be)
def test_malformed_points(pool): V.malformed_points(pool)
def test_bad_arguments(pool): V.bad_arguments(pool)
def test_blob_inputs(pool): V.blob_inputs(pool)
