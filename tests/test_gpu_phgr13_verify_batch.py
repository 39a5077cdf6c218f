"""Batch PHGR13 verification (tests/phgr13_verify_batch_cases.py) on the product library: the cases of the
host-emulation suite at N = 1, 7, 64 and 1000, and 4096 proofs of the 2^10 squaring chain with three invalid ones."""
import random

import pytest

from playsnark_b200 import api
from tests import phgr13_verify_batch_cases as V

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    b = api.Backend(0)
    yield b
    b.close()


@pytest.fixture(scope="module")
def pool(be):
    p = V.Pool(be, n=8, count=8)
    yield p
    p.close()


@pytest.mark.parametrize("N", [1, 7, 64, 1000])
def test_honest(pool, N): V.honest(pool, N)


@pytest.mark.parametrize("kind", V.MUTATIONS)
@pytest.mark.parametrize("N", [1, 7, 64, 1000])
def test_one_invalid(pool, N, kind):
    for pos in sorted({0, N // 2, N - 1}):
        V.one_invalid(pool, N, pos, kind)


@pytest.mark.parametrize("N", [7, 64, 1000])
def test_several_invalid(pool, N):
    V.several_invalid(pool, N, [1, N - 2])
    V.several_invalid(pool, N, sorted(random.Random(N).sample(range(N), min(N, 9))))


def test_all_invalid(pool): V.several_invalid(pool, 7, list(range(7)))
def test_weights_independent(pool): V.weights_independent(pool)
def test_matches_oracle(pool): V.matches_oracle(pool, 3)
def test_no_io(pool): V.no_io(pool.be)
def test_malformed_points(pool): V.malformed_points(pool, 7)
def test_bad_arguments(pool): V.bad_arguments(pool)
def test_blob_inputs(pool): V.blob_inputs(pool)


def test_chain_2p10_4096_proofs(be):
    """4096 proofs of the 2^10 chain (64 distinct device proofs, cycled) with 3 invalid at seeded positions: the batch is
    rejected and per_proof flags exactly those 3"""
    pool = V.Pool(be, n=1 << 10, count=64, seed=2)
    N = 4096
    blobs = [api._fr_bytes(v) for v in pool.ios]
    proofs = [pool.proofs[i % 64] for i in range(N)]
    blob = b"".join(blobs[i % 64] for i in range(N))
    assert pool.verify(proofs, blob) is True
    bad = sorted(random.Random(4096).sample(range(N), 3))
    for t, i in enumerate(bad):
        proofs, _ = V.mutate(proofs, [[0]] * N, i, ("hs", "wss", "gz")[t])
    hb = api.HostBuffer(be, blob)
    assert pool.verify(proofs, hb) is False
    assert pool.verify(proofs, hb, per_proof=True) == [i not in bad for i in range(N)]
    hb.close()
    pool.close()
