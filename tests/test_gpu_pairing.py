"""The verifiers' arithmetic as compiled for sm_100a (tests/device_pairing.cu), value by value against the oracle: the Fp6 /
Fp12 tower, the Frobenius map, pow_x, the Miller loop, the final exponentiation, the pairing-product check, the square
roots, the scalar multiplication and the subgroup check of decode -- the latter on points whose off-subgroup part has
small order (tests/pairing_cases.corpus), through the harness, the public base loader and the batch verifier.

Each test is a CONTRACT (holds for any correct implementation) or a PIN (holds for the current formulas only, and says
so: an optimisation that changes the formula replaces it on purpose).  test_host_pairing.py runs the same cases, reduced,
through the host build of the same harness."""
import random

import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api
from playsnark_b200._lib import PlaysnarkError
from tests import pairing_cases as PC
from tests import verify_batch_cases as V

pytestmark = pytest.mark.gpu

ROWS = 1 << 12
ROWS_INV = 1 << 10


@pytest.fixture(scope="module")
def h():
    hh = PC.Harness(device=True)
    yield hh
    hh.close()


@pytest.mark.parametrize("name", sorted(PC.TOWER_OPS))
def test_tower(h, name):
    """CONTRACT: Fp6 / Fp12 operations against the oracle on 2^12 rows (2^10 for the inversions)"""
    PC.tower_op(h, name, ROWS_INV if name.endswith("inv") else ROWS)


def test_frobenius(h):
    """CONTRACT: frob^k = x^(p^k), k = 1..12"""
    PC.frobenius(h, ROWS, 4)


def test_pow_x_cyclotomic(h):
    """CONTRACT"""
    PC.pow_x_cyclotomic(h, 64)


def test_pow_x_pin(h):
    """PIN: conj(a^|x|) on arbitrary elements"""
    PC.pow_x_any(h, 256)


def test_miller_loop_pin(h):
    """PIN: raw Miller values equal the oracle's"""
    PC.miller_values(h)


def test_final_exponentiation(h):
    """CONTRACT"""
    PC.final_exp_values(h, 24)


def test_final_exponentiation_algebra(h):
    """CONTRACT"""
    PC.final_exp_algebra(h, 8)


def test_pairing_values(h):
    """CONTRACT"""
    PC.pairing_values(h, 6)


def test_check_products(h):
    """CONTRACT"""
    PC.check_products(h)


def test_square_roots(h):
    """CONTRACT"""
    PC.square_roots(h, ROWS_INV)


def test_scalar_mul(h):
    """CONTRACT"""
    PC.scalar_mul(h)


def test_subgroup_corpus(h):
    """CONTRACT"""
    PC.subgroup_corpus(h)


# ---- the public paths -----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def be():
    b = api.Backend(0)
    yield b
    b.close()


def test_bases_load_corpus(be):
    """CONTRACT: ps_bases_load rejects every corpus point with PS_ERR_ENCODING while subgroup_check is on; with it off the
    point loads and exports as it came in (compressed and uncompressed)"""
    try:
        for group, label, pt, _ in PC.corpus():
            for fmt in (PC.FMT_COMPRESSED, PC.FMT_AFFINE):
                enc = PC.encode(group, pt, fmt)
                be.set_option("subgroup_check", 1)
                with pytest.raises(PlaysnarkError) as e:
                    be.load_bases(group, [enc], fmt=fmt)
                assert e.value.status == L.PS_ERR_ENCODING, label
                be.set_option("subgroup_check", 0)
                b = be.load_bases(group, [enc], fmt=fmt)
                assert b.export(fmt=fmt) == [enc], (label, fmt)
                b.close()
    finally:
        be.set_option("subgroup_check", 1)


@pytest.fixture(scope="module")
def pool(be):
    p = V.Pool(be, n=8, count=8)
    yield p
    p.close()


def _forge(p, which: str, T, group: int):
    if which == "A":
        return api.Groth16Proof(p.tp, O.g1_compress(O.g1_add(O.g1_decompress(p.A), T)), p.B, p.C)
    if which == "C":
        return api.Groth16Proof(p.tp, p.A, p.B, O.g1_compress(O.g1_add(O.g1_decompress(p.C), T)))
    return api.Groth16Proof(p.tp, p.A, O.g2_compress(O.g2_add(O.g2_decompress(p.B), T)), p.C)


@pytest.mark.parametrize("which,l", [("C", 3), ("A", 3), ("C", 11), ("A", 11), ("B", 13)])
def test_batch_small_order_forgery(pool, which, l):
    """CONTRACT: proof i of an honest batch of 8 with C_i, A_i or B_i moved by a point T of small order l, at the first,
    middle and last position.  The weights are multiples of l, so rho_i T = O: for A and C the combined equation still
    holds, and only the decode-time subgroup check of proof points rejects the forgery.  Expected,
    with the context's subgroup_check on and off (it governs key points only): the batch fails, per_proof flags exactly
    proof i, and the batch without it verifies.  Groth16Verify decodes its proof points under subgroup_check, so with
    the check on it reports the forged point as PS_ERR_ENCODING."""
    group = 2 if which == "B" else 1
    T = PC.small_torsion(group, l)
    rng = random.Random(l * 7 + ord(which))
    N = 8
    proofs, ios = pool.batch(N)
    w = [l * rng.randrange(1, (1 << 128) // l) for _ in range(N)]
    try:
        for pos in (0, N // 2, N - 1):
            forged = list(proofs)
            forged[pos] = _forge(proofs[pos], which, T, group)
            if which != "B":     # the weighted point the verifier sums is the honest one, so the combined equation holds
                X = O.g1_decompress(getattr(proofs[pos], which))
                assert PC.mul_unreduced(O.F1, w[pos], O.g1_add(X, T)) == PC.mul_unreduced(O.F1, w[pos], X)
            rest_p = [p for i, p in enumerate(forged) if i != pos]
            rest_io = [v for i, v in enumerate(ios) if i != pos]
            for sub in (1, 0):
                pool.be.set_option("subgroup_check", sub)
                assert pool.verify(forged, ios, weights=w) is False, (pos, sub)
                assert pool.verify(forged, ios, weights=w, per_proof=True) == [i != pos for i in range(N)], (pos, sub)
                assert pool.verify(rest_p, rest_io, weights=w[:pos] + w[pos + 1:]) is True
            pool.be.set_option("subgroup_check", 1)
            with pytest.raises(PlaysnarkError) as e:
                api.Groth16Verify(pool.tr, pool.q, forged[pos], ios[pos], backend=pool.be)
            assert e.value.status == L.PS_ERR_ENCODING
    finally:
        pool.be.set_option("subgroup_check", 1)
