"""CPU leg of test_gpu_pairing.py: the references and the small-order corpus themselves, and the same cases at reduced
size through the host build of tests/device_pairing.cu (g++ -DPS_HOST_EMU, carry flag emulated), so that the pairing and
codec functions can be checked and debugged on a machine without a GPU."""
import random

import pytest

from oracle import ps_oracle as O
from tests import pairing_cases as PC

P, R = O.P, O.R


# ---- references -----------------------------------------------------------------------------------------------------
def test_hard_part_decomposition():
    """3 (p^4 - p^2 + 1) / r = (x - 1)^2 (x + p) (x^2 + p^2 - 1) + 3 for x = -|x|: the chain final_exponentiation runs"""
    x = -O.BLS_X
    assert (P ** 4 - P ** 2 + 1) % R == 0
    assert 3 * (P ** 4 - P ** 2 + 1) // R == (x - 1) ** 2 * (x + P) * (x ** 2 + P ** 2 - 1) + 3


def test_frobenius_constants():
    """FROBk_C0 / FROBk_C1 of constants.cuh are xi^(k (p - 1) / 6) in Montgomery form, computed here from scratch"""
    for k in range(1, 6):
        g = PC.gamma(k)
        assert PC.header_constant("FROB%d_C0" % k) == g[0] * PC.RP % P, k
        assert PC.header_constant("FROB%d_C1" % k) == g[1] * PC.RP % P, k


def test_frobenius_reference():
    """the closed-form Frobenius of pairing_cases equals a^p, and pow_x's reference is a field power"""
    rng = random.Random(1)
    for a in PC.fp12_families(rng, 12)[:3] + [PC.rand_fp12(rng) for _ in range(3)]:
        assert PC.frob(a) == O.fp12_pow(a, P)
    g = PC.cyclotomic(PC.rand_fp12(rng))
    assert O.fp12_mul(g, O.fp12_conj(g)) == O.FP12_ONE
    assert PC.fp12_pow_x(g) == O.fp12_conj(O.fp12_pow(g, O.BLS_X))


def test_cofactors():
    """the factorisations the corpus is built on (h1 = (x - 1)^2 / 3; h2 from its polynomial in x)"""
    assert PC.H1 == 3 * 11 ** 2 * 10177 ** 2 * 859267 ** 2 * 52437899 ** 2
    assert PC.H2 == 13 ** 2 * 23 ** 2 * 2713 * 11953 * 262069 * PC.Q135
    assert len(str(PC.Q135)) == 135 and pow(3, PC.Q135 - 1, PC.Q135) == 1
    for h, primes in ((PC.H1, PC.H1_PRIMES), (PC.H2, PC.H2_PRIMES)):
        n = h
        for l, v in primes.items():
            assert n % l ** v == 0 and (n // l ** v) % l != 0
            n //= l ** v
        assert n == 1


def test_corpus_orders():
    """every corpus point lies on its curve, outside the prime-order subgroup, and has exactly the recorded order"""
    labels = set()
    for group, label, pt, order in PC.corpus():
        F = O.F1 if group == 1 else O.F2
        h = PC.H1 if group == 1 else PC.H2
        primes = list((PC.H1_PRIMES if group == 1 else PC.H2_PRIMES)) + [R]
        assert pt is not None and O.on_curve(F, pt), label
        assert not O.in_subgroup(F, pt), label
        assert PC.exact_order(F, pt, h * R, primes) == order, label
        labels.add((group, label))
    for l in PC.H1_PRIMES:
        assert (1, "T%d" % l) in labels and ((1, "S+T%d" % l) in labels)
    for l in PC.H2_PRIMES:
        assert (2, "T%d" % l if l < 1 << 32 else "Tq135") in labels
    assert PC.encode(1, (0, 2), PC.FMT_COMPRESSED) == b"\x80" + bytes(47)
    assert PC.encode(1, (0, P - 2), PC.FMT_COMPRESSED) == b"\xa0" + bytes(47)


@pytest.mark.parametrize("group,l", [(1, 11), (1, 10177), (2, 13), (2, 23)])
def test_corpus_l2_parts_are_not_cyclic(group, l):
    """for the primes with l^2 | h, [h r / l] Q = O for several curve points Q: the l-part is Z/l x Z/l and has no point
    of order l^2, which is why the corpus holds none"""
    F = O.F1 if group == 1 else O.F2
    N = (PC.H1 if group == 1 else PC.H2) * R
    pts = PC.curve_points(F)
    for _ in range(4):
        assert PC.mul_unreduced(F, N // l, next(pts)) is None


# ---- the cases, through the host build ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def h():
    hh = PC.Harness(device=False)
    yield hh
    hh.close()


@pytest.mark.parametrize("name", sorted(PC.TOWER_OPS))
def test_tower(h, name): PC.tower_op(h, name, 96)
def test_frobenius(h): PC.frobenius(h, 24, 1)
def test_pow_x_cyclotomic(h): PC.pow_x_cyclotomic(h, 4)
def test_pow_x_pin(h): PC.pow_x_any(h, 8)
def test_miller_loop_pin(h): PC.miller_values(h, limit=6)
def test_final_exponentiation(h): PC.final_exp_values(h, 10)
def test_final_exponentiation_algebra(h): PC.final_exp_algebra(h, 2)
def test_pairing_values(h): PC.pairing_values(h, 1)
def test_check_products(h): PC.check_products(h)
def test_square_roots(h): PC.square_roots(h, 96)
def test_scalar_mul(h): PC.scalar_mul(h)
def test_subgroup_corpus(h): PC.subgroup_corpus(h)
