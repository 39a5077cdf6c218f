"""Operands, references, the small-order point corpus and a loader for the pairing / codec harness (tests/device_pairing.cu),
shared by the GPU suite (test_gpu_pairing.py) and its CPU leg (test_host_pairing.py, the same harness compiled for the host).

Values cross the harness as raw Montgomery limbs: an Fp element v is the 12-limb integer v * 2^384 mod p; an Fp12 element
is 12 such elements in the oracle's tuple order (c0.c0.c0, c0.c0.c1, c0.c1.c0, ..., c1.c2.c1)."""
from __future__ import annotations

import ctypes as C
import functools
import os
import random
import re
import shutil
import tempfile

import numpy as np

from oracle import ps_oracle as O
from playsnark_b200 import build as B

P, R, X_ABS = O.P, O.R, O.BLS_X
RP = 1 << 384
RP_INV = pow(RP, -1, P)
F1, F2 = O.F1, O.F2

# operation codes of device_pairing.cu
FP6_MUL, FP6_INV, FP6_MUL_V, FP12_MUL, FP12_SQR, FP12_INV, FP12_CONJ, FP12_FROB, FP12_POW_X, FINAL_EXP = range(10)
FMT_COMPRESSED, FMT_AFFINE = 0, 1
ST_OK, ST_ENCODING, ST_SUBGROUP = 0, 2, 4


# ---- references -----------------------------------------------------------------------------------------------------
def fp12_pow_x(a):
    """a^x for the (negative) curve parameter x, as a field power: the inverse of a^|x|"""
    return O.fp12_inv(O.fp12_pow(a, X_ABS))


def gamma(k: int):
    """xi^(k (p - 1) / 6), xi = 1 + u: the Frobenius coefficient of w^k"""
    return O.fp2_pow((1, 1), k * (P - 1) // 6)


GAMMA = [gamma(k) for k in range(6)]


def frob(a):
    """a^p through the closed form: (c w^k)^p = conj(c) gamma_k w^k.  Checked against fp12_pow(a, p) by the CPU leg."""
    (a0, a2, a4), (a1, a3, a5) = a
    c = [F2.mul((x[0], (-x[1]) % P), GAMMA[k]) for k, x in enumerate((a0, a1, a2, a3, a4, a5))]
    return ((c[0], c[2], c[4]), (c[1], c[3], c[5]))


def frob_k(a, k: int):
    for _ in range(k):
        a = frob(a)
    return a


def fe_ref(f):
    """what final_exponentiation computes: f^(3 (p^12 - 1) / r), the cube of the oracle's final exponentiation"""
    e = O.final_exp(f)
    return O.fp12_mul(O.fp12_sqr(e), e)


def cyclotomic(f):
    """f^((p^6 - 1)(p^2 + 1)): an element of the cyclotomic subgroup (inverse = conjugate)"""
    f1 = O.fp12_mul(O.fp12_conj(f), O.fp12_inv(f))
    return O.fp12_mul(frob_k(f1, 2), f1)


def mul_unreduced(F, k: int, a):
    """k a by double-and-add over the bits of k as given (no reduction mod r): the loop of O.in_subgroup"""
    acc = (F.one, F.one, F.zero)
    if a is None or k == 0:
        return None
    base = O.to_jac(F, a)
    for bit in bin(k)[2:]:
        acc = O.jac_dbl(F, acc)
        if bit == "1":
            acc = O.jac_add(F, acc, base)
    return O.to_affine(F, acc)


# ---- limbs ----------------------------------------------------------------------------------------------------------
def fp_coeffs(a, kind: str):
    """the Fp coefficients of an oracle value in memory order; kind: fp, fp2, fp6, fp12"""
    if kind == "fp":
        return [a]
    if kind == "fp2":
        return [a[0], a[1]]
    if kind == "fp6":
        return [c for x in a for c in x]
    return [c for y in a for x in y for c in x]


def from_coeffs(c, kind: str):
    if kind == "fp":
        return c[0]
    if kind == "fp2":
        return (c[0], c[1])
    if kind == "fp6":
        return tuple((c[2 * j], c[2 * j + 1]) for j in range(3))
    return tuple(tuple((c[6 * i + 2 * j], c[6 * i + 2 * j + 1]) for j in range(3)) for i in range(2))


NCOEF = {"fp": 1, "fp2": 2, "fp6": 6, "fp12": 12}


def raw_to_array(raws) -> np.ndarray:
    """raw 384-bit limb integers -> uint32 array, 12 limbs each"""
    return np.frombuffer(b"".join(int(v).to_bytes(48, "little") for v in raws), dtype="<u4").copy()


def array_to_raw(arr: np.ndarray):
    b = arr.astype("<u4").tobytes()
    return [int.from_bytes(b[i:i + 48], "little") for i in range(0, len(b), 48)]


def to_array(vals, kind: str) -> np.ndarray:
    """oracle values (standard form) -> Montgomery limbs"""
    return raw_to_array([c * RP % P for v in vals for c in fp_coeffs(v, kind)])


def from_array(arr: np.ndarray, kind: str):
    """Montgomery limbs -> oracle values; a limb vector >= p is kept unreduced so that a comparison fails"""
    raw = array_to_raw(arr)
    n = NCOEF[kind]
    std = [v * RP_INV % P if v < P else v + (1 << 400) for v in raw]
    return [from_coeffs(std[i:i + n], kind) for i in range(0, len(std), n)]


def g1_array(pts) -> np.ndarray:
    """affine G1 points (None = infinity, stored (0, 0) as the device does)"""
    return to_array([c for p in pts for c in ((0, 0) if p is None else p)], "fp")


def g2_array(pts) -> np.ndarray:
    return to_array([c for p in pts for c in (((0, 0), (0, 0)) if p is None else p)], "fp2")


def points_from_array(arr: np.ndarray, group: int):
    kind = "fp" if group == 1 else "fp2"
    c = from_array(arr, kind)
    zero = 0 if group == 1 else (0, 0)
    return [None if c[i] == zero and c[i + 1] == zero else (c[i], c[i + 1]) for i in range(0, len(c), 2)]


def hexrow(v, kind: str) -> str:
    return " ".join("%096x" % c for c in fp_coeffs(v, kind))


# ---- operand families -----------------------------------------------------------------------------------------------
def raw_fp_values(rng: random.Random, count: int):
    """raw Montgomery limbs of Fp elements: every limb p - 1's, limbs saturated below p, uniform"""
    SAT = [0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF]
    out = []
    for i in range(count):
        m = i % 3
        if m == 0:
            out.append(P - 1 - rng.randrange(3))
        elif m == 1:
            v = sum(rng.choice(SAT) << (32 * j) for j in range(12))
            out.append(v % P)
        else:
            out.append(rng.randrange(P))
    return out


def std_of_raw(v: int) -> int:
    return v * RP_INV % P


def rand_fp(rng):
    return rng.randrange(P)


def rand_fp2(rng):
    return (rng.randrange(P), rng.randrange(P))


def rand_fp6(rng):
    return tuple(rand_fp2(rng) for _ in range(3))


def rand_fp12(rng):
    return (rand_fp6(rng), rand_fp6(rng))


Z2 = (0, 0)


def fp12_families(rng: random.Random, rows: int, nonzero: bool = False):
    """Fp12 operands: 0, 1, -1; elements with zero components (pure Fp, pure Fp2, pure Fp6, the line shape
    (A, B, 0) + (0, y, 0) w with y in Fp and in Fp2); coefficients whose raw limbs are p - 1 or saturated; uniform"""
    one, m1 = O.FP12_ONE, ((((P - 1), 0), Z2, Z2), (Z2, Z2, Z2))
    fixed = ([] if nonzero else [((Z2, Z2, Z2), (Z2, Z2, Z2))]) + [one, m1]
    out = list(fixed)
    k = 0
    while len(out) < rows:
        m = k % 8
        k += 1
        if m == 0:
            out.append((((rng.randrange(1, P), 0), Z2, Z2), (Z2, Z2, Z2)))
        elif m == 1:
            out.append(((rand_fp2(rng), Z2, Z2), (Z2, Z2, Z2)))
        elif m == 2:
            out.append((rand_fp6(rng), (Z2, Z2, Z2)))
        elif m == 3:
            out.append(((rand_fp2(rng), rand_fp2(rng), Z2), (Z2, (rng.randrange(1, P), 0), Z2)))
        elif m == 4:
            out.append(((rand_fp2(rng), rand_fp2(rng), Z2), (Z2, rand_fp2(rng), Z2)))
        elif m in (5, 6):      # raw limbs p - 1 / saturated / uniform per coefficient
            out.append(from_coeffs([std_of_raw(v) for v in raw_fp_values(rng, 12)], "fp12"))
        else:
            out.append(rand_fp12(rng))
    return out[:rows]


def fp6_families(rng: random.Random, rows: int, nonzero: bool = False):
    one, m1 = O.FP6_ONE, (((P - 1), 0), Z2, Z2)
    out = ([] if nonzero else [(Z2, Z2, Z2)]) + [one, m1]
    k = 0
    while len(out) < rows:
        m = k % 6
        k += 1
        if m == 0:
            out.append((((rng.randrange(1, P), 0), Z2, Z2)))
        elif m == 1:
            out.append((rand_fp2(rng), Z2, Z2))
        elif m == 2:
            out.append((rand_fp2(rng), rand_fp2(rng), Z2))
        elif m == 3:
            out.append((Z2, rand_fp2(rng), Z2))
        elif m == 4:
            out.append(from_coeffs([std_of_raw(v) for v in raw_fp_values(rng, 6)], "fp6"))
        else:
            out.append(rand_fp6(rng))
    return out[:rows]


def scalar_edges(rng: random.Random):
    """k in {1, 2, 3, r - 1, (r - 1) / 2, |x|, |x| +- 1, random}"""
    return [1, 2, 3, R - 1, (R - 1) // 2, X_ABS, X_ABS - 1, X_ABS + 1, rng.randrange(1, R)]


# ---- the small-order corpus ------------------------------------------------------------------------------------------
X = -X_ABS
H1 = (X - 1) ** 2 // 3                                                            # cofactor of G1 in E(Fp)
H2 = (X ** 8 - 4 * X ** 7 + 5 * X ** 6 - 4 * X ** 4 + 6 * X ** 3 - 4 * X ** 2 - 4 * X + 13) // 9   # of G2 in E'(Fp2)
H1_PRIMES = {3: 1, 11: 2, 10177: 2, 859267: 2, 52437899: 2}                       # prime -> exponent in H1
Q135 = H2 // (13 ** 2 * 23 ** 2 * 2713 * 11953 * 262069)                          # a 135-digit probable prime
H2_PRIMES = {13: 2, 23: 2, 2713: 1, 11953: 1, 262069: 1, Q135: 1}


def curve_points(F, start: int = 1):
    """the points (x, +-y) of the curve in order of x = start, start + 1, ... (G2: x = (x0, 1))"""
    x0 = start
    while True:
        x = x0 if F is F1 else (x0, 1)
        rhs = F.add(F.mul(F.sqr(x), x), F.b)
        y = O.fp_sqrt(rhs) if F is F1 else O.fp2_sqrt(rhs)
        if y is not None:
            yield (x, y)
        x0 += 1


def exact_order(F, pt, multiple: int, primes) -> int:
    """the order of pt, given a multiple of it and the primes dividing that multiple"""
    assert mul_unreduced(F, multiple, pt) is None
    n = multiple
    for l in primes:
        while n % l == 0 and mul_unreduced(F, n // l, pt) is None:
            n //= l
    return n


@functools.lru_cache(maxsize=None)
def corpus():
    """Deterministic points outside the prime-order subgroups, as a list of (group, label, point, order):
      - the l-primary part of a curve point for every prime l of the cofactor: [N / l^v] Q with N = h r and l^v the
        full power of l in N, retried over Q until it is not infinity.  No point of order l^2 exists for the primes
        with v = 2 (G1: 11, 10177, 859267, 52437899; G2: 13, 23): their l-parts are Z/l x Z/l, which
        test_host_pairing.test_corpus_l2_parts_are_not_cyclic checks, so every such component has order l;
      - [r] Q: a point with the whole cofactor part (order = the exponent of the cofactor group);
      - S + T for a subgroup point S and each T above except G2's 135-digit prime: order l r;
      - the G1 points (0, +-2) of order 3, whose compressed encodings are 0x80 / 0xA0 followed by zeros."""
    out = []
    for group, F, h, primes, start in ((1, F1, H1, H1_PRIMES, 1), (2, F2, H2, H2_PRIMES, 1)):
        N = h * R
        comps = {}
        for l, v in primes.items():
            for Q in curve_points(F, start):
                T = mul_unreduced(F, N // l ** v, Q)
                if T is not None:
                    break
            comps[l] = T
            out.append((group, "T%d" % l if l < 1 << 32 else "Tq135", T, l))
        Q = next(curve_points(F, start + 7))
        W = mul_unreduced(F, R, Q)
        out.append((group, "cofactor", W, exact_order(F, W, h, list(primes))))
        S = O.pt_mul(F, 0x5EED + group, O.G1_GEN if group == 1 else O.G2_GEN)
        for l, T in comps.items():
            if l < 1 << 32:
                out.append((group, "S+T%d" % l, O.pt_add(F, S, T), l * R))
    out.append((1, "(0,2)", (0, 2), 3))
    out.append((1, "(0,-2)", (0, P - 2), 3))
    return out


def subgroup_points(group: int, rng: random.Random):
    """+-G, +-2G, (r - 1) G and two random multiples"""
    F, g = (F1, O.G1_GEN) if group == 1 else (F2, O.G2_GEN)
    ks = [1, R - 1, 2, R - 2, rng.randrange(2, R), rng.randrange(2, R)]
    return [O.pt_mul(F, k, g) for k in ks]


def encode(group: int, pt, fmt: int) -> bytes:
    """zcash encoding; the (0, +-2) points go through the same code as any other"""
    if group == 1:
        return O.g1_compress(pt) if fmt == FMT_COMPRESSED else O.g1_affine_bytes(pt)
    return O.g2_compress(pt) if fmt == FMT_COMPRESSED else O.g2_affine_bytes(pt)


def small_torsion(group: int, l: int):
    return next(p for g, lab, p, o in corpus() if g == group and lab == "T%d" % l)


# ---- the harness ----------------------------------------------------------------------------------------------------
class Harness:
    """tests/device_pairing.cu loaded from the CUDA build (device=True: operands staged through torch on cuda:0) or the
    host build (operands passed as host arrays).  Every method takes and returns oracle values."""

    def __init__(self, device: bool):
        self.device = device
        out, self._tmp = B.TEST_BUILD, None
        so = B.harness_path(out, B.PAIRING_HARNESS, host=not device)
        # build() leaves the CUDA build in tests/_build; on a tree that cannot be written, a stale or missing harness is
        # compiled into a temporary directory instead
        if B.stale(so, B._deps(B.PAIRING_HARNESS)) and not B.can_write(out):
            out = self._tmp = tempfile.mkdtemp(prefix="device_pairing_")
        self.lib = C.CDLL(B.build_device_harness(out, source=B.PAIRING_HARNESS, host=not device))
        vp, i = C.c_void_p, C.c_int
        L = self.lib
        L.dp_is_device.argtypes = []
        L.dp_tower.argtypes = [i, i, vp, vp, vp, i]
        L.dp_miller.argtypes = [vp, vp, vp, i]
        L.dp_check.argtypes = [vp, vp, vp, vp, i]
        L.dp_sqrt.argtypes = [i, vp, vp, vp, i]
        L.dp_in_subgroup.argtypes = [i, vp, vp, i]
        L.dp_scalar_mul.argtypes = [i, i, vp, vp, vp, i]
        L.dp_decode.argtypes = [i, i, i, vp, vp, vp, vp, vp, i]
        assert L.dp_is_device() == (1 if device else 0)
        if device:
            import torch
            torch.zeros(1, device="cuda")      # the runtime is up before the first launch

    def close(self):
        if self._tmp:
            shutil.rmtree(self._tmp, ignore_errors=True)

    def _call(self, fn, args, outs):
        """args: ints or numpy arrays (inputs); outs: numpy arrays written by the call (returned, filled)"""
        if self.device:
            import torch
            keep, ptrs = [], []
            for a in list(args) + list(outs):
                if isinstance(a, np.ndarray):
                    t = torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).cuda() if a.size else torch.zeros(1, dtype=torch.uint8, device="cuda")
                    keep.append((a, t))
                    ptrs.append(t.data_ptr())
                else:
                    ptrs.append(a)
            rc = fn(*ptrs)
            assert rc == 0, "launch failed: CUDA error %d" % rc
            for a, t in keep[len(keep) - len(outs):]:
                if a.size:
                    a.view(np.uint8)[:] = t.cpu().numpy()[:a.nbytes]
        else:
            ptrs = [a.ctypes.data if isinstance(a, np.ndarray) else a for a in list(args) + list(outs)]
            rc = fn(*ptrs)
            assert rc == 0, "host harness returned %d" % rc
        return outs

    def tower(self, op: int, a, b=None, k: int = 0):
        kind = "fp6" if op <= FP6_MUL_V else "fp12"
        n = len(a)
        A = to_array(a, kind)
        Bv = to_array(b, kind) if b is not None else np.zeros(1, dtype="<u4")
        out = np.zeros(n * NCOEF[kind] * 12, dtype="<u4")
        f = lambda pa, pb, po: self.lib.dp_tower(op, k, pa, pb, po, n)
        self._call(f, [A, Bv], [out])
        return from_array(out, kind)

    def miller(self, Ps, Qs):
        n = len(Ps)
        out = np.zeros(n * 144, dtype="<u4")
        self._call(lambda p, q, o: self.lib.dp_miller(p, q, o, n), [g1_array(Ps), g2_array(Qs)], [out])
        return from_array(out, "fp12")

    def check(self, fs, counts):
        """PairingCheckK's verdicts and the final-exponentiated products, one check per count"""
        first = np.array([0] + list(np.cumsum(counts)), dtype="<u4")
        nc = len(counts)
        ok = np.zeros(nc, dtype=np.uint8)
        fe = np.zeros(nc * 144, dtype="<u4")
        fa = to_array(fs, "fp12") if fs else np.zeros(144, dtype="<u4")
        self._call(lambda f, fi, o, e: self.lib.dp_check(f, fi, o, e, nc), [fa, first], [ok, fe])
        return [bool(v) for v in ok], from_array(fe, "fp12")

    def sqrt(self, ext: int, vals):
        kind = "fp" if ext == 1 else "fp2"
        n = len(vals)
        out = np.zeros(n * 12 * ext, dtype="<u4")
        ok = np.zeros(n, dtype=np.uint8)
        self._call(lambda a, o, k: self.lib.dp_sqrt(ext, a, o, k, n), [to_array(vals, kind)], [out, ok])
        return from_array(out, kind), [bool(v) for v in ok]

    def in_subgroup(self, group: int, pts):
        n = len(pts)
        ok = np.zeros(n, dtype=np.uint8)
        arr = g1_array(pts) if group == 1 else g2_array(pts)
        self._call(lambda p, o: self.lib.dp_in_subgroup(group, p, o, n), [arr], [ok])
        return [bool(v) for v in ok]

    def scalar_mul(self, group: int, nlimbs: int, pts, ks):
        n = len(pts)
        arr = g1_array(pts) if group == 1 else g2_array(pts)
        karr = np.frombuffer(b"".join(int(k).to_bytes(32, "little") for k in ks), dtype="<u4").copy()
        out = np.zeros_like(arr)
        self._call(lambda p, k, o: self.lib.dp_scalar_mul(group, nlimbs, p, k, o, n), [arr, karr], [out])
        return points_from_array(out, group)

    def decode(self, group: int, fmt: int, subgroup: int, encs):
        """(points, status bytes, the points encoded again, the OR of the statuses)"""
        n = len(encs)
        per = {(1, 0): 48, (1, 1): 96, (2, 0): 96, (2, 1): 192}[(group, fmt)]
        assert all(len(e) == per for e in encs)
        inp = np.frombuffer(b"".join(encs), dtype=np.uint8).copy()
        pts = np.zeros(n * (24 if group == 1 else 48), dtype="<u4")
        st = np.zeros(n, dtype=np.uint8)
        again = np.zeros(n * per, dtype=np.uint8)
        err = np.zeros(1, dtype="<u4")
        self._call(lambda i, e, p, s, a: self.lib.dp_decode(group, fmt, subgroup, i, p, s, a, e, n), [inp, err], [pts, st, again])
        return (points_from_array(pts, group), [int(v) for v in st],
                [bytes(again[i * per:(i + 1) * per]) for i in range(n)])


def mismatches(got, want, labels=None, kind="fp12", operands=None, limit=3) -> str:
    """'' when equal; else the first differing rows with operands in hex"""
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    if len(got) != len(want):
        return "length %d != %d" % (len(got), len(want))
    if not bad:
        return ""
    lines = ["%d of %d rows differ" % (len(bad), len(got))]
    for i in bad[:limit]:
        lines.append("row %d%s" % (i, "" if labels is None else " (%s)" % labels[i]))
        for j, ops in enumerate(operands or []):
            lines.append("  operand %d: %s" % (j, hexrow(ops[i], kind)))
        lines.append("  got : %s" % (hexrow(got[i], kind) if not isinstance(got[i], (bool, int)) else got[i]))
        lines.append("  want: %s" % (hexrow(want[i], kind) if not isinstance(want[i], (bool, int)) else want[i]))
    return "\n".join(lines)


def header_constant(name: str) -> int:
    """an FpParams constant of constants.cuh as the integer its limbs spell"""
    path = os.path.join(B.CSRC, "constants.cuh")
    with open(path) as f:
        m = re.search(r"\b%s\(int i\) \{ constexpr uint32_t t\[12\] = \{([^}]*)\}" % name, f.read())
    limbs = [int(x.strip().rstrip("u"), 16) for x in m.group(1).split(",")]
    return sum(v << (32 * j) for j, v in enumerate(limbs))


# ---- cases (test_gpu_pairing.py at full size, test_host_pairing.py reduced) --------------------------------------------
# CONTRACT: holds for any correct implementation.  PIN: holds for the current formulas only; a change of formula may
# replace such a test on purpose.
TOWER_OPS = {"fp6_mul": (FP6_MUL, "fp6", 2), "fp6_inv": (FP6_INV, "fp6", 1), "fp6_mul_v": (FP6_MUL_V, "fp6", 1),
             "fp12_mul": (FP12_MUL, "fp12", 2), "fp12_sqr": (FP12_SQR, "fp12", 1), "fp12_inv": (FP12_INV, "fp12", 1),
             "fp12_conj": (FP12_CONJ, "fp12", 1)}
V6 = ((0, 0), (1, 0), (0, 0))          # v as an Fp6 element
FP6_ZERO, FP12_ZERO = O.FP6_ZERO, (O.FP6_ZERO, O.FP6_ZERO)
TOWER_REF = {"fp6_mul": O.fp6_mul, "fp6_inv": lambda a: a if a == FP6_ZERO else O.fp6_inv(a), "fp6_mul_v": lambda a: O.fp6_mul(a, V6),
             "fp12_mul": O.fp12_mul, "fp12_sqr": O.fp12_sqr, "fp12_inv": lambda a: a if a == FP12_ZERO else O.fp12_inv(a), "fp12_conj": O.fp12_conj}


def tower_op(h: Harness, name: str, rows: int, seed: int = 1):
    """CONTRACT: one tower operation against the oracle's (the product by v against a full product with v), on the
    operand families.  The inverse of zero is zero on both sides."""
    op, kind, arity = TOWER_OPS[name]
    fam = fp6_families if kind == "fp6" else fp12_families
    a = fam(random.Random(seed), rows)
    b = fam(random.Random(seed + 1000), rows)
    b = b[rows // 2:] + b[:rows // 2] if arity == 2 else None       # every family meets every other one
    got = h.tower(op, a, b)
    want = [TOWER_REF[name](x, y) for x, y in zip(a, b)] if arity == 2 else [TOWER_REF[name](x) for x in a]
    ops = [a, b] if arity == 2 else [a]
    msg = mismatches(got, want, kind=kind, operands=ops)
    assert not msg, "%s:\n%s" % (name, msg)


def frobenius(h: Harness, rows: int, pow_rows: int, seed: int = 2):
    """CONTRACT: fp12_frob applied k = 1..12 times is x -> x^(p^k): against the closed form on `rows` operands and against
    fp12_pow(a, p^k) itself on the first `pow_rows`; frob^6 is the conjugation and frob^12 the identity."""
    a = fp12_families(random.Random(seed), rows)
    want = list(a)
    pw = [a[i] for i in range(pow_rows)]
    for k in range(1, 13):
        got = h.tower(FP12_FROB, a, k=k)
        want = [frob(x) for x in want]
        pw = [O.fp12_pow(x, P) for x in pw]
        assert want[:pow_rows] == pw, "closed-form reference disagrees with a^(p^%d)" % k
        msg = mismatches(got, want, operands=[a])
        assert not msg, "frob^%d:\n%s" % (k, msg)
        if k == 6:
            assert got == [O.fp12_conj(x) for x in a]
        if k == 12:
            assert got == a


def pow_x_cyclotomic(h: Harness, rows: int, seed: int = 3):
    """CONTRACT: on the cyclotomic subgroup fp12_pow_x(g) = g^x, x = -|x| the curve parameter, as a field power"""
    g = [cyclotomic(f) for f in fp12_families(random.Random(seed), rows + 3)[3:]]     # f = 0, 1, -1 left out
    got = h.tower(FP12_POW_X, g)
    msg = mismatches(got, [fp12_pow_x(x) for x in g], operands=[g])
    assert not msg, msg


def pow_x_any(h: Harness, rows: int, seed: int = 4):
    """PIN: on arbitrary elements fp12_pow_x(a) = conj(a^|x|) (the conjugate is the inverse only on the cyclotomic
    subgroup; any other way of computing g^x there may differ here)"""
    a = fp12_families(random.Random(seed), rows)
    got = h.tower(FP12_POW_X, a)
    msg = mismatches(got, [O.fp12_conj(O.fp12_pow(x, X_ABS)) for x in a], operands=[a])
    assert not msg, msg


def miller_inputs(rng: random.Random):
    """(label, P, Q): generators, k G for the edge scalars on either side, -P and -Q, infinity on either side"""
    g1, g2 = O.G1_GEN, O.G2_GEN
    out = [("G1, G2", g1, g2)]
    for k in scalar_edges(rng):
        out.append(("%#x G1, G2" % k, O.g1_mul(k), g2))
        out.append(("G1, %#x G2" % k, g1, O.g2_mul(k)))
    a, b = O.g1_mul(rng.randrange(1, R)), O.g2_mul(rng.randrange(1, R))
    out += [("P, Q", a, b), ("-P, Q", O.pt_neg(F1, a), b), ("P, -Q", a, O.pt_neg(F2, b)),
            ("inf, Q", None, b), ("P, inf", a, None), ("inf, inf", None, None)]
    return out


def miller_values(h: Harness, seed: int = 5, limit: int = 0):
    """PIN: the raw Miller values equal the oracle's miller_loop (same line scaling and conjugation); infinity on either
    side gives one"""
    cases = miller_inputs(random.Random(seed))
    if limit:
        cases = cases[:limit] + cases[-3:]
    labels, Ps, Qs = zip(*cases)
    got = h.miller(list(Ps), list(Qs))
    want = [O.miller_loop(p, q) for p, q in zip(Ps, Qs)]
    msg = mismatches(got, want, labels=labels)
    assert not msg, msg
    for lab, v in zip(labels, got):
        if "inf" in lab:
            assert v == O.FP12_ONE, lab


def final_exp_values(h: Harness, rows: int, seed: int = 6):
    """CONTRACT: final_exponentiation(f) = f^(3 (p^12 - 1) / r) = final_exp(f)^3 on random values and the structured
    families (zero left out), and every Fp6 element maps to one"""
    rng = random.Random(seed)
    f = fp12_families(rng, rows, nonzero=True)
    got = h.tower(FINAL_EXP, f)
    msg = mismatches(got, [fe_ref(x) for x in f], operands=[f])
    assert not msg, msg
    sub = [(rand_fp6(rng), (Z2, Z2, Z2)), ((((5, 0), Z2, Z2)), (Z2, Z2, Z2)), (((P - 1, 0), Z2, Z2), (Z2, Z2, Z2))]
    assert h.tower(FINAL_EXP, sub) == [O.FP12_ONE] * len(sub)


def final_exp_algebra(h: Harness, rows: int, seed: int = 7):
    """CONTRACT: FE(a b) = FE(a) FE(b); FE(conj a) = conj(FE(a)) = FE(a)^-1 (the batch bisection's right child is
    parent * conj(left)); FE(a)^r = 1"""
    rng = random.Random(seed)
    a = [rand_fp12(rng) for _ in range(rows)]
    b = fp12_families(rng, rows, nonzero=True)
    ab = [O.fp12_mul(x, y) for x, y in zip(a, b)]
    fa, fb, fab, fca = (h.tower(FINAL_EXP, v) for v in (a, b, ab, [O.fp12_conj(x) for x in a]))
    for i in range(rows):
        assert fab[i] == O.fp12_mul(fa[i], fb[i]), "FE(a b) != FE(a) FE(b) at row %d" % i
        assert fca[i] == O.fp12_conj(fa[i]), "FE(conj a) != conj FE(a) at row %d" % i
        assert O.fp12_mul(fca[i], fa[i]) == O.FP12_ONE
        assert O.fp12_pow(fa[i], R) == O.FP12_ONE, "FE(a)^r != 1 at row %d" % i


def pairing_values(h: Harness, n_oracle: int, seed: int = 8):
    """CONTRACT: FE(miller(P, Q)) = e(P, Q)^3 for the oracle's pairing e; bilinearity e(aP, bQ) = e(P, Q)^(ab) for a, b
    from the edge scalars; e(G1, G2) != 1"""
    rng = random.Random(seed)
    pairs = [(O.G1_GEN, O.G2_GEN)] + [(O.g1_mul(rng.randrange(1, R)), O.g2_mul(rng.randrange(1, R)))
                                      for _ in range(n_oracle - 1)]
    fe = h.tower(FINAL_EXP, h.miller([p for p, _ in pairs], [q for _, q in pairs]))
    want = [O.fp12_mul(O.fp12_sqr(e), e) for e in (O.pairing(p, q) for p, q in pairs)]
    msg = mismatches(fe, want)
    assert not msg, msg
    base = fe[0]
    assert base != O.FP12_ONE and O.fp12_pow(base, R) == O.FP12_ONE
    ks = scalar_edges(rng)
    ab = [(ks[i], ks[(3 * i + 1) % len(ks)]) for i in range(len(ks))] + [(ks[i], ks[i]) for i in (3, 5)]
    got = h.tower(FINAL_EXP, h.miller([O.g1_mul(a) for a, _ in ab], [O.g2_mul(b) for _, b in ab]))
    for (a, b), v in zip(ab, got):
        assert v == O.fp12_pow(base, a * b % R), "e(%#x P, %#x Q) != e(P, Q)^ab" % (a, b)


def check_products(h: Harness, seed: int = 9):
    """CONTRACT: PairingCheckK over Miller values grouped by first[]: checks of 0, 1, 4 and 12 pairs return the oracle's
    product of pairings (cubed) and decide it against one; a check whose pairs cancel returns one and passes"""
    rng = random.Random(seed)
    counts = [0, 1, 4, 12, 2]
    Ps, Qs = [], []
    for c in counts[:-1]:
        for _ in range(c):
            Ps.append(O.g1_mul(rng.randrange(1, R)))
            Qs.append(O.g2_mul(rng.randrange(1, R)))
    a, q = O.g1_mul(rng.randrange(1, R)), O.g2_mul(rng.randrange(1, R))
    Ps += [a, O.pt_neg(F1, a)]
    Qs += [q, q]
    fs = h.miller(Ps, Qs)
    ok, fe = h.check(fs, counts)
    want, i = [], 0
    for c in counts:
        acc = O.FP12_ONE
        for j in range(i, i + c):
            acc = O.fp12_mul(acc, O.miller_loop(Ps[j], Qs[j]))
        want.append(fe_ref(acc))
        i += c
    msg = mismatches(fe, want, labels=["%d pairs" % c for c in counts])
    assert not msg, msg
    assert ok == [v == O.FP12_ONE for v in want] == [True, False, False, False, True]


def square_roots(h: Harness, rows: int, seed: int = 10):
    """CONTRACT: fp_sqrt / fp2_sqrt claim a root exactly for the squares (Euler's criterion on the element, on its norm in
    Fp2), and a claimed root squares back"""
    rng = random.Random(seed)
    for ext in (1, 2):
        if ext == 1:
            vals = [0, 1, P - 1, 4, P - 4] + [std_of_raw(v) for v in raw_fp_values(rng, rows // 2)]
            vals += [rng.randrange(P) ** 2 % P for _ in range(rows - len(vals))]
            is_sq = [pow(v, (P - 1) // 2, P) != P - 1 for v in vals]
            sq = lambda x: x * x % P
        else:
            vals = [(0, 0), (1, 0), (P - 1, 0), (0, 1), (0, P - 1), (4, 4)] + [rand_fp2(rng) for _ in range(rows // 2)]
            vals += [F2.sqr(rand_fp2(rng)) for _ in range(rows - len(vals))]
            is_sq = [pow((a * a + b * b) % P, (P - 1) // 2, P) != P - 1 for a, b in vals]
            sq = F2.sqr
        roots, ok = h.sqrt(ext, vals)
        for v, r, k, s in zip(vals, roots, ok, is_sq):
            assert k == s, "sqrt claim %s for %s (square: %s)" % (k, v, s)
            if k:
                assert sq(r) == v, "root of %s does not square back" % (v,)


def scalar_mul(h: Harness, seed: int = 11):
    """CONTRACT: xyzz_scalar_mul over 4 limbs (128-bit weights of the batch verifier) and 8 limbs (unreduced: r, r + 1 and
    2^256 - 1 included) against the oracle's double-and-add"""
    rng = random.Random(seed)
    for group, F, g in ((1, F1, O.G1_GEN), (2, F2, O.G2_GEN)):
        base = O.pt_mul(F, rng.randrange(2, R), g)
        for nl in (4, 8):
            top = 1 << (32 * nl)
            ks = [0, 1, 2, 3, top - 1, top >> 1, rng.randrange(top), rng.randrange(top)]
            if nl == 8:
                ks += [R, R + 1, R - 1, 2 * R + 5]
            pts = [base] * len(ks) + [None, g]
            ks += [5, 0]
            got = h.scalar_mul(group, nl, pts, ks)
            want = [mul_unreduced(F, k, p) for p, k in zip(pts, ks)]
            assert got == want, (group, nl, [i for i, (a, b) in enumerate(zip(got, want)) if a != b])


def subgroup_corpus(h: Harness, seed: int = 12):
    """CONTRACT: every corpus point is rejected by in_subgroup and by the decode kernels with subgroup checking (status 4,
    compressed and uncompressed) and passes them without (status 0, the point re-encodes byte for byte); subgroup points
    (+-G, +-2G, (r - 1) G, random) are accepted and decode to themselves"""
    rng = random.Random(seed)
    for group in (1, 2):
        bad = [(lab, p) for g, lab, p, _ in corpus() if g == group]
        good = subgroup_points(group, rng)
        labels = [lab for lab, _ in bad]
        pts = [p for _, p in bad]
        got = h.in_subgroup(group, pts + good)
        want = [O.in_subgroup(F1 if group == 1 else F2, p) for p in pts + good]
        assert want == [False] * len(pts) + [True] * len(good)
        assert got == want, [(l, v) for l, v in zip(labels + ["good"] * len(good), got)]
        for fmt in (FMT_COMPRESSED, FMT_AFFINE):
            encs = [encode(group, p, fmt) for p in pts + good]
            dec, st, again = h.decode(group, fmt, 1, encs)
            assert st == [ST_SUBGROUP] * len(pts) + [ST_OK] * len(good), list(zip(labels, st))
            assert dec == [None] * len(pts) + good
            assert again[len(pts):] == encs[len(pts):]
            dec, st, again = h.decode(group, fmt, 0, encs)
            assert st == [ST_OK] * len(encs), list(zip(labels, st))
            assert dec == pts + good
            assert again == encs, [l for l, a, e in zip(labels, again, encs) if a != e]
