"""Field and group arithmetic as compiled for sm_100a (tests/device_arith.cu) against Python integers and the oracle.

The host build (test_host_arith.py) runs the same templates with an emulated carry flag and the serial formulas in
place of the team group law; this suite runs the PTX carry chains, the inlined Fp2 tower of the G2 hot loop and the
four-lane team formulas of team.cuh.  Operands are edge values, values whose limbs saturate the carry chains, and
uniform values.  A mismatch is reported with its operands in hex and the tests/host_check.cpp function that replays
the same row through the host build: a row that fails here and passes there points at code generation, one that fails
in both at the algorithm.

The generators and references are plain Python: the tests without the gpu mark check them against the host build."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from oracle import ps_oracle as O
from playsnark_b200 import build as B

P, R = O.P, O.R
RP, RR = 1 << 384, 1 << 256                                 # Montgomery radices of Fp (12 limbs) and Fr (8 limbs)
FIELDS = {"fp": (0, P, 12, RP), "fr": (1, R, 8, RR)}
# operation codes of device_arith.cu
FE_OPS = {"mul": 0, "add": 1, "sub": 2, "sqr": 3, "neg": 4, "from_mont": 5, "to_mont": 6, "inv": 7, "inv_serial": 8,
          "mul_wide": 10, "mul2_wide": 11, "redc_wide": 12, "mul2_lazy": 13, "sqrt": 14, "neg_lazy": 15}
F2_OPS = {"mul": 0, "sqr": 1, "inv": 2, "inv_serial": 3}
DIFF_OPS = {"mul2_lazy": 0, "redc_wide": 1, "fp2_inline": 2}
G_MADD, G_ADD, G_DBL, G_ADD_TEAM, G_DBL_TEAM = range(5)

# limb values that saturate carry chains (full limbs, borrows, half-limb boundaries): the set
# test_host_arith.test_unreduced_products draws from
SAT = [0, 1, 0xFFFFFFFF, 0xFFFFFFFE, 0x80000000, 0x7FFFFFFF, 2]

ROWS = 1 << 16
ROWS_INV = 1 << 12
DIFF_ROWS = 1 << 28


# ---- operands --------------------------------------------------------------------------------------------------------
def edge_values(m, nl):
    """0, 1, 2, m-1, m-2, (m+-1)/2, R mod m, R^-1 mod m, a high power of two, and values whose limbs are all 0xFFFFFFFF
    under m's top limb (with that limb 0 and one below m's)"""
    rad = 1 << (32 * nl)
    low = (1 << (32 * (nl - 1))) - 1
    top = m >> (32 * (nl - 1))
    vals = [0, 1, 2, m - 1, m - 2, (m - 1) // 2, (m + 1) // 2, rad % m, pow(rad, -1, m), 1 << (m.bit_length() - 1),
            low, ((top - 1) << (32 * (nl - 1))) | low, rad * rad % m]
    return sorted(set(vals))


def sat_values(nrng, count, nl, bound):
    """`count` integers whose 32-bit limbs are drawn from SAT, reduced below `bound`"""
    if count <= 0:
        return []
    limbs = np.array(SAT, dtype="<u4")[nrng.integers(0, len(SAT), size=(count, nl))]
    raw = limbs.tobytes()
    w = 4 * nl
    return [int.from_bytes(raw[i * w:(i + 1) * w], "little") % bound for i in range(count)]


def operand_columns(m, nl, rows, seed, bounds, extra_edges=()):
    """len(bounds) operand columns of `rows` values, column j below bounds[j]: every pair of edge values for the first
    two columns (the others cycle through edges), then saturated limbs for half the remaining rows, then uniform ones"""
    rng = random.Random(seed)
    nrng = np.random.default_rng(seed)
    k = len(bounds)
    cols = [[] for _ in range(k)]
    edges = [[e for e in edge_values(m, nl) + list(extra_edges) if e < b] for b in bounds]
    E0, E1 = edges[0], edges[1 % k]
    for i, x in enumerate(E0):
        for j, y in enumerate(E1):
            if len(cols[0]) >= rows // 4:
                break
            row = [x, y] + [edges[c][(i * 3 + j * 5 + c) % len(edges[c])] for c in range(2, k)]
            for c in range(k):
                cols[c].append(row[c])
    n_sat = (rows - len(cols[0])) // 2
    n_uni = rows - len(cols[0]) - n_sat
    for c in range(k):
        cols[c] += sat_values(nrng, n_sat, nl, bounds[c])
        cols[c] += [rng.randrange(bounds[c]) for _ in range(n_uni)]
    return cols


def to_dev(vals, nl):
    import torch
    w = 4 * nl
    buf = bytearray(b"".join(v.to_bytes(w, "little") for v in vals))
    return torch.frombuffer(buf, dtype=torch.int32).cuda()


def from_dev(t, nl):
    raw = t.cpu().numpy().tobytes()
    w = 4 * nl
    return [int.from_bytes(raw[i * w:(i + 1) * w], "little") for i in range(len(raw) // w)]


# ---- element-wise cases: (field, op, std) -> operand bounds, reference, host_check replay -----------------------------------
def _inv(x, m):
    return pow(x, -1, m) if x % m else 0


def fe_case(field, op, std):
    """(bounds, reference(row) -> int, out_limbs, extra edges, host_check replay name or None)"""
    _, m, nl, rad = FIELDS[field]
    ri = pow(rad, -1, m)
    full = 1 << (32 * nl)
    if op == "mul_wide":
        return [full, full], lambda a, b: a * b, 2 * nl, [full - 1, full >> 1, 2 * m - 2, m], "hc_fp_mul_wide_raw"
    if op == "mul2_wide":     # a b + c d < 2^(64N)
        return ([full >> 1, full, full >> 1, full], lambda a, b, c, d: a * b + c * d, 2 * nl, [full - 1, (full >> 1) - 1, m],
                "hc_fp_mul2_wide_raw")
    if op == "redc_wide":     # T = hi R + lo < p R, given as (hi, lo)
        return [m, full], lambda hi, lo: ((hi << (32 * nl)) | lo) * ri % m, nl, [full - 1], "hc_fp_redc_wide_raw"
    if op == "mul2_lazy":
        return [m] * 4, lambda a, b, c, d: (a * b - c * d) * ri % m, nl, [], "hc_fp_mul2_lazy_raw"
    if op == "neg_lazy":      # p - a as a plain integer, 0 -> p
        return [m + 1], lambda a: m - a, nl, [m], None
    if op == "sqrt":
        return [m], lambda a: pow(a, (m + 1) // 4, m), nl, [], "hc_fp_sqrt"
    if op in ("inv", "inv_serial"):
        return [m], lambda a: _inv(a, m), nl, [], "hc_%s_%s" % (field, op)
    k = 1 if op in ("sqr", "neg", "from_mont", "to_mont") else 2
    if std:
        ref = {"mul": lambda a, b: a * b % m, "add": lambda a, b: (a + b) % m, "sub": lambda a, b: (a - b) % m,
               "sqr": lambda a: a * a % m, "neg": lambda a: -a % m}[op]
        replay = {"mul": "hc_%s_mul", "add": "hc_%s_add", "sub": "hc_%s_sub", "sqr": "hc_%s_sqr"}.get(op)
    else:
        ref = {"mul": lambda a, b: a * b * ri % m, "add": lambda a, b: (a + b) % m, "sub": lambda a, b: (a - b) % m,
               "sqr": lambda a: a * a * ri % m, "neg": lambda a: -a % m, "from_mont": lambda a: a * ri % m,
               "to_mont": lambda a: a * rad % m}[op]
        replay = {"mul": "hc_%s_montmul_raw", "sqr": "hc_%s_montsqr_raw"}.get(op)
    return [m] * k, ref, nl, [], (replay % field) if replay else None


FE_CASES = ([(f, op, std) for f in ("fp", "fr") for op in ("mul", "add", "sub", "sqr", "neg") for std in (0, 1)] +
            [(f, op, 0) for f in ("fp", "fr") for op in ("from_mont", "to_mont")] +
            [(f, op, 1) for f in ("fp", "fr") for op in ("inv", "inv_serial")] +
            [("fp", op, 0) for op in ("mul_wide", "mul2_wide", "redc_wide", "mul2_lazy", "neg_lazy")] + [("fp", "sqrt", 1)])


def fe_rows(field, op, std):
    return ROWS_INV if op in ("inv", "inv_serial", "sqrt") else ROWS


def fe_operands(field, op, std, rows):
    _, m, nl, _ = FIELDS[field]
    bounds, _, _, extra, _ = fe_case(field, op, std)
    seed = sum(map(ord, field + op)) * 2 + std
    return operand_columns(m, nl, rows, seed, bounds, extra)


def report(name, bad, replay=None):
    lines = ["%s: %d mismatching rows" % (name, len(bad))]
    for ops, got, want in bad[:6]:
        lines.append("  operands " + ", ".join(hex(x) for x in ops) + ": got %s want %s" % (hex(got) if isinstance(got, int) else got,
                                                                                         hex(want) if isinstance(want, int) else want))
    if replay:
        lines.append("  replay on the host build: host_check.%s" % replay)
    return "\n".join(lines)


def check_rows(cols, got, ref):
    bad = []
    for i, g in enumerate(got):
        ops = [c[i] for c in cols]
        w = ref(*ops)
        if g != w:
            bad.append((ops, g, w))
    return bad


# ---- Fp2 ------------------------------------------------------------------------------------------------------------
def fp2_operands(op, rows, seed):
    """Fp2 values (c0, c1); edge pairs, saturated limbs, uniform"""
    cols = operand_columns(P, 12, rows, seed, [P] * 4)
    a = list(zip(cols[0], cols[2]))
    b = list(zip(cols[1], cols[3]))
    return a, b


def fp2_ref(op):
    F = O.F2
    return {"mul": F.mul, "sqr": lambda a, b: F.sqr(a), "inv": lambda a, b: F.inv(a) if a != (0, 0) else (0, 0),
            "inv_serial": lambda a, b: F.inv(a) if a != (0, 0) else (0, 0)}[op]


def f2_flat(vals):
    out = []
    for c0, c1 in vals:
        out += [c0, c1]
    return out


# ---- differential rows, regenerated on the host ------------------------------------------------------------------
_M64 = (1 << 64) - 1
DIFF_SAT = sorted(SAT)       # the order of c_SAT in device_arith.cu


def _mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def diff_operand(seed, row, j, m=P, nl=12):
    """operand j of a row of da_diff, as the kernel generates it"""
    top = m >> (32 * (nl - 1))
    mask = 0xFFFFFFFF
    while mask >= top:
        mask >>= 1
    v = 0
    for k in range(nl):
        limb = DIFF_SAT[_mix64(seed ^ _mix64((row * 64 + j * 16 + k) & _M64)) % 7]
        if k == nl - 1:
            limb &= mask
        v |= limb << (32 * k)
    return v


# ---- group law -----------------------------------------------------------------------------------------------------
def _grp(g):
    return (O.F1, O.G1_GEN, 12) if g == 1 else (O.F2, O.G2_GEN, 24)


def mont_elem(F, x):
    if F is O.F1:
        return [x * RP % P]
    return [x[0] * RP % P, x[1] * RP % P]


def xyzz_limbs(F, pt, lam):
    """pt as XYZZ (x l^2, y l^3, l^2, l^3) in Montgomery form; None -> all zero"""
    if pt is None:
        return [0] * (4 if F is O.F1 else 8)
    l2 = F.sqr(lam)
    l3 = F.mul(l2, lam)
    out = []
    for v in (F.mul(pt[0], l2), F.mul(pt[1], l3), l2, l3):
        out += mont_elem(F, v)
    return out


def affine_limbs(F, pt):
    if pt is None:
        return [0] * (2 if F is O.F1 else 4)
    return mont_elem(F, pt[0]) + mont_elem(F, pt[1])


def decode_xyzz(F, vals):
    """Montgomery XYZZ limbs -> affine point (None for ZZ = 0); asserts canonical coordinates and ZZ^3 = ZZZ^2"""
    assert all(v < P for v in vals), "non-canonical coordinate (>= p): " + ", ".join(hex(v) for v in vals)
    ri = pow(RP, -1, P)
    std = [v * ri % P for v in vals]
    if F is O.F1:
        X, Y, ZZ, ZZZ = std
        if ZZ == 0:
            return None
    else:
        X, Y, ZZ, ZZZ = [(std[2 * i], std[2 * i + 1]) for i in range(4)]
        if ZZ == (0, 0):
            return None
    assert F.mul(F.sqr(ZZ), ZZ) == F.sqr(ZZZ), "XYZZ invariant ZZ^3 = ZZZ^2 broken"
    return (F.mul(X, F.inv(ZZ)), F.mul(Y, F.inv(ZZZ)))


def rand_elem(F, rng):
    if F is O.F1:
        return rng.randrange(1, P)
    return (rng.randrange(P), rng.randrange(1, P))


def group_cases(group, npts, seed):
    """(name, acc, q, lam_acc, lam_q, want) rows for addition / mixed addition, eight per base point, in an order where
    the eight teams of a warp take eight different branches"""
    F, gen, _ = _grp(group)
    rng = random.Random(seed)
    base = O.pt_mul(F, rng.randrange(1, R), gen)
    step = O.pt_mul(F, rng.randrange(1, R), gen)
    pts = []
    p = base
    for _ in range(npts + 1):
        pts.append(p)
        p = O.pt_add(F, p, step)
    rows = []
    unit = 1 if F is O.F1 else (1, 0)
    for i in range(npts):
        Pt, Q = pts[i], pts[i + 1]
        l1, l2 = rand_elem(F, rng), rand_elem(F, rng)
        P2 = O.pt_add(F, Pt, Pt)
        neg = O.pt_neg(F, Pt)
        rows += [
            ("P+P scaled", Pt, Pt, l1, l2, P2),
            ("P+P same limbs", Pt, Pt, unit, unit, P2),
            ("P+(-P)", Pt, neg, l1, l2, None),
            ("O+P", None, Pt, l1, l2, Pt),
            ("P+O", Pt, None, l1, l2, Pt),
            ("O+O", None, None, l1, l2, None),
            ("P+2P", Pt, P2, l1, l2, O.pt_add(F, Pt, P2)),
            ("P+Q", Pt, Q, l1, l2, O.pt_add(F, Pt, Q)),
        ]
    return rows


def dbl_cases(group, npts, seed):
    F, gen, _ = _grp(group)
    rng = random.Random(seed)
    unit = 1 if F is O.F1 else (1, 0)
    rows = []
    for _ in range(npts):
        Pt = O.pt_mul(F, rng.randrange(1, R), gen)
        P2 = O.pt_add(F, Pt, Pt)
        rows += [("2P scaled", Pt, rand_elem(F, rng), P2), ("2O", None, rand_elem(F, rng), None),
                 ("2P same limbs", Pt, unit, P2), ("2(2P)", P2, rand_elem(F, rng), O.pt_add(F, P2, P2))]
    return rows


# ---- tests that need no device: the generators and references against the host build -------------------------
def test_generators_and_references_on_host(host_check):
    """every element-wise case with a host_check counterpart, a few hundred rows, through the host build; the
    operands stay below their bounds"""
    for field, op, std in FE_CASES:
        bounds, ref, onl, _, replay = fe_case(field, op, std)
        _, m, nl, _ = FIELDS[field]
        cols = fe_operands(field, op, std, 300)
        for c, b in zip(cols, bounds):
            assert len(c) == 300 and all(0 <= x < b for x in c), (field, op, std)
        if replay is None:
            continue
        fn = getattr(host_check, replay)
        out = (C.c_uint32 * onl)()
        for i in range(300):
            ops = [c[i] for c in cols]
            if op == "redc_wide":
                args = [(C.c_uint32 * (2 * nl))(*[(((ops[0] << 384) | ops[1]) >> (32 * k)) & 0xFFFFFFFF for k in range(2 * nl)])]
            else:
                args = [(C.c_uint32 * nl)(*[(x >> (32 * k)) & 0xFFFFFFFF for k in range(nl)]) for x in ops]
            fn(*args, out)
            got = sum(int(v) << (32 * k) for k, v in enumerate(out))
            assert got == ref(*ops), report("%s %s std=%d" % (field, op, std), [(ops, got, ref(*ops))], replay)


def test_fp2_references_on_host(host_check):
    a, b = fp2_operands("mul", 200, 7)
    out = (C.c_uint32 * 24)()
    enc = lambda v: (C.c_uint32 * 24)(*[((v[0] | (v[1] << 384)) >> (32 * k)) & 0xFFFFFFFF for k in range(24)])
    dec = lambda o: (sum(int(x) << (32 * k) for k, x in enumerate(o[:12])), sum(int(x) << (32 * k) for k, x in enumerate(o[12:])))
    for x, y in zip(a, b):
        host_check.hc_fp2_mul(enc(x), enc(y), out); assert dec(out) == fp2_ref("mul")(x, y)
        host_check.hc_fp2_sqr(enc(x), out); assert dec(out) == fp2_ref("sqr")(x, y)


def test_diff_generator_on_host(host_check):
    """the in-kernel operand generator's values are field elements with saturating limbs, and both routes of the
    differential kernels agree on them in the host build"""
    out, out2 = (C.c_uint32 * 12)(), (C.c_uint32 * 12)()
    ri = pow(RP, -1, P)
    lim = lambda x: (C.c_uint32 * 12)(*[(x >> (32 * k)) & 0xFFFFFFFF for k in range(12)])
    for row in range(200):
        a, b, c, d = [diff_operand(0x5EED, row, j) for j in range(4)]
        assert all(x < P for x in (a, b, c, d))
        assert all(((x >> (32 * k)) & 0xFFFFFFFF) in SAT for x in (a, b, c, d) for k in range(11))
        host_check.hc_fp_mul2_lazy_raw(lim(a), lim(b), lim(c), lim(d), out)
        assert sum(int(v) << (32 * k) for k, v in enumerate(out)) == (a * b - c * d) * ri % P
    # the Fr variant masks its top limb below Fr's
    assert all(diff_operand(3, r, 0, R, 8) < R for r in range(100))


def test_group_cases_on_host(host_check):
    """the scaled XYZZ encodings decode to the intended points; the expectations are the oracle's sums"""
    for group in (1, 2):
        F, _, _ = _grp(group)
        for name, a, q, la, lq, want in group_cases(group, 3, seed=group):
            assert decode_xyzz(F, xyzz_limbs(F, a, la)) == a, name
            assert O.pt_add(F, a, q) == want, name


# ---- device ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    import shutil
    import tempfile
    import torch
    # build() leaves the harness in tests/_build; on a tree that cannot be written, a stale or missing one is compiled
    # into a temporary directory instead
    out, tmp = B.TEST_BUILD, None
    if B.stale(os.path.join(out, "libdevice_arith.so"), B._deps(B.DEVICE_HARNESS)) and not B.can_write(out):
        out = tmp = tempfile.mkdtemp(prefix="device_arith_")
    so = B.build_device_harness(out)
    lib = C.CDLL(so)
    vp, i = C.c_void_p, C.c_int
    lib.da_fe.argtypes = [i, i, i, vp, vp, vp, vp, vp, i]
    lib.da_fp2.argtypes = [i, i, vp, vp, vp, i]
    lib.da_diff.argtypes = [i, C.c_ulonglong, C.c_ulonglong, vp, vp, i]
    lib.da_group.argtypes = [i, i, vp, vp, vp, i]
    torch.zeros(1, device="cuda")      # the runtime is up before the first launch
    yield lib
    if tmp:
        shutil.rmtree(tmp, ignore_errors=True)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


@pytest.mark.gpu
@pytest.mark.parametrize("field,op,std", FE_CASES, ids=["%s-%s-%s" % (f, o, "std" if s else "raw") for f, o, s in FE_CASES])
def test_field_ops(dev, field, op, std):
    import torch
    code, m, nl, _ = FIELDS[field]
    rows = fe_rows(field, op, std)
    bounds, ref, onl, _, replay = fe_case(field, op, std)
    cols = fe_operands(field, op, std, rows)
    if op == "redc_wide":
        ins = [to_dev([(hi << 384) | lo for hi, lo in zip(cols[0], cols[1])], 2 * nl)]
    else:
        ins = [to_dev(c, nl) for c in cols]
    ins += [ins[0]] * (4 - len(ins))
    out = torch.zeros(rows * onl, dtype=torch.int32, device="cuda")
    assert dev.da_fe(code, FE_OPS[op], std, *[_ptr(t) for t in ins], _ptr(out), rows) == 0
    bad = check_rows(cols, from_dev(out, onl), ref)
    assert not bad, report("%s %s (%s)" % (field, op, "std" if std else "raw"), bad, replay)


F2_CASES = [(inl, op) for inl in (0, 1) for op in ("mul", "sqr", "inv", "inv_serial")]


@pytest.mark.gpu
@pytest.mark.parametrize("inlined,op", F2_CASES, ids=["%s-%s" % ("Fp2I" if i else "Fp2", o) for i, o in F2_CASES])
def test_fp2_ops(dev, inlined, op):
    import torch
    rows = ROWS_INV if "inv" in op else ROWS
    a, b = fp2_operands(op, rows, seed=11 + F2_OPS[op])
    out = torch.zeros(rows * 24, dtype=torch.int32, device="cuda")
    assert dev.da_fp2(inlined, F2_OPS[op], _ptr(to_dev(f2_flat(a), 12)), _ptr(to_dev(f2_flat(b), 12)), _ptr(out), rows) == 0
    got = from_dev(out, 12)
    ref = fp2_ref(op)
    bad = []
    for i in range(rows):
        g, w = (got[2 * i], got[2 * i + 1]), ref(a[i], b[i])
        if g != w:
            bad.append((list(a[i]) + list(b[i]), str(g), str(w)))
    assert not bad, report("%s %s" % ("Fp2I" if inlined else "Fp2", op), bad, "hc_fp2_%s" % op if op in ("mul", "sqr", "inv") else None)


@pytest.mark.gpu
@pytest.mark.parametrize("op", list(DIFF_OPS))
def test_differential_saturated(dev, op):
    """2^28 rows of saturated operands per pair of routes, generated and compared in the kernel"""
    import torch
    seed = 0xC0FFEE + DIFF_OPS[op]
    nbad = torch.zeros(1, dtype=torch.int64, device="cuda")
    rows_out = torch.zeros(16, dtype=torch.int64, device="cuda")
    assert dev.da_diff(DIFF_OPS[op], seed, DIFF_ROWS, _ptr(nbad), _ptr(rows_out), 16) == 0
    n = int(nbad.item())
    if n:
        lines = ["%s: %d of %d rows disagree" % (op, n, DIFF_ROWS)]
        ri = pow(RP, -1, P)
        for row in sorted(int(r) for r in rows_out[:min(n, 16)].tolist()):
            ops = [diff_operand(seed, row, j) for j in range(2 if op == "redc_wide" else 4)]
            if op == "mul2_lazy":
                want = "(a b - c d)/R = %s; replay host_check.hc_fp_mul2_lazy_raw / hc_fp_montmul_raw" % hex((ops[0] * ops[1] - ops[2] * ops[3]) * ri % P)
            elif op == "redc_wide":
                want = "a b / R = %s; replay host_check.hc_fp_mul_wide_raw + hc_fp_redc_wide_raw" % hex(ops[0] * ops[1] * ri % P)
            else:
                want = "Fp2 operands (a, b) x (c, d) in Montgomery form"
            lines.append("  row %d: %s -> %s" % (row, ", ".join(hex(x) for x in ops), want))
        pytest.fail("\n".join(lines))


def _run_group(dev, group, op, acc_rows, q_rows, n):
    import torch
    F, _, fl = _grp(group if group != 3 else 2)
    per = 4 * fl                      # limbs of one XYZZ point
    team = op in (G_ADD_TEAM, G_DBL_TEAM)
    out = torch.zeros(n * per * (4 if team else 1), dtype=torch.int32, device="cuda")
    acc = to_dev([v for r in acc_rows for v in r], 12)
    q = to_dev([v for r in q_rows for v in r], 12) if q_rows else acc
    assert dev.da_group(group, op, _ptr(acc), _ptr(q), _ptr(out), n) == 0
    vals = from_dev(out, 12)
    k = per // 12
    pts = [vals[i * k:(i + 1) * k] for i in range(len(vals) // k)]
    if not team:
        return [decode_xyzz(F, p) for p in pts]
    res = []
    for i in range(n):
        lanes = pts[4 * i:4 * i + 4]
        assert all(l == lanes[0] for l in lanes), "the four lanes of team %d hold different points" % i
        res.append(decode_xyzz(F, lanes[0]))
    return res


def _check_points(label, cases, got, want_of):
    bad = [(c[0], i) for i, (c, g) in enumerate(zip(cases, got)) if g != want_of(c)]
    assert not bad, "%s: %d wrong results, first: %s" % (label, len(bad), bad[:8])


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2])
def test_group_add(dev, group):
    """serial xyzz_add and the team's xyzz_add_t on the same XYZZ pairs, exceptional cases found through the cross
    products (equal points in different projective coordinates)"""
    F, _, _ = _grp(group)
    cases = group_cases(group, 64 if group == 1 else 32, seed=100 + group)
    acc = [xyzz_limbs(F, a, la) for _, a, _, la, _, _ in cases]
    q = [xyzz_limbs(F, b, lb) for _, _, b, _, lb, _ in cases]
    for op, label in ((G_ADD, "xyzz_add"), (G_ADD_TEAM, "xyzz_add_t")):
        got = _run_group(dev, group, op, acc, q, len(cases))
        _check_points("G%d %s" % (group, label), cases, got, lambda c: c[5])


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2, 3], ids=["g1", "g2", "g2-inlined"])
def test_group_madd(dev, group):
    """xyzz_madd (the bucket accumulation's step) with an XYZZ accumulator and an affine operand: acc == q doubles,
    acc == -q gives infinity, infinity on either side"""
    F, _, _ = _grp(1 if group == 1 else 2)
    cases = group_cases(1 if group == 1 else 2, 64 if group == 1 else 32, seed=200 + group)
    acc = [xyzz_limbs(F, a, la) for _, a, _, la, _, _ in cases]
    q = [affine_limbs(F, b) for _, _, b, _, _, _ in cases]
    got = _run_group(dev, group, G_MADD, acc, q, len(cases))
    _check_points("G%d xyzz_madd%s" % (min(group, 2), " (Fp2I)" if group == 3 else ""), cases, got, lambda c: c[5])


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 2])
def test_group_dbl(dev, group):
    F, _, _ = _grp(group)
    cases = dbl_cases(group, 32, seed=300 + group)
    acc = [xyzz_limbs(F, p, lam) for _, p, lam, _ in cases]
    for op, label in ((G_DBL, "xyzz_dbl"), (G_DBL_TEAM, "xyzz_dbl_t")):
        got = _run_group(dev, group, op, acc, None, len(cases))
        _check_points("G%d %s" % (group, label), cases, got, lambda c: c[3])
