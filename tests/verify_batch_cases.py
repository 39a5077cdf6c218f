"""Batch Groth16 verification (ps_g16_verify_batch / api.Groth16VerifyBatch), shared by the host-emulation suite
(test_emu_verify_batch.py, small batches) and the GPU suite (test_gpu_verify_batch.py, up to 4096 proofs).

Proofs come from the device prover on one squaring chain (helpers.squaring_chain: same circuit, witness x0 varies) under
a device setup; the oracle's pairing evaluates the combined equation the batch verifier decides."""
from __future__ import annotations

import ctypes as C
import dataclasses
import random

import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api
from playsnark_b200._lib import PlaysnarkError
from tests import helpers as H

MUTATIONS = ("A+G", "B+H", "C+G", "io_last", "io_other")


def chain_qap(n: int) -> api.SparseQAP:
    """the R1CS of helpers.squaring_chain(n, .) through the host mirror"""
    r = api.R1CS()
    r.NewInput("x0")
    r.NewOutput("x%d" % n)
    for i in range(1, n):
        r.NewVar("x%d" % i)
    for i in range(n):
        r.Mul("x%d" % i, "x%d" % i, "x%d" % (i + 1))
    return api.ToQAP(r)


class Pool:
    """`count` distinct device proofs of the n-gate squaring chain under one device setup, with their public inputs"""

    def __init__(self, be, n: int = 8, count: int = 6, seed: int = 1):
        self.be, self.n = be, n
        self.q = chain_qap(n)
        self.tr = api.NewGroth16TrustedSetup(self.q, backend=be, fmt=L.PS_FMT_COMPRESSED, export=True)
        diff = self.q.nbVars - self.q.nbIO
        rng = random.Random(seed)
        self.proofs, self.ios = [], []
        for k in range(count):
            _, wit = H.squaring_chain(n, 3 + k + 1000 * seed)
            self.proofs.append(api.Groth16Prove(self.tr, self.q, wit, rng.randrange(1, O.R), rng.randrange(1, O.R), backend=be))
            self.ios.append(wit[:diff])

    def batch(self, N: int):
        """N proofs (the pool cycled) and their io vectors"""
        return [self.proofs[i % len(self.proofs)] for i in range(N)], [list(self.ios[i % len(self.ios)]) for i in range(N)]

    def verify(self, proofs, ios, **kw):
        return api.Groth16VerifyBatch(self.tr, self.q, proofs, ios, backend=self.be, **kw)

    def close(self):
        self.tr.close()
        self.q.close()


def g1d(b):
    return O.g1_decompress(b)


def mutate(proofs, ios, i: int, kind: str):
    """proof i of the batch made invalid in place; returns (proofs, ios) as new lists"""
    proofs, ios = list(proofs), [list(v) for v in ios]
    p = proofs[i]
    if kind == "A+G":
        proofs[i] = api.Groth16Proof(p.tp, O.g1_compress(O.g1_add(g1d(p.A), O.G1_GEN)), p.B, p.C)
    elif kind == "B+H":
        proofs[i] = api.Groth16Proof(p.tp, p.A, O.g2_compress(O.g2_add(O.g2_decompress(p.B), O.G2_GEN)), p.C)
    elif kind == "C+G":
        proofs[i] = api.Groth16Proof(p.tp, p.A, p.B, O.g1_compress(O.g1_add(g1d(p.C), O.G1_GEN)))
    elif kind == "io_last":
        ios[i][-1] = (ios[i][-1] + 1) % O.R
    elif kind == "io_other":
        j = next(j for j in range(len(ios)) if ios[j] != ios[i]) if any(v != ios[i] for v in ios) else None
        ios[i] = list(ios[j]) if j is not None else [(v + 1) % O.R for v in ios[i]]
    else:
        raise KeyError(kind)
    return proofs, ios


def oracle_combined(tr, proofs, ios, weights) -> bool:
    """prod_i e(-w_i A_i, B_i) e(S Alpha, Beta2) e(L, Gamma) e(Cs, Delta2) == 1 with the oracle's pairing"""
    n_io = len(tr.IoLP)
    S = sum(weights) % O.R
    sj = [sum(w * io[j] for w, io in zip(weights, ios)) % O.R for j in range(n_io)]
    Lp = O.msm_naive(O.F1, sj, [g1d(p) for p in tr.IoLP])
    Cs = None
    for w, p in zip(weights, proofs):
        Cs = O.g1_add(Cs, O.g1_mul(w % O.R, g1d(p.C)))
    pairs = [(O.g1_mul((O.R - w) % O.R, g1d(p.A)), O.g2_decompress(p.B)) for w, p in zip(weights, proofs)]
    pairs += [(O.g1_mul(S, g1d(tr.Alpha)), O.g2_decompress(tr.Beta2)), (Lp, O.g2_decompress(tr.Gamma)),
              (Cs, O.g2_decompress(tr.Delta2))]
    f = O.FP12_ONE
    for a, b in pairs:
        if a is not None and b is not None:
            f = O.fp12_mul(f, O.pairing(a, b))
    return f == O.FP12_ONE


# ---- cases ---------------------------------------------------------------------------------------------------------
def honest(pool, N: int):
    """an honest batch is accepted with every verdict true; at N = 1 the decision is Groth16Verify's"""
    proofs, ios = pool.batch(N)
    assert pool.verify(proofs, ios) is True
    assert pool.verify(proofs, ios, per_proof=True) == [True] * N
    if N == 1:
        assert api.Groth16Verify(pool.tr, pool.q, proofs[0], ios[0], backend=pool.be) is True


def one_invalid(pool, N: int, pos: int, kind: str):
    """one mutated proof: the batch is rejected and only that index is flagged"""
    proofs, ios = mutate(*pool.batch(N), pos, kind)
    assert api.Groth16Verify(pool.tr, pool.q, proofs[pos], ios[pos], backend=pool.be) is False
    assert pool.verify(proofs, ios) is False
    want = [i != pos for i in range(N)]
    assert pool.verify(proofs, ios, per_proof=True) == want, (kind, pos)


def several_invalid(pool, N: int, positions, kinds=MUTATIONS):
    proofs, ios = pool.batch(N)
    for t, i in enumerate(positions):
        proofs, ios = mutate(proofs, ios, i, kinds[t % len(kinds)])
    assert pool.verify(proofs, ios) is False
    assert pool.verify(proofs, ios, per_proof=True) == [i not in set(positions) for i in range(N)]


def weights_applied(pool, D_scalar: int = 7):
    """C_0 + D, C_1 - D: both proofs are invalid, yet the sum of the C's is unchanged.  With weights (1, 1) the combined
    equation holds (the oracle agrees) and the batch is accepted; distinct weights and the library's own reject it."""
    proofs, ios = pool.batch(2)
    D = O.g1_mul(D_scalar)
    p0, p1 = proofs
    f0 = api.Groth16Proof(p0.tp, p0.A, p0.B, O.g1_compress(O.g1_add(g1d(p0.C), D)))
    f1 = api.Groth16Proof(p1.tp, p1.A, p1.B, O.g1_compress(O.g1_add(g1d(p1.C), O.pt_neg(O.F1, D))))
    forged = [f0, f1]
    assert oracle_combined(pool.tr, forged, ios, [1, 1]) is True
    assert pool.verify(forged, ios, weights=[1, 1]) is True
    assert oracle_combined(pool.tr, forged, ios, [3, 5]) is False
    assert pool.verify(forged, ios, weights=[3, 5]) is False
    assert pool.verify(forged, ios) is False
    assert pool.verify(forged, ios, per_proof=True) == [False, False]


def matches_oracle(pool, N: int = 2, seed: int = 5):
    """injected weights: the device's decision is the combined equation's, on an honest and on a mutated batch"""
    rng = random.Random(seed)
    proofs, ios = pool.batch(N)
    w = [rng.randrange(1, 1 << 128) for _ in range(N)]
    assert pool.verify(proofs, ios, weights=w) is oracle_combined(pool.tr, proofs, ios, w) is True
    bad_p, bad_io = mutate(proofs, ios, N - 1, "C+G")
    assert pool.verify(bad_p, bad_io, weights=w) is oracle_combined(pool.tr, bad_p, bad_io, w) is False


def _off_curve_g1() -> bytes:
    x = 1
    while O.fp_sqrt((x * x * x + 4) % O.P) is not None:
        x += 1
    b = bytearray(x.to_bytes(48, "big"))
    b[0] |= 0x80
    return bytes(b)


def _outside_subgroup_g1():
    """a point of E(Fp) outside the prime-order subgroup (the cofactor is not 1)"""
    x = 1
    while True:
        y = O.fp_sqrt((x * x * x + 4) % O.P)
        if y is not None and not O.in_subgroup(O.F1, (x, y)):
            assert O.on_curve(O.F1, (x, y))
            return O.g1_compress((x, y))
        x += 1


def _outside_subgroup_g2():
    """a point of the twist E'(Fp2) outside the prime-order subgroup"""
    F = O.F2
    x0 = 1
    while True:
        x = (x0, 1)
        rhs = F.add(F.mul(F.sqr(x), x), F.b)
        y = O.fp2_sqrt(rhs)
        if y is not None and not O.in_subgroup(F, (x, y)):
            assert O.on_curve(F, (x, y))
            return O.g2_compress((x, y))
        x0 += 1


def malformed_points(pool, N: int = 4):
    """a proof point off the curve or outside the subgroup marks only that proof invalid; the call succeeds and decides the
    other proofs -- also with the context's subgroup_check off, which governs key points only"""
    proofs, ios = pool.batch(N)
    off, out1, out2 = _off_curve_g1(), _outside_subgroup_g1(), _outside_subgroup_g2()
    p = list(proofs)
    p[0] = api.Groth16Proof(p[0].tp, off, p[0].B, p[0].C)
    p[1] = api.Groth16Proof(p[1].tp, p[1].A, p[1].B, out1)
    p[N - 1] = api.Groth16Proof(p[N - 1].tp, p[N - 1].A, out2, p[N - 1].C)
    want = [False, False] + [True] * (N - 3) + [False]
    try:
        for sub in (1, 0):
            pool.be.set_option("subgroup_check", sub)
            assert pool.verify(p, ios) is False
            assert pool.verify(p, ios, per_proof=True) == want
            honest_rest = [q for i, q in enumerate(p) if want[i]]
            assert pool.verify(honest_rest, [v for i, v in enumerate(ios) if want[i]]) is True
    finally:
        pool.be.set_option("subgroup_check", 1)


def bad_arguments(pool):
    """bad key point -> PS_ERR_ENCODING; zero weight -> ValueError / PS_ERR_ARG; io count mismatches -> ValueError;
    no proofs -> True"""
    proofs, ios = pool.batch(2)
    tr = pool.tr
    bad_tr = dataclasses.replace(tr, Gamma=bytes(96), _dev=None)          # no compression flag: does not decode
    with pytest.raises(PlaysnarkError) as e:
        api.Groth16VerifyBatch(bad_tr, pool.q, proofs, ios, backend=pool.be)
    assert e.value.status == L.PS_ERR_ENCODING
    with pytest.raises(ValueError):
        pool.verify(proofs, ios, weights=[1, 0])
    lib, n_io = pool.be.lib, len(tr.IoLP)
    ok = C.c_int(7)
    w = (1).to_bytes(16, "big") + bytes(16)
    st = lib.ps_g16_verify_batch(pool.be.ctx, tr.Alpha, tr.Beta2, tr.Gamma, tr.Delta2, b"".join(tr.IoLP), n_io, 2,
                                 b"".join(api._fr_bytes(v) for v in ios), proofs[0].A + proofs[1].A, proofs[0].B + proofs[1].B,
                                 proofs[0].C + proofs[1].C, w, C.byref(ok), None)
    assert st == L.PS_ERR_ARG
    bad_io = [list(v) for v in ios]
    bad_io[1] = bad_io[1][:-1]
    with pytest.raises(ValueError):
        pool.verify(proofs, bad_io)
    with pytest.raises(ValueError):
        pool.verify(proofs, ios[:1])
    with pytest.raises(ValueError):
        pool.verify(proofs, b"".join(api._fr_bytes(v) for v in ios)[:-32])
    assert pool.verify([], []) is True
    assert pool.verify([], [], per_proof=True) == []
    ok = C.c_int(7)
    assert lib.ps_g16_verify_batch(pool.be.ctx, tr.Alpha, tr.Beta2, tr.Gamma, tr.Delta2, b"".join(tr.IoLP), n_io, 0, None, None, None,
                                   None, None, C.byref(ok), None) == L.PS_OK and ok.value == 1


def blob_inputs(pool, N: int = 3):
    """ios as one wire-format blob and as a HostBuffer give the decisions of the list form"""
    proofs, ios = pool.batch(N)
    blob = b"".join(api._fr_bytes(v) for v in ios)
    assert pool.verify(proofs, blob) is True
    hb = api.HostBuffer(pool.be, blob)
    bad_p, _ = mutate(proofs, ios, 1, "A+G")
    assert pool.verify(bad_p, hb, per_proof=True) == [True, False, True]
    hb.close()
