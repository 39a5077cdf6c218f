"""Batch PHGR13 verification (ps_phgr13_verify_batch / api.PHGR13VerifyBatch), shared by the host-emulation suite
(test_emu_phgr13_verify_batch.py, N <= 5) and the GPU suite (test_gpu_phgr13_verify_batch.py, up to 4096 proofs).

Proofs come from the device prover on one squaring chain (helpers.squaring_chain: same circuit, witness x0 varies) under
a device setup with its verification key; the oracle's pairing evaluates the combined equation the batch verifier
decides (include/playsnark_b200.h, ps_phgr13_verify_batch)."""
from __future__ import annotations

import ctypes as C
import random

import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api
from playsnark_b200._lib import PlaysnarkError
from tests import helpers as H
from tests import verify_batch_cases as V

G1_FIELDS = ("hs", "vss", "yss", "vass", "wass", "yass", "gz")
MUTATIONS = G1_FIELDS + ("wss", "io_last", "io_other")


class Pool:
    """`count` distinct device proofs of the n-gate squaring chain under one device setup (with_vk=True)"""

    def __init__(self, be, n: int = 8, count: int = 5, seed: int = 1):
        self.be, self.n = be, n
        self.q = V.chain_qap(n)
        self.ek, self.vk, _ = api.NewPHGR13TrustedSetup(self.q, backend=be, with_vk=True)
        self.diff = self.q.nbVars - self.q.nbIO
        self.proofs, self.ios = [], []
        for k in range(count):
            _, wit = H.squaring_chain(n, 3 + k + 1000 * seed)
            self.proofs.append(api.PHGR13Prove(self.ek, self.q, wit, backend=be))
            self.ios.append(list(wit[:self.diff]))

    def batch(self, N: int):
        return [self.proofs[i % len(self.proofs)] for i in range(N)], [list(self.ios[i % len(self.ios)]) for i in range(N)]

    def verify(self, proofs, ios, **kw):
        return api.PHGR13VerifyBatch(self.vk, self.q, proofs, ios, backend=self.be, **kw)

    def verify_one(self, proof, io):
        return api.PHGR13Verify(self.vk, self.q, proof, io, backend=self.be)

    def close(self):
        self.ek.close()
        self.q.close()


def _replace(p, **kw):
    d = {f: getattr(p, f) for f in G1_FIELDS + ("wss",)}
    d.update(kw)
    return api.PHGR13Proof(**d)


def _g1_shift(b: bytes, D) -> bytes:
    return O.g1_compress(O.g1_add(O.g1_decompress(b), D))


def mutate(proofs, ios, i: int, kind: str):
    """proof i of the batch made invalid; returns (proofs, ios) as new lists"""
    proofs, ios = list(proofs), [list(v) for v in ios]
    p = proofs[i]
    if kind in G1_FIELDS:
        proofs[i] = _replace(p, **{kind: _g1_shift(getattr(p, kind), O.G1_GEN)})
    elif kind == "wss":
        proofs[i] = _replace(p, wss=O.g2_compress(O.g2_add(O.g2_decompress(p.wss), O.G2_GEN)))
    elif kind == "io_last":
        ios[i][-1] = (ios[i][-1] + 1) % O.R
    elif kind == "io_other":
        j = next((j for j in range(len(ios)) if ios[j] != ios[i]), None)
        ios[i] = list(ios[j]) if j is not None else [(v + 1) % O.R for v in ios[i]]
    else:
        raise KeyError(kind)
    return proofs, ios


def oracle_combined(vk, n_io, proofs, ios, weights) -> bool:
    """the combined equation of ps_phgr13_verify_batch with the oracle's pairing; weights = one 5-tuple per proof"""
    d1, d2 = O.g1_decompress, O.g2_decompress
    vs, ws, ys = [d1(b) for b in vk["vs"][:n_io]], [d2(b) for b in vk["ws"][:n_io]], [d1(b) for b in vk["ys"][:n_io]]
    mul1 = lambda k, b: O.pt_mul(O.F1, k % O.R, d1(b))
    acc = {k: None for k in ("X", "hs", "vss", "yss", "gz", "vy")}
    w3 = w5 = None
    pairs = []
    s = [0] * n_io
    for (r1, r2, r3, r4, r5), p, io in zip(weights, proofs, ios):
        gv = O.g1_add(O.msm_naive(O.F1, [r1 * v % O.R for v in io[:n_io]], vs), mul1(r1, p.vss))
        gw = O.g2_add(O.msm_naive(O.F2, [v % O.R for v in io[:n_io]], ws), d2(p.wss))
        pairs.append((gv, gw))
        for t, (k, b) in enumerate(((r2, p.vass), (r3, p.wass), (r4, p.yass), (O.R - r1, p.yss))):
            acc["X"] = O.g1_add(acc["X"], mul1(k, b))
        acc["hs"] = O.g1_add(acc["hs"], mul1(r1, p.hs))
        acc["vss"] = O.g1_add(acc["vss"], mul1(r2, p.vss))
        acc["yss"] = O.g1_add(acc["yss"], mul1(r4, p.yss))
        acc["gz"] = O.g1_add(acc["gz"], mul1(r5, p.gz))
        acc["vy"] = O.g1_add(acc["vy"], O.pt_mul(O.F1, r5 % O.R, O.g1_add(d1(p.vss), d1(p.yss))))
        w3 = O.g2_add(w3, O.pt_mul(O.F2, r3 % O.R, d2(p.wss)))
        w5 = O.g2_add(w5, O.pt_mul(O.F2, r5 % O.R, d2(p.wss)))
        for k in range(n_io):
            s[k] = (s[k] + r1 * io[k]) % O.R
    neg = lambda a: O.pt_neg(O.F1, a)
    X = O.g1_add(acc["X"], neg(O.msm_naive(O.F1, s, ys))) if n_io else acc["X"]
    pairs += [(X, O.G2_GEN), (neg(acc["hs"]), d2(vk["yts"])), (neg(acc["vss"]), d2(vk["av"])), (neg(acc["yss"]), d2(vk["ay"])),
              (acc["gz"], d2(vk["gamma"])), (neg(acc["vy"]), d2(vk["bgamma2"])), (neg(d1(vk["aw"])), w3),
              (neg(d1(vk["bgamma"])), w5)]
    f = O.FP12_ONE
    for a, b in pairs:
        if a is not None and b is not None:
            f = O.fp12_mul(f, O.pairing(a, b))
    return f == O.FP12_ONE


# ---- cases ---------------------------------------------------------------------------------------------------------
def honest(pool, N: int):
    """an honest batch is accepted with every verdict true; at N = 1 the verdict is PHGR13Verify's"""
    proofs, ios = pool.batch(N)
    assert pool.verify(proofs, ios) is True
    assert pool.verify(proofs, ios, per_proof=True) == [True] * N
    if N == 1:
        assert pool.verify_one(proofs[0], ios[0]) is True


def one_invalid(pool, N: int, pos: int, kind: str):
    """one mutated proof: PHGR13Verify rejects it, the batch is rejected and only that index is flagged"""
    proofs, ios = mutate(*pool.batch(N), pos, kind)
    assert pool.verify_one(proofs[pos], ios[pos]) is False, kind
    assert pool.verify(proofs, ios) is False, (kind, pos)
    assert pool.verify(proofs, ios, per_proof=True) == [i != pos for i in range(N)], (kind, pos)


def several_invalid(pool, N: int, positions, kinds=MUTATIONS):
    proofs, ios = pool.batch(N)
    for t, i in enumerate(positions):
        proofs, ios = mutate(proofs, ios, i, kinds[t % len(kinds)])
    assert pool.verify(proofs, ios) is False
    assert pool.verify(proofs, ios, per_proof=True) == [i not in set(positions) for i in range(N)]


def weights_independent(pool, D_scalar: int = 7):
    """Forgeries that only independent weights catch, each checked against the oracle's combined equation:
    hs_0 + D with hs_1 - D keeps sum rho1 hs when all weights are 1; vass_0 + D with yass_0 - D keeps the G2gen partner
    when rho2 = rho4 for that proof."""
    proofs, ios = pool.batch(2)
    D = O.g1_mul(D_scalar)
    negD = O.pt_neg(O.F1, D)
    f = [_replace(proofs[0], hs=_g1_shift(proofs[0].hs, D)), _replace(proofs[1], hs=_g1_shift(proofs[1].hs, negD))]
    ones = [(1,) * 5] * 2
    distinct = [(3, 5, 7, 11, 13), (17, 19, 23, 29, 31)]
    assert oracle_combined(pool.vk, pool.diff, f, ios, ones) is True
    assert pool.verify(f, ios, weights=ones) is True
    assert oracle_combined(pool.vk, pool.diff, f, ios, distinct) is False
    assert pool.verify(f, ios, weights=distinct) is False
    assert pool.verify(f, ios) is False
    assert pool.verify(f, ios, per_proof=True) == [False, False]
    g = [_replace(proofs[0], vass=_g1_shift(proofs[0].vass, D), yass=_g1_shift(proofs[0].yass, negD)), proofs[1]]
    assert pool.verify_one(g[0], ios[0]) is False
    same24 = [(3, 5, 7, 5, 13), (17, 19, 23, 29, 31)]
    assert oracle_combined(pool.vk, pool.diff, g, ios, same24) is True
    assert pool.verify(g, ios, weights=same24) is True
    assert oracle_combined(pool.vk, pool.diff, g, ios, distinct) is False
    assert pool.verify(g, ios, weights=distinct) is False
    assert pool.verify(g, ios, per_proof=True) == [False, True]


def matches_oracle(pool, N: int = 2, seed: int = 5):
    """injected weights: the device's decision is the combined equation's, on an honest and on a mutated batch"""
    rng = random.Random(seed)
    proofs, ios = pool.batch(N)
    w = [tuple(rng.randrange(1, 1 << 128) for _ in range(5)) for _ in range(N)]
    assert pool.verify(proofs, ios, weights=w) is oracle_combined(pool.vk, pool.diff, proofs, ios, w) is True
    bad_p, bad_io = mutate(proofs, ios, N - 1, "gz")
    assert pool.verify(bad_p, bad_io, weights=w) is oracle_combined(pool.vk, pool.diff, bad_p, bad_io, w) is False


def no_io_qap():
    """x1 = x0^2, x2 = x1^2 with x1, x2 both outputs: no intermediate variables, so the verification key has no public
    values (nbVars - nbIO = 0)"""
    r = api.R1CS()
    r.NewInput("x0")
    r.NewOutput("x1")
    r.NewOutput("x2")
    r.Mul("x0", "x0", "x1")
    r.Mul("x1", "x1", "x2")
    return api.ToQAP(r)


def no_io(be, seed: int = 6):
    """n_io = 0: gv = vss, gw = wss and no MSMs.  Honest proofs are accepted (with injected and with drawn weights),
    a mutated one is flagged alone, and each decision is the oracle's combined equation's"""
    q = no_io_qap()
    ek, vk, _ = api.NewPHGR13TrustedSetup(q, backend=be, with_vk=True)
    try:
        assert q.nbVars - q.nbIO == 0
        proofs = []
        for x0 in (3, 5, 7):
            proofs.append(api.PHGR13Prove(ek, q, [1, x0, x0 ** 2 % O.R, x0 ** 4 % O.R], backend=be))
        ios = [[] for _ in proofs]
        rng = random.Random(seed)
        w = [tuple(rng.randrange(1, 1 << 128) for _ in range(5)) for _ in proofs]
        verify = lambda ps, **kw: api.PHGR13VerifyBatch(vk, q, ps, ios[:len(ps)], backend=be, **kw)
        assert api.PHGR13Verify(vk, q, proofs[0], [], backend=be) is True
        assert oracle_combined(vk, 0, proofs, ios, w) is True
        assert verify(proofs, weights=w) is True
        assert verify(proofs) is True
        assert verify(proofs, per_proof=True) == [True, True, True]
        bad, _ = mutate(proofs, ios, 1, "wss")
        assert oracle_combined(vk, 0, bad, ios, w) is False
        assert verify(bad, weights=w) is False
        assert verify(bad, per_proof=True) == [True, False, True]
    finally:
        ek.close()
        q.close()


def malformed_points(pool, N: int = 5):
    """a proof point off the curve, outside the subgroup, or moved by a point of small order marks only that proof
    invalid; the call succeeds and decides the others -- with subgroup_check on and off (it governs key points only)"""
    from tests import pairing_cases as PCs
    proofs, ios = pool.batch(N)
    T3 = PCs.small_torsion(L.PS_G1, 3)
    p = list(proofs)
    p[0] = _replace(p[0], gz=V._off_curve_g1())
    p[1] = _replace(p[1], vass=V._outside_subgroup_g1())
    p[2] = _replace(p[2], yss=O.g1_compress(O.g1_add(O.g1_decompress(p[2].yss), T3)))
    p[N - 1] = _replace(p[N - 1], wss=V._outside_subgroup_g2())
    bad = {0, 1, 2, N - 1}
    want = [i not in bad for i in range(N)]
    try:
        for sub in (1, 0):
            pool.be.set_option("subgroup_check", sub)
            assert pool.verify(p, ios) is False
            assert pool.verify(p, ios, per_proof=True) == want
            rest = [i for i in range(N) if want[i]]
            assert pool.verify([p[i] for i in rest], [ios[i] for i in rest]) is True
    finally:
        pool.be.set_option("subgroup_check", 1)


def bad_arguments(pool):
    """bad key point / io >= r -> PS_ERR_ENCODING; zero weight -> ValueError / PS_ERR_ARG; count mismatches -> ValueError;
    no proofs -> True / []"""
    proofs, ios = pool.batch(2)
    bad_vk = dict(pool.vk, gamma=bytes(96))                        # no compression flag: does not decode
    with pytest.raises(PlaysnarkError) as e:
        api.PHGR13VerifyBatch(bad_vk, pool.q, proofs, ios, backend=pool.be)
    assert e.value.status == L.PS_ERR_ENCODING
    bad_io = b"".join(api._fr_bytes(v) for v in ios)
    bad_io = bad_io[:-32] + O.R.to_bytes(32, "big")
    with pytest.raises(PlaysnarkError) as e:
        pool.verify(proofs, bad_io)
    assert e.value.status == L.PS_ERR_ENCODING
    with pytest.raises(ValueError):
        pool.verify(proofs, ios, weights=[(1,) * 5, (1, 1, 0, 1, 1)])
    with pytest.raises(ValueError):
        pool.verify(proofs, ios, weights=[(1,) * 5, (1,) * 4])
    vk, n_io = pool.vk, pool.diff
    fixed = vk["av"] + vk["aw"] + vk["ay"] + vk["gamma"] + vk["bgamma"] + vk["bgamma2"] + vk["yts"]
    blob = b"".join(p.hs + p.vss + p.yss + p.vass + p.wass + p.yass + p.gz + p.wss for p in proofs)
    w = bytes(16 * 5 * 2 - 1) + b"\1"                               # proof 0's weights all zero
    ok = C.c_int(7)
    lib = pool.be.lib
    st = lib.ps_phgr13_verify_batch(pool.be.ctx, fixed, b"".join(vk["vs"][:n_io]), b"".join(vk["ws"][:n_io]), b"".join(vk["ys"][:n_io]),
                                    n_io, 2, b"".join(api._fr_bytes(v) for v in ios), blob, w, C.byref(ok), None)
    assert st == L.PS_ERR_ARG
    short = [list(v) for v in ios]
    short[1] = short[1][:n_io - 1]
    with pytest.raises(ValueError):
        pool.verify(proofs, short)
    with pytest.raises(ValueError):
        pool.verify(proofs, ios[:1])
    with pytest.raises(ValueError):
        pool.verify(proofs, b"".join(api._fr_bytes(v[:n_io]) for v in ios)[:-32])
    assert pool.verify([], []) is True
    assert pool.verify([], [], per_proof=True) == []
    ok = C.c_int(7)
    assert lib.ps_phgr13_verify_batch(pool.be.ctx, fixed, b"".join(vk["vs"][:n_io]), b"".join(vk["ws"][:n_io]),
                                      b"".join(vk["ys"][:n_io]), n_io, 0, None, None, None, C.byref(ok), None) == L.PS_OK
    assert ok.value == 1


def blob_inputs(pool, N: int = 3):
    """ios as one wire-format blob and as a HostBuffer give the decisions of the list form"""
    proofs, ios = pool.batch(N)
    blob = b"".join(api._fr_bytes(v[:pool.diff]) for v in ios)
    assert pool.verify(proofs, blob) is True
    hb = api.HostBuffer(pool.be, blob)
    bad_p, _ = mutate(proofs, ios, 1, "hs")
    assert pool.verify(bad_p, hb, per_proof=True) == [True, False, True]
    hb.close()
