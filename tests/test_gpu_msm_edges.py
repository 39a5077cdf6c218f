"""Degenerate MSM inputs through the product C ABI on the device (tests/msm_edge_cases.py), and the device-resident
MSM entry points: scalars in Montgomery form from ps_fr_upload, sub-ranges of a base set, and sums of partials."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api
from tests import msm_edge_cases as E, parity_cases as PC

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def be():
    lib = L.load()
    assert b"sm_100a" in lib.ps_version()      # the product build, not the host emulation
    b = api.Backend(0)
    before = b.launch_count()
    yield b
    assert b.launch_count() > before           # kernels really ran
    b.close()


WINDOWS = [(4, 1), (7, 100), (13, 1), (16, 16), (0, -1)]      # (window bits, tables); (0, -1): automatic, all tables
KINDS = ["rand", "ones", "small", "neg", "edge"]
SIZES = {L.PS_G1: [2, 3, 64, 1000, 4096, 1 << 14], L.PS_G2: [2, 17, 300, 4096]}


def _matrix():
    """every family on both groups and both tail paths (msm_team 0 / 1); sizes, scalar kinds, windows, the wave rounding
    and the scatter rotate so that each value meets several families"""
    out = []
    j = 0
    for fam in E.FAMILIES:
        for group in (L.PS_G1, L.PS_G2):
            for team in (0, 1):
                sizes = SIZES[group]
                wb, tables = WINDOWS[j % len(WINDOWS)]
                out.append((fam, group, sizes[j % len(sizes)], KINDS[(3 * j) % len(KINDS)], wb, tables, team,
                            (j // 2) % 2, 2 * ((j // 3) % 2)))
                j += 1
    return out


MATRIX = _matrix()


@pytest.mark.parametrize("fam,group,n,kind,wb,tables,team,wave_floor,scatter", MATRIX,
                         ids=["%s-g%d-n%d-%s-c%d-t%d-team%d-wf%d-sc%d" % m for m in MATRIX])
def test_msm_edge_matrix(be, fam, group, n, kind, wb, tables, team, wave_floor, scatter):
    E.msm_edge_check(be, group, n, fam, kind, wb, tables, team=team, wave_floor=wave_floor, scatter=scatter)


@pytest.mark.parametrize("fam,kind", [("same", "ones"), ("pm", "rand"), ("fold", "ones"), ("few", "small"),
                                      ("zero-sum", "rand"), ("inf-alt", "neg")])
@pytest.mark.parametrize("team", [0, 1])
def test_msm_edge_2p16_c4(be, fam, kind, team):
    # c = 4: 8 buckets per window, each spanning far more than RUN_MAX = 32 accumulation chunks, so the log-depth merge
    # of boundary partials adds up the degenerate sums
    E.msm_edge_check(be, L.PS_G1, 1 << 16, fam, kind, 4, 1, team=team)


@pytest.mark.parametrize("wb,tables", [(0, -1), (16, 1)])
def test_msm_edge_few_2p20(be, wb, tables):
    # large enough for the one-thread tails with the default options (more than 65536 merge items)
    E.msm_edge_check(be, L.PS_G1, 1 << 20, "few", "rand", wb, tables)


@pytest.mark.parametrize("fam", ["pm", "fold", "few"])
def test_msm_edge_g2_4096_c4(be, fam):
    E.msm_edge_check(be, L.PS_G2, 4096, fam, "ones", 4, 1, team=0)
    E.msm_edge_check(be, L.PS_G2, 4096, fam, "small", 4, 1, team=1)


# ---- device-resident entry points ------------------------------------------------------------------------------
def _limbs_le(torch, sc):
    """scalars as 8 little-endian 32-bit limbs each, on the device (ps_msm_device's layout)"""
    buf = bytearray(b"".join(s.to_bytes(32, "little") for s in sc))
    return torch.frombuffer(buf, dtype=torch.int32).cuda()


@pytest.mark.parametrize("log_n", [16, 20])
def test_msm_device_mont(be, log_n):
    """ps_msm_device_mont on scalars uploaded with ps_fr_upload (Montgomery limbs) equals ps_msm on the same scalars
    and the oracle"""
    import torch
    from oracle import c_oracle as CO
    F, gen, comp, _ = PC._grp(L.PS_G1)
    n = 1 << log_n
    rng = np.random.default_rng(log_n)
    ks = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    sc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    ks[:, 0] &= 0x3F
    sc[:, 0] &= 0x3F
    for i, v in enumerate([0, 1, O.R - 1, O.R - 2, (O.R - 1) // 2, (O.R + 1) // 2, 2]):   # both sides of the fold
        sc[i] = np.frombuffer(v.to_bytes(32, "big"), dtype=np.uint8)
    bases = be.bases_from_scalars(L.PS_G1, ks.tobytes(), 0, -1)
    want = comp(O.pt_mul(F, CO.fr_dot(ks, sc), gen))
    assert be.msm(bases, sc.tobytes()) == want
    d_mont = torch.zeros(n * 8, dtype=torch.int32, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    part = torch.zeros(192, dtype=torch.uint8, device="cuda")
    host = np.ascontiguousarray(sc)
    be._check(be.lib.ps_fr_upload(be.ctx, C.c_void_p(host.ctypes.data), n, C.c_void_p(d_mont.data_ptr()), C.c_void_p(status.data_ptr())))
    be._check(be.lib.ps_msm_device_mont(be.ctx, bases.handle, 0, C.c_void_p(d_mont.data_ptr()), n, C.c_void_p(part.data_ptr())))
    out = C.create_string_buffer(48)
    be._check(be.lib.ps_msm_combine(be.ctx, L.PS_G1, C.c_void_p(part.data_ptr()), 1, out))
    be.sync()
    assert int(status.item()) == 0
    assert out.raw == want
    bases.close()


@pytest.mark.parametrize("group,n", [(L.PS_G1, 5000), (L.PS_G2, 700)])
def test_msm_device_ranges_and_combine(be, group, n):
    """ps_msm_device over sub-ranges (first > 0, an empty one included) summed by ps_msm_combine equals the whole
    MSM; two partials that cancel exactly combine to the encoding of infinity"""
    import torch
    F, gen, comp, _ = PC._grp(group)
    per = 192 if group == L.PS_G1 else 384
    rng = random.Random(n)
    ks = [rng.randrange(1, O.R) for _ in range(n)]
    sc = PC.scalars_of("rand", n, rng)
    sc[:4] = [0, 1, O.R - 1, (O.R + 1) // 2]
    bases = be.bases_from_scalars(group, ks)
    want = comp(O.pt_mul(F, sum(k * s for k, s in zip(ks, sc)) % O.R, gen))
    assert be.msm(bases, sc) == want
    d_sc = _limbs_le(torch, sc)
    d_neg = _limbs_le(torch, [(O.R - s) % O.R for s in sc])
    cuts = [0, 1, 1, 37, n // 3, n // 3 + 1, n - 5, n]           # [1, 1) is empty
    parts = torch.zeros((len(cuts) - 1) * per, dtype=torch.uint8, device="cuda")
    ptr = lambda t, off: C.c_void_p(t.data_ptr() + off)
    for j, (lo, hi) in enumerate(zip(cuts, cuts[1:])):
        be._check(be.lib.ps_msm_device(be.ctx, bases.handle, lo, ptr(d_sc, 32 * lo), hi - lo, ptr(parts, per * j)))
    out = C.create_string_buffer(per // 4)
    be._check(be.lib.ps_msm_combine(be.ctx, group, ptr(parts, 0), len(cuts) - 1, out))
    assert out.raw == want
    # one range with s and with r - s: the two partials are negatives of each other
    lo, hi = 37, n // 3
    pair = torch.zeros(2 * per, dtype=torch.uint8, device="cuda")
    be._check(be.lib.ps_msm_device(be.ctx, bases.handle, lo, ptr(d_sc, 32 * lo), hi - lo, ptr(pair, 0)))
    be._check(be.lib.ps_msm_device(be.ctx, bases.handle, lo, ptr(d_neg, 32 * lo), hi - lo, ptr(pair, per)))
    be._check(be.lib.ps_msm_combine(be.ctx, group, ptr(pair, 0), 2, out))
    assert out.raw == comp(None)
    # and each of them alone is the MSM of that range
    be._check(be.lib.ps_msm_combine(be.ctx, group, ptr(pair, 0), 1, out))
    assert out.raw == comp(O.pt_mul(F, sum(k * s for k, s in zip(ks[lo:hi], sc[lo:hi])) % O.R, gen))
    bases.close()
