"""Host-side mirror of the reference's proving interface.

Names, argument meaning and error behaviour follow the Go package so that parity tests read like the
reference's own tests:
  Groth16Prove(tr, q, sol)          groth16.go:122
  PHGR13Prove(ek, qap, solution)    pinochio.go:207
  QAP.Quotient(sol) -> Quotient     qap.go:151         (raises ArithmeticError("apocalypse"))
  Poly.BlindEval -> BlindEval       algebra.go:348     (raises ValueError on length mismatch)
Scalars are Python ints mod r (the reference's kyber.Scalar); points are their MarshalBinary bytes
(48 B G1 / 96 B G2, zcash-compressed), which is also what crosses the C ABI.  This module holds no
arithmetic: every value is computed by the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import secrets
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

from . import _lib as L

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001

Vector = List[int]
Poly = List[int]


class HostBuffer:
    """Wire-format values in page-locked host memory (ps_host_alloc): what a caller who proves repeatedly
    marshals its witness into, so that the host-to-device copy runs at link speed.  Accepted wherever a
    Vector of Fr values is; len() is the number of 32-byte values."""

    def __init__(self, backend: "Backend", data):
        raw = _fr_bytes(data)
        self.lib, self.nbytes = backend.lib, len(raw)
        p = C.c_void_p()
        backend._check(self.lib.ps_host_alloc(max(1, self.nbytes), C.byref(p)))
        self.ptr = p
        C.memmove(p, raw, self.nbytes)

    def __len__(self):
        return self.nbytes // 32

    def close(self):
        if getattr(self, "ptr", None):
            self.lib.ps_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _fr_bytes(vals):
    """Fr values (ints, reduced mod r like Value.ToFieldElement) -> 32-byte big-endian rows; byte strings
    that are already in wire format pass through, a HostBuffer passes as its pointer."""
    if isinstance(vals, HostBuffer):
        return vals.ptr
    if isinstance(vals, (bytes, bytearray, memoryview)):
        return bytes(vals)
    if len(vals) >= 4096:
        # long vectors of small values (matrix coefficients): one vectorised pass instead of a to_bytes per element
        try:
            import numpy as np
            lo = np.array(vals, dtype=np.uint64)        # OverflowError on anything outside [0, 2^64)
            rows = np.zeros((len(vals), 32), dtype=np.uint8)
            rows[:, 24:] = lo.astype(">u8").view(np.uint8).reshape(-1, 8)
            return rows.tobytes()
        except (OverflowError, ImportError, TypeError, ValueError):
            pass
    return b"".join((int(v) % R).to_bytes(32, "big") for v in vals)


def _u32_array(vals):
    """index vectors for the C ABI (array('I') converts a list in one C loop; ctypes' (*vals) unpacks it argument by argument)"""
    import array
    a = array.array("I", vals) if len(vals) else array.array("I", [0])
    assert a.itemsize == 4
    return a


def _fr_list(buf: bytes) -> List[int]:
    return [int.from_bytes(buf[i:i + 32], "big") for i in range(0, len(buf), 32)]


def _join(x) -> bytes:
    """a list of per-point byte strings or one contiguous blob"""
    return bytes(x) if isinstance(x, (bytes, bytearray, memoryview)) else b"".join(x)


def _count(x, per: int) -> int:
    return len(x) // per if isinstance(x, (bytes, bytearray, memoryview)) else len(x)


class _DevHandle:
    """Owner of a resident device object (QAP, proving key): freed on close() / garbage collection, and when the
    host object is made resident on another backend."""

    def __init__(self, backend, handle, free_name: str):
        self.backend, self.handle, self._free = backend, handle, getattr(backend.lib, free_name)

    def close(self):
        if getattr(self, "handle", None):
            self._free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _resident_handle(obj, backend, build, free_name: str):
    """obj._dev caches one _DevHandle; a different backend frees the old handle first"""
    dev = getattr(obj, "_dev", None)
    if dev is not None and dev.backend is backend and dev.handle:
        return dev.handle
    if dev is not None:
        dev.close()
    obj._dev = _DevHandle(backend, build(), free_name)
    return obj._dev.handle


def _release(obj):
    """frees the device copy of a QAP / key object (it is rebuilt on the next use)"""
    dev = getattr(obj, "_dev", None)
    if dev is not None:
        dev.close()
        obj._dev = None


class Bases:
    """Device-resident []Commit (the blindedPoint argument of BlindEval)."""

    def __init__(self, backend: "Backend", handle, group: int):
        self.backend, self.handle, self.group = backend, handle, group

    def __len__(self):
        return self.backend.lib.ps_bases_len(self.handle)

    def export(self, first=0, count=None, fmt=L.PS_FMT_COMPRESSED, blob: bool = False):
        n = len(self) - first if count is None else count
        per = {(1, 0): 48, (1, 1): 96, (2, 0): 96, (2, 1): 192}[(self.group, fmt)]
        buf = C.create_string_buffer(max(1, n * per))
        self.backend._check(self.backend.lib.ps_bases_export(self.backend.ctx, self.handle, first, n, fmt, buf))
        raw = buf.raw[:n * per]
        return raw if blob else [raw[i * per:(i + 1) * per] for i in range(n)]

    def close(self):
        if self.handle:
            self.backend.lib.ps_bases_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Backend:
    """One context per process and GPU (ps_ctx)."""

    multi = False

    def __init__(self, device: int = 0, lib=None):
        self.lib = lib if lib is not None else L.load()
        ctx = C.c_void_p()
        self._check(self.lib.ps_ctx_create(device, C.byref(ctx)))
        self.ctx = ctx
        self.device = device

    def _check(self, status):
        L.check(self.lib, status)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.ps_ctx_destroy(self.ctx)
            self.ctx = None

    def set_option(self, name: str, value: int):
        self._check(self.lib.ps_ctx_set_option(self.ctx, name.encode(), value))

    def sync(self):
        self._check(self.lib.ps_ctx_sync(self.ctx))

    def set_stream(self, cuda_stream_ptr: int):
        self._check(self.lib.ps_ctx_set_stream(self.ctx, C.c_void_p(cuda_stream_ptr)))

    def launch_count(self) -> int:
        return int(self.lib.ps_launch_count())

    # ---- bases / MSM ----
    def load_bases(self, group: int, points, fmt: int = L.PS_FMT_COMPRESSED, window_bits: int = 0, tables: int = 1) -> Bases:
        per = {(1, 0): 48, (1, 1): 96, (2, 0): 96, (2, 1): 192}[(group, fmt)]
        buf = points if isinstance(points, (bytes, bytearray)) else b"".join(points)
        assert len(buf) % per == 0
        h = C.c_void_p()
        self._check(self.lib.ps_bases_load(self.ctx, group, bytes(buf), len(buf) // per, fmt, window_bits, tables, C.byref(h)))
        return Bases(self, h, group)

    def bases_from_scalars(self, group: int, scalars, window_bits: int = 0, tables: int = 1) -> Bases:
        buf = scalars if isinstance(scalars, (bytes, bytearray)) else _fr_bytes(scalars)
        h = C.c_void_p()
        self._check(self.lib.ps_bases_from_scalars(self.ctx, group, bytes(buf), len(buf) // 32, window_bits, tables, C.byref(h)))
        return Bases(self, h, group)

    def msm(self, bases: Bases, scalars) -> bytes:
        buf = scalars if isinstance(scalars, (bytes, bytearray)) else _fr_bytes(scalars)
        n = len(buf) // 32
        out = C.create_string_buffer(48 if bases.group == L.PS_G1 else 96)
        st = self.lib.ps_msm(self.ctx, bases.handle, bytes(buf), n, out)
        if st == L.PS_ERR_LENGTH:
            raise ValueError("mismatch of length between poly %d and blinded eval points %d" % (n, len(bases)))
        self._check(st)
        return out.raw

    def msm_rows(self, bases: Bases, scalars, rows: int) -> List[bytes]:
        """`rows` MSMs against the same bases in one call (ps_msm_rows): `scalars` = rows x len(bases) values, row-major
        (a flat list, a list of rows, or wire bytes); returns one compressed point per row."""
        if not isinstance(scalars, (bytes, bytearray)) and len(scalars) and isinstance(scalars[0], (list, tuple)):
            scalars = [v for row in scalars for v in row]
        buf = scalars if isinstance(scalars, (bytes, bytearray)) else _fr_bytes(scalars)
        if rows < 0 or (rows and len(buf) % (32 * rows)):
            raise ValueError("scalars do not split into %d rows" % rows)
        n = len(buf) // 32 // rows if rows else len(bases)
        per = 48 if bases.group == L.PS_G1 else 96
        out = C.create_string_buffer(max(1, rows * per))
        st = self.lib.ps_msm_rows(self.ctx, bases.handle, bytes(buf) or None, n, rows, out)
        if st == L.PS_ERR_LENGTH:
            raise ValueError("mismatch of length between poly %d and blinded eval points %d" % (n, len(bases)))
        self._check(st)
        return [out.raw[k * per:(k + 1) * per] for k in range(rows)]

    def prove_timing(self):
        t = (C.c_float * 6)()
        self._check(self.lib.ps_last_prove_timing(self.ctx, t))
        return {"quotient_ms": t[0], "msm_a_ms": t[1], "msm_c_ms": t[2], "encode_g1_ms": t[3], "wait_g2_ms": t[4], "total_ms": t[5]}

    def msm_timing(self):
        t = (C.c_float * 5)()
        self._check(self.lib.ps_last_msm_timing(self.ctx, t))
        return {"sort_ms": t[0], "accumulate_ms": t[1], "combine_ms": t[2], "reduce_ms": t[3], "total_ms": t[4]}

    # ---- NTT ----
    def ntt(self, values: Sequence[int], inverse: bool = False, coset: Optional[int] = None) -> List[int]:
        n = len(values)
        log_n = n.bit_length() - 1
        if n != 1 << log_n:
            raise ValueError("NTT size must be a power of two")
        buf = C.create_string_buffer(_fr_bytes(values), n * 32)
        cz = None if coset is None else (coset % R).to_bytes(32, "big")
        self._check(self.lib.ps_ntt_fr(self.ctx, buf, log_n, 1 if inverse else 0, cz))
        return _fr_list(buf.raw)


class MultiBases:
    """[]Commit sharded by point range over the devices of a MultiBackend"""

    def __init__(self, backend, handle, group):
        self.backend, self.handle, self.group = backend, handle, group

    def __len__(self):
        return self.backend.lib.ps_mbases_len(self.handle)

    def close(self):
        if self.handle:
            self.backend.lib.ps_mbases_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiBackend:
    """Several GPUs of one box behind one handle (ps_mctx): Groth16Prove(tr, q, sol, backend=MultiBackend([0..7]))
    is ONE library call; keys are sharded over the devices, the sparse QAP is replicated."""
    multi = True

    def __init__(self, devices: Sequence[int], lib=None):
        self.lib = lib if lib is not None else L.load()
        devs = (C.c_int * len(devices))(*devices)
        ctx = C.c_void_p()
        L.check(self.lib, self.lib.ps_mctx_create(devs, len(devices), C.byref(ctx)))
        self.ctx = ctx
        self.devices = list(devices)

    def _check(self, status):
        L.check(self.lib, status)

    def __len__(self):
        return len(self.devices)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.ps_mctx_destroy(self.ctx)
            self.ctx = None

    def set_option(self, name: str, value: int):
        self._check(self.lib.ps_mctx_set_option(self.ctx, name.encode(), value))

    def launch_count(self) -> int:
        return int(self.lib.ps_launch_count())

    def bases_from_scalars(self, group: int, scalars, window_bits: int = 0, tables: int = 1) -> MultiBases:
        buf = scalars if isinstance(scalars, (bytes, bytearray)) else _fr_bytes(scalars)
        h = C.c_void_p()
        self._check(self.lib.ps_mbases_from_scalars(self.ctx, group, bytes(buf), len(buf) // 32, window_bits, tables, C.byref(h)))
        return MultiBases(self, h, group)

    def load_bases(self, group: int, points, fmt: int = L.PS_FMT_COMPRESSED, window_bits: int = 0, tables: int = 1) -> MultiBases:
        per = {(1, 0): 48, (1, 1): 96, (2, 0): 96, (2, 1): 192}[(group, fmt)]
        buf = points if isinstance(points, (bytes, bytearray)) else b"".join(points)
        h = C.c_void_p()
        self._check(self.lib.ps_mbases_load(self.ctx, group, bytes(buf), len(buf) // per, fmt, window_bits, tables, C.byref(h)))
        return MultiBases(self, h, group)

    def msm(self, bases: MultiBases, scalars) -> bytes:
        buf = scalars if isinstance(scalars, (bytes, bytearray)) else _fr_bytes(scalars)
        n = len(buf) // 32 if not isinstance(buf, C.c_void_p) else len(scalars)
        out = C.create_string_buffer(48 if bases.group == L.PS_G1 else 96)
        st = self.lib.ps_mmsm(self.ctx, bases.handle, buf if isinstance(buf, C.c_void_p) else bytes(buf), n, out)
        if st == L.PS_ERR_LENGTH:
            raise ValueError("mismatch of length between poly %d and blinded eval points %d" % (n, len(bases)))
        self._check(st)
        return out.raw

    def timeline(self, dev: int = 0):
        """stage marks (ms since the start) of the last Groth16 proof on device `dev`"""
        buf = (C.c_float * 16)()
        cnt = C.c_int()
        self._check(self.lib.ps_mg16_last_timeline(self.ctx, dev, buf, 16, C.byref(cnt)))
        return [buf[i] for i in range(cnt.value)]


_default: Optional[Backend] = None


def default_backend() -> Backend:
    global _default
    if _default is None:
        _default = Backend(0)
    return _default


def set_default_backend(b: Optional[Backend]):
    global _default
    _default = b


def BlindEval(p: Poly, blinded: Bases, backend: Optional[Backend] = None) -> bytes:
    """Poly.BlindEval (algebra.go:348-359) against a resident base set."""
    return (backend or blinded.backend).msm(blinded, p)


# ---- R1CS / QAP types (r1cs.go:81-102, qap.go:10-27) ------------------------------------------------
class R1CS:
    """r1cs.go:81-174: gate matrices left / right / out (rows = gates, columns = variables) over the
    variable order [const, inputs..., outputs..., intermediates...] (mergeVars, r1cs.go:132-144).
    Host-side bookkeeping only; rows are kept sparse ({column: value})."""

    def __init__(self):
        self.inputs: List[str] = []
        self.outputs: List[str] = []
        self.intermediates: List[str] = []
        self._gates = []   # (left names->coef, right ..., out ...) by variable NAME, resolved in rows()

    @property
    def vars(self) -> List[str]:
        return ["const"] + self.inputs + self.outputs + self.intermediates

    def nbIO(self) -> int:                      # r1cs.go:108-110
        return 1 + len(self.inputs) + len(self.outputs)

    def NewInput(self, name: str): self.inputs.append(name)          # r1cs.go:112-115
    def NewOutput(self, name: str): self.outputs.append(name)        # r1cs.go:117-120
    def NewVar(self, name: str): self.intermediates.append(name)     # r1cs.go:122-125

    def IndexOf(self, name: str) -> int:                             # r1cs.go:21-28
        try:
            return self.vars.index(name)
        except ValueError:
            raise KeyError("plouf")

    def Mul(self, left: str, right: str, out: str):                  # r1cs.go:148-152
        self._gates.append(({left: 1}, {right: 1}, {out: 1}))

    def Add(self, var1: str, var2: str, out: str):                   # r1cs.go:156-164
        self._gates.append(({var1: 1, var2: 1}, {"const": 1}, {out: 1}))   # ConstraintOn marks 0/1 per name

    def AddConst(self, var1: str, add: int, out: str):               # r1cs.go:168-174
        row = {"const": 1, var1: 1}
        row["const"] = row["const"] * add
        self._gates.append((row, {"const": 1}, {out: 1}))

    def rows(self):
        """the three matrices as lists of {column index: Go int}"""
        idx = {n: i for i, n in enumerate(self.vars)}
        for names in self._gates:
            for d in names:
                for n in d:
                    if n not in idx:
                        raise KeyError("plouf")
        conv = lambda k: [{idx[n]: v for n, v in g[k].items() if v} for g in self._gates]
        return conv(0), conv(1), conv(2)


def ToQAP(circuit: R1CS) -> "SparseQAP":
    """ToQAP, qap.go:35-65.  The per-variable polynomials are not materialised (that costs O(m n^3)
    field operations and 3*m*n*32 bytes in the reference): the result keeps the gate matrices in CSR
    form and the device interpolates on {1..n} when proving.  Any nbGates >= 2 (the interpolation tree is built over
    the next power of two with dummy leaves, csrc/interp.cuh)."""
    left, right, out = circuit.rows()
    n = len(left)
    if n < 2:
        raise ValueError("a QAP needs at least two gates (got %d)" % n)

    def csr(m):
        rp, col, val = [0], [], []
        for row in m:
            for j in sorted(row):
                col.append(j); val.append(int(row[j]) % R)
            rp.append(len(col))
        return rp, col, val

    return SparseQAP(len(circuit.vars), circuit.nbIO(), n, csr(left), csr(right), csr(out))


@dataclass
class QAP:
    """qap.go:10-27: left/right/out are nbVars polynomials of nbGates coefficients (low degree
    first); z has nbGates+1."""
    nbVars: int
    nbIO: int
    nbGates: int
    left: List[Poly]
    right: List[Poly]
    out: List[Poly]
    z: Poly
    _dev: object = None

    def _resident(self, backend: Backend):
        def build():
            n, m = self.nbGates, self.nbVars
            if len(self.left) != m or len(self.right) != m or len(self.out) != m:
                raise ValueError("different number of solution variables than polynomials")
            for polys in (self.left, self.right, self.out):
                for p in polys:
                    if len(p) != n:
                        raise ValueError("QAP polynomial with %d coefficients, expected %d" % (len(p), n))
            if len(self.z) != n + 1:
                raise ValueError("z must have nbGates+1 coefficients")
            h = C.c_void_p()
            flat = lambda polys: b"".join(_fr_bytes(p) for p in polys)
            load = backend.lib.ps_mqap_load_dense if backend.multi else backend.lib.ps_qap_load_dense
            backend._check(load(backend.ctx, n, m, self.nbIO, flat(self.left), flat(self.right), flat(self.out), _fr_bytes(self.z),
                                C.byref(h)))
            return h
        return _resident_handle(self, backend, build, "ps_mqap_free" if backend.multi else "ps_qap_free")

    def close(self):
        _release(self)

    def Quotient(self, sol: Vector, backend: Optional[Backend] = None) -> Poly:
        return Quotient(self, sol, backend)


@dataclass
class SparseQAP:
    """The same object as QAP for circuits whose dense polynomials cannot be materialised
    (3*nbVars*nbGates*32 bytes): the R1CS gate matrices in CSR form (r1cs.go:96-101 holds them
    dense); the per-variable polynomials stay implicit as interpolants on {1..nbGates}
    (qap.go:67-93).  Any nbGates >= 2.  Each matrix is (row_ptr, col, val) with val as Fr integers."""
    nbVars: int
    nbIO: int
    nbGates: int
    left: tuple
    right: tuple
    out: tuple
    _dev: object = None

    @staticmethod
    def from_dense_rows(nbVars, nbIO, left, right, out):
        """rows of Go ints (Matrix, algebra.go:15) -> CSR; Value.ToFieldElement on the entries"""
        def csr(m):
            rp, col, val = [0], [], []
            for row in m:
                for j, v in enumerate(row):
                    if v:
                        col.append(j); val.append(int(v) % R)
                rp.append(len(col))
            return rp, col, val
        return SparseQAP(nbVars, nbIO, len(left), csr(left), csr(right), csr(out))

    def _resident(self, backend: Backend):
        def build():
            h = C.c_void_p()
            keep, args = [], []
            for rp, col, val in (self.left, self.right, self.out):
                if len(rp) != self.nbGates + 1:
                    raise ValueError("row_ptr must have nbGates+1 entries")
                a_rp, a_col = _u32_array(rp), _u32_array(col)
                b_val = _fr_bytes(val) or b"\0"
                keep += [a_rp, a_col, b_val]
                args += [C.c_void_p(a_rp.buffer_info()[0]), C.c_void_p(a_col.buffer_info()[0]), C.cast(C.c_char_p(b_val), C.c_void_p)]
            load = backend.lib.ps_mqap_load_r1cs if backend.multi else backend.lib.ps_qap_load_r1cs
            backend._check(load(backend.ctx, self.nbGates, self.nbVars, self.nbIO, *args, C.byref(h)))
            return h
        return _resident_handle(self, backend, build, "ps_mqap_free" if backend.multi else "ps_qap_free")

    def close(self):
        _release(self)

    def Quotient(self, sol: Vector, backend: Optional[Backend] = None) -> Poly:
        return Quotient(self, sol, backend)


def _sanity(q, sol):
    """QAP.sanityCheck, qap.go:177-189."""
    nsol = len(sol) // 32 if isinstance(sol, (bytes, bytearray, memoryview)) else len(sol)
    if nsol != q.nbVars:
        raise ValueError("different number of solution variables than left polynomials")


def Quotient(q: QAP, sol: Vector, backend: Optional[Backend] = None, return_abc: bool = False):
    """QAP.Quotient, qap.go:151-162."""
    b = backend or default_backend()
    _sanity(q, sol)
    h = q._resident(b)
    n = q.nbGates
    out = C.create_string_buffer(max(1, (n - 1) * 32))
    abc = C.create_string_buffer(3 * n * 32) if return_abc else None
    st = b.lib.ps_quotient(b.ctx, h, _fr_bytes(sol), out, abc)
    if st == L.PS_ERR_REMAINDER:
        raise ArithmeticError("apocalypse")
    b._check(st)
    hx = _fr_list(out.raw[:(n - 1) * 32])
    if return_abc:
        v = _fr_list(abc.raw)
        return hx, (v[:n], v[n:2 * n], v[2 * n:])
    return hx


# ---- Groth16 (groth16.go:30-61, 106-118) --------------------------------------------------------------
@dataclass
class Groth16Setup:
    """Prover-side fields of Groth16Setup; points as MarshalBinary bytes."""
    Alpha: bytes
    Beta: bytes
    Delta: bytes
    Xi: List[bytes]
    NioLP: List[bytes]
    XiT: List[bytes]
    Beta2: bytes
    Delta2: bytes
    Xi2: List[bytes]
    IoLP: List[bytes] = field(default_factory=list)   # verifier side, carried for completeness
    Gamma: bytes = b""
    fmt: int = L.PS_FMT_COMPRESSED    # PS_FMT_AFFINE for bulk keys (every point field then uncompressed)
    tw: Optional[dict] = None         # toxic waste, kept like the reference's Groth16Setup.tw (testing)
    _dev: object = None

    def _resident(self, backend: Backend):
        def build():
            g1b, g2b = (48, 96) if self.fmt == L.PS_FMT_COMPRESSED else (96, 192)
            n = _count(self.Xi, g1b)
            if _count(self.Xi2, g2b) != n or _count(self.XiT, g1b) != n - 1:
                raise ValueError("mismatch of length between poly and blinded eval points")
            h = C.c_void_p()
            j = _join
            load = backend.lib.ps_mg16_key_load if backend.multi else backend.lib.ps_g16_key_load
            backend._check(load(
                backend.ctx, n, _count(self.NioLP, g1b), self.fmt, j(self.Xi), j(self.Xi2), j(self.XiT), j(self.NioLP) or b"\0",
                self.Alpha, self.Beta, self.Delta, self.Beta2, self.Delta2, C.byref(h)))
            return h
        return _resident_handle(self, backend, build, "ps_mg16_key_free" if backend.multi else "ps_g16_key_free")

    def close(self):
        _release(self)


def NewGroth16TrustedSetup(qap, backend: Optional[Backend] = None, toxic=None, fmt: int = L.PS_FMT_AFFINE,
                           export: bool = True) -> "Groth16Setup":
    """NewGroth16TrustedSetup, groth16.go:64-101, computed on the device (ps_g16_setup).  `toxic` = (alpha, beta,
    delta, x, gamma); fresh randomness when omitted, kept in the result's `tw` like the reference's Groth16Setup.tw.
    The proving key stays resident on `backend`; with `export` the struct's point fields are filled as well
    (uncompressed blobs by default: they are what a key file or another backend would be loaded from)."""
    b = backend or default_backend()
    if toxic is None:
        toxic = tuple(secrets.randbelow(R - 1) + 1 for _ in range(5))
    qh = qap._resident(b)
    n, m, nio = qap.nbGates, qap.nbVars, qap.nbIO
    diff = m - nio
    kh = C.c_void_p()
    iolp = C.create_string_buffer(max(1, diff * 48))
    gamma = C.create_string_buffer(96)
    b._check(b.lib.ps_g16_setup(b.ctx, qh, _fr_bytes(list(toxic)), C.byref(kh), iolp, gamma))
    iolp_raw = iolp.raw          # ONE copy of the buffer (ctypes' .raw copies on every access)
    tr = Groth16Setup(Alpha=b"", Beta=b"", Delta=b"", Xi=b"", NioLP=b"", XiT=b"", Beta2=b"", Delta2=b"", Xi2=b"",
                      IoLP=[iolp_raw[i * 48:(i + 1) * 48] for i in range(diff)], Gamma=gamma.raw, fmt=fmt)
    tr.tw = dict(zip(("Alpha", "Beta", "Delta", "X", "Gamma"), toxic))
    tr._dev = _DevHandle(b, kh, "ps_g16_key_free")
    if export:
        g1b, g2b = (48, 96) if fmt == L.PS_FMT_COMPRESSED else (96, 192)
        bufs = {"xi": n * g1b, "xi2": n * g2b, "xit": (n - 1) * g1b, "niolp": nio * g1b, "alpha": g1b, "beta": g1b, "delta": g1b,
                "beta2": g2b, "delta2": g2b}
        cb = {k: C.create_string_buffer(max(1, v)) for k, v in bufs.items()}
        b._check(b.lib.ps_g16_key_export(b.ctx, kh, fmt, *[cb[k] for k in ("xi", "xi2", "xit", "niolp", "alpha", "beta", "delta",
                                                                            "beta2", "delta2")]))
        raw = {k: cb[k].raw[:bufs[k]] for k in bufs}
        tr.Xi, tr.Xi2, tr.XiT, tr.NioLP = raw["xi"], raw["xi2"], raw["xit"], raw["niolp"]
        tr.Alpha, tr.Beta, tr.Delta, tr.Beta2, tr.Delta2 = raw["alpha"], raw["beta"], raw["delta"], raw["beta2"], raw["delta2"]
    return tr


@dataclass
class Groth16ToxicProof:
    R: int
    S: int


@dataclass
class Groth16Proof:
    tp: Groth16ToxicProof
    A: bytes
    B: bytes
    C: bytes
    h: Optional[Poly] = None


def Groth16Prove(tr: Groth16Setup, q: QAP, sol: Vector, r: Optional[int] = None, s: Optional[int] = None,
                 backend: Optional[Backend] = None, want_h: bool = False) -> Groth16Proof:
    """Groth16Prove, groth16.go:122-211.  r, s default to fresh randomness (groth16.go:148,158) and
    are kept in the proof's tp like the reference; tests inject them."""
    b = backend or default_backend()
    _sanity(q, sol)
    if r is None:
        r = secrets.randbelow(R - 1) + 1
    if s is None:
        s = secrets.randbelow(R - 1) + 1
    kh, qh = tr._resident(b), q._resident(b)
    A, Bp, Cp = C.create_string_buffer(48), C.create_string_buffer(96), C.create_string_buffer(48)
    hb = C.create_string_buffer(max(1, (q.nbGates - 1) * 32)) if want_h else None
    if b.multi:
        if want_h:
            raise ValueError("want_h is a single-device debugging output")
        st = b.lib.ps_mg16_prove(b.ctx, kh, qh, _fr_bytes(sol), _fr_bytes([r]), _fr_bytes([s]), A, Bp, Cp)
    else:
        st = b.lib.ps_g16_prove(b.ctx, kh, qh, _fr_bytes(sol), _fr_bytes([r]), _fr_bytes([s]), A, Bp, Cp, hb)
    if st == L.PS_ERR_REMAINDER:
        raise ArithmeticError("apocalypse")
    if st == L.PS_ERR_LENGTH:
        raise ValueError("mismatch of length between poly and blinded eval points")
    b._check(st)
    return Groth16Proof(Groth16ToxicProof(r, s), A.raw, Bp.raw, Cp.raw,
                        _fr_list(hb.raw[:(q.nbGates - 1) * 32]) if want_h else None)


# ---- PHGR13 (pinochio.go:37-62, 180-203) -----------------------------------------------------------------
@dataclass
class PHGR13EvalKey:
    vs: List[bytes]
    ws: List[bytes]   # G2
    ys: List[bytes]
    vas: List[bytes]
    was: List[bytes]
    yas: List[bytes]
    gsi: List[bytes]
    vbs: List[bytes]
    wbs: List[bytes]  # typed []G2 in the reference but holds G1 points (pinochio.go:114,136)
    ybs: List[bytes]
    _dev: object = None

    def _resident(self, backend: Backend):
        def build():
            h = C.c_void_p()
            j = b"".join
            backend._check(backend.lib.ps_phgr13_key_load(
                backend.ctx, len(self.gsi) + 1, len(self.vs), L.PS_FMT_COMPRESSED, j(self.gsi), j(self.vs), j(self.ws),
                j(self.ys), j(self.vas), j(self.was), j(self.yas), j(self.vbs), j(self.wbs), j(self.ybs), C.byref(h)))
            return h
        return _resident_handle(self, backend, build, "ps_phgr13_key_free")

    def export(self):
        """fills the byte fields from the resident key (after NewPHGR13TrustedSetup)"""
        dev = self._dev
        n, nmid = self._shape
        b = dev.backend
        names = ("gsi", "vs", "ws", "ys", "vas", "was", "yas", "vbs", "wbs", "ybs")
        sizes = {k: (n - 1 if k == "gsi" else nmid) * (96 if k == "ws" else 48) for k in names}
        cb = {k: C.create_string_buffer(max(1, sizes[k])) for k in names}
        b._check(b.lib.ps_phgr13_key_export(b.ctx, dev.handle, L.PS_FMT_COMPRESSED, *[cb[k] for k in names]))
        for k in names:
            per = 96 if k == "ws" else 48
            raw = cb[k].raw[:sizes[k]]
            setattr(self, k, [raw[i:i + per] for i in range(0, len(raw), per)])
        return self

    def close(self):
        _release(self)


def NewPHGR13TrustedSetup(qap, backend: Optional[Backend] = None, toxic=None, with_vk: bool = False):
    """NewPHGR13TrustedSetup, pinochio.go:93-176, on the device (ps_phgr13_setup).  `toxic` = (s, av, aw, ay, rv, rw,
    beta, gamma) in the reference's sampling order.  Returns (PHGR13EvalKey resident on `backend`, vk dict or None,
    toxic); the evaluation key's byte fields are filled on demand by PHGR13EvalKey.export()."""
    b = backend or default_backend()
    if toxic is None:
        toxic = tuple(secrets.randbelow(R - 1) + 1 for _ in range(8))
    qh = qap._resident(b)
    m = qap.nbVars
    kh = C.c_void_p()
    fixed = C.create_string_buffer(576) if with_vk else None
    vs = C.create_string_buffer(m * 48) if with_vk else None
    ws = C.create_string_buffer(m * 96) if with_vk else None
    ys = C.create_string_buffer(m * 48) if with_vk else None
    b._check(b.lib.ps_phgr13_setup(b.ctx, qh, _fr_bytes(list(toxic)), C.byref(kh), fixed, vs, ws, ys))
    ek = PHGR13EvalKey(vs=[], ws=[], ys=[], vas=[], was=[], yas=[], gsi=[], vbs=[], wbs=[], ybs=[])
    ek._shape = (qap.nbGates, qap.nbIO)
    ek._dev = _DevHandle(b, kh, "ps_phgr13_key_free")
    vk = None
    if with_vk:
        f = fixed.raw
        cut = lambda raw, per: [raw[i:i + per] for i in range(0, len(raw), per)]
        vk = {"av": f[0:96], "aw": f[96:144], "ay": f[144:240], "gamma": f[240:336], "bgamma": f[336:384], "bgamma2": f[384:480],
              "yts": f[480:576], "vs": cut(vs.raw, 48), "ws": cut(ws.raw, 96), "ys": cut(ys.raw, 48)}
    return ek, vk, toxic


@dataclass
class PHGR13Proof:
    vss: bytes
    vass: bytes
    wss: bytes
    wass: bytes
    yss: bytes
    yass: bytes
    hs: bytes
    gz: bytes
    h: Optional[Poly] = None


def PHGR13Prove(ek: PHGR13EvalKey, qap: QAP, solution: Vector, backend: Optional[Backend] = None,
                want_h: bool = False) -> PHGR13Proof:
    """PHGR13Prove, pinochio.go:207-254."""
    b = backend or default_backend()
    _sanity(qap, solution)
    kh, qh = ek._resident(b), qap._resident(b)
    out = C.create_string_buffer(432)
    hb = C.create_string_buffer(max(1, (qap.nbGates - 1) * 32)) if want_h else None
    st = b.lib.ps_phgr13_prove(b.ctx, kh, qh, _fr_bytes(solution), out, hb)
    if st == L.PS_ERR_REMAINDER:
        raise ArithmeticError("apocalypse")
    if st == L.PS_ERR_LENGTH:
        raise ValueError("mismatch of length between poly and blinded eval points")
    b._check(st)
    o = out.raw
    g1 = [o[i * 48:(i + 1) * 48] for i in range(7)]  # hs vss yss vass wass yass gz
    return PHGR13Proof(hs=g1[0], vss=g1[1], yss=g1[2], vass=g1[3], wass=g1[4], yass=g1[5], gz=g1[6], wss=o[336:432],
                       h=_fr_list(hb.raw[:(qap.nbGates - 1) * 32]) if want_h else None)


# ---- verifiers (SURVEY 8 f4): pairing-product checks on the device --------------------------------------------
def PairingCheckBatch(g1_points: Sequence[bytes], g2_points: Sequence[bytes], counts: Sequence[int],
                      backend: Optional[Backend] = None) -> List[bool]:
    """For every check t: prod over its counts[t] consecutive pairs of e(P_i, Q_i) == 1 (compressed points).  What the
    reference's `Pair(...)` / `Equal` comparisons (curve.go:36-38) decide, with one side's G1 points negated."""
    b = backend or default_backend()
    if len(g1_points) != len(g2_points) or sum(counts) != len(g1_points):
        raise ValueError("pairs and counts disagree")
    ok = C.create_string_buffer(max(1, len(counts)))
    cnt = (C.c_uint32 * max(1, len(counts)))(*counts)
    b._check(b.lib.ps_pairing_check_batch(b.ctx, b"".join(g1_points), b"".join(g2_points), cnt, len(counts), L.PS_FMT_COMPRESSED, ok))
    return [ok.raw[i] == 1 for i in range(len(counts))]


def Groth16Verify(tr: Groth16Setup, q, p: "Groth16Proof", io: Vector, backend: Optional[Backend] = None) -> bool:
    """Groth16Verify, groth16.go:214-233.  `tr` needs its verifier side: Alpha, Beta2, Delta2 (compressed), IoLP and Gamma
    (always compressed; NewGroth16TrustedSetup fills them).  `io` = the public part of the solution, one per IoLP."""
    b = backend or default_backend()
    if tr.fmt != L.PS_FMT_COMPRESSED:
        raise ValueError("Groth16Verify takes the setup's points in compressed form (fmt = PS_FMT_COMPRESSED)")
    n_io = len(tr.IoLP)
    if len(io) < n_io:
        raise ValueError("different number of public inputs than IoLP elements")
    ok = C.c_int(0)
    b._check(b.lib.ps_g16_verify(b.ctx, _join(tr.Alpha), _join(tr.Beta2), tr.Gamma, _join(tr.Delta2), b"".join(tr.IoLP) or b"\0", n_io,
                                 _fr_bytes(list(io[:n_io])) or b"\0", p.A, p.B, p.C, C.byref(ok)))
    return ok.value == 1


def Groth16VerifyBatch(tr: Groth16Setup, q, proofs: Sequence["Groth16Proof"], ios, backend: Optional[Backend] = None,
                       weights: Optional[Sequence[int]] = None, per_proof: bool = False):
    """Groth16Verify for many proofs against one key, decided as ONE combined pairing-product check with random 128-bit
    weights (ps_g16_verify_batch).  `ios` = one public-input vector per proof (each at least as long as IoLP, like
    Groth16Verify's `io`), or one wire-format blob / HostBuffer of len(proofs) x len(IoLP) values, proof-major.
    `weights` (tests only) = one nonzero integer below 2^128 per proof; by default the library draws them from the
    operating system.  Returns True iff every proof verifies; with per_proof=True a list with one verdict per proof.
    A proof whose points do not decode, or lie outside the prime-order subgroup, is simply invalid."""
    b = backend or default_backend()
    if tr.fmt != L.PS_FMT_COMPRESSED:
        raise ValueError("Groth16VerifyBatch takes the setup's points in compressed form (fmt = PS_FMT_COMPRESSED)")
    n_io, n = len(tr.IoLP), len(proofs)
    if isinstance(ios, (HostBuffer, bytes, bytearray, memoryview)):
        nbytes = ios.nbytes if isinstance(ios, HostBuffer) else len(ios)
        if nbytes != n * n_io * 32:
            raise ValueError("different number of public inputs than IoLP elements")
        io_arg = _fr_bytes(ios)
    else:
        if len(ios) != n:
            raise ValueError("different number of proofs than public input vectors")
        for io in ios:
            if len(io) < n_io:
                raise ValueError("different number of public inputs than IoLP elements")
        io_arg = b"".join(_fr_bytes(list(io[:n_io])) for io in ios)
    w_arg = None
    if weights is not None:
        if len(weights) != n:
            raise ValueError("one weight per proof")
        if any(not 0 < int(w) < 1 << 128 for w in weights):
            raise ValueError("weights must be nonzero 128-bit integers")
        w_arg = b"".join(int(w).to_bytes(16, "big") for w in weights)
    ok = C.c_int(0)
    verdicts = C.create_string_buffer(max(1, n)) if per_proof else None
    st = b.lib.ps_g16_verify_batch(b.ctx, _join(tr.Alpha), _join(tr.Beta2), tr.Gamma, _join(tr.Delta2), b"".join(tr.IoLP) or b"\0",
                                   n_io, n, io_arg or None, b"".join(p.A for p in proofs) or None,
                                   b"".join(p.B for p in proofs) or None, b"".join(p.C for p in proofs) or None, w_arg,
                                   C.byref(ok), verdicts)
    if st == L.PS_ERR_ARG and weights is not None:
        raise ValueError("weights must be nonzero 128-bit integers")
    b._check(st)
    if per_proof:
        return [verdicts.raw[i] == 1 for i in range(n)]
    return ok.value == 1


def PHGR13Verify(vk: dict, qap, p: PHGR13Proof, io: Vector, backend: Optional[Backend] = None) -> bool:
    """PHGR13Verify, pinochio.go:281-375.  `vk` = the dict NewPHGR13TrustedSetup(..., with_vk=True) returns (av, aw, ay,
    gamma, bgamma, bgamma2, yts and the per-variable commitments vs / ws / ys); `io` = the first nbVars - nbIO values of
    the solution (the public ones in this reference's numbering)."""
    b = backend or default_backend()
    diff = qap.nbVars - qap.nbIO
    if len(io) < diff:
        raise ValueError("different number of public inputs than verification-key elements")
    fixed = vk["av"] + vk["aw"] + vk["ay"] + vk["gamma"] + vk["bgamma"] + vk["bgamma2"] + vk["yts"]
    proof = p.hs + p.vss + p.yss + p.vass + p.wass + p.yass + p.gz + p.wss
    ok = C.c_int(0)
    j = lambda xs: b"".join(xs[:diff]) or b"\0"
    b._check(b.lib.ps_phgr13_verify(b.ctx, fixed, j(vk["vs"]), j(vk["ws"]), j(vk["ys"]), diff, _fr_bytes(list(io[:diff])) or b"\0",
                                    proof, C.byref(ok)))
    return ok.value == 1


def PHGR13VerifyBatch(vk: dict, qap, proofs: Sequence[PHGR13Proof], ios, backend: Optional[Backend] = None,
                      weights=None, per_proof: bool = False):
    """PHGR13Verify for many proofs against one key, decided as ONE combined pairing-product check with five random
    128-bit weights per proof, one per equation (ps_phgr13_verify_batch).  `vk` as PHGR13Verify's; `ios` = one
    public-input vector per proof (each at least nbVars - nbIO long, like PHGR13Verify's `io`), or one wire-format blob /
    HostBuffer of len(proofs) x (nbVars - nbIO) values, proof-major.  `weights` (tests only) = one 5-tuple of nonzero
    integers below 2^128 per proof; by default the library draws them from the operating system.  Returns True iff every
    proof verifies; with per_proof=True a list with one verdict per proof.  A proof whose points do not decode, or lie
    outside the prime-order subgroup, is simply invalid."""
    b = backend or default_backend()
    n_io, n = qap.nbVars - qap.nbIO, len(proofs)
    if isinstance(ios, (HostBuffer, bytes, bytearray, memoryview)):
        nbytes = ios.nbytes if isinstance(ios, HostBuffer) else len(ios)
        if nbytes != n * n_io * 32:
            raise ValueError("different number of public inputs than verification-key elements")
        io_arg = _fr_bytes(ios)
    else:
        if len(ios) != n:
            raise ValueError("different number of proofs than public input vectors")
        for io in ios:
            if len(io) < n_io:
                raise ValueError("different number of public inputs than verification-key elements")
        io_arg = b"".join(_fr_bytes(list(io[:n_io])) for io in ios)
    w_arg = None
    if weights is not None:
        if len(weights) != n or any(len(w) != 5 for w in weights):
            raise ValueError("five weights per proof")
        if any(not 0 < int(x) < 1 << 128 for w in weights for x in w):
            raise ValueError("weights must be nonzero 128-bit integers")
        w_arg = b"".join(int(x).to_bytes(16, "big") for w in weights for x in w)
    fixed = vk["av"] + vk["aw"] + vk["ay"] + vk["gamma"] + vk["bgamma"] + vk["bgamma2"] + vk["yts"]
    blob = b"".join(p.hs + p.vss + p.yss + p.vass + p.wass + p.yass + p.gz + p.wss for p in proofs)
    j = lambda xs: b"".join(xs[:n_io]) or None
    ok = C.c_int(0)
    verdicts = C.create_string_buffer(max(1, n)) if per_proof else None
    st = b.lib.ps_phgr13_verify_batch(b.ctx, fixed, j(vk["vs"]), j(vk["ws"]), j(vk["ys"]), n_io, n, io_arg or None, blob or None,
                                      w_arg, C.byref(ok), verdicts)
    if st == L.PS_ERR_ARG and weights is not None:
        raise ValueError("weights must be nonzero 128-bit integers")
    b._check(st)
    if per_proof:
        return [verdicts.raw[i] == 1 for i in range(n)]
    return ok.value == 1
