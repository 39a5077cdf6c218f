#!/usr/bin/env python3
"""Benchmark of the prover hot path (contract: see the task statement / DESIGN.md section 6).

Headline metric (BASELINE.json): G1 MSM points/s -- the operation that dominates Groth16Prove / PHGR13Prove
(Poly.BlindEval, algebra.go:348-359) -- on synthetic data: bases k_i*G built on the device, scalars uniform
below 2^254 (< r).  One "step" = one MSM over the rank's point range.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--log-n L] [--impl reference] [--dump-outputs DIR]

N = 1: one MSM of 2^L points (default L = 24, configs[3] of BASELINE.json, the size the north-star's roofline
target is quoted on).  N > 1 (torchrun, one rank per GPU): every rank owns its own 2^L-point range (weak
scaling; the MSM shards by point range with no data-path collective), the partial points are all-gathered over
NCCL (192 B per rank) and summed on rank 0.  `value` = points/s with scalars resident in HBM (ps_msm_device);
`e2e` = the same through the reference-facing call with HOST buffers (pinned big-endian scalars in, compressed
point out).  Every timed configuration is first checked against the oracle (`parity`).

Secondary sections of the same JSON line (all of BASELINE.json's configs):
  g2_msm        G2 MSMs (2^20 and 2^22 points per GPU)
  msm_strong    N > 1: a FIXED 2^L-point G1 MSM split over the N ranks (strong scaling, next to the weak headline)
  groth16       full Groth16 prove of a 2^20-constraint sparse circuit: one GPU, or -- N > 1 -- all N GPUs behind ONE
                library call (ps_mg16_prove: key sharded, devices exchanging over NVLink peer memory)
  phgr13        full PHGR13 prove at 2^16 and 2^20 constraints (one GPU)
  small_configs the 2^10 repeated-squaring circuit (Groth16 + PHGR13) and a 2^16 sparse circuit
  cpu_baseline  the reference's algorithms restated in C (oracle/), timed on this box's host cores: BlindEval rate
                and the WHOLE reference flow (ToQAP -> setup -> Groth16Prove) at the sizes where it finishes
`--impl reference` times that CPU restatement of BlindEval on all host threads on a bounded sample.
`--dump-outputs DIR` writes the headline's result from its last timed step to DIR/g1_msm_point.npy: the compressed
point (summed over the ranks with N > 1) as its 48 byte values in float64.  The inputs are seeded, so two builds
run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
METRIC = "g1_msm_points_per_s"
UNIT = "points/s"
IMAD_PER_FP_MUL = 600.0      # 300 32x32->64 MACs as IMAD.LO/IMAD.HI pairs (SURVEY 8 d4)
FP_MUL_PER_MADD = 10.0       # XYZZ mixed addition, 8M + 2S


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


_T0 = time.perf_counter()
_STATE = {"section": "start", "line": None, "printed": False}


def progress(section: str):
    """one stderr line per section (the JSON line is printed once, at the end): where a slow or hung run stopped"""
    _STATE["section"] = section
    print("[bench %7.1fs] %s" % (time.perf_counter() - _T0, section), file=sys.stderr, flush=True)


def start_watchdog(limit_s: float):
    """The driver needs ONE JSON line within minutes.  If a secondary section (after the headline was measured) does
    not finish by `limit_s`, print the line as far as it got -- naming the section -- and leave; before the headline
    exists there is nothing to print and the run fails loudly."""
    def fire():
        import faulthandler
        faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
        line = _STATE["line"]
        if line is not None and not _STATE["printed"]:
            line["watchdog"] = "section %r did not finish within %.0f s; later sections are missing" % (_STATE["section"], limit_s)
            print(json.dumps(line), flush=True)
            os._exit(0)
        if _STATE.get("rank", 0) != 0:
            os._exit(0)
        print("bench.py: watchdog fired in section %r before the headline line existed" % _STATE["section"], file=sys.stderr, flush=True)
        os._exit(4)
    t = threading.Timer(limit_s, fire)
    t.daemon = True
    t.start()
    return t


def random_scalars_be(n: int, seed: int):
    """n uniform 254-bit scalars as big-endian 32-byte rows (numpy uint8 [n, 32])."""
    import numpy as np
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 0] &= 0x3F
    return a


def be_to_le_limbs(a):
    """[n, 32] big-endian bytes -> [n, 8] little-endian uint32 limbs (standard form)."""
    import numpy as np
    return np.ascontiguousarray(a[:, ::-1]).view("<u4").reshape(-1, 8).copy()


def expected_exponent(ks_be, sc_be) -> int:
    """sum_i k_i s_i mod r for the bases k_i*G and scalars s_i (oracle's C dot product; checker, untimed)"""
    from oracle import c_oracle as CO
    return CO.fr_dot(ks_be, sc_be)


def expected_point(group: int, e: int) -> bytes:
    from oracle import ps_oracle as O
    return O.g1_compress(O.g1_mul(e)) if group == 1 else O.g2_compress(O.g2_mul(e))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu_index, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- CPU legs: the reference's algorithms restated in C (oracle/), timed on the host cores -------------------------
def cpu_blind_eval(sample_log_n: int, threads: int, min_seconds: float, max_reps: int):
    """Poly.BlindEval (algebra.go:348-359: one bit-serial scalar multiplication per term) over 2^k points"""
    from oracle import c_oracle as CO, ps_oracle as O
    sample = 1 << sample_log_n
    sc = random_scalars_be(sample, 3)
    p0 = O.g1_mul(0x1234567 | 1)
    pts, acc = [], None
    for _ in range(sample):            # cheap distinct multiples of G (untimed setup)
        acc = O.g1_add(acc, p0)
        pts.append(acc)
    pbytes = b"".join(O.g1_affine_bytes(p) for p in pts)
    sbytes = sc.tobytes()
    CO.blind_eval_g1_mt(pbytes[:96 * 64], sbytes[:32 * 64], threads)
    reps, t0 = 0, time.perf_counter()
    while True:
        CO.blind_eval_g1_mt(pbytes, sbytes, threads)
        reps += 1
        if time.perf_counter() - t0 > min_seconds or reps >= max_reps:
            break
    dt = time.perf_counter() - t0
    return sample * reps / dt, reps, dt


def reference_arm(args):
    """the driver's reference arm: the CPU restatement of the reference's BlindEval on all host threads"""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from oracle import c_oracle as CO
    threads = CO.max_threads()
    sample = 1 << args.ref_log_n
    CO_rate, _, _ = cpu_blind_eval(min(args.ref_log_n, 8), threads, 0.0, 1)     # warm-up (small)
    del CO_rate
    from oracle import ps_oracle as O
    sc = random_scalars_be(sample, 3)
    p0 = O.g1_mul(0x1234567 | 1)
    pts, acc = [], None
    for _ in range(sample):
        acc = O.g1_add(acc, p0)
        pts.append(acc)
    pbytes = b"".join(O.g1_affine_bytes(p) for p in pts)
    sbytes = sc.tobytes()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        CO.blind_eval_g1_mt(pbytes, sbytes, threads)
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "G1 MSM 2^%d points/GPU, random 254-bit scalars" % args.log_n,
                   "sample": "2^%d points per step" % args.ref_log_n},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "Poly.BlindEval (algebra.go:348-359) restated in C (oracle/ps_prover.c), one bit-serial "
                                   "scalar-mul per term, 2^%d of the 2^%d points per step, spread over %d OpenMP threads "
                                   "(%d host cores present; the Go reference itself is single-threaded and cannot be built "
                                   "here: no Go toolchain)" % (args.ref_log_n, args.log_n, threads, os.cpu_count() or 0)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def cpu_groth16_flow(budget_s: float):
    """The WHOLE reference flow restated in C (ToQAP with per-variable Lagrange interpolation, NewGroth16TrustedSetup,
    Groth16Prove with its three sumBlind passes over G1 / G2, Quotient by schoolbook Mul + Div2) on the repeated-squaring
    circuit (config C2's shape), all host threads: end to end while ToQAP finishes, then prove-only with the QAP built
    by the fast path.  Every proof is compared with the Python oracle's closed form at n <= 32."""
    from oracle import c_oracle as CO, expect as E, ps_oracle as O
    threads = CO.max_threads()
    smp = O.Sampler(1)
    tox = [smp.fr() for _ in range(4)]
    r, s = smp.fr(), smp.fr()
    rows = []
    t_start = time.perf_counter()
    for k, fast in ((4, False), (5, False), (6, False), (7, True), (8, True), (9, True)):
        n = 1 << k
        if rows:   # predicted cost of this size from the previous one (prove ~ x4 per doubling, ToQAP ~ x16)
            prev = rows[-1]
            pred = prev["prove_s"] * 4.3 + (0 if fast else prev["to_qap_s"] * 16)
            if time.perf_counter() - t_start + pred > budget_s:
                break
        c, w = E.squaring_chain_r1cs(n, O.R - 1)
        A, B, Cc, h, sec = CO.groth16_flow(c, w, tox, r, s, threads, fast_qap=fast)
        row = {"gates": n, "variables": len(c.vars), "to_qap_s": None if fast else round(sec["to_qap_s"], 4),
               "setup_s": round(sec["setup_s"], 4), "prove_s": round(sec["prove_s"], 4),
               "to_qap": "fast path (untimed)" if fast else "reference algorithm (Interpolate per variable, qap.go:67-93)"}
        rows.append(row)
    return {"kind": "port", "cores": threads, "circuit": "repeated squaring, x0 = -1 (config C2's shape)", "runs": rows,
            "model": "prove ~ 3*m*n bit-serial scalar multiplications (one third in G2) + n^3/2 field operations in Div2; "
                     "ToQAP ~ 3*m*n*(n^2 + 380 n) field multiplications"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--log-n", type=int, default=24)
    ap.add_argument("--ref-log-n", type=int, default=14)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--tables", type=int, default=-1, help="precomputed window tables (-1 = all windows)")
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--g2-log-n", default="20,22", help="also time G2 MSMs of 2^k points per GPU (comma list, '' = skip)")
    ap.add_argument("--no-small-configs", action="store_true", help="skip the 2^10 / 2^16 prove latencies")
    ap.add_argument("--groth16-log-n", type=int, default=20,
                    help="also time a full Groth16 prove on a sparse synthetic circuit of 2^k constraints (0 = skip)")
    ap.add_argument("--phgr13-log-n", default="16,20", help="PHGR13 prove sizes (one GPU; '' = skip)")
    ap.add_argument("--cpu-budget-s", type=float, default=30.0, help="time budget of the CPU Groth16 flow")
    ap.add_argument("--watchdog-s", type=float, default=900.0, help="print the line as far as it got after this many seconds")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline MSM's result of the last timed step to DIR/g1_msm_point.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl != "reference":
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import playsnark_b200 as ps
    from playsnark_b200 import _lib as L

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    _STATE["rank"] = rank
    start_watchdog(args.watchdog_s)
    progress("init (rank %d of %d)" % (rank, world))
    dist = None
    host_group = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")       # host-side barrier for the one-call multi-GPU section
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    be = ps.Backend(local)
    stream = torch.cuda.current_stream()
    be.set_stream(stream.cuda_stream)
    lib = be.lib

    n = 1 << args.log_n
    progress("G1 bases 2^%d" % args.log_n)
    # synthetic inputs: bases k_i*G (fixed-base kernel on the device, untimed), scalars uniform < 2^254
    ks = random_scalars_be(n, 1000 + rank)
    sc_be = random_scalars_be(n, 2000 + rank)
    t0 = time.time()
    bases = be.bases_from_scalars(L.PS_G1, ks.tobytes(), args.window_bits, args.tables)
    be.sync()
    t_bases = time.time() - t0
    d_scalars = torch.from_numpy(be_to_le_limbs(sc_be).view(np.int32)).to(dev)
    h_scalars = torch.from_numpy(sc_be).pin_memory()            # e2e input: pinned host, wire format
    d_part = torch.zeros(192, dtype=torch.uint8, device=dev)
    d_all = torch.zeros(192 * world, dtype=torch.uint8, device=dev)
    d_stage = torch.empty((n, 8), dtype=torch.int32, device=dev) if world > 1 else None
    d_status = torch.zeros(4, dtype=torch.int32, device=dev)
    out = C.create_string_buffer(48)

    def step_resident():
        be._check(lib.ps_msm_device(be.ctx, bases.handle, 0, C.c_void_p(d_scalars.data_ptr()), n, C.c_void_p(d_part.data_ptr())))
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_part)

    def step_e2e():
        if world == 1:
            be._check(lib.ps_msm(be.ctx, bases.handle, C.c_void_p(h_scalars.data_ptr()), n, out))
            return out.raw
        # host scalars (wire format) -> device limbs with the library's own upload kernel -> partial -> gather ->
        # sum on rank 0 -> compressed point on the host.  ps_fr_upload leaves Montgomery limbs: mont = 1 below.
        be._check(lib.ps_fr_upload(be.ctx, C.c_void_p(h_scalars.data_ptr()), n, C.c_void_p(d_stage.data_ptr()),
                                   C.c_void_p(d_status.data_ptr())))
        be._check(lib.ps_msm_device_mont(be.ctx, bases.handle, 0, C.c_void_p(d_stage.data_ptr()), n, C.c_void_p(d_part.data_ptr())))
        dist.all_gather_into_tensor(d_all, d_part)
        if rank == 0:
            be._check(lib.ps_msm_combine(be.ctx, L.PS_G1, C.c_void_p(d_all.data_ptr()), world, out))
        return out.raw

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    progress("G1 warm-up + parity")
    for _ in range(args.warmup):
        step_resident()
    barrier()
    # Correctness gate on the exact configuration that is timed (same bases, scalars, window, scatter path): the
    # rank's partial must equal (sum_i k_i s_i mod r) * G, the exponent-level check of groth16_test.go:32-107.
    # The expectation comes from the oracle (checker only, untimed): a C dot product over Fr and one scalar-mul.
    exp_e = expected_exponent(ks, sc_be)
    be._check(lib.ps_msm_combine(be.ctx, L.PS_G1, C.c_void_p(d_part.data_ptr()), 1, out))
    parity = {"g1_2p%d_resident" % args.log_n: out.raw == expected_point(L.PS_G1, exp_e)}
    barrier()

    # integer-multiply peak measured on this device (MEASURED_PEAKS.json has no integer figure)
    v, ms_ = C.c_double(), C.c_double()
    be._check(lib.ps_bench_intpipe(be.ctx, 0, 2000, C.byref(v), C.byref(ms_)))
    imad_peak = v.value
    be._check(lib.ps_bench_fieldmul(be.ctx, 1, 1000, C.byref(v), C.byref(ms_)))
    fpmul_rate = v.value

    progress("G1 timed region")
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    launches0 = be.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phase = {"sort_ms": 0.0, "accumulate_ms": 0.0, "combine_ms": 0.0, "reduce_ms": 0.0, "total_ms": 0.0}
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = be.launch_count() - launches0
    tm = be.msm_timing()            # phases of the last step (CUDA events on the launching stream)
    for k in phase:
        phase[k] = tm[k]
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        # before the e2e steps, which reuse d_part with several ranks; d_all holds the last step's gathered partials
        be._check(lib.ps_msm_combine(be.ctx, L.PS_G1, C.c_void_p((d_all if world > 1 else d_part).data_ptr()), world, out))
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "g1_msm_point.npy"), np.frombuffer(out.raw, dtype=np.uint8).astype(np.float64))

    # e2e: host buffers in, host bytes out, copies inside the timed region
    progress("G1 e2e")
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world == 1:
        parity["g1_2p%d_e2e" % args.log_n] = res == expected_point(L.PS_G1, exp_e)
    else:
        exps = [None] * world
        dist.all_gather_object(exps, exp_e)
        if rank == 0:
            parity["g1_2p%d_x%d_e2e" % (args.log_n, world)] = res == expected_point(L.PS_G1, sum(exps) % R)

    # strong scaling next to the weak headline: ONE 2^L-point MSM split over the ranks (each rank the first 2^L / N of
    # its points, base set loaded with the window sized for that share), partials all-gathered, summed on rank 0
    strong = None
    if world > 1:
        progress("G1 strong scaling")
        ns = n // world
        bases_s = be.bases_from_scalars(L.PS_G1, ks[:ns].tobytes(), args.window_bits, args.tables)
        d_sc_s = d_scalars[:ns].contiguous()

        def step_strong():
            be._check(lib.ps_msm_device(be.ctx, bases_s.handle, 0, C.c_void_p(d_sc_s.data_ptr()), ns, C.c_void_p(d_part.data_ptr())))
            dist.all_gather_into_tensor(d_all, d_part)
        for _ in range(3):
            step_strong()
        barrier()
        be._check(lib.ps_msm_combine(be.ctx, L.PS_G1, C.c_void_p(d_part.data_ptr()), 1, out))
        parity["g1_strong_2p%d_over_%d" % (args.log_n, world)] = out.raw == expected_point(L.PS_G1, expected_exponent(ks[:ns], sc_be[:ns]))
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        s0.record(stream)
        for _ in range(args.steps):
            step_strong()
        s1.record(stream)
        barrier()
        info_s = (C.c_int * 4)()
        be._check(lib.ps_bases_info(bases_s.handle, info_s))
        strong = {"ms": s0.elapsed_time(s1), "c": info_s[0], "W": info_s[1]}
        bases_s.close()
        del d_sc_s
    del ks

    # secondary figures: G2 MSMs (same pipeline over Fp2), resident scalars, every rank its own range
    g2_runs = []
    for tok in [t for t in str(args.g2_log_n).split(",") if t.strip()]:
        k2 = int(tok)
        n2 = 1 << k2
        progress("G2 MSM 2^%d" % k2)
        ks2, sc2 = random_scalars_be(n2, 3000 + rank + 16 * k2), random_scalars_be(n2, 4000 + rank + 16 * k2)
        bases2 = be.bases_from_scalars(L.PS_G2, ks2.tobytes(), args.window_bits, args.tables)
        d_sc2 = torch.from_numpy(be_to_le_limbs(sc2).view(np.int32)).to(dev)
        d_part2 = torch.zeros(384, dtype=torch.uint8, device=dev)
        step2 = lambda: be._check(lib.ps_msm_device(be.ctx, bases2.handle, 0, C.c_void_p(d_sc2.data_ptr()), n2, C.c_void_p(d_part2.data_ptr())))
        for _ in range(3):
            step2()
        barrier()
        out2 = C.create_string_buffer(96)
        be._check(lib.ps_msm_combine(be.ctx, L.PS_G2, C.c_void_p(d_part2.data_ptr()), 1, out2))
        parity["g2_2p%d_resident" % k2] = out2.raw == expected_point(L.PS_G2, expected_exponent(ks2, sc2))
        del ks2, sc2
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(args.steps):
            step2()
        f1.record(stream)
        barrier()
        info2 = (C.c_int * 4)()
        be._check(lib.ps_bases_info(bases2.handle, info2))
        g2_runs.append({"log_n": k2, "ms": f0.elapsed_time(f1), "phases": be.msm_timing(), "c": info2[0], "W": info2[1]})
        bases2.close()
        del d_sc2
        torch.cuda.empty_cache()

    t = torch.tensor([ms_total, e2e_s * 1e3, strong["ms"] if strong else 0.0] + [g["ms"] for g in g2_runs], dtype=torch.float64, device=dev)
    ok = torch.tensor([1.0 if all(parity.values()) else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    ms_total, e2e_ms = float(t[0]), float(t[1])
    if strong:
        strong["ms"] = float(t[2])
    for i, g in enumerate(g2_runs):
        g["ms"] = float(t[3 + i])
    parity["all_ranks_ok"] = bool(ok.item() > 0.5)

    info_main = (C.c_int * 4)()
    be._check(lib.ps_bases_info(bases.handle, info_main))
    bases.close()
    del d_scalars, h_scalars, d_stage
    torch.cuda.empty_cache()
    if rank != 0:
        # rank 0 now drives ALL GPUs from one process (ps_mg16_prove); the other ranks release their devices and wait on the host
        be.close()
        dist.barrier(group=host_group)
        dist.destroy_process_group()
        return

    total_points = float(n) * world * args.steps
    value = total_points / (ms_total * 1e-3)
    e2e_value = total_points / (e2e_ms * 1e-3)

    # roofline of the dominant kernel (MsmAccumK): algorithmic IMAD = entries * madd * Fp-mul cost
    c_bits, W = info_main[0], info_main[1]
    madds = float(n) * W
    imad_alg = madds * FP_MUL_PER_MADD * IMAD_PER_FP_MUL
    accum_s = phase["accumulate_ms"] * 1e-3
    achieved = imad_alg / accum_s if accum_s > 0 else 0.0
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            tr = json.load(f)
        key = "g1_msm_2^%d" % args.log_n
        traffic = tr.get(key, {}).get("MsmAccumK_dram_bytes_per_launch")
    except (OSError, ValueError):
        pass
    gather_bytes = madds * 96.0 + madds * 4.0
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": "G1 MSM 2^%d points/GPU, random 254-bit scalars, resident bases" % args.log_n,
                   "window_bits": c_bits, "windows": W, "precomputed_tables": args.tables,
                   "l2": "inputs larger than L2 (scalars %d MB, bases >= %d MB per table)" % (n * 32 >> 20, n * 96 >> 20),
                   "parallelism": "point-range shard x%d, all-gather of 192 B partials" % world if world > 1 else "single GPU",
                   "bases_build_s": round(t_bases, 2)},
        "clocks": clocks,
        "parity": dict(parity, how="every timed configuration checked against (sum k_i s_i mod r)*G from the oracle "
                                   "(C dot product over Fr + one scalar multiplication), untimed"),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 32 * world, "d2h_bytes_per_step": 48,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "phases_ms_last_step": phase,
        "roofline": {"bound": "imad", "kernel": "MsmAccumK<Fp>", "achieved": achieved / 1e12, "peak": imad_peak / 1e12,
                     "unit": "TIMAD/s", "frac": achieved / imad_peak if imad_peak else None, "traffic": traffic,
                     "how": "algorithmic IMAD = n*W mixed adds x 10 Fp mul x 600 IMAD (IMAD.LO/HI pair accounting) / "
                            "CUDA-event time of the kernel; peak = IMAD issue rate measured live on this GPU "
                            "(ps_bench_intpipe, 'of measured'; MEASURED_PEAKS.json has no integer figure)",
                     "whole_msm_frac": (imad_alg / (phase["total_ms"] * 1e-3)) / imad_peak if phase["total_ms"] else None,
                     "fp_mul_per_s_microbench": fpmul_rate,
                     "hbm": {"achieved_gbs": gather_bytes / accum_s / 1e9 if accum_s else None,
                             "what": "base gather 96 B + entry 4 B per mixed add"}},
    }
    if strong:
        line["msm_strong"] = {"metric": "g1_msm_points_per_s", "scaling": "strong", "total_points": n, "n_gpus": world,
                              "points_per_gpu": n // world, "ms_per_step": strong["ms"] / args.steps,
                              "value": float(n) * args.steps / (strong["ms"] * 1e-3), "window_bits": strong["c"], "windows": strong["W"]}
    _STATE["line"] = line
    if g2_runs:
        def g2_entry(g):
            n2 = 1 << g["log_n"]
            acc2 = g["phases"]["accumulate_ms"] * 1e-3
            imad2 = float(n2) * g["W"] * 28.0 * IMAD_PER_FP_MUL     # G2 mixed add: 8 Fp2 mul + 2 Fp2 sqr = 28 Fp mul
            return {"metric": "g2_msm_points_per_s", "value": float(n2) * world * args.steps / (g["ms"] * 1e-3), "unit": UNIT,
                    "points_per_gpu": n2, "ms_per_step": g["ms"] / args.steps, "window_bits": g["c"], "windows": g["W"],
                    "phases_ms_last_step": g["phases"],
                    "roofline_frac_accumulate_kernel": (imad2 / acc2) / imad_peak if acc2 > 0 and imad_peak else None}
        line["g2_msm"] = g2_entry(g2_runs[0])
        for g in g2_runs[1:]:
            line["g2_msm_2p%d" % g["log_n"]] = g2_entry(g)
    if not args.no_cpu_baseline and world == 1:
        from oracle import c_oracle as CO
        threads = CO.max_threads()
        progress("CPU baseline: BlindEval")
        rate1, reps1, _ = cpu_blind_eval(10, 1, 3.0, 20)
        rate, reps, dt = cpu_blind_eval(args.ref_log_n, threads, 6.0, 40)
        line["cpu_baseline"] = {
            "value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d x Poly.BlindEval over 2^%d of the workload's points (oracle/ps_prover.c: bit-serial scalar-mul per "
                      "term as algebra.go:348-359), terms spread over %d OpenMP threads of %d host cores; single-threaded "
                      "(as the Go reference runs): %.0f points/s" % (reps, args.ref_log_n, threads, os.cpu_count() or 0, rate1),
            "single_thread_value": rate1}
        progress("CPU baseline: Groth16 flow")
        try:
            line["cpu_baseline"]["groth16_flow"] = cpu_groth16_flow(args.cpu_budget_s)
        except Exception as e:
            line["cpu_baseline"]["groth16_flow"] = {"error": repr(e)}
    if args.groth16_log_n:
        progress("Groth16 2^%d" % args.groth16_log_n)
        try:
            line["groth16"] = groth16_section(be, args, world)
        except Exception as e:  # the headline metric must still be reported
            line["groth16"] = {"error": repr(e)}
    if world == 1:
        sizes = [int(t) for t in str(args.phgr13_log_n).split(",") if t.strip()]
        if sizes:
            try:
                line["phgr13"] = phgr13_section(be, sizes)
            except Exception as e:
                line["phgr13"] = {"error": repr(e)}
        if not args.no_small_configs:
            try:
                line["small_configs"] = small_configs_section(be, line.get("cpu_baseline", {}).get("groth16_flow"))
            except Exception as e:
                line["small_configs"] = {"error": repr(e)}
    _STATE["printed"] = True
    print(json.dumps(line), flush=True)
    progress("done")
    if world > 1:
        dist.barrier(group=host_group)
        dist.destroy_process_group()
    if not parity["all_ranks_ok"]:
        print("bench.py: PARITY MISMATCH %r -- the numbers above are invalid" % parity, file=sys.stderr)
        sys.exit(3)


def _time_calls(fn, reps):
    fn()
    fn()
    best, t_all = 1e9, time.perf_counter()
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return (time.perf_counter() - t_all) / reps, best


def groth16_section(be, args, world):
    """BASELINE configs[2]/[4]: full Groth16 prove (sparse R1CS -> interpolation on {1..n} -> quotient -> 3 MSMs) on a
    synthetic circuit of 2^k constraints; the key comes from the device's own trusted setup (ps_g16_setup, untimed);
    parity = exponent-level recomputation from the toxic waste (groth16_test.go:32-107 at scale).  Timed through the
    reference-facing call with the witness in page-locked host memory (wire format) and the proof bytes back on the host.
    With several GPUs the SAME call runs on a MultiBackend: one library call per proof, key sharded over the devices."""
    import playsnark_b200 as ps
    from playsnark_b200 import synth
    from oracle import expect as E, ps_oracle as O
    k = args.groth16_log_n
    n = 1 << k
    sq, wit = synth.sparse_circuit(n, 7, n // 2)
    smp = O.Sampler(99)
    toxic = tuple(smp.fr() for _ in range(5))
    r, s = smp.fr(), smp.fr()
    progress("Groth16: setup on the device")
    t0 = time.perf_counter()
    tr = ps.NewGroth16TrustedSetup(sq, backend=be, toxic=toxic, export=world > 1)
    be.sync()
    t_setup = time.perf_counter() - t0
    progress("Groth16: prove")
    reps = max(3, args.steps)
    out = {"constraints": n, "variables": sq.nbVars, "nio_points": sq.nbIO, "n_gpus": world, "setup_on_device_s": round(t_setup, 2),
           "h2d_bytes_per_proof": 32 * sq.nbVars + 64, "d2h_bytes_per_proof": 192}
    if world == 1:
        wb = ps.HostBuffer(be, b"".join(v.to_bytes(32, "big") for v in wit))
        l0 = be.launch_count()
        avg, best = _time_calls(lambda: ps.Groth16Prove(tr, sq, wb, r, s, backend=be), reps)
        out["gpu_launches_per_proof"] = int((be.launch_count() - l0) // (reps + 2))
        pr = ps.Groth16Prove(tr, sq, wb, r, s, backend=be)
        out["device_ms"] = be.prove_timing()
        wb.close()
    else:
        sq.close(); tr.close()                      # device 0's single-device copies
        mb = ps.MultiBackend(list(range(world)))
        t0 = time.perf_counter()
        tr._resident(mb); sq._resident(mb)
        out["sharded_key_and_qap_load_s"] = round(time.perf_counter() - t0, 2)
        wb = ps.HostBuffer(be, b"".join(v.to_bytes(32, "big") for v in wit))
        l0 = mb.launch_count()
        avg, best = _time_calls(lambda: ps.Groth16Prove(tr, sq, wb, r, s, backend=mb), reps)
        out["gpu_launches_per_proof_all_devices"] = int((mb.launch_count() - l0) // (reps + 2))
        pr = ps.Groth16Prove(tr, sq, wb, r, s, backend=mb)
        marks = ["witness gathered", "subtree interpolated", "roots gathered", "top levels", "a, b swapped", "slice scalars (+ division on device 0)",
                 "MSMs (B_d at once, A_d + C_d after h)", "record ready", "combined + encoded"]
        out["timeline_ms"] = {"device%d" % d: dict(zip(marks, [round(x, 3) for x in mb.timeline(d)])) for d in (0, world - 1)}
        out["how"] = "ONE library call per proof (ps_mg16_prove): worker thread per GPU, exchanges over NVLink peer memory"
        wb.close()
        sq.close(); tr.close(); mb.close()
    out["proof_ms_e2e"] = avg * 1e3
    out["proof_ms_e2e_best"] = best * 1e3
    out["proofs_per_s_e2e"] = 1.0 / avg
    progress("Groth16: expectation")
    A, B, Cc, _, _ = E.groth16_expected(sq, wit, toxic, r, s)
    out["parity"] = ("A, B, C equal the exponent-level recomputation from the toxic waste"
                     if (pr.A, pr.B, pr.C) == (A, B, Cc) else "MISMATCH")
    out["cpu_reference"] = ("does not finish at this size: ToQAP is O(m n^3) field multiplications and the dense QAP "
                            "would need 3*m*n*32 bytes (BASELINE.md section 2); measured sizes under cpu_baseline.groth16_flow")
    if world == 1:
        sq.close(); tr.close()
    return out


def phgr13_section(be, sizes):
    """PHGR13Prove (pinochio.go:207-254) on sparse circuits of 2^k constraints: quotient + hs + eight sums over
    solution[diff:] (seven of them one batched G1 pipeline, wss on G2); key from ps_phgr13_setup; exponent-level parity."""
    import playsnark_b200 as ps
    from playsnark_b200 import synth
    from oracle import expect as E, ps_oracle as O
    res = {}
    for k in sizes:
        n = 1 << k
        progress("PHGR13 2^%d: circuit" % k)
        sq, wit = synth.sparse_circuit(n, 11 + k, n // 2)
        smp = O.Sampler(500 + k)
        toxic = tuple(smp.fr() for _ in range(8))
        progress("PHGR13 2^%d: setup" % k)
        t0 = time.perf_counter()
        ek, _, _ = ps.NewPHGR13TrustedSetup(sq, backend=be, toxic=toxic)
        be.sync()
        t_setup = time.perf_counter() - t0
        progress("PHGR13 2^%d: prove" % k)
        wb = ps.HostBuffer(be, b"".join(v.to_bytes(32, "big") for v in wit))
        avg, best = _time_calls(lambda: ps.PHGR13Prove(ek, sq, wb, backend=be), 5)
        pp = ps.PHGR13Prove(ek, sq, wb, backend=be)
        progress("PHGR13 2^%d: expectation" % k)
        want = E.phgr13_expected(sq, wit, toxic)
        okp = all(getattr(pp, f) == want[f] for f in O.PHGR13_FIELDS)
        res["2p%d" % k] = {"constraints": n, "mid_points": sq.nbIO, "prove_ms_e2e": avg * 1e3, "prove_ms_e2e_best": best * 1e3,
                           "setup_on_device_s": round(t_setup, 2),
                           "parity": "all eight elements equal the exponent-level recomputation" if okp else "MISMATCH"}
        wb.close(); ek.close(); sq.close()
    return res


def verify_section(be, q, w, toxic, ptoxic, r, s, pr, pp):
    """SURVEY 8 f4: Groth16Verify / PHGR13Verify on the device for the 2^10 chain's proofs (decisions: accept the honest
    proof, reject a wrong public input), and the throughput of the pairing-product checks for a batch of proofs."""
    import playsnark_b200 as ps
    from playsnark_b200 import _lib as L
    progress("verifiers")
    diff = q.nbVars - q.nbIO
    tr = ps.NewGroth16TrustedSetup(q, backend=be, toxic=toxic, fmt=L.PS_FMT_COMPRESSED, export=True)
    ek, vk, _ = ps.NewPHGR13TrustedSetup(q, backend=be, toxic=ptoxic, with_vk=True)
    io = w[:diff]
    bad = list(io); bad[-1] = (bad[-1] + 1) % R
    ok = (ps.Groth16Verify(tr, q, pr, io, backend=be) and not ps.Groth16Verify(tr, q, pr, bad, backend=be)
          and ps.PHGR13Verify(vk, q, pp, io, backend=be) and not ps.PHGR13Verify(vk, q, pp, bad, backend=be))
    _, g_best = _time_calls(lambda: ps.Groth16Verify(tr, q, pr, io, backend=be), 3)
    _, p_best = _time_calls(lambda: ps.PHGR13Verify(vk, q, pp, io, backend=be), 3)
    # a batch of Groth16 equations in one call: 4 pairs each (e(-A,B) e(Alpha,Beta2) e(b1,Gamma) e(C,Delta2) == 1 with b1 = 0
    # replaced by the honest pairs of this proof is not available host-side, so the batch repeats e(aG,bH) e(-abG,H) == 1)
    from oracle import ps_oracle as O
    a_, b_ = 0x1234567, 0x7654321
    g1a, g1ab = O.g1_compress(O.g1_mul(a_)), O.g1_compress(O.g1_mul((-a_ * b_) % R))
    g2b, g2g = O.g2_compress(O.g2_mul(b_)), O.g2_compress(O.g2_mul(1))
    batch = 2048
    P1, Q2 = [g1a, g1ab, g1a, g1ab] * batch, [g2b, g2g, g2b, g2g] * batch
    res = ps.PairingCheckBatch(P1, Q2, [4] * batch, backend=be)
    _, b_best = _time_calls(lambda: ps.PairingCheckBatch(P1, Q2, [4] * batch, backend=be), 2)
    tr.close(); ek.close()
    return {"decisions": "honest proofs accepted, wrong public input rejected (Groth16 and PHGR13)" if ok and all(res) else "MISMATCH",
            "groth16_verify_ms": g_best * 1e3, "phgr13_verify_ms": p_best * 1e3,
            "batch": {"checks": batch, "pairs_per_check": 4, "ms": b_best * 1e3, "checks_per_s": batch / b_best,
                      "what": "ps_pairing_check_batch: one thread per Miller loop and per final exponentiation"}}


def small_configs_section(be, cpu_flow):
    """BASELINE configs[1] and [2]: the 2^10 repeated-squaring circuit (Groth16 and PHGR13) and a 2^16-constraint sparse
    circuit (Groth16); keys from the device setups, exponent-level parity, end-to-end latency through the
    reference-facing calls.  Where the CPU flow was measured on the same circuit shape its time stands beside ours."""
    import playsnark_b200 as ps
    from playsnark_b200 import synth
    from oracle import expect as E, ps_oracle as O
    out = {}
    smp = O.Sampler(2)
    toxic = tuple(smp.fr() for _ in range(5))
    ptoxic = tuple(smp.fr() for _ in range(8))
    r, s = smp.fr(), smp.fr()
    cpu_by_n = {row["gates"]: row for row in (cpu_flow or {}).get("runs", [])} if isinstance(cpu_flow, dict) else {}
    for k in (4, 6, 8, 10):
        n = 1 << k
        progress("chain circuit 2^%d" % k)
        c, w = synth.squaring_chain(n, -1)
        q = ps.ToQAP(c)
        tr = ps.NewGroth16TrustedSetup(q, backend=be, toxic=toxic, export=False)
        ek, _, _ = ps.NewPHGR13TrustedSetup(q, backend=be, toxic=ptoxic)
        wb = b"".join(v.to_bytes(32, "big") for v in w)
        _, g_best = _time_calls(lambda: ps.Groth16Prove(tr, q, wb, r, s, backend=be), 5)
        _, p_best = _time_calls(lambda: ps.PHGR13Prove(ek, q, wb, backend=be), 5)
        pr = ps.Groth16Prove(tr, q, wb, r, s, backend=be)
        pp = ps.PHGR13Prove(ek, q, wb, backend=be)
        A, B, Cc, _, _ = E.groth16_expected(q, w, toxic, r, s)
        want = E.phgr13_expected(q, w, ptoxic)
        okp = (pr.A, pr.B, pr.C) == (A, B, Cc) and all(getattr(pp, f) == want[f] for f in O.PHGR13_FIELDS)
        row = {"gates": n, "variables": q.nbVars, "groth16_prove_ms": g_best * 1e3, "phgr13_prove_ms": p_best * 1e3,
               "parity": "Groth16 A, B, C and the eight PHGR13 elements equal the exponent-level recomputation" if okp else "MISMATCH"}
        if n in cpu_by_n:
            row["cpu_port_groth16_prove_s"] = cpu_by_n[n]["prove_s"]
            row["speedup_vs_cpu_port_prove"] = cpu_by_n[n]["prove_s"] / g_best
        out["chain_2p%d" % k] = row
        if k == 10:
            try:
                out["verify"] = verify_section(be, q, w, toxic, ptoxic, r, s, pr, pp)
            except Exception as e:
                out["verify"] = {"error": repr(e)}
        tr.close(); ek.close(); q.close()
    k = 16
    progress("sparse circuit 2^16")
    nn = 1 << k
    sq, wit = synth.sparse_circuit(nn, 7, nn // 2)
    tr = ps.NewGroth16TrustedSetup(sq, backend=be, toxic=toxic, export=False)
    wb = ps.HostBuffer(be, b"".join(v.to_bytes(32, "big") for v in wit))
    _, best = _time_calls(lambda: ps.Groth16Prove(tr, sq, wb, r, s, backend=be), 5)
    pr = ps.Groth16Prove(tr, sq, wb, r, s, backend=be)
    A, B, Cc, _, _ = E.groth16_expected(sq, wit, toxic, r, s)
    out["c3_sparse_2p16"] = {"groth16_prove_ms": best * 1e3, "device_ms": be.prove_timing(),
                             "parity": "A, B, C equal the exponent-level recomputation" if (pr.A, pr.B, pr.C) == (A, B, Cc) else "MISMATCH"}
    wb.close(); tr.close(); sq.close()
    return out


if __name__ == "__main__":
    main()
