"""PHGR13VerifyBatch of the C++ host mirror (playsnark_b200/host/playsnark.hpp) on the README circuit: a device setup
and proof, then the batch [proof, proof, proof with hs + G] gives the verdicts [1, 1, 0].  Setup, proof and the C++
program run on the host-emulation build on CPU and, under -m gpu, on the product library."""
import os
import subprocess

import pytest

from oracle import ps_oracle as O
from playsnark_b200 import _lib as L, api, build as B
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")


def run_against(libpath, exe_name):
    os.makedirs(BUILD, exist_ok=True)
    exe = os.path.join(BUILD, exe_name)
    src = os.path.join(ROOT, "tests", "phgr13_verify_batch_cpp_test.cpp")
    libdir, libfile = os.path.split(libpath)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, src, "-L" + libdir, "-l:" + libfile, "-Wl,-rpath," + libdir])
    be = api.Backend(0, lib=L.bind(libpath))
    try:
        c = O.create_r1cs()
        w = O.create_witness(c)
        q = H.mirror_qap(O.to_qap(c))
        ek, vk, _ = api.NewPHGR13TrustedSetup(q, backend=be, with_vk=True)
        p = api.PHGR13Prove(ek, q, w, backend=be)
        diff = q.nbVars - q.nbIO
        ek.close()
        q.close()
    finally:
        be.close()
    hs_plus_g = O.g1_compress(O.g1_add(O.g1_decompress(p.hs), O.G1_GEN))
    toks = [vk[k].hex() for k in ("av", "aw", "ay", "gamma", "bgamma", "bgamma2", "yts")] + [str(diff)]
    toks += [b.hex() for k in ("vs", "ws", "ys") for b in vk[k][:diff]]
    toks += [getattr(p, f).hex() for f in ("hs", "vss", "yss", "vass", "wass", "yass", "gz", "wss")] + [hs_plus_g.hex()]
    toks += [str(v) for v in w[:diff]]
    tok = os.path.join(BUILD, "phgr13_verify_batch_tokens_%s.txt" % exe_name)
    with open(tok, "w") as f:
        f.write("\n".join(toks) + "\n")
    res = subprocess.run([exe, tok], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = {l.split()[0]: l.split()[1:] for l in res.stdout.strip().split("\n")}
    assert got["ok"] == ["0"] and got["verdicts"] == ["1", "1", "0"]
    assert got["honest"] == ["1"] and got["single"] == ["1"] and got["short"] == ["mismatch"]


def test_cpp_phgr13_verify_batch_emulated():
    run_against(B.build_host_emulation(BUILD), "phgr13_verify_batch_cpp_test_emu")


@pytest.mark.gpu
def test_cpp_phgr13_verify_batch_gpu():
    run_against(B.LIB, "phgr13_verify_batch_cpp_test_gpu")
