"""Groth16VerifyBatch of the C++ host mirror (playsnark_b200/host/playsnark.hpp) on the README circuit's golden key and
proof: the batch [proof, proof, proof with C + G] gives the verdicts [1, 1, 0].  Linked against the host-emulation build
on CPU and, under -m gpu, against the product library."""
import os
import subprocess

import pytest

from oracle import ps_oracle as O
from playsnark_b200 import build as B
from tests.parity_cases import gold

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")


def run_against(libpath, exe_name):
    os.makedirs(BUILD, exist_ok=True)
    exe = os.path.join(BUILD, exe_name)
    src = os.path.join(ROOT, "tests", "verify_batch_cpp_test.cpp")
    libdir, libfile = os.path.split(libpath)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-o", exe, src, "-L" + libdir, "-l:" + libfile, "-Wl,-rpath," + libdir])
    g = gold("readme_circuit")
    k = g["groth16"]
    n_io = g["nb_vars"] - g["nb_io"]
    assert len(k["IoLP"]) == n_io
    c_plus_g = O.g1_compress(O.g1_add(O.g1_decompress(bytes.fromhex(k["C"])), O.G1_GEN)).hex()
    toks = [k["Alpha"], k["Beta2"], k["Gamma"], k["Delta2"], str(n_io)] + k["IoLP"] + [k["A"], k["B"], k["C"], c_plus_g]
    toks += [str(v) for v in g["witness"][:n_io]]
    tok = os.path.join(BUILD, "verify_batch_tokens_%s.txt" % exe_name)
    with open(tok, "w") as f:
        f.write("\n".join(toks) + "\n")
    res = subprocess.run([exe, tok], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = {l.split()[0]: l.split()[1:] for l in res.stdout.strip().split("\n")}
    assert got["ok"] == ["0"] and got["verdicts"] == ["1", "1", "0"]
    assert got["honest"] == ["1"] and got["single"] == ["1"] and got["short"] == ["mismatch"]


def test_cpp_verify_batch_emulated():
    run_against(B.build_host_emulation(BUILD), "verify_batch_cpp_test_emu")


@pytest.mark.gpu
def test_cpp_verify_batch_gpu():
    run_against(B.LIB, "verify_batch_cpp_test_gpu")
