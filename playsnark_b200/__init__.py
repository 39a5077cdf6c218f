"""playsnark_b200 -- B200-native backend for the proving path of nikkolasg/playsnark.

Host-side mirror of the reference's prover interface (Groth16Prove / PHGR13Prove over its R1CS / QAP
/ key types) on top of the C ABI in include/playsnark_b200.h; all arithmetic runs in hand-written
sm_100a CUDA kernels (playsnark_b200/csrc).
"""
from .api import (  # noqa: F401
    MultiBackend, MultiBases, NewGroth16TrustedSetup, NewPHGR13TrustedSetup,
    R, Backend, Bases, HostBuffer, Groth16Proof, Groth16Setup, PHGR13EvalKey, PHGR13Proof, QAP, SparseQAP, R1CS, Groth16Prove,
    PHGR13Prove, Quotient, BlindEval, ToQAP, default_backend, set_default_backend, Groth16Verify, Groth16VerifyBatch, PHGR13Verify, PHGR13VerifyBatch, PairingCheckBatch,
)
from ._lib import PlaysnarkError  # noqa: F401
