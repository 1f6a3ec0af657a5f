"""Generates tests/golden/ref_math_golden.npz (SVD) and ref_stress_golden.npz (constitutive models) from the REFERENCE's own
3x3 SVD and constitutive models.

Run in the container that has /root/reference:  bash oracle/build_ref.sh && python tests/golden/make_ref_math_golden.py
oracle/_ref/libclaymore_ref_math.so is the reference's svd.cuh / constitutive_models.cuh compiled for the host by
oracle/ref_math_host.cpp (the sources are included where they lie; nothing is copied).  The vectors pin the oracle
(tests/test_oracle_cpu.py compares bitwise) and travel to the GPU box, where /root/reference does not exist.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_binding as ob  # noqa: E402  (only for the material defaults)


def main():
    ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libclaymore_ref_math.so"))
    ref.ref_svd3.argtypes = [C.c_void_p] * 4
    ref.ref_compute_stress.argtypes = [C.c_int] + [C.c_void_p] * 4
    rng = np.random.default_rng(20260924)
    n = 4000
    scales = rng.choice([1e-3, 1e-2, 0.1, 0.3, 1.0], size=n)
    F = (np.eye(3)[None] + scales[:, None, None] * rng.standard_normal((n, 3, 3))).astype(np.float32).reshape(n, 9)
    F[:8] = np.stack([np.eye(3).reshape(9) * s for s in (1.0, 0.9, 1.1, 0.5, 2.0, 1.0, 1.0, 1.0)]).astype(np.float32)
    F[5] = np.diag([1.2, 0.9, 0.95]).reshape(9)
    F[6] = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], np.float32).T.reshape(9)   # pure rotation
    F[7] = np.diag([1.0, 1.0, -1.0]).reshape(9)                                    # reflection
    U, S, V = np.zeros((n, 9), np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 9), np.float32)
    for i in range(n):
        ref.ref_svd3(F[i].ctypes.data, U[i].ctypes.data, S[i].ctypes.data, V[i].ctypes.data)
    svd = dict(F=F, U=U, S=S, V=V)
    # a second, independently seeded set at three strain scales (tests/test_oracle_cpu.py: fresh vectors)
    rng_fresh = np.random.default_rng(7)
    fresh = np.stack([(np.eye(3) + rng_fresh.choice([0.01, 0.1, 1.0]) * rng_fresh.standard_normal((3, 3))).astype(np.float32).reshape(-1) for _ in range(3000)])
    svd["fresh_F"] = fresh
    svd["fresh_U"], svd["fresh_S"], svd["fresh_V"] = np.zeros((3000, 9), np.float32), np.zeros((3000, 3), np.float32), np.zeros((3000, 9), np.float32)
    for i in range(3000):
        ref.ref_svd3(fresh[i].ctypes.data, svd["fresh_U"][i].ctypes.data, svd["fresh_S"][i].ctypes.data, svd["fresh_V"][i].ctypes.data)
    out = {}
    cfg = ob.make_config(domain_bits=8)
    log_jp_in = rng.uniform(-0.05, 0.02, size=n).astype(np.float32)
    out["log_jp_in"] = log_jp_in
    small = (np.eye(3)[None] + np.minimum(scales, 0.3)[:, None, None] * rng.standard_normal((n, 3, 3))).astype(np.float32).reshape(n, 9)
    out["F_stress"] = small
    for mat, name in ((ob.FIXED_COROTATED, "fc"), (ob.SAND, "sand"), (ob.NACC, "nacc")):
        pb = ob.default_buffer(cfg, mat)
        params = np.array([pb.volume, pb.mu, pb.lambda_, pb.bm, pb.xi, pb.beta, pb.msqr, 0, pb.cohesion, pb.yield_surface, pb.hardening_on, pb.volume_correction], np.float32)
        Fo, PF, LJ = small.copy(), np.zeros((n, 9), np.float32), log_jp_in.copy()
        for i in range(n):
            lj = LJ[i:i + 1]
            ref.ref_compute_stress(mat, params.ctypes.data, Fo[i].ctypes.data, PF[i].ctypes.data, lj.ctypes.data)
        out[f"{name}_F_out"], out[f"{name}_PF"], out[f"{name}_log_jp_out"] = Fo, PF, LJ
    # two files, each under 1 MB
    for name, data in (("ref_math_golden.npz", svd), ("ref_stress_golden.npz", out)):
        np.savez_compressed(os.path.join(HERE, name), **data)
        print("wrote", os.path.join(HERE, name), {k: v.shape for k, v in data.items()})


if __name__ == "__main__":
    main()
