"""Helpers shared by the GPU parity tests: the CUDA path is always reached through the C ABI
(distributedfft_b200 -> libdfft.so); oracle/ is only the checker."""
import ctypes as C
import os

import numpy as np
import torch

import distributedfft_b200 as dfft
from oracle import dft_oracle as O

CDT = {dfft.F64: torch.complex128, dfft.F32: torch.complex64}
RDT = {dfft.F64: torch.float64, dfft.F32: torch.float32}
NPC = {dfft.F64: np.complex128, dfft.F32: np.complex64}
NPR = {dfft.F64: np.float64, dfft.F32: np.float32}
TOL = {dfft.F64: O.TOL["f64"], dfft.F32: O.TOL["f32"]}
PNAME = {dfft.F64: "double", dfft.F32: "float"}

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# single-GPU cuFFT spectra of the comparisons below, at the positions of sample_index (tests/golden/make_cufft_golden.py)
CUFFT_GOLDEN = os.path.join(ROOT, "tests", "golden", "cufft_sample.npz")
CUFFT_SHAPES = [(128, 128, 128), (256, 128, 64)]
FULL_SIZE_CASES = ["512_c2c_f64_slab", "1024_r2c_f64_slab", "1024_c2c_f32_pencil", "1024_r2c_f64_zyx"]


def dev(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t: torch.Tensor) -> np.ndarray:
    return t.detach().cpu().numpy()


def make_plan(cls, prec, transform, shape, partition=None, comm=None, comm_method=dfft.CommunicationMethod.Peer2Peer):
    cfg = dfft.Configurations(comm_method=comm_method, comm_method2=comm_method)
    plan = cls(cfg, comm if comm is not None else dfft.Comm(), precision=PNAME[prec], transform="c2c" if transform == dfft.C2C else "r2c")
    plan.initFFT(dfft.GlobalSize(*shape), partition, True)
    return plan


def cufft_lib():
    """oracle/_ref/libcufft_ref.so (single-GPU cufftPlan3d, built by `make -C oracle`), or None when it is not built."""
    path = os.path.join(ROOT, "oracle", "_ref", "libcufft_ref.so")
    if not os.path.exists(path):
        return None
    lib = C.CDLL(path)
    lib.cufft_ref_3d.restype = C.c_int
    lib.cufft_ref_3d.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_int]
    return lib


def cufft_key(kind, prec, shape):
    return f"{kind}_{PNAME[prec]}_{shape[0]}x{shape[1]}x{shape[2]}"


def sample_index(n, k=2048):
    """Fixed positions (sorted flat indices drawn by a seed-0 generator) at which the golden spectra are stored."""
    return np.sort(np.random.default_rng(0).choice(n, size=min(k, n), replace=False))


def sampled(t: torch.Tensor) -> np.ndarray:
    return host(t.reshape(-1)[torch.from_numpy(sample_index(t.numel())).to(t.device)])


def full_size_input(kind, prec, n):
    """uniform[0,255) input of the full-size comparisons, from torch's generator seeded 99 on the device"""
    g = torch.Generator(device="cuda").manual_seed(99)
    shape = (n, n, n)
    if kind == "c2c":
        return torch.complex(torch.rand(shape, generator=g, device="cuda", dtype=RDT[prec]) * 255,
                             torch.rand(shape, generator=g, device="cuda", dtype=RDT[prec]) * 255)
    return torch.rand(shape, generator=g, device="cuda", dtype=RDT[prec]) * 255
