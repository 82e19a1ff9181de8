"""Generates tests/golden/cufft_sample.npz: what single-GPU cuFFT (cufftPlan3d, the oracle of the reference's
testcase 1, through oracle/_ref/libcufft_ref.so) computes on the inputs of the cuFFT comparisons in
tests/test_gpu_plan.py, kept at the positions of common.sample_index so that the file stays small and those
comparisons run without the cuFFT helper.  The full-size cases also keep their input at the same positions, which
pins torch's seeded generator.  Needs a GPU and the build; run from the repo root:
    python tests/golden/make_cufft_golden.py [out.npz]"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import torch  # noqa: E402

import distributedfft_b200 as dfft  # noqa: E402
from common import (CDT, CUFFT_GOLDEN, CUFFT_SHAPES, FULL_SIZE_CASES, NPC, NPR, cufft_key, cufft_lib, dev,  # noqa: E402
                    full_size_input, sampled)
from oracle import dft_oracle as O  # noqa: E402


def cufft(lib, prec, kind, x, out_shape):
    ref = torch.empty(out_shape, dtype=CDT[prec], device="cuda")
    ms = C.c_float()
    assert lib.cufft_ref_3d(1 if prec == dfft.F64 else 0, 0 if kind == "c2c" else 2, *x.shape, ref.data_ptr(), x.data_ptr(), C.byref(ms), 1) == 0
    return ref


def main(path):
    lib = cufft_lib()
    assert lib is not None, "oracle/_ref/libcufft_ref.so is not built (make -C oracle)"
    out = {}
    for prec in (dfft.F64, dfft.F32):
        for shape in CUFFT_SHAPES:
            nzo = shape[2] // 2 + 1
            out[cufft_key("r2c", prec, shape)] = sampled(cufft(lib, prec, "r2c", dev(O.real_input(shape, dtype=NPR[prec])), (*shape[:2], nzo)))
            out[cufft_key("c2c", prec, shape)] = sampled(cufft(lib, prec, "c2c", dev(O.complex_input(shape, dtype=NPC[prec])), shape))
    for case in FULL_SIZE_CASES:
        n, kind, pname, _ = case.split("_")
        n = int(n)
        prec = dfft.F64 if pname == "f64" else dfft.F32
        x = full_size_input(kind, prec, n)
        out[case] = sampled(cufft(lib, prec, kind, x, (n, n, n if kind == "c2c" else n // 2 + 1)))
        out[case + "_in"] = sampled(x)
        del x
        torch.cuda.empty_cache()
    np.savez_compressed(path, **out)
    print("written", path, {k: (v.dtype.name, v.shape) for k, v in out.items()})


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else CUFFT_GOLDEN)
