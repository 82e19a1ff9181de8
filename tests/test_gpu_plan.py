"""Whole-plan parity on one GPU: the reference's testcases 1 (vs a single 3D transform), 3 (round trip)
and 4 (spectral Laplacian), plus the pencil partial transforms (-f 1 / -f 2), through the C ABI."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import distributedfft_b200 as dfft
from oracle import dft_oracle as O
from common import (CDT, CUFFT_GOLDEN, CUFFT_SHAPES, FULL_SIZE_CASES, NPC, NPR, RDT, TOL, cufft_key, cufft_lib, dev,
                    full_size_input, host, make_plan, sampled)

pytestmark = pytest.mark.gpu

CLASSES = [dfft.MPIcuFFT_Slab, dfft.MPIcuFFT_Slab_Z_Then_YX, dfft.MPIcuFFT_Pencil]


def _part(cls):
    return dfft.Pencil_Partition(1, 1) if cls is dfft.MPIcuFFT_Pencil else None


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("prec", [dfft.F64, dfft.F32])
@pytest.mark.parametrize("shape", [(128, 128, 128), (32, 64, 16), (8, 4, 256), (256, 16, 32)])
def test_c2c_forward_inverse(cls, prec, shape):
    """BASELINE config 1 (128^3 complex-double forward+inverse) and friends."""
    plan = make_plan(cls, prec, dfft.C2C, shape, _part(cls))
    x = O.complex_input(shape, dtype=NPC[prec])
    xin = dev(x)
    out = torch.empty(shape, dtype=CDT[prec], device="cuda")
    plan.execC2C(out, xin, dfft.FORWARD)
    ref = O.fft_c2c(x)
    assert O.rel_l2(host(out), ref) < TOL[prec]
    assert np.array_equal(host(xin), x), "forward must leave the input intact"
    back = torch.empty_like(out)
    plan.execC2C(back, out, dfft.INVERSE)
    assert O.rel_l2(host(back), x.astype(np.complex128) * np.prod(shape)) < TOL[prec]
    plan.destroy()


@pytest.mark.parametrize("cls", CLASSES)
@pytest.mark.parametrize("prec", [dfft.F64, dfft.F32])
@pytest.mark.parametrize("shape", [(128, 128, 128), (16, 32, 64), (64, 8, 4), (4, 4, 512)])
def test_r2c_c2r(cls, prec, shape):
    """testcase 1 (forward vs single 3D transform) and testcase 3 (round trip)."""
    plan = make_plan(cls, prec, dfft.R2C, shape, _part(cls))
    nx, ny, nz = shape
    nzo = nz // 2 + 1
    assert plan.getInSize() == [nx, ny, nz] and plan.getOutSize() == [nx, ny, nzo]
    x = O.real_input(shape, dtype=NPR[prec])
    xin = dev(x)
    out = torch.empty((nx, ny, nzo), dtype=CDT[prec], device="cuda")
    assert out.numel() * out.element_size() >= plan.getDomainSize()
    plan.execR2C(out, xin)
    assert O.rel_l2(host(out), O.fft_r2c(x)) < TOL[prec]
    back = torch.empty_like(xin)
    plan.execC2R(back, out)
    assert O.rel_l2(host(back), x.astype(np.float64) * np.prod(shape)) < TOL[prec]
    plan.destroy()


@pytest.mark.parametrize("prec", [dfft.F64, dfft.F32])
@pytest.mark.parametrize("d", [1, 2])
def test_pencil_partial(prec, d):
    """pencil -f 1 / -f 2 (tests/src/pencil/random_dist_1D.cu:319-350, random_dist_2D.cu:321-352)."""
    shape = (16, 32, 64)
    plan = make_plan(dfft.MPIcuFFT_Pencil, prec, dfft.R2C, shape, dfft.Pencil_Partition(1, 1))
    x = O.real_input(shape, dtype=NPR[prec])
    out = torch.empty((16, 32, 33), dtype=CDT[prec], device="cuda")
    plan.execR2C(out, dev(x), d)
    ref = O.fft_r2c(x, d)
    assert O.rel_l2(host(out), ref) < TOL[prec]
    back = torch.empty(shape, dtype=RDT[prec], device="cuda")
    plan.execC2R(back, dev(ref.astype(NPC[prec])), d)
    scale = 64 * (32 if d == 2 else 1)
    assert O.rel_l2(host(back), x.astype(np.float64) * scale) < TOL[prec]
    plan.destroy()


@pytest.mark.parametrize("cls", CLASSES)
def test_laplacian(cls):
    """testcase 4 (random_dist_default.cu:625-758): inverse(coeff * forward(sin sin sin)) = -3 sqrt(N) f."""
    shape = (64, 64, 64)
    plan = make_plan(cls, dfft.F64, dfft.R2C, shape, _part(cls))
    f = O.sine_input(shape)
    out = torch.empty((64, 64, 33), dtype=torch.complex128, device="cuda")
    plan.execR2C(out, dev(f))
    size, start = plan.getOutSize(), plan.getOutStart()
    out *= dev(O.laplacian_coefficients(64, 64, 64, start, size))
    back = torch.empty(shape, dtype=torch.float64, device="cuda")
    plan.execC2R(back, out)
    expect = O.laplacian_expected(shape)
    err = np.abs(host(back) - expect)
    # the reference records avg abs err 7e-7 on amplitude 1e5 at 1024^3 (eval/benchmarks/**/numerical_8.csv)
    assert err.max() / np.abs(expect).max() < 1e-12
    plan.destroy()


@pytest.mark.parametrize("prec", [dfft.F64, dfft.F32])
@pytest.mark.parametrize("shape", CUFFT_SHAPES)
def test_vs_cufft_single_gpu(prec, shape):
    """The reference's own oracle: cufftPlan3d on one GPU (random_dist_default.cu:300-303,337,365-371), at the positions
    stored in tests/golden/cufft_sample.npz and, when oracle/_ref/libcufft_ref.so is built, element by element."""
    golden = np.load(CUFFT_GOLDEN)
    lib = cufft_lib()
    nx, ny, nz = shape
    nzo = nz // 2 + 1
    ms = C.c_float()
    x = dev(O.real_input(shape, dtype=NPR[prec]))
    plan = make_plan(dfft.MPIcuFFT_Slab, prec, dfft.R2C, shape)
    out = torch.empty((nx, ny, nzo), dtype=CDT[prec], device="cuda")
    plan.execR2C(out, x)
    assert O.rel_l2(sampled(out), golden[cufft_key("r2c", prec, shape)]) < TOL[prec]
    if lib is not None:
        ref = torch.empty_like(out)
        assert lib.cufft_ref_3d(1 if prec == dfft.F64 else 0, 2, nx, ny, nz, ref.data_ptr(), x.data_ptr(), C.byref(ms), 1) == 0
        assert O.rel_l2(host(out), host(ref)) < TOL[prec]
    # complex
    xc = dev(O.complex_input(shape, dtype=NPC[prec]))
    planc = make_plan(dfft.MPIcuFFT_Slab, prec, dfft.C2C, shape)
    outc = torch.empty_like(xc)
    planc.execC2C(outc, xc, dfft.FORWARD)
    assert O.rel_l2(sampled(outc), golden[cufft_key("c2c", prec, shape)]) < TOL[prec]
    if lib is not None:
        refc = torch.empty_like(xc)
        assert lib.cufft_ref_3d(1 if prec == dfft.F64 else 0, 0, nx, ny, nz, refc.data_ptr(), xc.data_ptr(), C.byref(ms), 1) == 0
        assert O.rel_l2(host(outc), host(refc)) < TOL[prec]
    plan.destroy(); planc.destroy()


def _build_and_run(tmp_path, compiler_cmd, src, name):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / name)
    libdir = os.path.join(root, "distributedfft_b200")
    subprocess.run([*compiler_cmd, "-std=c++17", "-I" + os.path.join(root, "include"), "-I/usr/local/cuda/include",
                    os.path.join(root, "tests", "cpp", src), "-o", exe, "-L" + libdir, "-ldfft",
                    "-L/usr/local/cuda/lib64", "-lcudart"] + (["-Xlinker", "-rpath," + libdir] if compiler_cmd[0].endswith("nvcc") else ["-Wl,-rpath," + libdir]),
                   check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "PASSED" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def test_cpp_shim_caller(tmp_path):
    """Reference-shaped C++ caller over include/dfft.hpp (MPIcuFFT_Slab<double> etc.): round trip + Laplacian, with
    plain cudaMemcpy from pageable memory right before the execs (no synchronisation)."""
    _build_and_run(tmp_path, ["g++"], "slab_shim_test.cpp", "slab_shim_test")


def test_cpp_shim_kernel_then_exec(tmp_path):
    """The reference's testcase 4 call pattern (random_dist_default.cu:704-724): cudaMemcpyAsync on the default stream,
    execR2C, a default-stream kernel scaling the spectrum, execC2R directly behind it — no host synchronisation.  The
    synchronous execs must be ordered behind the caller's default-stream work like cuFFT on the legacy stream."""
    _build_and_run(tmp_path, ["/usr/local/cuda/bin/nvcc", "-gencode", "arch=compute_100a,code=sm_100a"], "slab_shim_kernel_test.cu", "slab_shim_kernel_test")


def test_sync_exec_is_ordered_after_default_stream_work():
    """Fill / scale the buffers on torch's current (= legacy default) stream with a long-running kernel and call the
    synchronous execs without any host synchronisation in between."""
    shape = (256, 256, 256)
    plan = make_plan(dfft.MPIcuFFT_Slab, dfft.F64, dfft.R2C, shape)
    f = dev(O.sine_input(shape))
    out = torch.empty((256, 256, 129), dtype=torch.complex128, device="cuda")
    coef = dev(O.laplacian_coefficients(256, 256, 256, plan.getOutStart(), plan.getOutSize()))
    expect = O.laplacian_expected(shape)
    big = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
    for _ in range(3):
        x = torch.zeros_like(f)
        big.normal_()                      # ~ms of default-stream work queued in front ...
        x.copy_(f)                         # ... of the kernel that produces the input
        plan.execR2C(out, x)               # synchronous exec: must see the finished input
        big.normal_()
        out *= coef                        # default-stream kernel, then the inverse straight behind it
        back = torch.empty(shape, dtype=torch.float64, device="cuda")
        plan.execC2R(back, out)
        err = np.abs(host(back) - expect).max() / np.abs(expect).max()
        assert err < 1e-10  # rounding at 256^3 is ~5e-12 (k^2 amplification); a missed ordering edge gives O(1)
    plan.destroy()


def _gpu_rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    """relative L2 distance evaluated on the device in chunks (full-size arrays never travel to the host)"""
    a = a.reshape(-1); b = b.reshape(-1)
    num = 0.0; den = 0.0
    step = 1 << 26
    for i in range(0, a.numel(), step):
        d = (a[i:i + step] - b[i:i + step])
        num += float((d.real.double() ** 2 + d.imag.double() ** 2).sum()) if d.is_complex() else float((d.double() ** 2).sum())
        r = b[i:i + step]
        den += float((r.real.double() ** 2 + r.imag.double() ** 2).sum()) if r.is_complex() else float((r.double() ** 2).sum())
    return (num / den) ** 0.5


@pytest.mark.parametrize("case", FULL_SIZE_CASES)
def test_full_size_vs_cufft(case):
    """The reference's testcase 1 has no size cap (random_dist_default.cu:300-303,337,365-371): distributed result ==
    single-GPU cufftPlan3d.  BASELINE config 2 (512^3 complex-double), the single-GPU image of configs 3/5 (1024^3,
    R2C double incl. the inverse) and a 1024^3 complex-float pencil plan, compared at the positions stored in
    tests/golden/cufft_sample.npz and, when oracle/_ref/libcufft_ref.so is built, on the device element by element."""
    golden = np.load(CUFFT_GOLDEN)
    lib = cufft_lib()
    n, kind, pname, dec = case.split("_")
    n = int(n)
    prec = dfft.F64 if pname == "f64" else dfft.F32
    shape = (n, n, n)
    cls = {"slab": dfft.MPIcuFFT_Slab, "pencil": dfft.MPIcuFFT_Pencil, "zyx": dfft.MPIcuFFT_Slab_Z_Then_YX}[dec]
    part = dfft.Pencil_Partition(1, 1) if dec == "pencil" else None
    x = full_size_input(kind, prec, n)
    assert np.array_equal(sampled(x), golden[case + "_in"]), "torch's seeded generator no longer gives the stored input"
    ms = C.c_float()
    if kind == "c2c":
        plan = make_plan(cls, prec, dfft.C2C, shape, part)
        out = torch.empty_like(x)
        plan.execC2C(out, x, dfft.FORWARD)
    else:
        plan = make_plan(cls, prec, dfft.R2C, shape, part)
        out = torch.empty((n, n, n // 2 + 1), dtype=CDT[prec], device="cuda")
        plan.execR2C(out, x)
    assert O.rel_l2(sampled(out), golden[case]) < TOL[prec]
    if lib is not None:
        ref = torch.empty_like(out)
        assert lib.cufft_ref_3d(1 if prec == dfft.F64 else 0, 0 if kind == "c2c" else 2, n, n, n, ref.data_ptr(), x.data_ptr(), C.byref(ms), 1) == 0
        assert _gpu_rel_l2(out, ref) < TOL[prec]
        del ref
    back = torch.empty_like(x)
    if kind == "c2c":
        plan.execC2C(back, out, dfft.INVERSE)
    else:
        plan.execC2R(back, out)
    back /= float(n) ** 3
    assert _gpu_rel_l2(back, x) < TOL[prec]
    plan.destroy()
    del x, out, back
    torch.cuda.empty_cache()


def test_full_size_roundtrip_512():
    """BASELINE config 2 size (512^3 complex-double, one GPU): size-independent properties —
    forward->inverse round trip, Parseval, and linearity against a second input."""
    shape = (512, 512, 512)
    plan = make_plan(dfft.MPIcuFFT_Slab, dfft.F64, dfft.C2C, shape)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.complex(torch.rand(shape, generator=g, device="cuda", dtype=torch.float64), torch.rand(shape, generator=g, device="cuda", dtype=torch.float64))
    X = torch.empty_like(x)
    plan.execC2C(X, x, dfft.FORWARD)
    n = float(np.prod(shape))
    e_x = float((x.abs() ** 2).sum())
    e_X = float((X.abs() ** 2).sum())
    assert abs(e_X / (n * e_x) - 1) < 1e-12  # Parseval
    assert abs(complex(X[0, 0, 0]) - complex(x.sum())) / abs(complex(x.sum())) < 1e-12  # DC bin
    back = torch.empty_like(x)
    plan.execC2C(back, X, dfft.INVERSE)
    err = float((back / n - x).abs().max())
    assert err < 1e-12
    plan.destroy()


def test_timer_csv_schema(tmp_path):
    """Phase-timer CSV in the reference's on-disk schema (src/timer.cpp:58-101): header ',0,1,..,P-1,',
    one row per section, blank line between execs; warm-up execs are skipped; file name as in
    mpicufft_slab.cpp:99-103."""
    cfg = dfft.Configurations(warmup_rounds=1, benchmark_dir=str(tmp_path))
    plan = dfft.MPIcuFFT_Slab(cfg, dfft.Comm(), precision="double", transform="r2c")
    plan.initFFT(dfft.GlobalSize(32, 32, 32), None, True)
    x = dev(O.real_input((32, 32, 32)))
    out = torch.empty((32, 32, 17), dtype=torch.complex128, device="cuda")
    for _ in range(3):
        plan.execR2C(out, x)
    path = tmp_path / "slab_default" / "test_0_0_0_32_32_32_1_1.csv"
    assert path.exists()
    lines = path.read_text().split("\n")
    assert lines[0] == ",0,"
    blocks = [b for b in "\n".join(lines[1:]).split("\n\n") if b.strip()]
    assert len(blocks) == 2  # 3 execs - 1 warm-up
    rows = [r.split(",") for r in blocks[0].strip().split("\n")]
    names = [r[0] for r in rows]
    assert names[0] == "init" and names[-1] == "Run complete" and "2D FFT Y-Z-Direction" in names and "1D FFT X-Direction" in names
    assert len(names) == 14
    vals = {r[0]: float(r[1]) for r in rows}
    assert 0 < vals["2D FFT Y-Z-Direction"] <= vals["1D FFT X-Direction"] <= vals["Run complete"]
    steps = plan.stepTimes()
    assert [l for l, _ in steps] == ["z pass (R2C)", "y pass", "x pass"]
    plan.destroy()


def test_plan_tune_single_rank_has_no_alternatives():
    """dfft_plan_tune on one rank: nothing to choose (no exchange), the plan keeps working"""
    shape = (64, 32, 128)
    cfg = dfft.Configurations(send_method=dfft.SendMethod.Streams)
    plan = dfft.MPIcuFFT_Slab(cfg, dfft.Comm(), precision="double", transform="r2c")
    plan.initFFT(dfft.GlobalSize(*shape), None, True)
    x = dev(O.real_input(shape))
    out = torch.empty((64, 32, 65), dtype=torch.complex128, device="cuda")
    rep = plan.tune(out, x, dfft.FORWARD, 2)
    assert "no alternatives" in rep
    plan.execR2C(out, x)
    assert O.rel_l2(host(out), O.fft_r2c(host(x))) < 1e-10
    plan.destroy()


def test_step_timeline():
    """dfft_get_timeline: (label, stream, begin, end) of every step of the last timed exec"""
    shape = (64, 64, 64)
    plan = make_plan(dfft.MPIcuFFT_Slab, dfft.F64, dfft.C2C, shape)
    x = dev(O.complex_input(shape))
    out = torch.empty(shape, dtype=torch.complex128, device="cuda")
    plan.enableTimer(True)
    plan.execC2C(out, x, dfft.FORWARD)
    tl = plan.timeline()
    assert [l for l, _, _, _ in tl] == ["z pass", "y pass", "x pass"]
    assert all(st == 0 and 0 <= b <= e for _, st, b, e in tl)
    assert tl[0][3] <= tl[1][2] + 1e-3 and tl[1][3] <= tl[2][2] + 1e-3  # sequential schedule: one after the other
    plan.destroy()


@pytest.mark.parametrize("argv", [
    ["slab", "-nx", "64", "-ny", "64", "-nz", "64", "-t", "1", "-d"],
    ["slab", "-nx", "64", "-ny", "32", "-nz", "128", "-t", "3", "-s", "Z_Then_YX", "-i", "2"],
    ["slab", "-nx", "64", "-ny", "64", "-nz", "64", "-t", "4", "-d", "-comm", "All2All"],
    ["pencil", "-nx", "32", "-ny", "64", "-nz", "64", "-p1", "1", "-p2", "1", "-t", "1", "-f", "2", "-d"],
    ["pencil", "-nx", "64", "-ny", "64", "-nz", "64", "-p1", "1", "-p2", "1", "-t", "4", "-d"],
    ["slab", "-nx", "64", "-ny", "64", "-nz", "64", "-t", "0", "-i", "2", "-w", "1"],
    ["slab", "-nx", "64", "-ny", "64", "-nz", "64", "-t", "2", "-d"],
    ["slab", "-nx", "512", "-ny", "256", "-nz", "512", "-t", "1", "-d"],          # testcase 1 above 256^3: vs cufftPlan3d
    ["pencil", "-nx", "256", "-ny", "512", "-nz", "512", "-p1", "1", "-p2", "1", "-t", "1"],
])
def test_cli_testcases(argv, capsys):
    """The reference's CLI testcases 0-4 (tests/src/slab/main.cpp, tests/src/pencil/main.cpp) on one rank."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("dfft_cli", os.path.join(root, "tests", "cli.py"))
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    assert cli.main(argv) == 0
    out = capsys.readouterr().out
    assert "Result" in out or "Run complete" in out


def test_host_executor_pipeline():
    """HostExecutor: pinned host in -> device -> transform -> pinned host out, pipelined over submits."""
    shape = (32, 64, 128)
    plan = make_plan(dfft.MPIcuFFT_Slab, dfft.F64, dfft.R2C, shape)
    hx = dfft.HostExecutor(plan, dfft.FORWARD)
    ins = [O.real_input(shape, seed=s) for s in (1, 2, 3, 4, 5)]
    hin = [torch.from_numpy(a.copy()).pin_memory() for a in ins]
    hout = [torch.empty(32 * 64 * 65, dtype=torch.complex128).pin_memory() for _ in ins]
    for o, i in zip(hout, hin):
        hx.submit(o, i)
    hx.wait()
    for o, a in zip(hout, ins):
        assert O.rel_l2(o.numpy().reshape(32, 64, 65), O.fft_r2c(a)) < 1e-10
    # inverse through the host path
    hb = dfft.HostExecutor(plan, dfft.INVERSE)
    back = torch.empty(32 * 64 * 128, dtype=torch.float64).pin_memory()
    hb.submit(back, hout[2])
    hb.wait()
    assert O.rel_l2(back.numpy().reshape(shape), ins[2] * np.prod(shape)) < 1e-10
    plan.destroy()


def test_caller_supplied_work_area():
    """initFFT(.., allocate=false) + setWorkArea(device) — mpicufft_slab.cpp:236-281: the caller owns the arena."""
    shape = (32, 32, 64)
    plan = dfft.MPIcuFFT_Slab(dfft.Configurations(), dfft.Comm(), precision="double", transform="r2c")
    plan.initFFT(dfft.GlobalSize(*shape), None, False)
    x = dev(O.real_input(shape))
    out = torch.empty((32, 32, 33), dtype=torch.complex128, device="cuda")
    from distributedfft_b200._lib import DfftError
    with pytest.raises(DfftError):
        plan.execR2C(out, x)  # no work area yet
    arena = torch.empty(plan.getWorkSizeDevice(), dtype=torch.uint8, device="cuda")
    plan.setWorkArea(arena)
    assert plan.getWorkAreaDevice() == arena.data_ptr()
    plan.execR2C(out, x)
    assert O.rel_l2(host(out), O.fft_r2c(host(x))) < 1e-10
    plan.destroy()
    assert arena.numel() > 0  # still ours


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_against_committed_golden_vectors(name):
    """CUDA path vs tests/golden/golden_small.npz (generated by tests/golden/make_golden.py from the pinned oracle)."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_small.npz"))
    shape = tuple(int(v) for v in g[f"{name}_shape"])
    nzo = shape[2] // 2 + 1
    xr = O.real_input(shape, seed=1234)
    assert np.array_equal(xr.ravel()[:16], g[f"{name}_real_head"])
    plan = make_plan(dfft.MPIcuFFT_Pencil, dfft.F64, dfft.R2C, shape, dfft.Pencil_Partition(1, 1))
    out = torch.empty((shape[0], shape[1], nzo), dtype=torch.complex128, device="cuda")
    for d, key in ((3, "r2c"), (1, "r2c_d1"), (2, "r2c_d2")):
        plan.execR2C(out, dev(xr), d)
        assert O.rel_l2(host(out), g[f"{name}_{key}"]) < 1e-10, key
    plan.destroy()
    planc = make_plan(dfft.MPIcuFFT_Slab, dfft.F64, dfft.C2C, shape)
    outc = torch.empty(shape, dtype=torch.complex128, device="cuda")
    planc.execC2C(outc, dev(O.complex_input(shape, seed=1234)), dfft.FORWARD)
    assert O.rel_l2(host(outc), g[f"{name}_c2c"]) < 1e-10
    planc.destroy()
