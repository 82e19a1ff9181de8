#!/usr/bin/env python
"""bench.py — distributed 3D FFT throughput on B200 (BASELINE.json metric: GFLOP/s = 5*Ntot*log2(Ntot)/t
for a complex transform, and ms/transform).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (libdfft.so)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port (scipy pocketfft)
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # one rank per GPU, NCCL / NVLink peer stores
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's spectrum (seeded sample)

A step is ONE forward complex-double 3D transform of the workload grid through the reference-shaped plan
API (MPIcuFFT_Slab.execC2C).  Workload (weak scaling, 512^3 points per GPU — BASELINE configs[1] at N=1,
configs[2] at N=8): N=1 512x512x512, N=2 1024x512x512, N=4 1024x1024x512, N=8 1024x1024x1024, slab
decomposition (2D y,z FFT -> transpose -> 1D x FFT).  Inputs are synthetic uniform[0,255) complex
values, resident in HBM for `value`; `e2e` adds the pinned-host -> device copy of the input block and the
device -> host copy of the spectrum block inside the timed region.  Arrays are >= 2 GiB per GPU, far
larger than the 126 MB L2, so no L2 flush is needed between iterations.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WEAK_SHAPES = {1: (512, 512, 512), 2: (1024, 512, 512), 4: (1024, 1024, 512), 8: (1024, 1024, 1024)}


def workload_name(shape, prec="f64", transform="c2c", decomp="slab"):
    """config.workload — the SAME string in both arms (ours and --impl reference)."""
    return (f"{shape[0]}x{shape[1]}x{shape[2]} complex-{'double' if prec == 'f64' else 'float'} "
            f"{'C2C' if transform == 'c2c' else 'R2C'} forward 3D FFT, {decomp} decomposition")


def metric_name(transform="c2c"):
    return ("3D FFT GFLOP/s (5*Ntot*log2(Ntot)/t, complex-double forward)" if transform == "c2c"
            else "3D FFT GFLOP/s (2.5*Ntot*log2(Ntot)/t, R2C forward)")


def flops_c2c(shape):
    n = shape[0] * shape[1] * shape[2]
    return 5.0 * n * math.log2(n)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(gpu_index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            # "under load": upper half of the samples
            load = sm[len(sm) // 2:]
            out["sm_mhz"] = load[len(load) // 2]
            out["sm_max_mhz"] = max(mx)
            out["samples"] = len(sm)
        out["reasons"] = sorted(reasons)
        return out


DUMP_VALUES = 1 << 21  # complex values written by --dump-outputs over all ranks: 32 MiB as float64 pairs


def dump_outputs(path, out, osz, rank, world):
    """--dump-outputs: the spectrum block that the last timed forward step left in `out`, as <path>/spectrum_rank<r>.npy,
    float64 [n, 2] (real, imag).  A block of more than DUMP_VALUES / world values is sampled at fixed positions (the
    sorted flat indices drawn by a seed-0 generator), so two builds with the same arguments compare value for value."""
    import numpy as np
    import torch

    n = osz[0] * osz[1] * osz[2]
    k = DUMP_VALUES // world
    flat = out[:n]
    if n > k:
        idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"spectrum_rank{rank}.npy"), torch.view_as_real(flat).to(torch.float64).cpu().numpy())


_CPU_INPUT = {}


def claim_all_cores():
    """The CPU arm must use every host core it can.  Launchers clamp it: torchrun exports OMP_NUM_THREADS=1 and a
    parent may have pinned this process.  Undo both before numpy / scipy are imported; report what we got."""
    n = os.cpu_count() or 1
    try:
        os.sched_setaffinity(0, range(n))
    except Exception:
        pass
    try:
        usable = len(os.sched_getaffinity(0))
    except Exception:
        usable = n
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[k] = str(usable)
    return usable


def cpu_fft_sample(shape, reps=1, cores=None):
    """The CPU arm: oracle port = pocketfft (scipy.fft.fftn, all usable host cores) on complex128.
    Returns (seconds per transform, cores asked for, sample description, effective parallelism = CPU time / wall time).
    The synthetic input is generated once."""
    import resource

    import numpy as np
    import scipy.fft as sfft

    cores = cores or claim_all_cores()
    x = _CPU_INPUT.get(shape)
    if x is None:
        rng = np.random.default_rng(0)
        x = np.empty(shape, dtype=np.complex128)
        x.real = rng.random(shape) * 255
        x.imag = rng.random(shape) * 255
        _CPU_INPUT.clear()
        _CPU_INPUT[shape] = x
    best, par = None, None
    for _ in range(reps):
        r0 = resource.getrusage(resource.RUSAGE_SELF)
        t0 = time.perf_counter()
        y = sfft.fftn(x, workers=cores)
        dt = time.perf_counter() - t0
        r1 = resource.getrusage(resource.RUSAGE_SELF)
        if best is None or dt < best:
            best = dt
            par = ((r1.ru_utime - r0.ru_utime) + (r1.ru_stime - r0.ru_stime)) / dt
        del y
    return best, cores, f"scipy.fft.fftn {shape[0]}x{shape[1]}x{shape[2]} complex128, workers={cores}", par


def bounded_cpu_shape(shape):
    # cap the CPU sample at 512^3 points (a few seconds of pocketfft on a host's cores); GFLOP/s is size-normalised
    s = list(shape)
    while s[0] * s[1] * s[2] > 512 ** 3:
        k = max(range(3), key=lambda i: s[i])
        s[k] //= 2
    return tuple(s)


def run_reference(args, shape):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = claim_all_cores()
    cshape = bounded_cpu_shape(shape)
    for _ in range(args.warmup):
        cpu_fft_sample(cshape, cores=cores)
    t0 = time.perf_counter()
    secs, pars = [], []
    for _ in range(args.steps):
        sec, cores, desc, par = cpu_fft_sample(cshape, cores=cores)
        secs.append(sec)
        pars.append(par)
    total = time.perf_counter() - t0
    sec = sum(secs) / len(secs)      # transform time only (input generation is outside the timed region)
    ms = sec * 1e3
    val = flops_c2c(cshape) / sec / 1e9
    sample = desc if cshape == tuple(shape) else desc + f" (bounded sample of the {shape[0]}x{shape[1]}x{shape[2]} workload; GFLOP/s is size-normalised)"
    line = {
        "impl": "reference", "metric": metric_name("c2c"), "value": val, "unit": "GFLOP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(shape, args.prec, args.transform, args.decomp), "cpu_sample": sample,
                   "threads_used": cores, "threads_effective": sum(pars) / len(pars), "host_cpus": os.cpu_count(),
                   "note": "the reference has no CPU path (MPI+cuFFT only, SURVEY.md F1); this arm is the oracle port, pocketfft on the host cores"},
        "cpu_baseline": {"value": val, "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": total,
    }
    print(json.dumps(line), flush=True)



def parity_check(dfft, make_plan_for, comm_world, rank, world, local, prec, transform, decomp, full_plan, full_in, full_out):
    """Driver-visible correctness BEFORE the timed region, on every rank:
      (a) a 256-point-edge global grid of the same decomposition / precision / exchange path, filled with the oracle's
          index-hashed input, each rank's output block against numpy's 3D transform (the oracle);
      (b) at the full workload size, on the very buffers that are timed: DC bin = sum of the input, and Parseval
          (sum |X|^2 = N * sum |x|^2; R2C: Hermitian weights) reduced over all ranks.
    Returns a dict; ok == False makes bench.py exit non-zero."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from oracle import dft_oracle as O

    f64 = prec == "f64"
    tol = 1e-10 if f64 else 1e-5
    c2c = transform == "c2c"
    res = {"tolerance": tol}
    # (a) small global grid against the oracle
    small = (256, 256, 256) if world <= 8 else (512, 256, 256)
    plan, _ = make_plan_for(small)
    isz, ist, osz, ost = plan.getInSize(), plan.getInStart(), plan.getOutSize(), plan.getOutStart()
    cdt = torch.complex128 if f64 else torch.complex64
    es = 16 if f64 else 8
    if c2c:
        xg = O.complex_input(small)
        ref = O.fft_c2c(xg)
        xin = torch.from_numpy(np.ascontiguousarray(O.block(xg, ist, isz)).astype(np.complex128 if f64 else np.complex64)).cuda()
    else:
        xg = O.real_input(small)
        ref = O.fft_r2c(xg)
        xin = torch.from_numpy(np.ascontiguousarray(O.block(xg, ist, isz)).astype(np.float64 if f64 else np.float32)).cuda()
    out = torch.empty(plan.getDomainSize() // es, dtype=cdt, device="cuda")
    n_out = osz[0] * osz[1] * osz[2]
    stream = torch.cuda.current_stream()
    if c2c:
        plan.execC2C(out, xin, dfft.FORWARD, stream=stream)
    else:
        plan.execR2C(out, xin, stream=stream)
    plan.wait()
    got = out[:n_out].cpu().numpy().reshape(osz)
    blk = O.block(ref, ost, osz)
    err = float(np.linalg.norm((got - blk).ravel()) / np.linalg.norm(blk.ravel()))
    # inverse of the oracle's block must give back the input block (unnormalised)
    back = torch.empty_like(xin)
    spec = torch.zeros_like(out)
    spec[:n_out] = torch.from_numpy(np.ascontiguousarray(blk).astype(np.complex128 if f64 else np.complex64)).cuda().reshape(-1)
    if c2c:
        plan.execC2C(back, spec, dfft.INVERSE, stream=stream)
    else:
        plan.execC2R(back, spec, stream=stream)
    plan.wait()
    nsm = float(small[0] * small[1] * small[2])
    xin_h = xin.cpu().numpy().astype(np.complex128 if c2c else np.float64)
    err_inv = float(np.linalg.norm((back.cpu().numpy() / nsm - xin_h).ravel()) / np.linalg.norm(xin_h.ravel()))
    plan.destroy()
    del out, spec, back, xin
    t = torch.tensor([err, err_inv], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["small_grid"] = {"shape": list(small), "rel_l2_forward_max_over_ranks": float(t[0]), "rel_l2_inverse_max_over_ranks": float(t[1]),
                         "checker": "numpy fftn / rfftn on the oracle's index-hashed input (oracle/dft_oracle.py)"}
    ok = float(t[0]) < tol and float(t[1]) < tol
    # (b) full size, the timed buffers
    osz = full_plan.getOutSize()
    ost = full_plan.getOutStart()
    n_out = osz[0] * osz[1] * osz[2]
    if c2c:
        full_plan.execC2C(full_out, full_in, dfft.FORWARD, stream=stream)
    else:
        full_plan.execR2C(full_out, full_in, stream=stream)
    full_plan.wait()
    X = full_out[:n_out].reshape(osz)
    sx = full_in.sum().to(torch.complex128)
    e_in = (full_in.abs().double() ** 2).sum() if c2c else (full_in.double() ** 2).sum()
    if c2c:
        e_out = (X.real.double() ** 2 + X.imag.double() ** 2).sum()
    else:
        # Hermitian half spectrum: bins kz = 0 and kz = Nz/2 count once, the others twice
        p2 = X.real.double() ** 2 + X.imag.double() ** 2
        w = torch.full((osz[2],), 2.0, device="cuda", dtype=torch.float64)
        gz0 = ost[2]
        nzc_global = full_plan.global_size.Nz // 2 + 1
        for k in range(osz[2]):
            if gz0 + k == 0 or gz0 + k == nzc_global - 1:
                w[k] = 1.0
        e_out = (p2 * w).sum()
    dc = X[0, 0, 0].to(torch.complex128) if (ost[0] == 0 and ost[1] == 0 and ost[2] == 0) else torch.zeros((), dtype=torch.complex128, device="cuda")
    v = torch.stack([sx.real, sx.imag, e_in.to(torch.float64), e_out.to(torch.float64), dc.real, dc.imag])
    if world > 1:
        dist.all_reduce(v)
    gs = full_plan.global_size
    ntot = float(gs.Nx) * gs.Ny * gs.Nz
    s_in = complex(float(v[0]), float(v[1]))
    dcv = complex(float(v[4]), float(v[5]))
    dc_err = abs(dcv - s_in) / abs(s_in)
    pars_err = abs(float(v[3]) / (ntot * float(v[2])) - 1.0)
    res["full_size"] = {"shape": [gs.Nx, gs.Ny, gs.Nz], "dc_bin_rel_err": dc_err, "parseval_rel_err": pars_err,
                        "note": "on the timed buffers: X[0,0,0] == sum(x), sum|X|^2 == N sum|x|^2, reduced over all ranks"}
    tol_full = 1e-10 if f64 else 2e-4  # f32 sums over 2^29+ values in float32 accumulate rounding
    ok = ok and dc_err < tol_full and pars_err < tol_full
    res["ok"] = bool(ok)
    return res


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="dfft", choices=["dfft", "reference"])
    ap.add_argument("--shape", default=None, help="Nx,Ny,Nz (default: weak-scaling table)")
    ap.add_argument("--decomp", default="slab", choices=["slab", "z_then_yx", "pencil"])
    ap.add_argument("--p1", type=int, default=0)
    ap.add_argument("--p2", type=int, default=0)
    ap.add_argument("--comm", default="Peer2Peer", choices=["Peer2Peer", "All2All"])
    ap.add_argument("--send", default="auto", choices=["auto", "Sync", "Streams"], help="Streams = overlapped schedule (default for N > 1)")
    ap.add_argument("--prec", default="f64", choices=["f64", "f32"])
    ap.add_argument("--transform", default="c2c", choices=["c2c", "r2c"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-tune", action="store_true", help="keep the default overlapped schedule instead of measuring the candidates at plan time")
    ap.add_argument("--no-parity", action="store_true", help="skip the correctness checks in front of the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output block (sampled above 2M values) to DIR/spectrum_rank<r>.npy")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "dfft" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.shape:
        shape = tuple(int(v) for v in args.shape.split(","))
    else:
        n = args.gpus
        shape = WEAK_SHAPES.get(n, (512 * n, 512, 512))
    if args.impl == "reference":
        return run_reference(args, shape)

    import numpy as np
    import torch
    import torch.distributed as dist

    import distributedfft_b200 as dfft

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    own_pg = False
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        own_pg = True
    comm = dfft.Comm.from_torch_distributed(local)
    f64 = args.prec == "f64"
    cdt = torch.complex128 if f64 else torch.complex64
    rdt = torch.float64 if f64 else torch.float32
    es = 16 if f64 else 8
    cm = dfft.CommunicationMethod.Peer2Peer if args.comm == "Peer2Peer" else dfft.CommunicationMethod.All2All
    send = args.send if args.send != "auto" else ("Streams" if world > 1 else "Sync")
    sm = dfft.SendMethod.Streams if send == "Streams" else dfft.SendMethod.Sync
    cfg = dfft.Configurations(comm_method=cm, comm_method2=cm, send_method=sm)
    c2c = args.transform == "c2c"

    def make_plan(config, shape=shape):
        if args.decomp == "pencil":
            p1 = args.p1 or (2 if world >= 2 else 1)
            p2 = args.p2 or world // p1
            pl = dfft.MPIcuFFT_Pencil(config, comm, precision="double" if f64 else "float", transform=args.transform)
            pl.initFFT(dfft.GlobalSize(*shape), dfft.Pencil_Partition(p1, p2), True)
            return pl, f"pencil{p1}x{p2}"
        cls = dfft.MPIcuFFT_Slab if args.decomp == "slab" else dfft.MPIcuFFT_Slab_Z_Then_YX
        pl = cls(config, comm, precision="double" if f64 else "float", transform=args.transform)
        pl.initFFT(dfft.GlobalSize(*shape), None, True)
        return pl, f"{args.decomp}{world}"

    plan, par = make_plan(cfg)
    isz, osz = plan.getInSize(), plan.getOutSize()
    n_in = isz[0] * isz[1] * isz[2]
    dom = plan.getDomainSize() // es
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    if c2c:
        x = torch.complex(torch.rand(n_in, generator=g, device="cuda", dtype=rdt) * 255, torch.rand(n_in, generator=g, device="cuda", dtype=rdt) * 255)
    else:
        x = torch.rand(n_in, generator=g, device="cuda", dtype=rdt) * 255
    out = torch.empty(dom, dtype=cdt, device="cuda")
    stream = torch.cuda.current_stream()

    def step():
        if c2c:
            plan.execC2C(out, x, dfft.FORWARD, stream=stream)
        else:
            plan.execR2C(out, x, stream=stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    tuned = None
    if world > 1 and send == "Streams" and not args.no_tune and hasattr(plan, "tune"):
        # plan-time measurement (dfft_plan_tune): sequential vs overlapped schedules with different SM shares for the
        # exchanging pass, on the buffers of this run; the choice is fixed before any timed step
        tuned = {"forward": plan.tune(out, x, dfft.FORWARD, 3)}
    parity = None
    if not args.no_parity:
        parity = parity_check(dfft, lambda shp: make_plan(cfg, shp), comm, rank, world, local, args.prec, args.transform, args.decomp, plan, x, out)
        if not parity["ok"]:
            if rank == 0:
                print(json.dumps({"error": "parity check failed", "parity": parity}), flush=True)
            sys.exit(3)
    for _ in range(args.warmup):
        step()
    plan.wait()
    sampler = ClockSampler(local) if rank == 0 else None  # keeps sampling through the breakdown and e2e loops
    total_ms = timed(step, args.steps)
    plan.wait()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, osz, rank, world)
    launches = plan.lastLaunchCount() * args.steps
    ms_step = total_ms / args.steps
    # inverse transform of the same grid (reported beside the headline; BASELINE config 1 names forward+inverse)
    inv_steps = max(3, min(args.steps, 10))
    back = torch.empty_like(x)
    if tuned is not None:
        tuned["inverse"] = plan.tune(back, out, dfft.INVERSE, 3)  # the inverse leaves its input (the spectrum) intact
    if c2c:
        inv = lambda: plan.execC2C(back, out, dfft.INVERSE, stream=stream)
    else:
        inv = lambda: plan.execC2R(back, out, stream=stream)
    for _ in range(2):
        inv()
    plan.wait()
    ms_inverse = timed(inv, inv_steps) / inv_steps
    plan.wait()
    del back
    step()  # restore the forward result in `out`
    plan.wait()
    fl = flops_c2c(shape) * (1.0 if c2c else 0.5)
    value = fl / (ms_step * 1e-3) / 1e9

    # per-step breakdown (separate loop: CUDA events between the steps of one exec).  The overlapped
    # (Streams) schedule has no meaningful per-step times, so the breakdown runs the sequential schedule.
    if send == "Streams":
        bplan, _ = make_plan(dfft.Configurations(comm_method=cm, comm_method2=cm, send_method=dfft.SendMethod.Sync))
    else:
        bplan = plan

    def bstep():
        if c2c:
            bplan.execC2C(out, x, dfft.FORWARD, stream=stream)
        else:
            bplan.execR2C(out, x, stream=stream)

    bplan.enableTimer(True)
    reps = max(3, min(10, args.steps))
    acc_steps, acc_cum, bd_acc = None, None, None
    for _ in range(reps):
        barrier()
        bstep()
        bplan.wait()
        st = bplan.stepTimes()
        pt = bplan.phaseTimes()
        bd = bplan.lastBreakdown()
        acc_steps = [t for _, t in st] if acc_steps is None else [a + t for a, (_, t) in zip(acc_steps, st)]
        acc_cum = [t for _, t in pt] if acc_cum is None else [a + t for a, (_, t) in zip(acc_cum, pt)]
        bd_acc = dict(bd) if bd_acc is None else {k: bd_acc[k] + bd[k] for k in bd}
    bplan.enableTimer(False)
    seq_ms = bd_acc["total_ms"] / reps
    if bplan is not plan:
        bplan.destroy()
    timeline = None
    if send == "Streams" and hasattr(plan, "timeline"):
        # where every step of the overlapped schedule ran (stream, begin, end) — rank 0's view of one exec
        plan.enableTimer(True)
        for _ in range(2):
            barrier()
            step()
            plan.wait()
        try:
            timeline = [{"step": l, "stream": st_, "begin_ms": round(b0, 4), "end_ms": round(e0, 4)} for l, st_, b0, e0 in plan.timeline()]
        except Exception:
            timeline = None
        plan.enableTimer(False)
    labels = [n for n, _ in st]
    step_ms = [a / reps for a in acc_steps]
    names = [n for n, _ in pt]
    cum = [a / reps for a in acc_cum]
    bd_avg = {k: v / reps for k, v in bd_acc.items()}
    hbm_peak, peak_src = measured_peaks()
    ntot_local = shape[0] * shape[1] * shape[2] / world
    nzc = shape[2] if c2c else shape[2] // 2 + 1
    cplx_bytes = es * shape[0] * shape[1] * nzc / world   # one complex array of the local share
    real_bytes = (es // 2) * ntot_local
    passes = []
    for lab, ms in zip(labels, step_ms):
        if "pass" not in lab or "tail" in lab:
            continue
        if lab.startswith("z pass") and not c2c:
            b = real_bytes + cplx_bytes          # R2C: read reals, write Nz/2+1 complex
        else:
            b = 2.0 * cplx_bytes                 # one read + one write of the local complex array
        passes.append({"step": lab, "ms": ms, "algorithmic_bytes": b, "gbs": b / (ms * 1e-3) / 1e9, "frac": b / (ms * 1e-3) / 1e9 / hbm_peak})
    fft_ms = bd_avg["fft_ms"]
    tot_bytes = sum(q["algorithmic_bytes"] for q in passes)
    # HBM roofline: the dominant LOCAL pass.  With peers the scattering passes (slab: y; pencil: z and y) are bound by
    # NVLink, not HBM — they are reported in roofline.nvlink against the link peak instead.
    if world > 1 and args.comm == "Peer2Peer":
        xch = ("y pass",) if args.decomp == "slab" else (("z pass", "z pass (R2C)") if args.decomp == "z_then_yx" else ("z pass", "z pass (R2C)", "y pass"))
        local = [q for q in passes if q["step"] not in xch] or passes
    else:
        local = passes
    dom = max(local, key=lambda q: q["ms"])
    # DRAM bytes per launch of the dominant pass, read from the committed ncu --set full capture of this workload
    # (profiles/r02/bench_traffic.json, written from profiles/r02/ncu_full_final_kernels.csv); null for other workloads
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02", "bench_traffic.json")))
        key = f"{shape[0]}x{shape[1]}x{shape[2]} {args.prec} {args.transform} {args.decomp} n{world}"
        traffic = tj["workloads"].get(key, {}).get(dom["step"])
    except Exception:
        traffic = None
    roofline = {"bound": "hbm", "achieved": dom["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["frac"], "traffic": traffic,
                "peak_source": peak_src, "kernel": f"dominant FFT pass: {dom['step']} ({dom['ms']:.3f} ms per launch; algorithmic bytes = one read + one write of the local array)",
                "all_passes": passes, "all_passes_achieved": tot_bytes / (fft_ms * 1e-3) / 1e9, "all_passes_frac": tot_bytes / (fft_ms * 1e-3) / 1e9 / hbm_peak,
                "fft_ms": fft_ms, "exchange_ms": bd_avg["exchange_ms"], "steps_ms": dict(zip([f"{i}:{l}" for i, l in enumerate(labels)], step_ms)),
                "phases_cumulative_ms": dict(zip(names, cum)), "overlap_timeline": timeline}
    if world > 1:
        def link(sent, t_x, note):
            return {"bytes_sent_per_gpu": sent, "transfer_ms": t_x, "gbs_per_direction": (sent / (t_x * 1e-3) / 1e9) if t_x else None,
                    "peak_nominal": 900.0, "peak_measured_peer_copy": 770.0, "eff_vs_nominal": (sent / (t_x * 1e-3) / 1e9 / 900.0) if t_x else None,
                    "note": note}
        a2a = [ms for lab, ms in zip(labels, step_ms) if "all-to-all" in lab]
        pass_ms = {q["step"]: q["ms"] for q in passes}
        if args.decomp == "pencil":
            p1 = args.p1 or 2
            p2 = args.p2 or world // p1
            t1 = a2a[0] if a2a else next((ms for lab, ms in pass_ms.items() if lab.startswith("z pass")), None)
            t2 = a2a[1] if len(a2a) > 1 else pass_ms.get("y pass")
            roofline["nvlink"] = [link(cplx_bytes * (p2 - 1) / p2, t1, "first transposition (row group): scattered by the z pass (Peer2Peer) or NCCL step"),
                                  link(cplx_bytes * (p1 - 1) / p1, t2, "second transposition (column group): scattered by the y pass (Peer2Peer) or NCCL step")]
        else:
            t_x = max(a2a) if a2a else (pass_ms.get("y pass") if args.decomp == "slab" else next((ms for lab, ms in pass_ms.items() if lab.startswith("z pass")), None))
            roofline["nvlink"] = link(cplx_bytes * (world - 1) / world, t_x,
                                      "Peer2Peer: the scattering pass stores straight into the peers' slots, so its duration is the transfer time")

    cpu = None
    cufft_ms = None
    if rank == 0 and world == 1:
        if not args.no_cpu:
            cs = bounded_cpu_shape(shape)
            sec, cores, desc, eff_par = cpu_fft_sample(cs, reps=1)
            cpu = {"value": flops_c2c(cs) / sec / 1e9, "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": desc, "ms": sec * 1e3,
                   "threads_effective": eff_par}
        ref = os.path.join(ROOT, "oracle", "_ref", "libcufft_ref.so")
        if os.path.exists(ref):
            try:
                lib = C.CDLL(ref)
                lib.cufft_ref_3d.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_float), C.c_int]
                msf = C.c_float()
                if lib.cufft_ref_3d(1 if f64 else 0, 0 if c2c else 2, shape[0], shape[1], shape[2], out.data_ptr(), x.data_ptr(), C.byref(msf), 10) == 0:
                    cufft_ms = float(msf.value)
            except Exception:
                cufft_ms = None

    # end-to-end through the public host-buffer API (HostExecutor): every step copies its input block from pinned
    # host memory, transforms it and copies the spectrum block back; consecutive steps are pipelined (the D2H of
    # step i overlaps the H2D of step i+1), all inside the timed region
    def run_e2e():
        hin = dfft.pinned_empty(x.numel(), x.dtype, local)   # pages on the GPU's own NUMA node
        hin.copy_(x)
        n_out = osz[0] * osz[1] * osz[2]
        hout = dfft.pinned_empty(n_out, cdt, local)
        hx = dfft.HostExecutor(plan, dfft.FORWARD)
        for _ in range(2):
            hx.submit(hout, hin)
        hx.wait()
        ksteps = max(3, min(args.steps, 10))
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(hx.s_in)
        for _ in range(ksteps):
            hx.submit(hout, hin)
        e1.record(hx.s_out)
        hx.wait()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        tms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        t = float(tms.item()) / ksteps
        # sanity: the spectrum that arrived on the host is the device result
        chk = float((hout[:1024].cuda() - hx.d_out[(hx.count - 1) & 1][:1024]).abs().max())
        return {"value": fl / (t * 1e-3) / 1e9, "unit": "GFLOP/s", "ms_per_step": t, "wall_ms_per_step": wall_ms / ksteps,
                "h2d_bytes_per_step": int(x.numel() * x.element_size() * world), "d2h_bytes_per_step": int(n_out * es * world),
                "pipeline": "H2D(i+1) overlaps D2H(i); 2 device buffer sets", "host_equals_device": chk == 0.0,
                "pinned_numa_cpus": len(dfft.gpu_local_cpus(local) or []) or None}

    def make_line(e2e, clocks):
        return {
            "metric": metric_name(args.transform),
            "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.prec, "data": "synthetic",
            "config": {"workload": workload_name(shape, args.prec, args.transform, args.decomp),
                       "parallelism": par, "parity": parity, "tuned_schedule": tuned, "comm_method": args.comm, "send_method": send, "sequential_schedule_ms": seq_ms, "ms_inverse": ms_inverse, "points_per_gpu": int(ntot_local),
                       "l2_policy": "inputs (>= 2 GiB per GPU) exceed the 126 MB L2; no flush needed",
                       "gflops_literal_5N3log2N_edge": (5.0 * shape[0] * shape[1] * shape[2] * math.log2(shape[0]) / (ms_step * 1e-3) / 1e9)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "cufft_1gpu_ms": cufft_ms,
        }

    # The e2e leg runs last and is guarded: should it fail or stall on some rank, the measured line is still printed.
    e2e = None
    if not args.no_e2e:
        import threading
        finished = threading.Event()

        def watchdog():
            if not finished.wait(240):
                if rank == 0:
                    print(json.dumps(make_line({"error": "e2e leg did not finish within 240 s"}, sampler.stop() if sampler else None)), flush=True)
                os._exit(0)

        threading.Thread(target=watchdog, daemon=True).start()
        try:
            e2e = run_e2e()
        except Exception as ex:  # report, do not lose the device-resident measurement
            finished.set()
            if rank == 0:
                print(json.dumps(make_line({"error": repr(ex)[:300]}, sampler.stop() if sampler else None)), flush=True)
            os._exit(0)
        finished.set()
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        print(json.dumps(make_line(e2e, clocks)), flush=True)
    plan.destroy()
    comm.destroy()
    del x, out
    torch.cuda.empty_cache()
    if own_pg:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
