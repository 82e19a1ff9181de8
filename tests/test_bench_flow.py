"""Runs bench.py's whole single-GPU control flow on the CPU with the CUDA bits and the library mocked, so that a
slip in the reporting code (it cannot be executed without a GPU otherwise) is caught by the CPU suite: the JSON line
must carry every key the contract names."""
import json
import os
import sys
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Event:
    def __init__(self, *a, **k): pass
    def record(self, *a): pass
    def elapsed_time(self, other): return 2.0
    def synchronize(self): pass


class _Stream:
    cuda_stream = 0
    def wait_event(self, e): pass
    def synchronize(self): pass


def _fake_dfft():
    m = types.ModuleType("distributedfft_b200")

    class CM:
        Peer2Peer, All2All = 0, 1

    class SM:
        Sync, Streams = 0, 1

    class Configurations:
        def __init__(self, **kw): self.__dict__.update(kw)

    class GlobalSize:
        def __init__(self, *s): self.s = s

    class Comm:
        @classmethod
        def from_torch_distributed(cls, dev=None): return cls()
        def destroy(self): pass

    class Plan:
        precision, transform = 1, 1
        def __init__(self, cfg, comm, precision="double", transform="c2c"): self.t = transform
        def initFFT(self, gs, part, alloc): self.s = gs.s
        def getInSize(self): return list(self.s)
        def getOutSize(self): return [self.s[0], self.s[1], self.s[2] if self.t == "c2c" else self.s[2] // 2 + 1]
        def getDomainSize(self): return self.s[0] * self.s[1] * self.s[2] * 16
        def execC2C(self, *a, **k): pass
        def execR2C(self, *a, **k): pass
        def execC2R(self, *a, **k): pass
        def wait(self): pass
        def lastLaunchCount(self): return 3
        def enableTimer(self, on): pass
        def stepTimes(self): return [("z pass", 0.5), ("y pass", 0.7), ("x pass", 0.6)]
        def phaseTimes(self): return [("2D FFT Y-Z-Direction", 1.2), ("1D FFT X-Direction", 1.8), ("Run complete", 1.8)]
        def lastBreakdown(self): return {"fft_ms": 1.8, "exchange_ms": 0.0, "total_ms": 1.8}
        def destroy(self): pass

    class HostExecutor:
        def __init__(self, plan, direction):
            self.s_in, self.s_out, self.count = _Stream(), _Stream(), 0
            self.d_out = [torch.zeros(2048, dtype=torch.complex128)] * 2
        def submit(self, o, i): self.count += 1
        def wait(self): pass

    m.CommunicationMethod, m.SendMethod, m.Configurations, m.GlobalSize, m.Comm = CM, SM, Configurations, GlobalSize, Comm
    m.MPIcuFFT_Slab = m.MPIcuFFT_Slab_Z_Then_YX = m.MPIcuFFT_Pencil = Plan
    m.Pencil_Partition = lambda a, b: (a, b)
    m.HostExecutor = HostExecutor
    m.pinned_empty = lambda n, dtype, device=None: torch.empty(n, dtype=dtype)
    m.gpu_local_cpus = lambda device: None
    m.FORWARD, m.INVERSE = -1, 1
    return m


@pytest.mark.parametrize("extra", [[], ["--transform", "r2c"], ["--no-e2e", "--no-cpu"], ["WORLD=8"], ["WORLD=8", "--decomp", "pencil", "--p1", "2", "--p2", "4", "--prec", "f32"],
                                   ["WORLD=2", "--comm", "All2All", "--send", "Sync"], ["--dump-outputs", "DUMP"]])
def test_bench_single_gpu_flow_with_mocks(monkeypatch, capsys, tmp_path, extra):
    extra = [str(tmp_path / "dump") if a == "DUMP" else a for a in extra]
    world = 1
    if extra and extra[0].startswith("WORLD="):
        world = int(extra.pop(0).split("=")[1])
    monkeypatch.setitem(sys.modules, "distributedfft_b200", _fake_dfft())
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: _Stream())
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)
    real_gen, real_rand, real_empty, real_tensor = torch.Generator, torch.rand, torch.empty, torch.tensor

    def strip(kw):
        kw.pop("device", None); kw.pop("pin_memory", None)
        return kw
    monkeypatch.setattr(torch, "Generator", lambda *a, **k: real_gen())
    monkeypatch.setattr(torch, "rand", lambda *a, **k: real_rand(*a, **strip(k)))
    monkeypatch.setattr(torch, "empty", lambda *a, **k: real_empty(*a, **strip(k)))
    monkeypatch.setattr(torch, "tensor", lambda *a, **k: real_tensor(*a, **strip(k)))
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(torch.Tensor, "data_ptr", lambda self: 0)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    monkeypatch.delenv("RANK", raising=False)
    if world > 1:  # one rank of a torchrun launch, torch.distributed mocked
        import torch.distributed as dist
        monkeypatch.setenv("WORLD_SIZE", str(world)); monkeypatch.setenv("RANK", "0"); monkeypatch.setenv("LOCAL_RANK", "0")
        monkeypatch.setattr(dist, "is_initialized", lambda: True)
        monkeypatch.setattr(dist, "barrier", lambda *a, **k: None)
        monkeypatch.setattr(dist, "all_reduce", lambda *a, **k: None)
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    monkeypatch.setattr(bench, "ClockSampler", lambda idx: types.SimpleNamespace(stop=lambda: {"sm_mhz": 1900.0, "sm_max_mhz": 1965.0, "reasons": []}))
    monkeypatch.setattr(bench, "DUMP_VALUES", 1000)  # below the 32^3 block: the sampled path
    monkeypatch.setattr(bench, "cpu_fft_sample", lambda shape, reps=1, cores=None: (0.5, 8, "mock sample", 7.5))
    monkeypatch.setattr(os.path, "exists", lambda p, _e=os.path.exists: False if p.endswith("libcufft_ref.so") else _e(p))
    if world > 1:
        # per-step labels of a multi-rank slab / pencil plan
        steps = [("entry rendezvous", 0.02), ("z pass", 0.6), ("y pass", 2.7), ("rendezvous 2", 0.01), ("x pass", 0.9)]
        if "All2All" in extra:
            steps = [("z pass", 0.6), ("y pass", 1.0), ("nccl all-to-all", 3.2), ("x pass", 0.9)]
        monkeypatch.setattr(sys.modules["distributedfft_b200"].MPIcuFFT_Slab, "stepTimes", lambda self: steps)
        monkeypatch.setattr(sys.modules["distributedfft_b200"].MPIcuFFT_Slab, "lastBreakdown", lambda self: {"fft_ms": 4.2, "exchange_ms": 0.03, "total_ms": 4.3})
    bench.main(["--gpus", str(world), "--steps", "4", "--warmup", "3", "--shape", "32,32,32", "--no-parity", *extra])
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == world and line["gpu_launches"] == 12 and line["config"]["workload"].startswith("32x32x32")
    if world > 1:
        nv = line["roofline"]["nvlink"]
        nv = nv if isinstance(nv, list) else [nv]
        assert all(x["gbs_per_direction"] and x["gbs_per_direction"] > 0 for x in nv)
        assert len(nv) == (2 if "pencil" in extra else 1)
        assert line["cpu_baseline"] is None and line["config"]["send_method"] == ("Sync" if "Sync" in extra else "Streams")
        return
    if "--dump-outputs" in extra:
        import numpy as np
        a = np.load(tmp_path / "dump" / "spectrum_rank0.npy")
        assert a.dtype == np.float64 and a.shape == (1000, 2)
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in line["roofline"]
    if "--no-e2e" not in extra:
        assert set(("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step")) <= set(line["e2e"])
        assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == 8
    else:
        assert line["e2e"] is None and line["cpu_baseline"] is None
