"""bench.py's measurement loops executed on the CPU (stand-in device at the C-ABI boundary, gloo, small state): the driver runs
bench.py on boxes this container cannot reach, so every leg both arms share -- api_loop, the local-manager leg, the JSON
assembly helpers -- is at least executed here.  Numbers are meaningless; only "it runs and verifies" is checked."""
import sys
import types
from pathlib import Path

import pytest
import torch

from _fake_device import FakeCudaTensor, fake_device

ROOT = Path(__file__).resolve().parent.parent


class _Event:
    def __init__(self, *a, **k):
        pass

    def record(self, *a):
        pass

    def synchronize(self):
        pass

    def elapsed_time(self, other):
        return 1.0


@pytest.fixture
def bench(monkeypatch):
    sys.path.insert(0, str(ROOT))
    import bench as B

    monkeypatch.setattr(B, "max_over_ranks", lambda x: float(x))
    monkeypatch.setattr(B, "min_over_ranks", lambda x: float(x))
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: types.SimpleNamespace(cuda_stream=0, synchronize=lambda: None))
    return B


def _small_state(fake=True):
    g = torch.Generator().manual_seed(3)
    wrap = FakeCudaTensor.wrap if fake else (lambda t: t)
    model = {f"l{i}": wrap(torch.randn(65 + i, 33, generator=g)) for i in range(4)}
    opt = {i: {"exp_avg": wrap(torch.randn(65 + i, 33, generator=g)), "step": wrap(torch.tensor(float(i)))} for i in range(4)}
    return {"model": model, "optimizer": {"state": opt}}


def test_engine_arm_loops(bench, monkeypatch, built_library, shm_dir, dist_1rank):
    B = bench
    with fake_device(monkeypatch) as (engine, lib):
        sd = _small_state()
        tensors = B.flatten(sd)
        total = sum(t.numel() * t.element_size() for t in tensors)
        arm = B.EngineArm(False)
        try:
            rows = []
            stall, safe, persist = B.api_loop(arm, sd, shm_dir / "ckpt.pt", steps=3, warmup=1, persist_steps=1, trace_rows=rows)
            assert len(stall) == len(safe) == len(persist) == 3 and all(0 < a <= b <= c for a, b, c in zip(stall, safe, persist))
            loaded = B.flatten(torch.load(shm_dir / "ckpt.pt", weights_only=False))
            assert len(loaded) == len(tensors) and all(B.bits_equal(a, b.as_subclass(torch.Tensor)) for a, b in zip(loaded, tensors))
        finally:
            arm.close()
        leg = B.local_manager_leg("engine", sd, tensors, total, 0, False)
        assert leg["restore_verify"] == "bit-exact" and leg["restore_s"] > 0 and leg["local_save_persist_s"] >= leg["local_save_stall_ms"] / 1e3
        assert not any(s.busy for s in engine._slots)


def test_reference_arm_loops(bench, tmp_path, dist_1rank, monkeypatch):
    B = bench
    sd = _small_state(fake=False)
    arm = B.ReferenceArm(False)
    stall, safe, persist = B.api_loop(arm, sd, tmp_path / "ref.pt", steps=3, warmup=1, persist_steps=2)
    arm.close()
    assert len(stall) == 3 and len(persist) == 2 and arm.trace() is None
    got = B.flatten(torch.load(tmp_path / "ref.pt", weights_only=False))
    assert all(B.bits_equal(a, b) for a, b in zip(got, B.flatten(sd)))
    # the local leg of the reference arm restores with tensor.to("cuda"): only its save half runs without a GPU
    from oracle import reference_port as rp

    res = rp.reference_local_save(B.fresh_containers(sd), tmp_path / "iter_0000001_0_local.pt")
    assert res["total"] >= res["stall"] > 0


def test_workload_matches_the_survey():
    sys.path.insert(0, str(ROOT))
    import bench as B

    shapes = B.llama3_8b_shard_shapes()
    params = sum(int(torch.tensor(s).prod()) for _, s in shapes)
    assert len(shapes) == 291 and params == 1_003_782_656  # SURVEY 8(d): 1/8 row shard of Llama-3-8B
    assert set(B.WORKLOADS) == {"c2", "c3"} and "16.06 GB" in B.WORKLOADS["c2"]


def _args(B, **over):
    import argparse

    ns = argparse.Namespace(gpus=1, steps=2, warmup=3, impl="engine", config="c2", narrow=False, persist_steps=1, load_reps=1, scale=1.0,
                            baseline_sample_gb=0.001, no_cpu_baseline=True, no_verify=False, no_restore=False, no_training_loop=True,
                            no_ceiling=True, no_c3_kernel=False, traffic_bytes=None, dump_outputs=None)
    for k, v in over.items():
        setattr(ns, k, v)
    return ns


def test_run_arm_assembles_the_same_config_in_both_arms(bench, monkeypatch, built_library, dist_1rank):
    """The whole of run_arm (minus the GEMM loop and the PCIe ceiling, which need a GPU) on the stand-in device: the JSON line
    of both arms is assembled without error, carries the contract's keys, and `config` is identical in both (the driver
    compares it to decide whether the two arms measured the same thing)."""
    import json

    B = bench
    monkeypatch.setattr(B, "ClockSampler", lambda idx: types.SimpleNamespace(__enter__=lambda: None, __exit__=lambda *a: None, summary=lambda: {"sm_mhz": None}))
    with fake_device(monkeypatch) as (engine, lib):
        def state(dev, seed=0, scale=1.0):
            sd = _small_state()
            return sd, sum(t.numel() * t.element_size() for t in B.flatten(sd))

        monkeypatch.setattr(B, "llama3_8b_shard_state", state)
        eng = B.run_arm(_args(B), 0, 1, 0)
        c3 = B.run_arm(_args(B, config="c3", narrow=True, no_restore=True), 0, 1, 0)
    monkeypatch.setattr(B, "llama3_8b_shard_state", lambda dev, seed=0, scale=1.0: (_small_state(False), sum(t.numel() * t.element_size() for t in B.flatten(_small_state(False)))))
    ref = B.run_arm(_args(B, impl="reference", no_restore=True), 0, 1, 0)
    for line in (eng, c3, ref):
        json.dumps(line)
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "stall_device_ms",
                    "data", "config", "e2e", "gpu_launches", "stall_ms", "impl", "clocks"):
            assert key in line, key
        assert line["ms_per_step"] > 0 and line["value"] >= 0 and line["e2e"]["value"] >= 0 and line["verify"] == "bit-exact"  # (KB-sized state)
    assert eng["config"] == ref["config"] and eng["config"]["workload"] == B.WORKLOADS["c2"]
    assert eng["impl"] == "engine" and ref["impl"] == "reference" and ref["gpu_launches"] == 0 and eng["gpu_launches"] > 0
    assert eng["roofline"]["bound"] == "hbm" and eng["roofline"]["algorithmic_bytes_per_launch"] > 0 and "roofline" not in ref and "cpu_baseline" in ref
    assert "error" not in eng["c3_kernel_roofline"] and eng["c3_kernel_roofline"]["algorithmic_bytes_per_launch"] > 0 and "c3_kernel_roofline" not in c3
    assert eng["restore_verify"] == "bit-exact" and c3["config"]["workload"] == B.WORKLOADS["c3"] and c3["dtype"].startswith("f32->bf16")


def test_dump_outputs_writes_the_last_checkpoint(bench, monkeypatch, built_library, dist_1rank, tmp_path):
    """--dump-outputs: run_arm writes the checkpoint of its last timed step as float32 .npy files named by key path, whole
    when small, else the first 16 elements plus a seeded sample at the same positions in every run; non-finite elements are
    written as 0 and recorded in a .nonfinite.npy beside them."""
    import numpy as np

    B = bench
    monkeypatch.setattr(B, "ClockSampler", lambda idx: types.SimpleNamespace(__enter__=lambda: None, __exit__=lambda *a: None, summary=lambda: {"sm_mhz": None}))
    with fake_device(monkeypatch) as (engine, lib):
        monkeypatch.setattr(B, "llama3_8b_shard_state", lambda dev, seed=0, scale=1.0: (_small_state(), sum(t.numel() * t.element_size() for t in B.flatten(_small_state()))))
        B.run_arm(_args(B, config="c3", narrow=True, no_restore=True, no_c3_kernel=True, dump_outputs=str(tmp_path / "c3")), 0, 1, 0)
    sd = _small_state(fake=False)
    names = {f"model.l{i}" for i in range(4)} | {f"optimizer.state.{i}.{k}" for i in range(4) for k in ("exp_avg", "step")}
    assert {p.stem for p in (tmp_path / "c3").iterdir()} == names
    got = np.load(tmp_path / "c3" / "model.l2.npy")
    assert got.dtype == np.float32 and np.array_equal(got, sd["model"]["l2"].to(torch.bfloat16).float().reshape(-1).numpy())

    big = {"w": torch.randn(5000, generator=torch.Generator().manual_seed(1), dtype=torch.float64), "h": torch.arange(300, dtype=torch.bfloat16)}
    big["w"][1:4] = torch.tensor([float("inf"), float("-inf"), float("nan")], dtype=torch.float64)
    torch.save(big, tmp_path / "big.pt")
    monkeypatch.setattr(B, "DUMP_SAMPLE", 100)
    for run in ("a", "b"):
        B.dump_outputs(tmp_path / "big.pt", tmp_path / run)
    w, h = np.load(tmp_path / "a" / "w.npy"), np.load(tmp_path / "a" / "h.npy")
    kind = np.load(tmp_path / "a" / "w.nonfinite.npy")
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == ["h.npy", "w.nonfinite.npy", "w.npy"]
    assert w.dtype == kind.dtype == np.float64 and w.shape == kind.shape == (100,) and np.array_equal(w, np.load(tmp_path / "b" / "w.npy"))
    assert np.isfinite(w).all() and list(w[1:4]) == [0, 0, 0] and list(kind[:5]) == [0, 1, -1, 2, 0] and not kind[4:].any()
    finite = big["w"].numpy()[np.isfinite(big["w"].numpy())]
    assert w[0] == big["w"][0] and np.array_equal(w[4:16], big["w"][4:16].numpy()) and np.isin(w[4:], finite).all() and len(np.unique(w[4:])) == 96
    assert h.dtype == np.float32 and h.shape == (100,) and np.array_equal(h[:16], np.arange(16))


def test_d2h_ceiling_control_flow(bench, monkeypatch, dist_1rank):
    """The PCIe-ceiling leg needs a GPU for its number, not for its control flow: the buffer is allocated under the affinity of
    the GPU's NUMA node and the affinity is put back, every rank reaches both barriers, and a measurement that fails on this
    rank comes back as "not measured" instead of taking the bench line down (or leaving the other ranks in a collective)."""
    import os

    B = bench
    real_empty = torch.empty
    seen = {}

    def empty(*a, **k):
        if k.get("device") is not None:
            k["device"] = "cpu"
        else:
            seen["affinity_at_host_alloc"] = os.sched_getaffinity(0)
        return real_empty(*a, **k)

    monkeypatch.setattr(torch, "empty", empty)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    before = os.sched_getaffinity(0)
    one = sorted(before)[0]
    monkeypatch.setattr(B, "_numa_cpus_of_gpu", lambda idx: [one])
    dev = torch.device("cuda", 0)
    out = _ceiling_with_small_buffers(B, dev)
    assert seen["affinity_at_host_alloc"] == {one} and os.sched_getaffinity(0) == before
    assert out["per_gpu_min_GBps"] > 0 and out["per_gpu_max_GBps"] >= out["per_gpu_min_GBps"] and "NUMA" in out["what"] and "unbound" not in out["what"]
    # node unknown: measured unbound, and said so
    monkeypatch.setattr(B, "_numa_cpus_of_gpu", lambda idx: None)
    out = _ceiling_with_small_buffers(B, dev)
    assert out["per_gpu_min_GBps"] > 0 and "unbound" in out["what"] and os.sched_getaffinity(0) == before
    # the allocation fails on this rank: both barriers are still reached, the result says why there is no number
    def broken(*a, **k):
        raise RuntimeError("out of pinned memory")

    monkeypatch.setattr(torch.Tensor, "pin_memory", broken)
    monkeypatch.setattr(B, "_numa_cpus_of_gpu", lambda idx: [one])
    barriers = []
    real_barrier = B.dist.barrier
    monkeypatch.setattr(B.dist, "barrier", lambda *a, **k: (barriers.append(1), real_barrier(*a, **k))[1])
    out = _ceiling_with_small_buffers(B, dev)
    assert out["per_gpu_min_GBps"] is None and "out of pinned memory" in out["what"] and len(barriers) == 2
    assert os.sched_getaffinity(0) == before


def _ceiling_with_small_buffers(B, dev):
    class Tiny(int):  # d2h_ceiling computes ``gib << 30`` bytes: 4 KiB instead of GiBs here
        def __lshift__(self, n):
            return 4096

    return B.d2h_ceiling(dev, 1, gib=Tiny(1), reps=2)


def test_numa_cpus_of_gpu_reads_sysfs(bench, monkeypatch, tmp_path):
    """PCI address from the device properties -> numa_node -> cpulist ("0-3,8-9"); anything missing means "unknown"."""
    import builtins

    B = bench
    props = types.SimpleNamespace(pci_domain_id=0, pci_bus_id=0x1B, pci_device_id=0)
    monkeypatch.setattr(torch.cuda, "get_device_properties", lambda i: props)
    files = {"/sys/bus/pci/devices/0000:1b:00.0/numa_node": "1\n", "/sys/devices/system/node/node1/cpulist": "0-3,8-9,12\n"}
    real_open = builtins.open

    def fake_open(path, *a, **k):
        if str(path) in files:
            p = tmp_path / str(path).strip("/").replace("/", "_")
            p.write_text(files[str(path)])
            return real_open(p, *a, **k)
        if str(path).startswith("/sys/"):
            raise FileNotFoundError(path)
        return real_open(path, *a, **k)

    monkeypatch.setattr(builtins, "open", fake_open)
    assert B._numa_cpus_of_gpu(0) == [0, 1, 2, 3, 8, 9, 12]
    files["/sys/bus/pci/devices/0000:1b:00.0/numa_node"] = "-1\n"
    assert B._numa_cpus_of_gpu(0) is None
    props.pci_bus_id = 0x2C  # no such device in sysfs
    assert B._numa_cpus_of_gpu(0) is None


def _w_run_arm_two_ranks(rank, world, out_dir):
    """One rank of a two-rank ``run_arm`` (engine arm, every leg the driver's N>1 runs execute except the GEMM loop and the
    PCIe ceiling) on the stand-in device with gloo collectives."""
    import json

    import torch.distributed as dist

    sys.path.insert(0, str(ROOT))
    import bench as B

    mp_ = pytest.MonkeyPatch()

    def over(op):
        def reduce(x):
            t = torch.tensor([float(x)], dtype=torch.float64)
            dist.all_reduce(t, op=op)
            return t.item()

        return reduce

    try:
        mp_.setattr(B, "max_over_ranks", over(dist.ReduceOp.MAX))
        mp_.setattr(B, "min_over_ranks", over(dist.ReduceOp.MIN))
        mp_.setattr(torch.cuda, "Event", _Event)
        mp_.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
        mp_.setattr(torch.cuda, "current_stream", lambda *a, **k: types.SimpleNamespace(cuda_stream=0, synchronize=lambda: None))
        mp_.setattr(B, "ClockSampler", lambda idx: types.SimpleNamespace(__enter__=lambda: None, __exit__=lambda *a: None, summary=lambda: {"sm_mhz": None}))
        with fake_device(mp_) as (engine, lib):
            def state(dev, seed=0, scale=1.0):
                g = torch.Generator().manual_seed(seed)  # (the bench seeds every rank differently: 1234 + rank)
                sd = {"model": {f"l{i}": FakeCudaTensor.wrap(torch.randn(65 + i, 33, generator=g)) for i in range(4)},
                      "optimizer": {"state": {i: {"exp_avg": FakeCudaTensor.wrap(torch.randn(65 + i, 33, generator=g)),
                                                  "step": FakeCudaTensor.wrap(torch.tensor(float(i)))} for i in range(4)}}}
                return sd, sum(t.numel() * t.element_size() for t in B.flatten(sd))

            mp_.setattr(B, "llama3_8b_shard_state", state)
            line = B.run_arm(_args(B), rank, world, 0)
        with open(f"{out_dir}/line{rank}.json", "w") as fh:
            json.dump(line, fh)
    finally:
        mp_.undo()


def test_run_arm_on_two_ranks(tmp_path, built_library):
    """The driver launches bench.py on 2, 4 and 8 ranks: every collective of run_arm (barriers of the loops, max / min over
    ranks, the local manager's find_latest gathers with ONE session id for all ranks) must line up across ranks.  Executed here
    on two gloo ranks with the stand-in device; both ranks assemble the same whole-job line."""
    import json

    from _mp import run_ranks

    run_ranks(_w_run_arm_two_ranks, 2, str(tmp_path), timeout=300.0)
    lines = [json.load(open(tmp_path / f"line{r}.json")) for r in range(2)]
    for line in lines:
        assert line["n_gpus"] == 2 and line["verify"] in ("bit-exact", "skipped") and line["restore_verify"] == "bit-exact"
        assert line["local_save_stall_ms"] >= 0 and line["restore_s"] > 0 and line["gpu_launches"] > 0
    assert lines[0]["verify"] == "bit-exact"  # (rank 0 checks its file)
    for key in ("value", "ms_per_step", "stall_ms", "restore_s", "local_save_persist_s", "config"):
        assert lines[0][key] == lines[1][key], key  # max over ranks: the same number on every rank


def test_a_failing_local_leg_is_reported_inside_the_line(bench, monkeypatch, built_library, dist_1rank):
    """The stall / e2e numbers are measured before the local-manager leg: an exception there (on every rank alike, e.g. the
    session-id assertion of the first 2-GPU run) must not cost the whole line."""
    import json

    B = bench
    monkeypatch.setattr(B, "ClockSampler", lambda idx: types.SimpleNamespace(__enter__=lambda: None, __exit__=lambda *a: None, summary=lambda: {"sm_mhz": None}))

    def broken(*a, **k):
        raise AssertionError("session == self.session_id")

    monkeypatch.setattr(B, "local_manager_leg", broken)
    with fake_device(monkeypatch) as (engine, lib):
        monkeypatch.setattr(B, "llama3_8b_shard_state", lambda dev, seed=0, scale=1.0: (_small_state(), sum(t.numel() * t.element_size() for t in B.flatten(_small_state()))))
        line = B.run_arm(_args(B, no_c3_kernel=True), 0, 1, 0)
    json.dumps(line)
    assert "session == self.session_id" in line["local_leg_error"] and line["restore_GBps"] is None
    assert line["value"] > 0 and line["e2e"]["value"] > 0 and line["verify"] == "bit-exact" and line["roofline"]["algorithmic_bytes_per_launch"] > 0
