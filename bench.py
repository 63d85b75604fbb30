#!/usr/bin/env python
"""Benchmark of the checkpoint-snapshot hot path (BASELINE.json metric), one process per GPU.

    python bench.py --gpus N --steps K --warmup W                    # this repo's engine, config C2
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own path (oracle port), same loop
    python bench.py --config c3 ...                                  # C3: fp32->bf16 narrowing in the pack kernel
    python bench.py --config c4 --gpus 8 ...                         # C4/C5: replicated local checkpoints (bench_c4.py)

Workload (every N: weak scaling, no data-path collective for C2/C3): per rank a 1/8 row shard of Llama-3-8B in 4 fp32
copies (param, main_param, exp_avg, exp_avg_sq) = 1164 tensors, 16,060,522,496 B, plus 291 scalar fp32 `step` tensors,
synthetic values (SURVEY.md 8d).

BOTH arms run the SAME loop (``api_loop``) over the same state dict on EVERY rank; only the object behind it differs:
the product's ``TorchAsyncCheckpoint`` or the port of the reference's ``TorchAsyncCheckpoint`` flow
(``oracle/reference_port.py``).  One step = one checkpoint of the whole state dict through ``async_save(state_dict, path)``.

  value       state bytes of all ranks / STALL: the wall time ``async_save`` keeps the training stream blocked (from the
              call until an event recorded on the training stream right after it has completed).  The state is resident
              in HBM when the timed region starts; this is the "snapshot GB/s" a training loop sees.  ms_per_step = that
              stall (mean of the K steps, max over ranks).  stall_device_ms = the same span timed on the device (CUDA events
              recorded on the training stream right before and after the call).
  e2e         same metric until the snapshot bytes are SAFE IN HOST MEMORY (the D2H of the whole snapshot is inside the
              timed region): PCIe-bound in both arms.
  stall_beside_training_ms   the same stall measured inside a running GEMM loop (SURVEY 8d): extra wall time of a window of
              training steps when one checkpoint is taken in the middle of it.
  persist_s   until ``finalize_async_save(blocking=True)`` returned (file loadable by ``torch.load``);
  restore_s   ``LocalCheckpointManager.find_latest() + load()`` of the same state from its local checkpoint file.
  roofline    (engine arm) the pack kernel alone: algorithmic HBM bytes of one launch (2*S; 1.5*S_in when narrowing) /
              its duration, K back-to-back launches timed with CUDA events on the launching stream, against the measured
              copy peak in MEASURED_PEAKS.json.  This kernel rate is NOT the headline; it explains the stall.
  cpu_baseline (engine arm, N=1) a short run of the reference loop on the same box, for the record.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "nvidia-resiliency-ext_b200"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "checkpoint_snapshot_GBps"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
WORKLOADS = {
    "c2": "C2: 16.06 GB Llama-3-8B-shaped param+Adam state_dict per rank (1164 fp32 tensors + 291 scalar steps), "
          "snapshot through TorchAsyncCheckpoint.async_save -> pinned host -> file on /dev/shm",
    "c3": "C3: 16.06 GB Llama-3-8B-shaped param+Adam state_dict per rank (1164 fp32 tensors + 291 scalar steps), "
          "fp32->bf16 narrow in the pack kernel, snapshot through TorchAsyncCheckpoint.async_save -> pinned host -> file on /dev/shm",
}


# ----------------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------------
def llama3_8b_shard_shapes():
    """1/8 row shard (dim0 / 8) of every Llama-3-8B tensor (vocab 128256, hidden 4096, 32 layers, ffn 14336, 32/8
    heads): 291 tensors, 1,003,782,656 parameters per rank (SURVEY.md 8d)."""
    shapes = [("embed", (16032, 4096))]
    for layer in range(32):
        for name, shp in (("q", (512, 4096)), ("k", (128, 4096)), ("v", (128, 4096)), ("o", (512, 4096)),
                          ("gate", (1792, 4096)), ("up", (1792, 4096)), ("down", (512, 14336)), ("ln1", (512,)), ("ln2", (512,))):
            shapes.append((f"layers.{layer}.{name}", shp))
    shapes += [("final_ln", (512,)), ("lm_head", (16032, 4096))]
    return shapes


def llama3_8b_shard_state(device, seed=1234, scale=1.0):
    """{"model": {name: p}, "optimizer": {"state": {i: {main_param, exp_avg, exp_avg_sq, step}}}} (SURVEY.md 8d)."""
    g = torch.Generator(device=device).manual_seed(seed)
    model, opt = {}, {}
    total = 0
    for i, (name, shp) in enumerate(llama3_8b_shard_shapes()):
        if scale != 1.0 and len(shp) == 2:
            shp = (max(1, int(shp[0] * scale)), shp[1])
        p = torch.empty(shp, dtype=torch.float32, device=device).normal_(0, 0.02, generator=g)
        m = p.clone()
        ea = torch.empty(shp, dtype=torch.float32, device=device).normal_(0, 1e-3, generator=g)
        es = torch.empty(shp, dtype=torch.float32, device=device).uniform_(0, 1e-6, generator=g)
        if i == 1:  # edge values for the narrowing path
            flat = ea.view(-1)
            flat[:6] = torch.tensor([float("inf"), float("-inf"), float("nan"), -0.0, 1e-40, -1e-45], device=device)
        model[name] = p
        opt[i] = {"main_param": m, "exp_avg": ea, "exp_avg_sq": es, "step": torch.tensor(float(1000 + i), device=device)}
        total += 4 * p.numel() * 4 + 4
    return {"model": model, "optimizer": {"state": opt}}, total


def fresh_containers(sd):
    """New nested containers around the same tensors (LocalCheckpointManager.save rewrites the container it is given)."""
    return {"model": dict(sd["model"]), "optimizer": {"state": {k: dict(v) for k, v in sd["optimizer"]["state"].items()}}}


def flatten(sd):
    out = []

    def walk(x):
        for v in (x.values() if isinstance(x, dict) else x):
            if isinstance(v, (dict, list)):
                walk(v)
            elif isinstance(v, torch.Tensor):
                out.append(v)

    walk(sd)
    return out


# ----------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        if shutil.which("nvidia-smi"):
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)

            def pump():
                for ln in self.proc.stdout:
                    self.lines.append(ln)

            threading.Thread(target=pump, daemon=True).start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < 5.0:  # nvidia-smi needs a moment (longer on 8-GPU boxes)
                time.sleep(0.05)
        return self

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:  # noqa: BLE001
            pass
    return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(label_prefix):
    """dram read+write bytes per launch of the dominant kernel from the newest committed `ncu --set full` summary, with the
    commit that summary was captured at (the number is a cross-check, not a live measurement)."""
    for name in ("r02_ncu_walk_summary.json", "r01_ncu_walk_summary.json"):
        p = ROOT / "profiles" / name
        try:
            doc = json.load(open(p))
            for k in doc["kernels"]:
                if k["label"].startswith(label_prefix):
                    return float(k["traffic_bytes"]), f"profiles/{name} (ncu --set full, same state, one launch; captured at commit {doc.get('commit', 'round 1')})"
        except Exception:  # noqa: BLE001
            continue
    return None, None


def init_dist(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    return rank, world, local


def max_over_ranks(x: float) -> float:
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item()


def min_over_ranks(x: float) -> float:
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return t.item()


def mean(xs):
    return sum(xs) / len(xs)


def median(xs):
    s = sorted(xs)
    return s[len(s) // 2]


def shm_dir(rank, tag="bench"):
    base = Path("/dev/shm") if os.access("/dev/shm", os.W_OK) else Path("/tmp")
    d = base / f"nvrx_b200_{tag}_{os.getpid()}_{rank}"
    d.mkdir(parents=True, exist_ok=True)
    return d


def bits_equal(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and (
        a.numel() == 0 or torch.equal(a.contiguous().view(-1).view(torch.uint8), b.contiguous().view(-1).view(torch.uint8)))


DUMP_SAMPLE = 8192  # elements kept per tensor: 1455 tensors x 8192 x 4 B = 48 MB, within the 64 MB a dump may take


def dump_outputs(path, out_dir):
    """Writes the checkpoint file ``path``, as ``torch.load`` returns it, to ``out_dir/<key path>.npy`` (e.g.
    ``optimizer.state.0.exp_avg.npy``), flattened, as float32 (float64 stays float64).  A tensor of more than DUMP_SAMPLE
    elements is sampled: its first 16 elements (the narrowing edge values sit there) and the rest at positions drawn with a fixed
    seed, so two builds run with the same arguments write the same positions.  Every value written is finite: a non-finite
    element (the workload holds +-inf and NaN on purpose) is written as 0, and ``<key path>.nonfinite.npy`` beside it says
    which ones it replaced (same positions: 0 finite, 1 +inf, -1 -inf, 2 NaN); tensors without any get no such file."""
    import numpy as np

    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(0)
    loaded = torch.load(path, weights_only=False, mmap=True)

    def walk(x, prefix):
        for k, v in (x.items() if isinstance(x, dict) else enumerate(x)):
            if isinstance(v, (dict, list, tuple)):
                walk(v, f"{prefix}{k}.")
            elif isinstance(v, torch.Tensor):
                flat = v.reshape(-1)
                if flat.numel() > DUMP_SAMPLE:
                    rest = rng.choice(flat.numel() - 16, DUMP_SAMPLE - 16, replace=False) + 16
                    flat = flat[torch.from_numpy(np.concatenate([np.arange(16), np.sort(rest)]))]
                values = (flat if flat.dtype == torch.float64 else flat.float()).numpy()
                if not np.isfinite(values).all():
                    kind = np.isposinf(values) * 1.0 - np.isneginf(values) + np.isnan(values) * 2.0
                    np.save(out_dir / f"{prefix}{k}.nonfinite.npy", kind.astype(values.dtype))
                    values = np.where(np.isfinite(values), values, 0).astype(values.dtype)
                np.save(out_dir / f"{prefix}{k}.npy", values)

    walk(loaded, "")


# ----------------------------------------------------------------------------------------------------
# the two arms behind one interface
# ----------------------------------------------------------------------------------------------------
class EngineArm:
    """The product: nvidia_resiliency_ext.checkpointing.async_ckpt.torch_ckpt.TorchAsyncCheckpoint (public API)."""

    name = "engine"
    writes_every_step = True

    def __init__(self, narrow):
        from nvidia_resiliency_ext.checkpointing.async_ckpt.torch_ckpt import TorchAsyncCheckpoint

        self.ckpt = TorchAsyncCheckpoint(persistent_queue=True, narrow_fp32_to_bf16=narrow)

    def save(self, sd, path, write=True):
        self.ckpt.async_save(sd, path)

    def host_safe(self):
        for snap in list(self.ckpt._pending.values()):
            snap.wait()  # CPU wait on the drain's event: bytes are in pinned host memory

    def trace(self):
        from nvidia_resiliency_ext.checkpointing.b200.engine import SnapshotEngine

        tr = SnapshotEngine.get().trace
        return dict(tr) if tr else None

    def finalize(self):
        self.ckpt.finalize_async_save(blocking=True, no_dist=True)

    def close(self):
        self.ckpt.close()


class ReferenceArm:
    """The reference's flow (oracle/reference_port.py, port of async_ckpt/torch_ckpt.py:43-53 + core.py:318-355)."""

    name = "reference"
    writes_every_step = False

    def __init__(self, narrow):
        from oracle.reference_port import ReferenceAsyncCheckpoint

        self.ckpt = ReferenceAsyncCheckpoint()  # the reference has no narrowing: C3's reference arm is C2's

    def save(self, sd, path, write=True):
        self.ckpt.async_save(sd, path, write=write)

    def host_safe(self):
        pass  # async_save returned after torch.cuda.synchronize(): the host copies are complete

    def trace(self):
        return None

    def finalize(self):
        self.ckpt.finalize(blocking=True)

    def close(self):
        self.ckpt.finalize(blocking=True)


def api_loop(arm, sd, path, steps, warmup, persist_steps, trace_rows=None, device_ms=None):
    """K checkpoints through ``arm``; per step: stall, time to host-safe, time to persisted (only when the step wrote)."""
    ev = torch.cuda.Event()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stall, safe, persist = [], [], []
    # ``device_ms`` (a list to fill): the same stall as the DEVICE saw it, CUDA events around the call on the training stream
    for it in range(warmup + steps):
        write = arm.writes_every_step or it >= warmup + steps - persist_steps
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev0.record()
        arm.save(sd, path, write)
        t_ret = time.perf_counter()
        ev1.record()
        ev.record()
        ev.synchronize()  # the training stream is free again here
        t1 = time.perf_counter()
        if it >= warmup and device_ms is not None:
            device_ms.append(ev0.elapsed_time(ev1))
        if it >= warmup and trace_rows is not None:
            tr = arm.trace()
            if tr:
                trace_rows.append({"to_snapshot_ms": (tr["enter"] - t0) * 1e3, "plan_ms": (tr["planned"] - tr["enter"]) * 1e3,
                                   "enqueue_ms": (tr["launched"] - tr["planned"]) * 1e3, "after_launch_ms": (t_ret - tr["launched"]) * 1e3,
                                   "gpu_tail_ms": (t1 - t_ret) * 1e3})
        arm.host_safe()
        t2 = time.perf_counter()
        arm.finalize()
        t3 = time.perf_counter()
        if it >= warmup:
            stall.append(t1 - t0)
            safe.append(t2 - t0)
            if write:
                persist.append(t3 - t0)
    return stall, safe, persist


class TrainingLoop:
    """Dummy training step (SURVEY 8d): a fixed number of bf16 8192^3 GEMMs on the current stream."""

    def __init__(self, dev, step_ms=30.0):
        self.a = torch.randn(8192, 8192, dtype=torch.bfloat16, device=dev)
        self.b = torch.randn(8192, 8192, dtype=torch.bfloat16, device=dev)
        self.c = torch.empty(8192, 8192, dtype=torch.bfloat16, device=dev)
        self.gemms = 8
        ms = self._time(3)
        self.gemms = max(4, int(round(self.gemms * step_ms / max(ms, 1e-3))))
        self.step_ms = self._time(5)

    def step(self, n=1):
        for _ in range(n * self.gemms):
            torch.mm(self.a, self.b, out=self.c)

    def _time(self, n):
        self.step(2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        self.step(n)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / n


def stall_beside_training(arm, sd, path, loop, reps, before=10, after=30):
    """Extra wall time of a window of ``before + after`` training steps when ONE checkpoint is taken after ``before`` of
    them (device idle at both ends of the window).  The window is longer than the background drain, so the number holds
    everything the checkpoint costs the training loop: the call, the pack kernel(s) in stream order, and whatever the
    side-stream D2H takes away from the GEMMs."""
    base, with_ckpt = [], []
    for r in range(reps + 1):
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop.step(before + after)
        torch.cuda.synchronize()
        t_base = time.perf_counter() - t0
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop.step(before)
        arm.save(sd, path, arm.writes_every_step)
        loop.step(after)
        torch.cuda.synchronize()
        t_with = time.perf_counter() - t0
        arm.host_safe()
        arm.finalize()
        if r > 0:  # first repetition warms up
            base.append(t_base)
            with_ckpt.append(t_with)
    return (median(with_ckpt) - median(base)) * 1e3, median(base) * 1e3


def _numa_cpus_of_gpu(index):
    """CPUs of the NUMA node GPU ``index`` hangs off (sysfs), or None."""
    try:
        props = torch.cuda.get_device_properties(index)
        bdf = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        return cpus or None
    except Exception:  # noqa: BLE001
        return None


def d2h_ceiling(dev, world, gib=4, reps=4):
    """What the box gives N concurrent plain device->pinned-host copies (cudaMemcpyAsync into a cudaHostAlloc buffer, all
    ranks at once): the PCIe / host-memory ceiling the e2e number can be judged against.  The buffer is allocated while the
    thread is bound to the CPUs next to the GPU: where a pinned buffer lands is otherwise a lottery, and a buffer on the other
    socket halves the rate when all 8 GPUs copy (16-21 instead of 39 GB/s per GPU on this pool's 8-GPU box,
    profiles/r02_d2h_ceiling_8gpu.jsonl)."""
    n, rate, err, cpus, src, dst = gib << 30, None, None, None, None, None
    try:
        src = torch.empty(n, dtype=torch.uint8, device=dev)
        cpus, before = _numa_cpus_of_gpu(dev.index), None
        try:
            if cpus:
                before = os.sched_getaffinity(0)
                os.sched_setaffinity(0, cpus)
            dst = torch.empty(n, dtype=torch.uint8).pin_memory()
            dst.fill_(0)
        finally:
            if before is not None:
                os.sched_setaffinity(0, before)
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
    except Exception as exc:  # noqa: BLE001 - a ceiling that cannot be measured must not take the bench line with it
        err = exc
    dist.barrier()  # (every rank reaches the collectives whatever happened to its own measurement)
    if err is None:
        try:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize()
            rate = reps * n / (time.perf_counter() - t0) / 1e9
        except Exception as exc:  # noqa: BLE001
            err = exc
    dist.barrier()
    if min_over_ranks(0.0 if rate is None else 1.0) < 0.5:
        return {"per_gpu_min_GBps": None, "per_gpu_max_GBps": None, "what": f"not measured on every rank ({err!r})"}
    return {"per_gpu_min_GBps": round(min_over_ranks(rate), 2), "per_gpu_max_GBps": round(max_over_ranks(rate), 2),
            "what": f"{world} concurrent plain pinned-memory D2H copies, {reps} x {gib} GiB each (cudaHostAlloc buffer on the GPU's NUMA "
                    f"node{'' if cpus else ' -- node unknown, unbound'}, cudaMemcpyAsync)"}


def local_manager_leg(arm_name, sd, tensors, total, rank, narrow):
    """C5 on every rank independently (no replication): local checkpoint save through ``LocalCheckpointManager`` and
    restore with ``find_latest() + load()``; the reference arm runs the port of the same two flows."""
    root = shm_dir(rank, "local")
    ev = torch.cuda.Event()
    out = {}
    try:
        if arm_name == "engine":
            from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue
            from nvidia_resiliency_ext.checkpointing.local.basic_state_dict import BasicTensorAwareStateDict
            from nvidia_resiliency_ext.checkpointing.local.ckpt_managers.local_manager import LocalCheckpointManager

            from nvidia_resiliency_ext.checkpointing.b200.engine import SnapshotEngine

            mgr = LocalCheckpointManager(root, session_id="bench")
            q = AsyncCallsQueue(persistent=False)
            # like TorchAsyncCheckpoint.warmup(): staging and host slot for THIS state exist before the timed save (the async
            # loop above may have run on narrowed, i.e. smaller, snapshots; the reference arm's pinned cache is warm from its loop)
            from nvidia_resiliency_ext.checkpointing.b200 import ptzip

            eng = SnapshotEngine.get()
            # exactly what save() will ask for (container geometry + room for the container's tail): a slot the async loop left
            # qualifies as it is; only a loop that ran on narrowed (half-size) snapshots makes this create one, untimed
            sizes = [t.numel() * t.element_size() for t in tensors]
            span = ptzip.slot_offsets(sizes)[1]
            need = -(-span // 512) * 512 + ptzip.slot_tail_room(len(sizes))
            eng._ensure_staging(need)
            eng._release(eng._acquire_slot(need))
            tasd = BasicTensorAwareStateDict(fresh_containers(sd))
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            req = mgr.save(tasd, 1, is_async=True)
            ev.record()
            ev.synchronize()
            t1 = time.perf_counter()
            q.schedule_async_request(req)
            q.maybe_finalize_async_calls(blocking=True, no_dist=False)
            t2 = time.perf_counter()
            q.close()
            del tasd, req
            mgr2 = LocalCheckpointManager(root, session_id="bench")
            torch.cuda.synchronize()
            dist.barrier()
            t3 = time.perf_counter()
            latest = mgr2.find_latest()
            loaded, cid = mgr2.load()
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            got = list(loaded.tensors)
            ok = latest == 1 and cid[0] == 1
        else:
            from oracle.reference_port import reference_local_load, reference_local_save

            path = root / "iter_0000001_0_local.pt"
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            res = reference_local_save(fresh_containers(sd), path)
            t1, t2 = t0 + res["stall"], t0 + res["total"]
            torch.cuda.synchronize()
            dist.barrier()
            t3 = time.perf_counter()
            loaded = reference_local_load(path)
            torch.cuda.synchronize()
            t4 = time.perf_counter()
            got = flatten(loaded.state_dict)
            ok = True
        ok = ok and len(got) == len(tensors)
        for a, b in list(zip(got, tensors))[:: max(1, len(tensors) // 48)]:
            ok = ok and a.is_cuda and bits_equal(a, b)
        del loaded, got
        out = {
            "local_save_stall_ms": round(max_over_ranks(t1 - t0) * 1e3, 2),
            "local_save_persist_s": round(max_over_ranks(t2 - t0), 3),
            "restore_s": round(max_over_ranks(t4 - t3), 3),
            "restore_verify": "bit-exact" if ok else "MISMATCH",
        }
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


def kernel_leg(args, tensors, local):
    """The pack kernel alone: K back-to-back launches, CUDA events on the launching stream, max over ranks."""
    from nvidia_resiliency_ext.checkpointing.b200.engine import Event, SnapshotEngine

    engine = SnapshotEngine.get(local, host_slots=2)
    stream = torch.cuda.current_stream().cuda_stream
    mask = SnapshotEngine._narrow_mask(tensors, args.narrow)
    plan = engine._plan_for(tensors, mask)
    staging = engine._ensure_staging(plan.staging_bytes)
    for _ in range(max(args.warmup, 3)):
        plan.pack(staging.ptr, stream)
    e0, e1 = Event(local, True), Event(local, True)
    torch.cuda.synchronize()
    dist.barrier()
    e0.record(stream)
    for _ in range(args.steps):
        plan.pack(staging.ptr, stream)
    e1.record(stream)
    e1.synchronize()
    kernel_ms = max_over_ranks(e0.elapsed_ms(e1) / args.steps)
    torch.cuda.synchronize()
    dist.barrier()
    return engine, plan, kernel_ms


def run_arm(args, rank, world, local):
    dev = torch.device("cuda", local)
    sd, total = llama3_8b_shard_state(dev, seed=1234 + rank, scale=args.scale)
    tensors = flatten(sd)
    engine_arm = args.impl == "engine"
    clocks = ClockSampler(local)
    clocks.__enter__()
    launches = 0
    engine = plan = None
    kernel_ms = None
    c3_kernel = None
    if engine_arm:
        engine, plan, kernel_ms = kernel_leg(args, tensors, local)
        launches += args.steps
        if not args.narrow and not args.no_c3_kernel:
            # config C3's kernel in the same line (the driver only runs the default config): the narrowing pack alone, same timing
            try:
                import copy

                a3 = copy.copy(args)
                a3.narrow = True
                _, plan3, ms3 = kernel_leg(a3, tensors, local)
                peak3, _ = hbm_peak()
                c3_kernel = {
                    "kernel": "nvrx::walk_ldg<pack> (fp32->bf16 narrow)", "kernel_ms": round(ms3, 4),
                    "algorithmic_bytes_per_launch": plan3.algorithmic_bytes, "achieved": round(plan3.algorithmic_bytes / (ms3 * 1e-3) / 1e9, 1),
                    "peak": peak3, "unit": "GB/s", "frac": round(plan3.algorithmic_bytes / (ms3 * 1e-3) / 1e9 / peak3, 4),
                    "packed_bytes_per_rank": plan3.staging_bytes, "timing": f"{args.steps} back-to-back launches, CUDA events, max over ranks",
                }
                launches += args.steps
            except Exception as exc:  # noqa: BLE001 - an extra; must not take the C2 line with it
                c3_kernel = {"error": repr(exc)}
        launches_before = engine.launches

    arm = (EngineArm if engine_arm else ReferenceArm)(args.narrow)
    out_dir = shm_dir(rank)
    path = out_dir / "ckpt.pt"  # one file per rank, overwritten every step
    trace_rows = [] if os.environ.get("NVRX_B200_TRACE", "0") == "1" else None
    device_ms = []
    stall, safe, persist = api_loop(arm, sd, path, args.steps, args.warmup, args.persist_steps, trace_rows, device_ms)
    clocks.__exit__(None, None, None)
    stall_s = max_over_ranks(mean(stall))  # the K timed steps, mean -> ms_per_step
    safe_s = max_over_ranks(mean(safe))
    persist_s = max_over_ranks(median(persist)) if persist else None
    linked = bool(path.exists() and os.stat(path).st_nlink > 1)  # the file IS the pinned slot (zero-copy publish)

    # spot-check the last file against the live state (bit-exact unless narrowed)
    check = "skipped"
    if rank == 0 and not args.no_verify and path.exists():
        loaded = torch.load(path, weights_only=False, mmap=True)
        lt = flatten(loaded)
        ok = len(lt) == len(tensors)
        for a, b in list(zip(lt, tensors))[:: max(1, len(tensors) // 64)]:
            narrowed = engine_arm and args.narrow and b.dtype == torch.float32 and b.numel() > 0
            ok &= bits_equal(a, b.to(torch.bfloat16).cpu() if narrowed else b.cpu())
        check = "bit-exact" if ok else "MISMATCH"
        del loaded, lt
    if rank == 0 and args.dump_outputs:
        dump_outputs(path, args.dump_outputs)

    load_ms = base_ms = None
    if not args.no_training_loop:
        loop = TrainingLoop(dev)
        load_ms, base_ms = stall_beside_training(arm, sd, path, loop, args.load_reps)
        load_ms, base_ms = max_over_ranks(load_ms), max_over_ranks(base_ms)
        del loop
    arm.close()
    shutil.rmtree(out_dir, ignore_errors=True)
    local_leg = {}
    if not args.no_restore:
        try:
            local_leg = local_manager_leg(args.impl, sd, tensors, total, rank, args.narrow)
        except Exception as exc:  # noqa: BLE001 - the headline numbers above are measured: a failure here is reported in the line
            import traceback

            traceback.print_exc()
            local_leg = {"local_leg_error": repr(exc)}
    ceiling = None if args.no_ceiling else d2h_ceiling(dev, world)
    if engine_arm:
        launches += engine.launches - launches_before

    line = {
        "metric": METRIC,
        "value": round(world * total / stall_s / 1e9, 1),
        "unit": "GB/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": round(stall_s * 1e3, 4),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u8" if not (args.narrow and engine_arm) else "f32->bf16 (rne) + u8",
        "data": "synthetic",
        "impl": args.impl,
        "value_definition": "state bytes of all ranks / training-stream stall of async_save (state resident in HBM; until the "
                            "training stream is free again), public API, same loop in both arms",
        "config": {
            "workload": WORKLOADS[args.config],
            "state_bytes_per_rank": total,
            "tensors": len(tensors),
            "l2": "inputs (16 GB) >> L2 (126 MB); no flush needed",
            "scale": args.scale,
        },  # identical in both arms (the driver compares it); what differs between the arms is under "path" / "engine"
        "path": ("nvidia_resiliency_ext...TorchAsyncCheckpoint.async_save (pack kernel on the training stream, side-stream drain, "
                 "writer process follows the drain)" if engine_arm else
                 "reference flow (oracle/reference_port.py): per-tensor pinned D2H + torch.cuda.synchronize() + fork + torch.save"
                 + ("; the reference has no narrowing, it saves fp32" if args.narrow else "")),
        "e2e": {
            "value": round(world * total / safe_s / 1e9, 2),
            "unit": "GB/s",
            "h2d_bytes_per_step": int(len(tensors) * 32) if engine_arm else 0,
            "d2h_bytes_per_step": int(plan.staging_bytes) if engine_arm else int(total),
            "definition": "state bytes of all ranks / wall time from async_save() until the snapshot is safe in host memory",
            "per_gpu_GBps": round(total / safe_s / 1e9, 2),
            "d2h_ceiling": ceiling,
        },
        "stall_ms": round(stall_s * 1e3, 3),
        "stall_device_ms": round(max_over_ranks(mean(device_ms)), 3) if device_ms else None,
        "stall_beside_training_ms": None if load_ms is None else round(load_ms, 3),
        "training_window_ms": None if base_ms is None else round(base_ms, 1),
        "persist_s": None if persist_s is None else round(persist_s, 3),
        "persist_GBps": None if persist_s is None else round(world * total / persist_s / 1e9, 2),
        "persist_mode": ("zero-copy link" if linked else "parallel copy") if engine_arm else "torch.save in the forked child (1 core per rank)",
        "persist_steps": len(persist),
        **local_leg,
        "restore_GBps": round(world * total / local_leg["restore_s"] / 1e9, 2) if local_leg.get("restore_s") else None,
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "verify": check,
        "host_cores_on_box": os.cpu_count(),
    }
    if trace_rows:
        line["stall_breakdown_ms"] = {k: round(mean([r[k] for r in trace_rows]), 3) for k in trace_rows[0]}
    if engine_arm:
        peak, peak_src = hbm_peak()
        algo = plan.algorithmic_bytes
        achieved = algo / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = (args.traffic_bytes, "command line") if args.traffic_bytes else ncu_traffic("pack LDG narrow" if args.narrow else "pack TMA")
        line["engine"] = {"packed_bytes_per_rank": plan.staging_bytes, "walker": os.environ.get("NVRX_B200_VARIANT", "auto")}
        line["roofline"] = {
            "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo,
            "kernel": "nvrx::walk_tma<pack>" if not args.narrow else "nvrx::walk_ldg<pack> (narrow)",
            "kernel_ms": round(kernel_ms, 4), "device_snapshot_GBps": round(world * total / (kernel_ms * 1e-3) / 1e9, 1),
            "timing": f"{args.steps} back-to-back launches of the whole-state pack, CUDA events on the launching stream, max over ranks",
        }
        if c3_kernel is not None:
            line["c3_kernel_roofline"] = c3_kernel
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(sd, total, args.baseline_sample_gb)
    else:
        line["cpu_baseline"] = {
            "value": line["value"], "unit": "GB/s", "cores": 1, "kind": "port",
            "sample": f"every step, every rank: full-state per-tensor pinned D2H + torch.cuda.synchronize() (the stall); the forked "
                      f"torch.save child (1 core per rank of {os.cpu_count()}) ran on the last {len(persist)} step(s) on the full state",
        }
        line["e2e"]["h2d_bytes_per_step"] = 0
        line["e2e"]["d2h_bytes_per_step"] = 0
        line["gpu_launches"] = 0
    return line


def cpu_baseline(sd, total, sample_gb):
    """A short run of the reference loop (same ``api_loop``) on this box: stall on the full state, persistence on a bounded
    sample of the tensors."""
    from oracle import snapshot_oracle as orc

    arm = ReferenceArm(False)
    out = shm_dir(0, "cpubase")
    stall, safe, _ = api_loop(arm, sd, out / "x.pt", 2, 1, 0)
    arm.close()
    tensors = flatten(sd)
    sample, acc = {}, 0
    for i, t in enumerate(tensors):
        if acc + t.numel() * 4 > sample_gb * 1e9:
            continue
        sample[f"t{i}"] = t
        acc += t.numel() * 4
    res = orc.reference_fork_save(sample, out / "sample.pt")
    shutil.rmtree(out, ignore_errors=True)
    persist_rate = acc / (res["total"] - res["d2h"]) / 1e9
    d2h = mean(stall)
    return {
        "value": round(total / d2h / 1e9, 2), "unit": "GB/s", "cores": 1, "kind": "port",
        "sample": f"reference loop, 2 steps on the full state: per-tensor pinned D2H + cuda sync (stall {d2h*1e3:.0f} ms); fork + "
                  f"torch.save timed on {acc/1e9:.2f} GB of the tensors ({persist_rate:.2f} GB/s, 1 core)",
        "stall_ms": round(d2h * 1e3, 1), "persist_GBps_1core": round(persist_rate, 2), "host_cores_on_box": os.cpu_count(),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4"])
    ap.add_argument("--narrow", action="store_true", help="alias of --config c3: fp32->bf16 in the pack kernel")
    ap.add_argument("--persist-steps", type=int, default=1, help="reference arm: how many of the steps run the forked torch.save")
    ap.add_argument("--load-reps", type=int, default=3, help="repetitions of the stall-beside-training measurement")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the state (debug only; numbers at != 1.0 are not C2)")
    ap.add_argument("--baseline-sample-gb", type=float, default=2.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-restore", action="store_true")
    ap.add_argument("--no-training-loop", action="store_true")
    ap.add_argument("--no-ceiling", action="store_true")
    ap.add_argument("--no-c3-kernel", action="store_true", help="skip the C3 (narrowing) kernel-only leg of the default run")
    ap.add_argument("--traffic-bytes", type=float, default=None, help="dram read+write bytes per launch from the ncu capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write rank 0's checkpoint of the last step to DIR/<key path>.npy (sampled, see dump_outputs)")
    args, rest = ap.parse_known_args()
    if args.dump_outputs and args.config == "c4":
        raise SystemExit("--dump-outputs covers the configs c2 and c3")
    if args.narrow:
        args.config = "c3"
    args.narrow = args.config == "c3"
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else max(args.warmup, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the snapshot path has no CPU fallback)")
    rank, world, local = init_dist(args.gpus)
    if args.config == "c4":
        import bench_c4

        line = bench_c4.run(args, rest, rank, world, local)
    else:
        line = run_arm(args, rank, world, local)
    if rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
