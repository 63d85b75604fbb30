"""Helper to run a function on N local ranks (gloo on CPU, NCCL when the ranks own GPUs)."""
import os
import sys
import traceback

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import PKG_ROOT, ROOT, free_port


def _entry(rank, world, port, backend, fn, args, errq):
    for p in (str(ROOT), str(PKG_ROOT), str(ROOT / "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["RANK"], os.environ["WORLD_SIZE"], os.environ["LOCAL_RANK"] = str(rank), str(world), str(rank)
    try:
        if backend == "nccl":
            torch.cuda.set_device(rank)
        dist.init_process_group(backend, rank=rank, world_size=world)
        fn(rank, world, *args)
        dist.barrier()
        dist.destroy_process_group()
    except Exception:  # noqa: BLE001
        errq.put((rank, traceback.format_exc()))
        raise


def run_ranks(fn, world: int, *args, backend: str = "gloo", timeout: float = 150.0):
    ctx = mp.get_context("spawn")
    errq = ctx.SimpleQueue()
    port = free_port()
    procs = [ctx.Process(target=_entry, args=(r, world, port, backend, fn, args, errq)) for r in range(world)]
    # gloo ranks run the host-only paths: they must not see this machine's GPUs, or they would take the device paths, whose
    # point-to-point payloads gloo cannot send.  The children inherit the environment at start.
    hidden = os.environ.get("CUDA_VISIBLE_DEVICES")
    if backend == "gloo":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""
    try:
        for p in procs:
            p.start()
    finally:
        if backend == "gloo":
            if hidden is None:
                del os.environ["CUDA_VISIBLE_DEVICES"]
            else:
                os.environ["CUDA_VISIBLE_DEVICES"] = hidden
    for p in procs:
        p.join(timeout)
    errors = []
    while not errq.empty():
        errors.append(errq.get())
    hung = [p for p in procs if p.is_alive()]
    for p in hung:
        p.kill()
    assert not hung, "ranks hung"
    assert not errors, "\n".join(f"[rank {r}]\n{tb}" for r, tb in errors)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
