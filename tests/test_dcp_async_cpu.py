"""torch.distributed.checkpoint through FileSystemWriterAsync, CPU only (gloo): the files must be byte-identical to a
synchronous ``dcp.save`` of the same state dict, and ``dcp.load`` must give the values back.  Mirrors the scenarios of the
reference's tests/checkpointing/unit/test_async_writer.py (sync-vs-async equality, cached-plan reuse, failure propagation)."""
import filecmp
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.distributed.checkpoint as dcp
from torch.distributed.checkpoint import CheckpointException, DefaultSavePlanner, FileSystemReader, FileSystemWriter

from _mp import run_ranks


def _state(rank=0, step=0):
    g = torch.Generator().manual_seed(100 + rank)
    return {
        "model": {
            "w": torch.randn(33, 17, generator=g) + step,
            "b": torch.arange(7, dtype=torch.int64) * (rank + 1),
            "h": torch.randn(5, 3, generator=g).to(torch.bfloat16),
            "empty": torch.empty(0, 4),
        },
        "opt": {"step": torch.tensor(3 + step), "lr": 0.125, "name": f"adam{rank}"},
    }


def _async_save(state, path, queue, planner=None, writer_kw=None, **kw):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncRequest
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync
    from nvidia_resiliency_ext.checkpointing.async_ckpt.state_dict_saver import (
        save_state_dict_async_finalize,
        save_state_dict_async_plan,
    )

    writer = FileSystemWriterAsync(path, thread_count=2, **(writer_kw or {}))
    ret = save_state_dict_async_plan(state, writer, None, 0, planner=planner or DefaultSavePlanner(), **kw)
    save_fn, preload_fn, save_args = writer.get_save_function_and_args()
    assert save_fn is not None and getattr(save_fn, "nvrx_drain_aware", False)
    req = AsyncRequest(save_fn, save_args, [lambda: save_state_dict_async_finalize(*ret)], preload_fn=preload_fn)
    queue.schedule_async_request(req)
    return ret


def _same_files(a, b):
    cmp = filecmp.dircmp(a, b)
    assert not cmp.left_only and not cmp.right_only, (cmp.left_only, cmp.right_only)
    data = [f for f in cmp.common_files if f.endswith(".distcp")]
    assert data
    match, mismatch, errors = filecmp.cmpfiles(a, b, data, shallow=False)
    assert not mismatch and not errors, (mismatch, errors)


def _loaded_equals(path, expect):
    got = {k: ({kk: (torch.zeros_like(vv) if isinstance(vv, torch.Tensor) else None) for kk, vv in v.items()}) for k, v in expect.items()}
    dcp.load(got, storage_reader=FileSystemReader(path))
    for k, sub in expect.items():
        for kk, vv in sub.items():
            if isinstance(vv, torch.Tensor):
                assert got[k][kk].dtype == vv.dtype and torch.equal(got[k][kk], vv), (k, kk)
            else:
                assert got[k][kk] == vv, (k, kk)


@pytest.mark.parametrize("persistent", [False])  # the persistent worker is covered by the golden-fixture test below
def test_async_dcp_matches_sync_save(tmp_path, dist_1rank, persistent):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue

    state = _state()
    sync_dir, async_dir = tmp_path / "sync", tmp_path / "async"
    dcp.save(state, storage_writer=FileSystemWriter(sync_dir, thread_count=2), planner=DefaultSavePlanner())
    q = AsyncCallsQueue(persistent=persistent)
    try:
        _async_save(state, async_dir, q)
        # the trainer may change its tensors as soon as the request is scheduled
        state["model"]["w"].add_(1000.0)
        state["model"]["b"].zero_()
        q.maybe_finalize_async_calls(blocking=True, no_dist=False)
        assert q.get_num_unfinalized_calls() == 0
    finally:
        q.close()
    _same_files(sync_dir, async_dir)
    _loaded_equals(async_dir, _state())


def _two_rank_job(rank, world, root):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue
    from nvidia_resiliency_ext.checkpointing.async_ckpt.state_dict_saver import (
        CheckpointMetadataCache,
        get_metadata_caching_status,
    )

    q = AsyncCallsQueue(persistent=False)
    cache = CheckpointMetadataCache()
    for step in range(3):
        state = {f"r{rank}": _state(rank, step)["model"], "shared": {"s": torch.full((4,), float(step))}}
        sync_dir, async_dir = os.path.join(root, f"sync{step}"), os.path.join(root, f"async{step}")
        dcp.save(state, storage_writer=FileSystemWriter(sync_dir, thread_count=2), planner=DefaultSavePlanner())
        ret = _async_save(state, async_dir, q, enable_cache=True, metadata_cache=cache)
        # plans are identical from the second save on: the third one must have skipped the exchange
        assert cache.validated_cache_reuse == (step >= 1), (step, cache.get_metadata_caching_status())
        assert (ret[1] is not None) == (rank == 0)
        q.maybe_finalize_async_calls(blocking=True)
        dist.barrier()
        if rank == 0:
            _same_files(sync_dir, async_dir)
            assert {f[:4] for f in os.listdir(async_dir) if f.endswith(".distcp")} == {"__0_", "__1_"}
        got = {f"r{rank}": {k: torch.zeros_like(v) for k, v in state[f"r{rank}"].items()}, "shared": {"s": torch.zeros(4)}}
        dcp.load(got, storage_reader=FileSystemReader(async_dir))
        for k, v in state[f"r{rank}"].items():
            assert torch.equal(got[f"r{rank}"][k], v), (step, k)
        assert torch.equal(got["shared"]["s"], state["shared"]["s"])
    assert get_metadata_caching_status() is None  # the process-wide cache was never created
    if rank == 0:
        # metadata written from the cached plan (3rd save) describes the same checkpoint as the planned one (1st save)
        import pickle
        from dataclasses import fields

        mds = []
        for step in (0, 2):
            with open(os.path.join(root, f"async{step}", ".metadata"), "rb") as fh:
                mds.append(pickle.load(fh))
        for f in fields(mds[0]):
            if f.name not in ("storage_data", "storage_meta"):
                assert getattr(mds[0], f.name) == getattr(mds[1], f.name), f.name
        assert set(mds[0].storage_data) == set(mds[1].storage_data)
    q.close()


def test_async_dcp_two_ranks_with_plan_cache(tmp_path):
    run_ranks(_two_rank_job, 2, str(tmp_path))


def _failing_job(rank, world, root):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue

    q = AsyncCallsQueue(persistent=False)
    target = os.path.join(root, "ckpt")
    state = {f"r{rank}": {"w": torch.ones(8) * rank}}
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync
    from nvidia_resiliency_ext.checkpointing.async_ckpt.state_dict_saver import (
        save_state_dict_async_finalize,
        save_state_dict_async_plan,
    )

    writer = FileSystemWriterAsync(target, thread_count=1)
    ret = save_state_dict_async_plan(state, writer, None, 0)
    save_fn, preload_fn, save_args = writer.get_save_function_and_args()
    if rank == 1:
        # rank 1's writer process cannot create its file: the directory is replaced by a plain file
        dist.barrier()
        import shutil

        shutil.rmtree(target)
        open(target, "w").close()
        dist.barrier()
    else:
        dist.barrier()
        dist.barrier()
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncRequest

    q.schedule_async_request(AsyncRequest(save_fn, save_args, [], preload_fn=preload_fn))
    q.maybe_finalize_async_calls(blocking=True)
    with pytest.raises(CheckpointException) as err:
        save_state_dict_async_finalize(*ret)
    if rank == 0:
        assert 1 in err.value.failures and "Worker failure" in str(err.value)
    else:
        assert "Worker failure" not in str(err.value)
    assert not os.path.exists(os.path.join(target, ".metadata"))
    q.close()


def test_async_dcp_write_failure_raises_everywhere(tmp_path):
    run_ranks(_failing_job, 2, str(tmp_path))


def test_writer_process_reads_cuda_items_from_the_snapshot_slot(tmp_path, built_library):
    """Writer side of the engine path without a GPU: the slot content is produced by the oracle's pack, the progress word
    is advanced by a thread (as the side stream would), and the write function must wait for it and write the same file
    as a synchronous save of the tensors."""
    import ctypes as C
    import multiprocessing
    import threading
    import time

    from oracle.snapshot_oracle import pack_oracle
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync
    from nvidia_resiliency_ext.checkpointing.async_ckpt.state_dict_saver import save_state_dict_async_plan
    from nvidia_resiliency_ext.checkpointing.b200.engine import HostBuffer, PackedLayout

    state = _state()
    sync_dir, async_dir = tmp_path / "sync", tmp_path / "async"
    # per_thread_copy_ahead=0: with one thread and a CUDA device present, PyTorch's writer would switch to its copy-ahead
    # loader, which writes the items in order of size; the writer process never copies ahead (its items are on the host)
    dcp.save(state, storage_writer=FileSystemWriter(sync_dir, thread_count=1, per_thread_copy_ahead=0), planner=DefaultSavePlanner())

    writer = FileSystemWriterAsync(async_dir, thread_count=1)
    _, metadata, dist_wrapper = save_state_dict_async_plan(state, writer, None, 0)
    payload = writer._payload
    # pretend every tensor item was on the GPU: move it from the host staging into a packed slot
    tensor_idx = [i for i, v in payload["host"].items() if isinstance(v, torch.Tensor)]
    tensors = [payload["host"].pop(i) for i in tensor_idx]
    packed, offs, sizes = pack_oracle(tensors)
    names = {torch.float32: "float32", torch.int64: "int64", torch.bfloat16: "bfloat16"}
    layout = PackedLayout(
        shapes=[tuple(t.shape) for t in tensors], dtypes=[names[t.dtype] for t in tensors],
        src_dtypes=[names[t.dtype] for t in tensors], offsets=list(offs), packed_nbytes=list(sizes), total_bytes=len(packed),
    )
    hb = HostBuffer.create(max(len(packed), 4096), name=f"/nvrx_dcp_{os.getpid()}", pin=False, prefault_threads=1)
    try:
        payload["snapshot"] = {"shm_name": hb.name, "progress_target": 7, "layout": layout}
        payload["cuda_indices"] = tensor_idx

        def drain():
            time.sleep(0.2)
            hb.as_tensor(len(packed)).numpy()[:] = packed
            C.c_uint64.from_address(hb.progress_ptr).value = 7

        t = threading.Thread(target=drain)
        t.start()
        results = multiprocessing.get_context("spawn").Manager().Queue()
        FileSystemWriterAsync.write_preloaded_data(writer._ctor, 1, None, "test-save", 0, payload, results)
        t.join()
        rank, save_id, outcome = results.get(timeout=10)
        assert rank == 0 and isinstance(outcome, list) and len(outcome) == len(payload["plan"].items), outcome
        writer.finish(metadata, [outcome])
    finally:
        hb.close()
    _same_files(sync_dir, async_dir)
    _loaded_equals(async_dir, _state())


def test_writer_rejects_unsupported_modes(tmp_path):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync

    with pytest.raises(NotImplementedError):
        FileSystemWriterAsync(tmp_path, single_file_per_rank=False)
    with pytest.raises(NotImplementedError):
        FileSystemWriterAsync(tmp_path, use_msc=True)
    w = FileSystemWriterAsync(tmp_path)
    assert w.get_save_function_and_args() == (None, None, [])
    assert w.retrieve_write_results() == []
    with pytest.raises(NotImplementedError):
        w.write_data(None, None)


def test_cached_metadata_reader(tmp_path, dist_1rank):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.cached_metadata_filesystem_reader import CachedMetadataFileSystemReader

    state = _state()
    dcp.save(state, storage_writer=FileSystemWriter(tmp_path / "a"), planner=DefaultSavePlanner())
    CachedMetadataFileSystemReader.clear_metadata_cache()
    first = CachedMetadataFileSystemReader(tmp_path / "a").read_metadata()
    os.rename(tmp_path / "a" / ".metadata", tmp_path / "a" / ".moved")  # a second read from disk would fail
    assert CachedMetadataFileSystemReader(str(tmp_path / "a")).read_metadata() is first
    with pytest.raises(Exception):
        CachedMetadataFileSystemReader(tmp_path / "a", cache_metadata=False).read_metadata()
    os.rename(tmp_path / "a" / ".moved", tmp_path / "a" / ".metadata")
    got = {k: {kk: (torch.zeros_like(vv) if isinstance(vv, torch.Tensor) else None) for kk, vv in v.items()} for k, v in state.items()}
    dcp.load(got, storage_reader=CachedMetadataFileSystemReader(tmp_path / "a"))
    assert torch.equal(got["model"]["w"], state["model"]["w"]) and got["opt"]["name"] == "adam0"
    CachedMetadataFileSystemReader.clear_metadata_cache(tmp_path / "a")
    assert CachedMetadataFileSystemReader(tmp_path / "a").read_metadata() is not first
    CachedMetadataFileSystemReader.clear_metadata_cache()


def test_separation_hint_splits_files(tmp_path, dist_1rank):
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync

    state = _state()
    q = AsyncCallsQueue(persistent=False)
    try:
        _async_save(state, tmp_path / "ckpt", q, writer_kw={"separation_hint": "opt"})
        q.maybe_finalize_async_calls(blocking=True)
    finally:
        q.close()
    files = sorted(f for f in os.listdir(tmp_path / "ckpt") if f.endswith(".distcp"))
    assert [f for f in files if f.startswith("opt__0_")] and [f for f in files if f.startswith("__0_")], files
    md = FileSystemReader(tmp_path / "ckpt").read_metadata()
    for index, info in md.storage_data.items():
        assert info.relative_path.startswith("opt") == index.fqn.startswith("opt"), (index, info)
    _loaded_equals(tmp_path / "ckpt", _state())
    with pytest.raises(AssertionError, match="thread_count"):
        w = FileSystemWriterAsync(tmp_path / "x", thread_count=1, separation_hint="opt")
        w.prepare_write_data(None, None)


def test_matches_the_references_own_async_checkpoint(tmp_path, dist_1rank):
    """tests/golden/dcp_reference was written by the REFERENCE's FileSystemWriterAsync path (make_golden.py::gen_dcp) for
    dcp_inputs.pt.  Our writer must produce the same checkpoint: same values when loaded, same metadata, and -- on the
    PyTorch version the fixture was made with -- the same bytes."""
    import pickle
    from dataclasses import fields

    from conftest import GOLDEN
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue

    state = torch.load(GOLDEN / "dcp_inputs.pt", weights_only=False)
    q = AsyncCallsQueue(persistent=True)
    try:
        _async_save(state, tmp_path / "ours", q)
        q.maybe_finalize_async_calls(blocking=True)
    finally:
        q.close()

    def loaded(path):
        got = {k: {kk: (torch.zeros_like(vv) if isinstance(vv, torch.Tensor) else None) for kk, vv in v.items()} for k, v in state.items()}
        dcp.load(got, storage_reader=FileSystemReader(path))
        return got

    ref, ours = loaded(GOLDEN / "dcp_reference"), loaded(tmp_path / "ours")
    for k, sub in state.items():
        for kk, vv in sub.items():
            if isinstance(vv, torch.Tensor):
                assert torch.equal(ref[k][kk], vv) and torch.equal(ours[k][kk], vv) and ours[k][kk].dtype == ref[k][kk].dtype
            else:
                assert ref[k][kk] == ours[k][kk] == vv
    mds = []
    for d in (GOLDEN / "dcp_reference", tmp_path / "ours"):
        with open(d / ".metadata", "rb") as fh:
            mds.append(pickle.load(fh))
    for f in fields(mds[1]):
        if f.name not in ("storage_data", "storage_meta") and hasattr(mds[0], f.name):
            assert getattr(mds[0], f.name) == getattr(mds[1], f.name), f.name
    assert {k: (v.relative_path, v.offset, v.length) for k, v in mds[0].storage_data.items()} == {
        k: (v.relative_path, v.offset, v.length) for k, v in mds[1].storage_data.items()
    }
    if (GOLDEN / "dcp_reference" / "torch_version.txt").read_text() == torch.__version__:
        names = sorted(f for f in os.listdir(GOLDEN / "dcp_reference") if f.endswith(".distcp"))
        assert names == sorted(f for f in os.listdir(tmp_path / "ours") if f.endswith(".distcp"))
        _, mismatch, errors = filecmp.cmpfiles(GOLDEN / "dcp_reference", tmp_path / "ours", names, shallow=False)
        assert not mismatch and not errors, (mismatch, errors)


def test_abort_with_a_pending_dcp_save_and_resume(tmp_path, dist_1rank):
    """In-process restart: abort_nvrx_checkpoint() stops the writer workers of every queue, also with a DCP save in flight; the
    queues work again afterwards and a queue dropped right after an abort shuts down cleanly (reference
    test_async_writer.py::test_async_cp_with_multiple_queue_and_abort[_followed_by_delete])."""
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue, AsyncRequest, abort_nvrx_checkpoint

    state = _state()
    q_dcp, q_plain = AsyncCallsQueue(persistent=True), AsyncCallsQueue(persistent=False)
    try:
        _async_save(state, tmp_path / "a", q_dcp)
        q_plain.schedule_async_request(AsyncRequest(torch.save, ({"x": torch.arange(4)}, tmp_path / "plain_a.pt"), []))
        q_dcp.maybe_finalize_async_calls(blocking=True)
        q_plain.maybe_finalize_async_calls(blocking=True, no_dist=True)
        _loaded_equals(tmp_path / "a", _state())

        abort_nvrx_checkpoint()
        for q in (q_dcp, q_plain):
            caller = q._get_async_caller()
            assert caller is None or caller._debug_is_async_process_running() is False
            assert q.get_num_unfinalized_calls() == 0

        # seamless resume: same queues, new workers
        _async_save(state, tmp_path / "b", q_dcp)
        q_plain.schedule_async_request(AsyncRequest(torch.save, ({"x": torch.arange(4)}, tmp_path / "plain_b.pt"), []))
        q_dcp.maybe_finalize_async_calls(blocking=True)
        q_plain.maybe_finalize_async_calls(blocking=True, no_dist=True)
        _loaded_equals(tmp_path / "b", _state())
        assert torch.equal(torch.load(tmp_path / "plain_b.pt")["x"], torch.arange(4))
        assert q_dcp._get_async_caller()._debug_is_async_process_running() is True

        # an exception in the trainer right after scheduling, abort, then the queue object goes away
        _async_save(state, tmp_path / "c", q_dcp)
        abort_nvrx_checkpoint()
        q_dcp.__del__()
    finally:
        q_dcp.close()
        q_plain.close()


class _DecentralPlanner(DefaultSavePlanner):
    """A planner that finishes its plan on its own (what Megatron-Core's planner offers): every rank owns disjoint keys."""

    can_run_decentralized_global_plan = True

    def create_decentralized_global_plan(self, local_plan):
        return local_plan


def _decentral_job(rank, world, root):
    import pickle

    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue
    from nvidia_resiliency_ext.checkpointing.async_ckpt.state_dict_saver import CheckpointMetadataCache

    q = AsyncCallsQueue(persistent=False)
    gathers = []
    from torch.distributed.checkpoint.utils import _DistWrapper

    real_gather = _DistWrapper.gather_object
    _DistWrapper.gather_object = lambda self, obj: (gathers.append(type(obj).__name__), real_gather(self, obj))[1]

    def save(step, cache):
        state = {f"r{rank}": _state(rank, step)["model"]}
        path = os.path.join(root, f"d{step}")
        ret = _async_save(state, path, q, planner=_DecentralPlanner(), enable_cache=True, metadata_cache=cache)
        q.maybe_finalize_async_calls(blocking=True)
        dist.barrier()
        got = {f"r{rank}": {k: torch.zeros_like(v) for k, v in state[f"r{rank}"].items()}}
        dcp.load(got, storage_reader=FileSystemReader(path))
        assert all(torch.equal(got[f"r{rank}"][k], v) for k, v in state[f"r{rank}"].items()), step
        return path, ret

    cache = CheckpointMetadataCache()
    path0, ret0 = save(0, cache)
    assert gathers.count("SavePlan") == 1  # plans gathered once for the metadata, never scattered
    with open(os.path.join(path0, ".metadata"), "rb") as fh:
        md = pickle.load(fh)
    assert len(md.all_local_plans) == world  # stored for a job that resumes from this checkpoint
    # "resume": a fresh cache seeded with the loaded metadata -> no plan exchange at all, the coordinator re-uses the metadata
    resumed = CheckpointMetadataCache()
    resumed.set_cached_global_metadata(md)
    path1, ret1 = save(1, resumed)
    assert gathers.count("SavePlan") == 1 and resumed.validated_loaded_metadata_reuse
    assert (ret1[1] is not None) == (rank == 0)
    # a changed structure is noticed by every rank: back to gathering
    resumed2 = CheckpointMetadataCache()
    resumed2.set_cached_global_metadata(md)
    state = {f"r{rank}": dict(_state(rank, 2)["model"], extra=torch.ones(3 + rank))}
    _async_save(state, os.path.join(root, "d2"), q, planner=_DecentralPlanner(), enable_cache=True, metadata_cache=resumed2)
    q.maybe_finalize_async_calls(blocking=True)
    assert gathers.count("SavePlan") == 2 and not resumed2.validated_loaded_metadata_reuse
    _DistWrapper.gather_object = real_gather
    q.close()


def test_decentralized_planning_and_reuse_of_loaded_metadata(tmp_path):
    run_ranks(_decentral_job, 2, str(tmp_path))


def test_result_of_an_abandoned_save_is_not_taken_for_the_next_one(tmp_path, dist_1rank):
    """The write-results queue is process-wide.  A save whose writer reported but whose trainer never asked (abort between the
    two) must not hand its results to the following save -- that would put the wrong storage offsets into ``.metadata``."""
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue

    q = AsyncCallsQueue(persistent=False)
    try:
        abandoned = {"other": {"z": torch.arange(5)}}
        ret = _async_save(abandoned, tmp_path / "abandoned", q)
        import time

        # the writer of the abandoned save runs to completion and reports ...

        deadline = time.time() + 60
        while not any(f.endswith(".distcp") for f in os.listdir(tmp_path / "abandoned")) and time.time() < deadline:
            time.sleep(0.05)
        time.sleep(0.5)
        q.close(abort=True)  # ... but the trainer aborts before finalizing: nobody retrieves that report
        del ret
        q = AsyncCallsQueue(persistent=False)
        state = _state()
        _async_save(state, tmp_path / "next", q)
        q.maybe_finalize_async_calls(blocking=True)
        _loaded_equals(tmp_path / "next", _state())
    finally:
        q.close()


def _failing_open(path, mode="rb"):
    raise OSError("worker critical failure during open()")


def _counting_open(path, mode="rb"):
    with open(os.path.join(os.path.dirname(path), "opened.log"), "a") as log:
        log.write(os.path.basename(path) + "\n")
    return open(path, mode)


def test_open_file_hook_and_daemon_multiproc_setup(tmp_path, dist_1rank):
    """Reference tests/checkpointing/unit/test_async_writer.py:180-231: a user ``open_file`` is what the writer process opens this
    rank's files with (a failing one surfaces as "Worker failure" at finalize); multi-process file IO from a daemonic worker is
    reported as "Invalid Setup!"."""
    from torch.distributed.checkpoint import CheckpointException

    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue
    from nvidia_resiliency_ext.checkpointing.async_ckpt.filesystem_async import FileSystemWriterAsync

    FileSystemWriterAsync._cached_identifiers.clear()
    FileSystemWriterAsync._shm_tensor_cache.clear()
    q = AsyncCallsQueue(persistent=False)
    try:
        _async_save(_state(), tmp_path / "counted", q, writer_kw={"open_file": _counting_open})
        q.maybe_finalize_async_calls(blocking=True, no_dist=False)
        assert any(n.endswith(".distcp") for n in (tmp_path / "counted" / "opened.log").read_text().split())
        _loaded_equals(tmp_path / "counted", _state())
        _async_save(_state(), tmp_path / "broken", q, writer_kw={"open_file": _failing_open})
        with pytest.raises(CheckpointException) as err:
            q.maybe_finalize_async_calls(blocking=True, no_dist=False)
        assert "Worker failure" in str(err.value)
    finally:
        q.close()
    q = AsyncCallsQueue(persistent=True, is_daemon=True)
    try:
        _async_save(_state(), tmp_path / "daemon", q, writer_kw={"is_multiproc_io": True})
        with pytest.raises(CheckpointException) as err:
            q.maybe_finalize_async_calls(blocking=True, no_dist=False)
        assert "Invalid Setup!" in str(err.value)
    finally:
        q.close()
