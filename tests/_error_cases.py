"""Misuse and edge scenarios of the checkpointing API, runnable on CPU (one-rank gloo world), shared by
tests/golden/make_behaviour_golden.py (runs the REFERENCE) and tests/test_behaviour_golden_cpu.py (runs the mirror): what is
raised (type and message) or returned must be the same.  Every scenario gets a fresh temporary directory."""
import os
import re


def _outcome(fn):
    try:
        return {"returns": _plain(fn())}
    except BaseException as exc:  # noqa: BLE001 - the raised type is the point
        return {"raises": type(exc).__name__, "message": _scrub(str(exc))}


_TMP_ROOTS = []  # the directories scenarios() was given: a temporary directory need not live under /tmp


def _scrub(text):
    roots = "".join(re.escape(r) + r"[^\s'\"]*|" for r in _TMP_ROOTS)
    text = re.sub(roots + r"/tmp/[^\s'\"]+|/dev/shm/[^\s'\"]+", "<path>", text)
    return re.sub(r"0x[0-9a-f]+", "<addr>", text)


def _plain(x):
    import torch

    if isinstance(x, torch.Tensor):
        return {"tensor": x.tolist(), "dtype": str(x.dtype)}
    if isinstance(x, dict):
        return {str(k): _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, (int, float, str, bool)) or x is None:
        return x
    return f"<{type(x).__name__}>"


def _write_text(path, text):
    with open(path, "w") as fh:
        fh.write(text)


def _raise_value_error(msg):
    raise ValueError(msg)


def scenarios(tmp):
    """name -> outcome.  Imports happen inside: the caller decides which ``nvidia_resiliency_ext`` is on sys.path."""
    import torch

    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncRequest
    from nvidia_resiliency_ext.checkpointing.local.basic_state_dict import BasicTensorAwareStateDict
    from nvidia_resiliency_ext.checkpointing.local.ckpt_managers.local_manager import LocalCheckpointManager
    from nvidia_resiliency_ext.checkpointing.local.replication.group_utils import parse_group_sequence

    _TMP_ROOTS[:] = [os.path.realpath(tmp), os.path.abspath(tmp)]
    out = {}
    counter = [0]

    def fresh():
        counter[0] += 1
        d = os.path.join(tmp, f"d{counter[0]}")
        os.makedirs(d)
        return d

    def tasd():
        return BasicTensorAwareStateDict({"iteration": 5, "names": ["a", "b"], "nested": {"lr": 0.5}})

    # ---- BasicTensorAwareStateDict ---------------------------------------------------------------------------------
    out["tasd_rejects_host_tensors"] = _outcome(lambda: BasicTensorAwareStateDict({"w": torch.zeros(2)}))
    out["tasd_without_tensors_pops_nothing"] = _outcome(lambda: tasd().pop_tensors())

    def twice():
        t = tasd()
        t.pop_tensors()
        return t.pop_tensors()

    out["tasd_pop_twice"] = _outcome(twice)
    out["tasd_insert_when_not_hollow"] = _outcome(lambda: tasd().insert_tensors([]))
    out["tasd_init_when_not_hollow"] = _outcome(lambda: tasd().init_tensors())

    def hollow(method, *args):
        t = tasd()
        t.pop_tensors()
        return getattr(t, method)(*args)

    out["tasd_copy_to_cpu_when_hollow"] = _outcome(lambda: hollow("copy_tensors_to_cpu"))
    out["tasd_restore_device_when_hollow"] = _outcome(lambda: hollow("restore_tensor_device"))

    def tensors_when_hollow():
        t = tasd()
        t.pop_tensors()
        return list(t.tensors)

    out["tasd_tensors_when_hollow"] = _outcome(tensors_when_hollow)

    def roundtrip():
        t = tasd()
        flags = [t.is_hollow]
        payload = t.pop_tensors()
        flags.append(t.is_hollow)
        t.insert_tensors(payload)
        flags.append(t.is_hollow)
        return flags, t.state_dict, list(t.tensors)

    out["tasd_hollow_flags_roundtrip"] = _outcome(roundtrip)

    # ---- LocalCheckpointManager --------------------------------------------------------------------------------------
    out["manager_load_before_find_latest"] = _outcome(lambda: LocalCheckpointManager(fresh()).load())
    out["manager_find_latest_on_empty_directory"] = _outcome(lambda: LocalCheckpointManager(fresh()).find_latest())
    out["manager_negative_iteration"] = _outcome(lambda: LocalCheckpointManager(fresh())._ckpt_id(-1))
    out["manager_ckpt_id"] = _outcome(lambda: LocalCheckpointManager(fresh(), session_id="s")._ckpt_id(12))

    def save_find_load():
        root = fresh()
        mgr = LocalCheckpointManager(root)
        res = mgr.save(tasd(), 3, is_async=False)
        latest = mgr.find_latest()
        loaded, cid = mgr.load()
        names = sorted(os.path.relpath(os.path.join(dp, f), root) for dp, _, fs in os.walk(root) for f in fs)
        return res, latest, list(cid), loaded.state_dict, names

    out["manager_sync_save_find_load"] = _outcome(save_find_load)

    def other_session():
        root = fresh()
        LocalCheckpointManager(root, session_id="one").save(tasd(), 3, is_async=False)
        return LocalCheckpointManager(root, session_id="two").find_latest()

    out["manager_other_session_sees_nothing"] = _outcome(other_session)

    def keeps_only_latest():
        root = fresh()
        mgr = LocalCheckpointManager(root)
        for it in (1, 2, 5):
            mgr.save(tasd(), it, is_async=False)
        import time

        time.sleep(1.0)  # removal of older iterations may run in the background
        return mgr.find_latest(), sorted(f for _, _, fs in os.walk(root) for f in fs)

    out["manager_keeps_only_the_latest_iteration"] = _outcome(keeps_only_latest)

    def older_iteration():
        mgr = LocalCheckpointManager(fresh())
        mgr.save(tasd(), 5, is_async=False)
        mgr.find_latest()  # (latest_iteration is invalid right after a save: this makes 5 known)
        return mgr.save(tasd(), 3, is_async=False)

    out["manager_refuses_an_older_iteration"] = _outcome(older_iteration)

    def dirty_file():
        mgr = LocalCheckpointManager(fresh())
        mgr._ensure_dir()
        mgr._local_ckpt_path_from_id(mgr._ckpt_id(3), True).touch()
        return mgr.save(tasd(), 3, is_async=False)

    out["manager_dirty_file_of_the_same_id"] = _outcome(dirty_file)

    def dirty_is_invisible_and_cleaned():
        mgr = LocalCheckpointManager(fresh())
        mgr._ensure_dir()
        dirty = mgr._local_ckpt_path_from_id(mgr._ckpt_id(3), True)
        dirty.touch()
        seen = (dirty.name, mgr.find_latest())
        mgr._cleanup_failed_save(3)
        return seen, sorted(p.name for p in mgr.local_ckpt_dir.iterdir())

    out["manager_dirty_files_are_invisible_and_removed"] = _outcome(dirty_is_invisible_and_cleaned)

    def load_after_file_vanished():
        mgr = LocalCheckpointManager(fresh())
        mgr.save(tasd(), 4, is_async=False)
        mgr.find_latest()
        for p in mgr.local_ckpt_dir.iterdir():
            p.unlink()
        return mgr.load()

    out["manager_load_after_the_file_vanished"] = _outcome(load_after_file_vanished)

    # ---- AsyncRequest ------------------------------------------------------------------------------------------------
    def frozen():
        r = AsyncRequest(print, ("x",), [])
        r2 = r.freeze()
        return r.is_frozen, r2.is_frozen, r2.add_finalize_fn(print)

    out["async_request_frozen_rejects_finalize_fns"] = _outcome(frozen)

    def finalize_order():
        seen = []
        r = AsyncRequest(print, (), [lambda: seen.append(1)])
        r.add_finalize_fn(lambda: seen.append(2))
        for fn in r.finalize_fns:
            fn()
        return seen

    out["async_request_finalize_fns_keep_order"] = _outcome(finalize_order)

    # ---- AsyncCallsQueue with a persistent worker (host functions only) -----------------------------------------------
    from nvidia_resiliency_ext.checkpointing.async_ckpt.core import AsyncCallsQueue

    def queue_flow():
        d = fresh()
        q = AsyncCallsQueue(persistent=True, cpu_shm_mode=True)  # (the reference worker needs no CUDA device in this mode)
        seen = []
        try:
            idx0 = q.schedule_async_request(AsyncRequest(_write_text, (os.path.join(d, "a.txt"), "A"), [lambda: seen.append("fin0")]))
            idx1 = q.schedule_async_request(AsyncRequest(_write_text, (os.path.join(d, "b.txt"), "B"), [lambda: seen.append("fin1")]))
            pending = q.get_num_unfinalized_calls()
            done = q.maybe_finalize_async_calls(blocking=True, no_dist=True)
            left = q.get_num_unfinalized_calls()
            again = q.maybe_finalize_async_calls(blocking=True, no_dist=True)
            files = sorted((f, open(os.path.join(d, f)).read()) for f in os.listdir(d))
            return idx0, idx1, pending, done, left, again, seen, files
        finally:
            q.close()

    out["queue_two_requests_finalize_in_order"] = _outcome(queue_flow)

    def queue_sync_request():
        d = fresh()
        seen = []
        r = AsyncRequest(_write_text, (os.path.join(d, "s.txt"), "S"), [lambda: seen.append("fin")])
        r.execute_sync()
        return seen, open(os.path.join(d, "s.txt")).read()

    out["request_execute_sync_runs_fn_and_finalizers"] = _outcome(queue_sync_request)

    # ---- parse_group_sequence ----------------------------------------------------------------------------------------
    for name, kw in {
        "jump_zero": dict(replication_jump=0, replication_factor=2, world_size=8),
        "factor_zero": dict(replication_jump=1, replication_factor=0, world_size=8),
        "world_not_divisible": dict(replication_jump=2, replication_factor=3, world_size=8),
        "jump4_factor2_world8": dict(replication_jump=4, replication_factor=2, world_size=8),
        "jump1_factor4_world8": dict(replication_jump=1, replication_factor=4, world_size=8),
        "factor1": dict(replication_jump=1, replication_factor=1, world_size=4),
    }.items():
        out[f"group_sequence_{name}"] = _outcome(lambda kw=kw: parse_group_sequence(**kw))
    return out
