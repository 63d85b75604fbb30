"""Drop-in check of the API surface (SURVEY 8b): every public function, class, method, property and parameter of the
reference's checkpointing modules on the path (tests/golden/api_surface.json, dumped by importing the reference,
tests/golden/make_api_golden.py) exists in the mirror with the same parameter names, order, kinds and defaults.  The mirror
may ADD parameters only if they have defaults (existing call sites keep working)."""
import importlib.util
import json

import pytest
import torch

from conftest import GOLDEN

_spec = importlib.util.spec_from_file_location("make_api_golden", GOLDEN / "make_api_golden.py")
_gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(_gen)

# reference names the mirror leaves out on purpose (reason next to each); everything else must be there
_W = "checkpointing.async_ckpt.filesystem_async."
WAIVED = {
    # worker-side internals of the reference's DCP writer: statics that pass its "write bucket" tuples (tensors as CUDA IPC
    # handles or per-tensor shm) between get_save_function_and_args() and the writer process.  Nothing outside that file calls
    # them (reference tests and docs included); here the writer process gets ONE payload (plan + snapshot slot name) and reads
    # the packed slot, so the bucket plumbing has no counterpart.  What callers use -- the constructor and its options,
    # prepare_write_data, get_save_function_and_args, retrieve_write_results, finish, the cache class methods -- is compared.
    _W + "ConsistentDataIdentifier": "key object of the reference's worker-side bucket cache",
    _W + "FileSystemWriterAsync.preload_tensors": "static: (write buckets, non_blocking) -> per-tensor D2H; replaced by the snapshot engine",
    _W + "FileSystemWriterAsync.write_preloaded_data": "static: one thread's bucket loop",
    _W + "FileSystemWriterAsync.write_preloaded_data_multiproc": "static: bucket fan-out over forked processes",
    _W + "FileSystemWriterAsync.write_preloaded_data_multithread": "static: bucket fan-out over threads",
    _W + "FileSystemWriterAsync.write_preloaded_data_proc": "static: one process's bucket loop",
}

# defaults the reference computes when its module is imported, i.e. from the machine it runs on: the golden holds their value
# on the machine it was dumped on (no GPU), so they are compared with the same expression evaluated here
_S = "checkpointing.local.replication.strategies."
IMPORT_TIME_DEFAULTS = {
    (_S + "CliqueReplicationStrategy.from_replication_params", "replication_jump"): lambda: repr(torch.cuda.device_count()),
    (_S + "LazyCliqueReplicationStrategy.__init__", "replication_jump"): lambda: repr(torch.cuda.device_count()),
}


def _compare_params(where, ref, got, problems):
    if ref is None or got is None:
        return
    got_by_name = {p["name"]: p for p in got}
    ref_names = [p["name"] for p in ref]
    for p in ref:
        g = got_by_name.get(p["name"])
        if g is None:
            if p["kind"] in ("VAR_POSITIONAL", "VAR_KEYWORD"):
                continue
            problems.append(f"{where}: parameter {p['name']!r} is missing")
            continue
        if g["kind"] != p["kind"]:
            problems.append(f"{where}: parameter {p['name']!r} is {g['kind']}, the reference has {p['kind']}")
        want = IMPORT_TIME_DEFAULTS[where, p["name"]]() if (where, p["name"]) in IMPORT_TIME_DEFAULTS else p["default"]
        if g["default"] != want:
            problems.append(f"{where}: default of {p['name']!r} is {g['default']}, the reference has {want}")
    positional = [p["name"] for p in got if p["kind"] in ("POSITIONAL_ONLY", "POSITIONAL_OR_KEYWORD") and p["name"] in ref_names]
    want_positional = [p["name"] for p in ref if p["kind"] in ("POSITIONAL_ONLY", "POSITIONAL_OR_KEYWORD") and p["name"] in got_by_name]
    if positional != want_positional:
        problems.append(f"{where}: positional order {positional} differs from the reference's {want_positional}")
    # an added positional parameter in front of / between the reference's would shift positional call sites
    seen_ref = 0
    for p in got:
        if p["name"] in ref_names:
            seen_ref += 1
        elif p["kind"] in ("POSITIONAL_ONLY", "POSITIONAL_OR_KEYWORD"):
            if seen_ref < len(want_positional):
                problems.append(f"{where}: added positional parameter {p['name']!r} sits before reference parameters")
            if p["default"] is None:
                problems.append(f"{where}: added parameter {p['name']!r} has no default")
        elif p["kind"] == "KEYWORD_ONLY" and p["default"] is None:
            problems.append(f"{where}: added keyword-only parameter {p['name']!r} has no default")


def test_mirror_has_the_references_api_surface():
    golden = json.load(open(GOLDEN / "api_surface.json"))
    assert sorted(golden) == sorted(_gen.MODULES)
    mirror = _gen.surface()  # the same walk over THIS repo's package (conftest puts it on sys.path)
    import nvidia_resiliency_ext

    assert "nvidia-resiliency-ext_b200" in nvidia_resiliency_ext.__file__
    problems = []
    for module, names in golden.items():
        for name, ref in names.items():
            where = f"{module.split('nvidia_resiliency_ext.')[1]}.{name}"
            if where in WAIVED:
                continue
            got = mirror[module].get(name)
            if got is None:
                problems.append(f"{where}: missing")
                continue
            if got["type"] != ref["type"]:
                problems.append(f"{where}: is a {got['type']}, the reference has a {ref['type']}")
                continue
            if ref["type"] == "function":
                _compare_params(where, ref["params"], got["params"], problems)
                continue
            for base in ref["bases"]:
                if base not in got["bases"] and base not in ("ABC", "Generic", "NamedTuple", "tuple"):
                    problems.append(f"{where}: base class {base} is missing (has {got['bases']})")
            for mname, rm in ref["members"].items():
                mwhere = f"{where}.{mname}"
                if mwhere in WAIVED:
                    continue
                gm = got["members"].get(mname)
                if gm is None:
                    # inherited from a base of the mirror's own is as good as defined here
                    cls = getattr(importlib.import_module(module), name)
                    if hasattr(cls, mname):
                        continue
                    problems.append(f"{mwhere}: missing")
                    continue
                if gm["kind"] != rm["kind"]:
                    problems.append(f"{mwhere}: is a {gm['kind']}, the reference has a {rm['kind']}")
                    continue
                if rm["kind"] in ("method", "staticmethod", "classmethod"):
                    _compare_params(mwhere, rm["params"], gm["params"], problems)
                    if rm.get("abstract") and not gm.get("abstract"):
                        problems.append(f"{mwhere}: abstract in the reference, concrete here")
    assert not problems, "\n".join(problems)
