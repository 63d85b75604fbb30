"""Parity of the CUDA hot path (called through the C ABI) against the oracle.  Bit-exact: this is byte work.
Run on the B200 box: ``pytest -m gpu``."""
import numpy as np
import pytest
import torch

from oracle import snapshot_oracle as orc

pytestmark = pytest.mark.gpu

VARIANTS = {"ldg": 1, "tma": 2}


def _plan(tensors, narrow=False, **kw):
    from nvidia_resiliency_ext.checkpointing.b200.engine import Plan

    ptrs = [t.data_ptr() if t.numel() else 0 for t in tensors]
    nbytes = [t.numel() * t.element_size() for t in tensors]
    flags = [1 if m else 0 for m in orc.narrow_mask(tensors, narrow)]
    return Plan(ptrs, nbytes, flags, device=torch.cuda.current_device(), **kw)


def _staging(nbytes):
    return torch.zeros(max(nbytes, 512), dtype=torch.uint8, device="cuda")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def ragged_tensors(seed=1):
    """Every source alignment class (0..15) x sizes around the vector / tile boundaries, carved out of one flat
    buffer -- the 'views into a flat param buffer at 4-byte offsets' case of SURVEY 8(d) and worse."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    flat = torch.randint(0, 256, (24 << 20,), dtype=torch.uint8, device="cuda", generator=g)
    sizes = [0, 1, 3, 4, 15, 16, 17, 31, 32, 33, 47, 63, 64, 100, 255, 1000, 1023, 1024, 4095, 4096, 4097, 32768, 32769,
             65536 + 5, (1 << 20) + 13]
    out, cur = [], 0
    for mis in range(16):
        for s in sizes:
            cur = (cur + 15) // 16 * 16 + mis
            out.append(flat[cur : cur + s])
            cur += s
    assert cur < flat.numel()
    return out


def typed_tensors(seed=2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = torch.randn(70001, device="cuda", generator=g)
    return [
        f[:5000].clone(), f[1:4098], f[3:3 + 32768], torch.tensor(7.0, device="cuda"),
        torch.randn(33, 17, device="cuda", generator=g).to(torch.bfloat16),
        torch.randn(9, 5, device="cuda", generator=g).to(torch.float16),
        torch.randn(11, device="cuda", generator=g).to(torch.float64),
        torch.randint(-1000, 1000, (1025,), device="cuda", generator=g, dtype=torch.int64),
        torch.randint(0, 2, (77,), device="cuda", generator=g).bool(),
        torch.randint(-128, 127, (513,), device="cuda", generator=g, dtype=torch.int8),
        torch.empty(0, 3, device="cuda"),
        torch.randn(4, 3, 2, 5, device="cuda", generator=g),
    ]


@pytest.mark.parametrize("variant", ["ldg", "tma"])
@pytest.mark.parametrize("tile", [4096, 32768, 65536])
def test_pack_matches_oracle_ragged(built_library, variant, tile):
    tensors = ragged_tensors() + typed_tensors()
    plan = _plan(tensors, tile_bytes=tile, variant=VARIANTS[variant])
    exp, offs, packed = orc.pack_oracle(tensors)
    assert list(plan.offsets) == offs and list(plan.packed_nbytes) == packed and plan.staging_bytes == exp.size
    assert plan.algorithmic_bytes == 2 * sum(t.numel() * t.element_size() for t in tensors)
    stg = _staging(plan.staging_bytes)
    plan.pack(stg.data_ptr(), _stream())
    torch.cuda.synchronize()
    got = stg[: plan.staging_bytes].cpu().numpy()
    assert np.array_equal(got, exp)
    plan.close()


@pytest.mark.parametrize("variant", ["ldg", "tma"])
@pytest.mark.parametrize("tile", [4096, 32768])
def test_scatter_roundtrip_into_other_alignments(built_library, variant, tile):
    tensors = ragged_tensors(seed=3)
    plan = _plan(tensors, tile_bytes=tile, variant=VARIANTS[variant])
    stg = _staging(plan.staging_bytes)
    plan.pack(stg.data_ptr(), _stream())
    nbytes = [t.numel() for t in tensors]
    flat = torch.zeros(sum(nbytes) + 32 * len(tensors) + 64, dtype=torch.uint8, device="cuda")
    dsts, c = [], 0
    for i, nb in enumerate(nbytes):
        c = (c + 15) // 16 * 16 + (i * 7 + 5) % 16  # destination alignment differs from the source's
        dsts.append(flat[c : c + nb])
        c += nb
    guard = flat.clone()
    plan.update_ptrs([d.data_ptr() if d.numel() else 0 for d in dsts])
    plan.scatter(stg.data_ptr(), _stream())
    torch.cuda.synchronize()
    for d, t in zip(dsts, tensors):
        assert torch.equal(d, t)
    # nothing outside the destinations was touched
    mask = torch.ones_like(flat, dtype=torch.bool)
    for d in dsts:
        if d.numel():
            off = d.data_ptr() - flat.data_ptr()
            mask[off : off + d.numel()] = False
    assert torch.equal(flat[mask], guard[mask])
    plan.close()


@pytest.mark.parametrize("tile", [4096, 65536])
def test_narrow_pack_and_widen_scatter(built_library, tile):
    g = torch.Generator(device="cuda").manual_seed(4)
    base = torch.randn(900_000, device="cuda", generator=g) * 0.02
    edge = torch.tensor([float("inf"), float("-inf"), float("nan"), -0.0, 0.0, 1e-40, -1e-45, 3.3895314e38, -3.4e38, 1.0, 1.00390625,
                         1.005859375, 1.0078125, 65504.0, 1e-6, 2.0**-126, 2.0**-133], device="cuda")
    base[: edge.numel()] = edge
    base[100] = torch.tensor([0x7F800001], dtype=torch.int32, device="cuda").view(torch.float32)[0]  # signalling NaN
    sq = torch.rand(300_000, device="cuda", generator=g) * 1e-38  # denormal-range magnitudes (Adam exp_avg_sq like)
    tensors = [base[:300_001], base[300_001 + 1 : 300_001 + 1 + 8193], base[400_003:400_003 + 77], sq, torch.tensor(3.0, device="cuda"),
               torch.randint(0, 9, (100,), device="cuda", generator=g), torch.empty(0, device="cuda")]
    plan = _plan(tensors, narrow=True, tile_bytes=tile)
    exp, offs, packed = orc.pack_oracle(tensors, narrow=True)
    assert list(plan.offsets) == offs and list(plan.packed_nbytes) == packed
    assert plan.algorithmic_bytes == sum(t.numel() * t.element_size() for t in tensors) + sum(packed)
    stg = _staging(plan.staging_bytes)
    plan.pack(stg.data_ptr(), _stream())
    torch.cuda.synchronize()
    got = stg[: plan.staging_bytes].cpu().numpy()
    assert np.array_equal(got, exp)  # oracle (numpy RNE, NaN -> 0x7FFF)
    # and bit-equal to PyTorch's own conversion on the device
    for t, off, nb, m in zip(tensors, offs, packed, orc.narrow_mask(tensors, True)):
        if t.numel():
            ref = (t.to(torch.bfloat16) if m else t).contiguous().view(-1).view(torch.uint8)
            assert torch.equal(stg[off : off + nb], ref)
    outs = [torch.full_like(t, 7) for t in tensors]
    plan.update_ptrs([o.data_ptr() if o.numel() else 0 for o in outs])
    plan.scatter(stg.data_ptr(), _stream())
    torch.cuda.synchronize()
    for o, t, m in zip(outs, tensors, orc.narrow_mask(tensors, True)):
        want = t.to(torch.bfloat16).to(torch.float32) if m else t
        assert o.dtype == t.dtype
        assert o.numel() == 0 or torch.equal(o.contiguous().view(-1).view(torch.uint8), want.contiguous().view(-1).view(torch.uint8))
    plan.close()


def test_empty_and_degenerate_plans(built_library):
    from nvidia_resiliency_ext.checkpointing.b200._cabi import SnapError
    from nvidia_resiliency_ext.checkpointing.b200.engine import Plan

    p = Plan([], [], None, device=0)
    assert p.staging_bytes == 0 and p.n_tiles == 0
    p.pack(_staging(0).data_ptr(), _stream())
    p.close()
    z = [torch.empty(0, device="cuda"), torch.empty(0, 5, device="cuda")]
    p = _plan(z)
    assert p.staging_bytes == 0 and list(p.offsets) == [0, 0]
    p.pack(_staging(0).data_ptr(), _stream())
    p.close()
    t = torch.ones(10, device="cuda")
    with pytest.raises(SnapError):
        Plan([t.data_ptr()], [40], None, device=0, align=24)  # not a power of two
    with pytest.raises(SnapError):
        Plan([t.data_ptr()], [40], None, device=0, tile_bytes=1000)
    with pytest.raises(SnapError):
        Plan([0], [40], None, device=0)  # null pointer with bytes
    with pytest.raises(SnapError):
        Plan([t.data_ptr() + 2], [8], [1], device=0)  # narrow needs 4-byte alignment
    p = _plan([t])
    with pytest.raises(SnapError):
        p.pack(_staging(1024).data_ptr() + 16, _stream())  # staging must be 512-aligned
    p.close()
    torch.cuda.synchronize()


def test_many_small_tensors_like_reference_cleanup_test(built_library):
    """16384 x (128,128) fp32 = 1 GiB (reference tests/checkpointing/unit/test_cleanup.py:46): many segments."""
    g = torch.Generator(device="cuda").manual_seed(5)
    big = torch.empty(4096 * 128 * 128, device="cuda").random_(generator=g)
    tensors = list(big.view(4096, 128, 128).unbind(0))
    for variant in (1, 2):
        plan = _plan(tensors, variant=variant)
        stg = _staging(plan.staging_bytes)
        plan.pack(stg.data_ptr(), _stream())
        torch.cuda.synchronize()
        assert plan.staging_bytes == big.numel() * 4  # 64 KiB segments: no padding at align 512
        assert torch.equal(stg.view(torch.float32), big)
        plan.close()


def test_full_size_c2_roundtrip_properties(built_library):
    """BASELINE config C2 (16.06 GB, 1164 fp32 tensors + 291 steps): size-independent checks -- per-tensor
    checksums survive pack -> scatter, and packing is insensitive to the walker."""
    import time

    from bench import llama3_8b_shard_state

    free, _ = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip("needs ~50 GB of free HBM")
    marks = [("start", time.perf_counter())]

    def mark(name):
        torch.cuda.synchronize()
        marks.append((name, time.perf_counter()))

    sd, total = llama3_8b_shard_state(torch.device("cuda"), seed=1234)
    tensors = orc.flatten_tensors(sd)
    assert len(tensors) == 1455 and total == 16_060_522_496 + 291 * 4
    mark("state")

    def checksums():
        # one reduction per tensor, results gathered with a single sync
        return torch.stack([t.view(-1).view(torch.int32).sum(dtype=torch.int64) for t in tensors]).cpu()

    sums = checksums()
    mark("checksums")
    plan = _plan(tensors, variant=2)
    stg = _staging(plan.staging_bytes)
    mark("plan+staging")
    plan.pack(stg.data_ptr(), _stream())
    mark("pack tma")
    # checksum of the packed buffer == sum of per-tensor checksums (gaps are zero)
    assert stg[: plan.staging_bytes].view(torch.int32).sum(dtype=torch.int64).item() == int(sums.sum())
    mark("packed checksum")
    plan.set_variant(1)
    stg2 = _staging(plan.staging_bytes)
    plan.pack(stg2.data_ptr(), _stream())
    mark("pack ldg")
    assert torch.equal(stg, stg2)
    mark("compare walkers")
    del stg2
    for t in tensors:
        t.zero_()
    plan.scatter(stg.data_ptr(), _stream())
    mark("scatter")
    assert torch.equal(checksums(), sums)
    mark("checksums 2")
    plan.close()
    print("".join(f"{b:18s} {tb - ta:8.3f} s\n" for (a, ta), (b, tb) in zip(marks, marks[1:])))  # shown by pytest -s / -rP


@pytest.mark.parametrize("chunk_mb,ring,threads", [(4, 2, 3), (64, 4, 16)])
def test_fill_from_fd_pipeline_matches_the_file(tmp_path, chunk_mb, ring, threads):
    """nvrx_fill_from_fd (file -> pinned ring -> device staging): ragged extents at unaligned file offsets, extents larger than
    a chunk, empty ones, more chunks than ring slots; the device bytes of every extent equal the file's, bit for bit."""
    import ctypes as C
    import os

    from nvidia_resiliency_ext.checkpointing.b200 import _cabi

    rng = np.random.default_rng(chunk_mb)
    blob = rng.integers(0, 256, size=40 << 20, dtype=np.uint8)
    path = tmp_path / "blob.bin"
    blob.tofile(path)
    sizes = [0, 1, 15, 16, 4097, 1 << 20, (5 << 20) + 3, 0, 512, (9 << 20) + 1, 77, 3 << 20]
    file_offs, stg_offs, cur_f, cur_s = [], [], 13, 0
    for s in sizes:
        file_offs.append(cur_f)
        cur_s = (cur_s + 511) // 512 * 512
        stg_offs.append(cur_s)
        cur_f += s + 7
        cur_s += s
    total = (cur_s + 511) // 512 * 512
    stg = torch.full((total,), 0xAB, dtype=torch.uint8, device="cuda")
    u64 = lambda v: (C.c_uint64 * len(v))(*v)  # noqa: E731
    fd = os.open(path, os.O_RDONLY)
    try:
        for _ in range(2):  # second call reuses the ring
            _cabi.check(_cabi.lib().nvrx_fill_from_fd(stg.data_ptr(), total, fd, len(sizes), u64(stg_offs), u64(sizes), u64(file_offs),
                                                      chunk_mb << 20, ring, threads, torch.cuda.current_device(), _stream()), "nvrx_fill_from_fd")
            torch.cuda.synchronize()
            got = stg.cpu().numpy()
            for s, fo, so in zip(sizes, file_offs, stg_offs):
                assert np.array_equal(got[so : so + s], blob[fo : fo + s]), (s, fo, so)
    finally:
        os.close(fd)
    # a file shorter than the extents say is an error, not garbage
    fd = os.open(path, os.O_RDONLY)
    try:
        rc = _cabi.lib().nvrx_fill_from_fd(stg.data_ptr(), total, fd, 1, u64([0]), u64([4096]), u64([blob.size - 100]), 0, 0, 2,
                                           torch.cuda.current_device(), _stream())
        assert rc == _cabi.E_SYS
    finally:
        os.close(fd)
