"""Offload engine (save_blocks / load_blocks) through the reference-shaped handlers: bit-exact round trips,
reference file layout, host-arena tier, skip-existing, cancel and failure behaviour."""
import hashlib
import math
import os
import shutil
import struct
import tempfile
import time

import numpy as np
import pytest

from oracle import offload_oracle as oo

pytestmark = pytest.mark.gpu

# one directory per test process: on a machine shared by several users a fixed name may belong to someone else
TMP_DIR = os.path.join(tempfile.gettempdir(), f"kvb-shared-kv-test-{os.getpid()}")


def _kv_tensors(torch, num_layers, num_blocks, block_size, num_heads, head_size, dtype, seed=42):
    """Same construction as the reference test (tests/test_fs_backend.py:45-58): (2, N, bs, H, D) per layer."""
    torch.manual_seed(seed)
    shape = (2, num_blocks, block_size, num_heads, head_size)
    return [torch.rand(shape, dtype=dtype, device="cuda") for _ in range(num_layers)]


def _canonical(torch, kv_tensors):
    """K and V halves of every layer as (num_blocks, page_bytes) int8 views (tests/test_fs_backend.py:61-97)."""
    out = []
    for t in kv_tensors:
        n = t.shape[1]
        half = t.stride(1) * t.element_size()
        raw = torch.tensor([], dtype=torch.int8, device=t.device).set_(t.untyped_storage()).view(2, n, half)
        out.extend(raw.unbind(0))
    return out


def _hash(tokens):
    buf = b"".join(struct.pack("<I", int(t) & 0xFFFFFFFF) for t in tokens)
    return int.from_bytes(hashlib.sha256(buf).digest()[:8], "big").to_bytes(8, "little")


def _hashes(n, start=0):
    return [_hash(range(100 + (start + i) * 100, 117 + (start + i) * 100)) for i in range(n)]


def _wait(handler, job_id, timeout=20.0):
    t0 = time.time()
    while time.time() - t0 < timeout:
        for r in handler.get_finished():
            if r.job_id == job_id:
                return r
        time.sleep(0.002)
    raise TimeoutError(job_id)


def _mapper(kvb, bpf, root=TMP_DIR, dtype="torch.float16"):
    return kvb.file_mapper.FileMapper(root, "llama3-70b", 16, bpf, 1, 1, 1, 0, dtype)


@pytest.fixture(autouse=True)
def _clean():
    shutil.rmtree(TMP_DIR, ignore_errors=True)
    yield
    shutil.rmtree(TMP_DIR, ignore_errors=True)


@pytest.mark.parametrize("tier", ["file", "host_arena"])
@pytest.mark.parametrize("gpu_blocks_per_file", [1, 2, 4, 8])
@pytest.mark.parametrize("start_idx", [0, 3])
def test_roundtrip_param(kvb, torch_cuda, tier, gpu_blocks_per_file, start_idx):
    """Mirror of test_fs_backend_roundtrip_param (tests/test_fs_backend.py:353-411): Llama-70B-like shapes,
    8 blocks, write all, read back blocks start_idx.. into a zeroed cache, bit-exact."""
    torch = torch_cuda
    W, M = kvb.worker, kvb.mediums
    num_layers, block_size, num_heads, head_size, num_blocks = 80, 16, 64, 128, 8
    original = _kv_tensors(torch, num_layers, num_blocks, block_size, num_heads, head_size, torch.float16)
    restored = [torch.zeros_like(t) for t in original]
    write_ids, read_ids = list(range(num_blocks)), list(range(start_idx, num_blocks))
    fm = _mapper(kvb, gpu_blocks_per_file)
    extra = {"tier": tier, "host_arena_bytes": 1 << 30}
    put_files = math.ceil(len(write_ids) / gpu_blocks_per_file)
    hashes = _hashes(put_files)

    h_put = W.StorageOffloadingHandlers(_canonical(torch, original), fm, 16, gpu_blocks_per_file, 8, extra_config=extra)
    put = h_put.gpu_to_storage_handler
    assert put.transfer_async(1, (M.GPULoadStoreSpec(write_ids), M.SharedStorageLoadStoreSpec(hashes)))
    r = _wait(put, 1)
    assert r.success and r.transfer_size > 0 and r.transfer_time > 0 and r.transfer_type == ("GPU", "SHARED_STORAGE")
    for h in hashes:
        assert h_put.engine.exists(fm.get_file_name(h))
        if tier == "file":
            assert os.path.exists(fm.get_file_name(h))

    if tier == "file":   # a second engine (fresh process state) reads what the first one wrote
        h_get = W.StorageOffloadingHandlers(_canonical(torch, restored), fm, 16, gpu_blocks_per_file, 8, extra_config=extra)
        get = h_get.storage_to_gpu_handler
    else:                # the arena lives inside the engine: reuse it, but load into the zeroed cache
        h_get = None
        eng = h_put.engine
        pool2 = kvb.pool.KVPool(_canonical(torch, restored))
    get_files = math.ceil(len(read_ids) / gpu_blocks_per_file)
    get_hashes = hashes[len(hashes) - get_files:]
    if tier == "file":
        assert get.transfer_async(2, (M.SharedStorageLoadStoreSpec(get_hashes), M.GPULoadStoreSpec(read_ids)))
        r = _wait(get, 2)
        assert r.success and r.transfer_type == ("SHARED_STORAGE", "GPU")
        for o_t, r_t in zip(original, restored):
            for b in read_ids:
                assert torch.equal(o_t[:, b], r_t[:, b])
            for b in range(start_idx):
                assert int(r_t[:, b].abs().sum()) == 0        # blocks that were not requested stay untouched
    else:
        # zero the source cache, load back into it through the same engine, compare with a saved copy
        saved = [t.clone() for t in original]
        for t in original:
            t.zero_()
        get = h_put.storage_to_gpu_handler
        assert get.transfer_async(2, (M.SharedStorageLoadStoreSpec(get_hashes), M.GPULoadStoreSpec(read_ids)))
        assert _wait(get, 2).success
        for s_t, o_t in zip(saved, original):
            for b in read_ids:
                assert torch.equal(s_t[:, b], o_t[:, b])
            for b in range(start_idx):
                assert int(o_t[:, b].abs().sum()) == 0


def test_file_bytes_match_reference_layout(kvb, torch_cuda):
    """The bytes on disk are the reference CPU-path image: max(bpf*block,16MiB) long, blocks tail-aligned."""
    torch = torch_cuda
    T, N, frag, bpf = 6, 32, 4096, 4
    g = torch.Generator(device="cuda").manual_seed(1)
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda", generator=g) for _ in range(T)]
    np_t = [t.cpu().numpy() for t in tensors]
    eng = kvb.engine.StorageOffloadEngine(4, bpf, tensors, 3, "disabled", 0.0)
    os.makedirs(TMP_DIR, exist_ok=True)
    groups = [[5, 9], [1, 2, 3, 4], [31, 0, 30, 7]]                # first file partial, like the handlers produce
    files = [f"{TMP_DIR}/a/b/f{i}.bin" for i in range(3)]
    assert eng.async_store_gpu_blocks(7, files, groups)
    eng.wait_job(7)   # NB: wait cancels *queued* work only; poll below confirms completion
    t0 = time.time()
    done = []
    while not done and time.time() - t0 < 10:
        done = [j for j in eng.get_finished() if j[0] == 7]
    assert done == [(7, True)]
    for f, ids in zip(files, groups):
        if not os.path.exists(f):
            continue
        img = np.fromfile(f, dtype=np.uint8)
        assert np.array_equal(img, oo.file_image(np_t, ids, bpf))
    # partial tail read: asking the 4-block file for its last 2 blocks returns blocks 3 and 4's data
    zero = [torch.zeros_like(t) for t in tensors]
    eng2 = kvb.engine.StorageOffloadEngine(2, bpf, zero, 1, "disabled", 0.0)
    if os.path.exists(files[1]):
        assert eng2.async_load_gpu_blocks(8, [files[1]], [[10, 11]])
        while not eng2.get_finished():
            time.sleep(0.001)
        for z, t in zip(zero, tensors):
            assert torch.equal(z[10], t[3]) and torch.equal(z[11], t[4])
    eng.shutdown()
    eng2.shutdown()


def test_store_skips_existing_and_counts(kvb, torch_cuda):
    torch = torch_cuda
    tensors = [torch.randint(0, 256, (16, 1024), dtype=torch.uint8, device="cuda") for _ in range(3)]
    for tier in ("file", "host_arena"):
        eng = kvb.engine.StorageOffloadEngine(2, 2, tensors, 1, "disabled", 0.0, tier=tier, host_arena_bytes=1 << 24)
        f = [f"{TMP_DIR}/{tier}/x.bin", f"{TMP_DIR}/{tier}/y.bin"]
        assert eng.async_store_gpu_blocks(1, f, [[0, 1], [2, 3]])
        while not eng.get_finished():
            time.sleep(0.001)
        keep = [t.clone() for t in tensors]
        for t in tensors:
            t[0:4] = 7                                            # change the blocks, store again under the same names
        assert eng.async_store_gpu_blocks(2, f, [[0, 1], [2, 3]])
        while not eng.get_finished():
            time.sleep(0.001)
        st = eng.stats()
        assert st["files_stored"] == 2 and st["files_skipped_existing"] == 2   # second store wrote nothing
        for t in tensors:
            t[0:4] = 0
        assert eng.async_load_gpu_blocks(3, f, [[0, 1], [2, 3]])
        while not eng.get_finished():
            time.sleep(0.001)
        for t, k in zip(tensors, keep):
            assert torch.equal(t[0:4], k[0:4])                   # the FIRST version is what the tier holds
        eng.shutdown()


def test_missing_file_load_reporting(kvb, torch_cuda):
    torch = torch_cuda
    tensors = [torch.zeros((8, 512), dtype=torch.uint8, device="cuda")]
    # reference behaviour: read failures are swallowed, job still succeeds (storage_offload.cpp:378-383)
    eng = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.0)
    assert eng.async_load_gpu_blocks(1, [f"{TMP_DIR}/nope.bin"], [[0]])
    res = []
    while not res:
        res = eng.get_finished()
    assert res == [(1, True)] and eng.stats()["load_failures"] == 1
    eng.shutdown()
    strict = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.0, strict_load_errors=True)
    assert strict.async_load_gpu_blocks(2, [f"{TMP_DIR}/nope.bin"], [[0]])
    res = []
    while not res:
        res = strict.get_finished()
    assert res == [(2, False)]
    # invalid submissions are refused up front (False), not crashed on
    assert not strict.async_store_gpu_blocks(3, ["a"], [[99]])          # block id out of range
    assert not strict.async_store_gpu_blocks(4, ["a"], [[0, 1]])        # more blocks than gpu_blocks_per_file
    strict.wait_job(12345)                                               # unknown job: returns
    strict.shutdown()


def test_many_jobs_priority_and_wait(kvb, torch_cuda):
    """Several concurrent jobs in both directions; every job is reported exactly once."""
    torch = torch_cuda
    T, N, frag, bpf = 8, 256, 8192, 4
    g = torch.Generator(device="cuda").manual_seed(3)
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda", generator=g) for _ in range(T)]
    ref = [t.clone() for t in tensors]
    eng = kvb.engine.StorageOffloadEngine(4, bpf, tensors, 3, "disabled", 0.0, tier="host_arena",
                                          host_arena_bytes=N * T * frag * 2, chunk_bytes=1 << 20)
    perm = np.random.default_rng(0).permutation(N)
    jobs = {}
    for j in range(8):
        ids = perm[j * 32:(j + 1) * 32]
        files = [f"job{j}/f{i}" for i in range(8)]
        groups = [ids[i * 4:(i + 1) * 4].tolist() for i in range(8)]
        jobs[j] = (files, groups)
        assert eng.async_store_gpu_blocks(j, files, groups)
    seen = {}
    t0 = time.time()
    while len(seen) < 8 and time.time() - t0 < 30:
        for jid, ok in eng.get_finished():
            assert jid not in seen
            seen[jid] = ok
    assert seen == {j: True for j in range(8)}
    for t in tensors:
        t.zero_()
    for j in range(8):
        assert eng.async_load_gpu_blocks(100 + j, *jobs[j])
    for j in range(8):
        eng.wait_job(100 + j)
    fin = dict(eng.get_finished())
    assert fin == {100 + j: True for j in range(8)}
    for t, r in zip(tensors, ref):
        assert torch.equal(t, r)
    st = eng.stats()
    assert st["bytes_stored"] == st["bytes_loaded"] == N * T * frag
    eng.shutdown()


def test_arena_eviction_lru(kvb, torch_cuda):
    torch = torch_cuda
    tensors = [torch.randint(0, 256, (8, 1 << 16), dtype=torch.uint8, device="cuda")]
    eng = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.0, tier="host_arena",
                                          host_arena_bytes=3 << 16)      # room for 3 blocks
    for i in range(5):
        assert eng.async_store_gpu_blocks(i, [f"k{i}"], [[i]])
        while not eng.get_finished():
            time.sleep(0.001)
    assert [eng.exists(f"k{i}") for i in range(5)] == [False, False, True, True, True]
    eng.shutdown()


def test_wait_job_cancels_queued_writes(kvb, torch_cuda):
    """Mirror of the reference's test_wait_job_cancels_queued_writes (tests/test_priority_queue.py:644-731):
    one worker, many files queued behind it, wait() returns quickly, the job still reports success and most
    files were never written."""
    torch = torch_cuda
    T, N, frag = 8, 48, 1 << 20
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda") for _ in range(T)]
    eng = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.0, chunk_bytes=T * frag)  # 1 file per task
    files = [f"{TMP_DIR}/cancel/{i}.bin" for i in range(40)]
    assert eng.async_store_gpu_blocks(1, files, [[i] for i in range(40)])
    t0 = time.time()
    eng.wait_job(1)
    dt = time.time() - t0
    fin = eng.get_finished()
    assert fin == [(1, True)]                       # cancelled job still reports success
    written = sum(os.path.exists(f) for f in files)
    assert dt < 2.0 and written < 40, (dt, written)
    # what was written is complete and correct (no torn files: tmp + rename)
    for i, f in enumerate(files):
        if os.path.exists(f):
            img = np.fromfile(f, dtype=np.uint8)
            assert np.array_equal(img, oo.file_image([t.cpu().numpy() for t in tensors], [i], 1))
            break
    eng.shutdown()


def test_write_queue_limit_drops_excess_writes(kvb, torch_cuda):
    """Mirror of test_write_queue_limit_drops_excess_writes (tests/test_priority_queue.py:557-641): after one write
    primed the EMA, a tiny max_write_queued_seconds makes most files of a large job hit the drop path; the job still
    succeeds and the dropped files do not exist."""
    torch = torch_cuda
    T, N, frag = 4, 64, 1 << 20
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda") for _ in range(T)]
    eng = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.01, chunk_bytes=T * frag)
    assert eng.async_store_gpu_blocks(0, [f"{TMP_DIR}/drop/prime.bin"], [[0]])
    while not eng.get_finished():
        time.sleep(0.001)
    files = [f"{TMP_DIR}/drop/{i}.bin" for i in range(50)]
    assert eng.async_store_gpu_blocks(1, files, [[1 + i] for i in range(50)])
    res = []
    t0 = time.time()
    while not res and time.time() - t0 < 30:
        res = eng.get_finished()
    assert res == [(1, True)]
    written = sum(os.path.exists(f) for f in files)
    st = eng.stats()
    assert st["writes_dropped"] == 50 - written, (written, st)
    if written == 50:   # limit = threads*budget/avg_write rounds to 0 ("no limit") on very slow storage, as in the reference
        pytest.skip("storage too slow/fast for the 10 ms budget to produce a non-zero queue limit")
    eng.shutdown()


def test_reads_overtake_queued_writes(kvb, torch_cuda):
    """Loads go to the high-priority queue (storage_offload.cpp:413): a load submitted after a pile of stores
    finishes before the pile drains (reference: test_priority_completion_order, tests/test_priority_queue.py:96)."""
    torch = torch_cuda
    T, N, frag = 4, 128, 1 << 20
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda") for _ in range(T)]
    eng = kvb.engine.StorageOffloadEngine(2, 1, tensors, 1, "disabled", 0.0, chunk_bytes=T * frag)
    assert eng.async_store_gpu_blocks(0, [f"{TMP_DIR}/prio/seed.bin"], [[0]])
    while not eng.get_finished():
        time.sleep(0.001)
    for j in range(1, 5):
        files = [f"{TMP_DIR}/prio/w{j}_{i}.bin" for i in range(25)]
        assert eng.async_store_gpu_blocks(j, files, [[1 + (j - 1) * 25 + i] for i in range(25)])
    assert eng.async_load_gpu_blocks(99, [f"{TMP_DIR}/prio/seed.bin"], [[127]])
    order = []
    t0 = time.time()
    while len(order) < 5 and time.time() - t0 < 60:
        order.extend(j for j, ok in eng.get_finished() if ok)
        time.sleep(0.0005)
    assert sorted(order) == [1, 2, 3, 4, 99]
    assert order.index(99) < 4, order               # the read did not wait behind every queued write
    assert all(torch.equal(t[127], t[0]) for t in tensors)
    eng.shutdown()


@pytest.mark.parametrize("tier", ["file", "host_arena"])
def test_direct_host_io_roundtrip(kvb, torch_cuda, tier):
    """direct_host_io: the gather kernel's bulk stores land in pinned host memory (fused gather+D2H) and the scatter
    kernel reads it back (fused H2D+scatter); same files / arena entries, same bytes as the staged path."""
    torch = torch_cuda
    T, N, frag, bpf = 16, 96, 16384, 4
    g = torch.Generator(device="cuda").manual_seed(21)
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda", generator=g) for _ in range(T)]
    ref = [t.clone() for t in tensors]
    ids = np.random.default_rng(2).permutation(N)[:70]
    groups = [ids[:2].tolist()] + [ids[2 + 4 * i: 6 + 4 * i].tolist() for i in range(17)]
    files = [f"{TMP_DIR}/direct/{tier}/{i}.bin" for i in range(len(groups))]
    eng = kvb.engine.StorageOffloadEngine(3, bpf, tensors, 2, "disabled", 0.0, tier=tier, host_arena_bytes=1 << 28,
                                          chunk_bytes=1 << 20, direct_host_io=True)
    assert eng.async_store_gpu_blocks(1, files, groups)
    while not eng.get_finished():
        time.sleep(0.001)
    if tier == "file":
        np_t = [t.cpu().numpy() for t in ref]
        for f, grp in zip(files, groups):
            assert np.array_equal(np.fromfile(f, dtype=np.uint8), oo.file_image(np_t, grp, bpf))
    for t in tensors:
        t.zero_()
    assert eng.async_load_gpu_blocks(2, files, groups)
    while not eng.get_finished():
        time.sleep(0.001)
    idt = torch.from_numpy(ids).cuda()
    for t, r in zip(tensors, ref):
        assert torch.equal(t[idt], r[idt])
        mask = torch.ones(N, dtype=torch.bool, device="cuda")
        mask[idt] = False
        assert int(t[mask].sum()) == 0
    st = eng.stats()
    assert st["bytes_stored"] == st["bytes_loaded"] == 70 * T * frag
    eng.shutdown()


@pytest.mark.parametrize("tier", ["file", "host_arena"])
def test_missing_file_does_not_block_other_files(kvb, torch_cuda, tier):
    """The reference runs one task per file (storage_offload.cpp:373-419): a missing file fails alone, the other files
    of the same job are still loaded.  Same here although several files share one GPU chunk."""
    torch = torch_cuda
    tensors = [torch.randint(1, 256, (16, 4096), dtype=torch.uint8, device="cuda") for _ in range(3)]
    ref = [t.clone() for t in tensors]
    eng = kvb.engine.StorageOffloadEngine(2, 2, tensors, 1, "disabled", 0.0, tier=tier, host_arena_bytes=1 << 24,
                                          strict_load_errors=True)
    files = [f"{TMP_DIR}/partial/{tier}/{i}.bin" for i in range(3)]
    groups = [[0, 1], [2, 3], [4, 5]]
    assert eng.async_store_gpu_blocks(1, [files[0], files[2]], [groups[0], groups[2]])      # file 1 never stored
    while not eng.get_finished():
        time.sleep(0.001)
    for t in tensors:
        t.zero_()
    assert eng.async_load_gpu_blocks(2, files, groups)
    res = []
    while not res:
        res = eng.get_finished()
    assert res == [(2, False)]                                   # strict mode reports the failure ...
    for t, r in zip(tensors, ref):
        assert torch.equal(t[[0, 1, 4, 5]], r[[0, 1, 4, 5]])     # ... but the files that exist were loaded
        assert int(t[[2, 3]].sum()) == 0
    st = eng.stats()
    assert st["files_loaded"] == 2 and st["load_failures"] == 1
    eng.shutdown()


@pytest.mark.parametrize("mode", ["read_write", "bb_read_write", "write_only", "read_only"])
def test_gds_tier_format_and_roundtrip(kvb, torch_cuda, mode):
    """gds_mode: stores write the reference's GDS file format (gds_file_io.cpp:238-330: exactly n x block_bytes,
    head-aligned, [block][tensor][fragment]) from the packed HBM chunk with one cuFile call per file; loads read the
    FIRST n blocks (:386-414).  Modes route reads / writes like the reference (storage_offload.cpp:111-146)."""
    torch = torch_cuda
    T, N, frag, bpf = 5, 40, 8192, 4
    g = torch.Generator(device="cuda").manual_seed(3)
    tensors = [torch.randint(0, 256, (N, frag), dtype=torch.uint8, device="cuda", generator=g) for _ in range(T)]
    np_t = [t.cpu().numpy() for t in tensors]
    root = f"{TMP_DIR}/gds_{mode}"
    shutil.rmtree(root, ignore_errors=True)
    eng = kvb.engine.StorageOffloadEngine(4, bpf, tensors, 3, mode, 0.0, strict_load_errors=True)
    groups = [[7, 3], [11, 12, 13, 14], [39, 0, 20, 5], [9]]
    files = [f"{root}/x/f{i}.bin" for i in range(len(groups))]
    assert eng.async_store_gpu_blocks(1, files, groups)
    t0 = time.time()
    done = []
    while not done and time.time() - t0 < 20:
        done = [j for j in eng.get_finished() if j[0] == 1]
    assert done == [(1, True)]
    writes_gds = mode in ("read_write", "bb_read_write", "write_only")
    for f, ids in zip(files, groups):
        img = np.fromfile(f, dtype=np.uint8)
        if writes_gds:
            assert np.array_equal(img, oo.pack_blocks(np_t, ids))           # nothing but the payload, from offset 0
        else:
            assert np.array_equal(img, oo.file_image(np_t, ids, bpf))       # CPU-path image (tail-aligned, full size)
    reads_gds = mode in ("read_write", "bb_read_write", "read_only")
    if reads_gds != writes_gds:
        eng.shutdown()
        return            # mixed modes only agree on full files in the reference too; the formats are checked above
    zero = [torch.zeros_like(t) for t in tensors]
    eng2 = kvb.engine.StorageOffloadEngine(2, bpf, zero, 1, mode, 0.0, strict_load_errors=True)
    dst = [[1, 2], [21, 22, 23, 24], [30, 31, 32, 33], [8]]
    assert eng2.async_load_gpu_blocks(2, files, dst)
    done = []
    t0 = time.time()
    while not done and time.time() - t0 < 20:
        done = [j for j in eng2.get_finished() if j[0] == 2]
    assert done == [(2, True)]
    for ids, to in zip(groups, dst):
        for a, b in zip(ids, to):
            for z, t in zip(zero, tensors):
                assert torch.equal(z[b], t[a])
    # a shorter read takes the FIRST blocks of a GDS file
    assert eng2.async_load_gpu_blocks(3, [files[1]], [[35, 36]])
    done = []
    while not done and time.time() - t0 < 40:
        done = [j for j in eng2.get_finished() if j[0] == 3]
    assert done == [(3, True)]
    for z, t in zip(zero, tensors):
        assert torch.equal(z[35], t[11]) and torch.equal(z[36], t[12])
    eng.shutdown()
    eng2.shutdown()


@pytest.mark.parametrize("tier", ["file", "host_arena"])
def test_manager_lookup_is_one_library_call(kvb, torch_cuda, tier):
    """SharedStorageOffloadingManager.lookup (manager.py:43-53): consecutive hits from the start, stopping at the first
    miss — through kvb_engine_lookup_prefix, against the reference's per-block loop on the same state."""
    torch = torch_cuda
    bpf = 2
    tensors = [torch.randint(0, 256, (64, 4096), dtype=torch.uint8, device="cuda") for _ in range(4)]
    kw = dict(tier=tier, host_arena_bytes=8 << 20) if tier == "host_arena" else {}
    eng = kvb.engine.StorageOffloadEngine(2, bpf, tensors, 1, "disabled", 0.0, **kw)
    fm = _mapper(kvb, bpf)
    hashes = _hashes(24)
    files = [fm.get_file_name(h) for h in hashes]
    present = [0, 1, 2, 3, 4, 6, 7, 10]                      # a hole at 5: the prefix is 5 long whatever comes after
    assert eng.async_store_gpu_blocks(1, [files[i] for i in present], [[2 * i, 2 * i + 1] for i in present])
    while not eng.get_finished():
        time.sleep(0.001)
    mgr = kvb.manager.SharedStorageOffloadingManager(fm, engine=eng)
    loop = kvb.manager.SharedStorageOffloadingManager(fm, exists=eng.exists)          # the reference's loop
    for start in (0, 1, 5, 6, 10, 11):
        assert mgr.lookup(hashes[start:]) == loop.lookup(hashes[start:]), start
    assert mgr.lookup(hashes) == 5 and mgr.lookup(hashes[6:]) == 2 and mgr.lookup(hashes[5:]) == 0 and mgr.lookup([]) == 0
    assert eng.lookup_prefix([files[0], files[1]]) == 2
    eng.shutdown()


def test_arena_miss_fails_the_load(kvb, torch_cuda):
    """The reference swallows a vanished FILE (storage_offload.cpp:378-383).  An entry the host arena's own LRU dropped
    is a different thing — nothing was restored — and must fail the job without any strict flag."""
    torch = torch_cuda
    tensors = [torch.randint(0, 256, (8, 1 << 16), dtype=torch.uint8, device="cuda")]
    eng = kvb.engine.StorageOffloadEngine(1, 1, tensors, 1, "disabled", 0.0, tier="host_arena", host_arena_bytes=2 << 16)
    for i in range(3):                                       # room for 2: k0 is evicted by k2
        assert eng.async_store_gpu_blocks(i, [f"k{i}"], [[i]])
        while not eng.get_finished():
            time.sleep(0.001)
    assert not eng.exists("k0")
    assert eng.async_load_gpu_blocks(10, ["k0"], [[0]])
    res = []
    while not res:
        res = eng.get_finished()
        time.sleep(0.001)
    assert res == [(10, False)] and eng.stats()["load_failures"] == 1
    eng.shutdown()


def test_engine_that_cannot_allocate_its_workers_fails_at_construction(kvb, torch_cuda):
    """Worker resources (a packed HBM chunk per worker) are part of construction: asking for more than the device has is a
    constructor error, not a load that quietly restores nothing later."""
    torch = torch_cuda
    tensors = [torch.randint(0, 256, (8, 1 << 16), dtype=torch.uint8, device="cuda")]
    free, _total = torch.cuda.mem_get_info()
    per_worker = (free // 4 + (1 << 30)) // (1 << 16) * (1 << 16)       # 8 workers x > free/4: cannot fit
    with pytest.raises(Exception) as ei:
        kvb.engine.StorageOffloadEngine(8, 1, tensors, 1, "disabled", 0.0, tier="host_arena", host_arena_bytes=4 << 16,
                                        chunk_bytes=per_worker)
    assert "do not fit" in str(ei.value) or "NOMEM" in str(ei.value) or "-3" in str(ei.value)
    # and the device is still usable afterwards
    ok = kvb.engine.StorageOffloadEngine(2, 1, tensors, 1, "disabled", 0.0, tier="host_arena", host_arena_bytes=4 << 16)
    ok.shutdown()
