#!/usr/bin/env python
"""bench.py — KV-block offload throughput (save + load) on N x B200, one process per GPU.

Metric (BASELINE.json): KV-block offload GB/s (save+load); blocks/sec.
Workload at N=1 = BASELINE config #2: Llama-3-8B fp16 paged KV, 16-token blocks
  64 canonical tensors x (12288 blocks x 32768 B), 10 000 random non-contiguous block ids,
  one step = save the 10 000 blocks + load them back (2 x 20.97 GB of payload).
Every rank runs the same workload on its own GPU / KV partition (weak scaling, no data-path collective).

  value     device-resident: paged pool -> packed HBM (gather kernel) and back (scatter kernel); inputs in HBM.
            It has NO host leg: compare it with the HBM roofline, not with the reference arm.
  e2e       through the reference-facing engine API (StorageOffloadEngine.async_store_gpu_blocks /
            async_load_gpu_blocks), tier = host_arena (pinned host DRAM): D2H of every saved block and H2D of every
            loaded block inside the timed region.  This is the north-star host tier.
  e2e_file_tier  the same API writing the REFERENCE'S on-disk format to /dev/shm, at every N, on the same blocks per step
            as the reference arm: the like-for-like number against `--impl reference`.
  roofline  gather kernel: 2 x payload bytes / CUDA-event time per launch vs the measured HBM copy peak.
  extras    config1 / config5 (index path), config3 (70B-fp8 block shape), migration (+ migration_70b) at N > 1,
            ingest, manager_lookup — computed in the same run, each asserting parity before it reports a number.
  cpu_baseline / --impl reference: the UNMODIFIED reference engine (oracle/_ref, built from /root/reference's own
            csrc) storing to and loading from /dev/shm with its default per-(block x tensor) cudaMemcpyAsync path.
            At N > 1 every rank runs its own reference engine on its own GPU (storage_offload.cpp:160-167) and the
            line reports the aggregate.  `config.blocks_per_step` is the number of blocks it really moved per step.
"""
from __future__ import annotations

import argparse
import importlib
import importlib.util
import json
import os
import shutil
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import bench_extras as bx  # noqa: E402

# ---- workload: BASELINE config #2 -------------------------------------------------------------------------
T_TENSORS = 64          # K and V of 32 layers
FRAG_BYTES = 32768      # 16 tok x 8 kv heads x 128 x fp16
POOL_BLOCKS = int(os.environ.get("KVB_BENCH_POOL_BLOCKS", "12288"))   # env overrides exist ONLY for ncu captures
N_BLOCKS = int(os.environ.get("KVB_BENCH_BLOCKS", "10000"))           # (a reduced run says so in config)
BLOCK_BYTES = T_TENSORS * FRAG_BYTES          # 2 MiB
BLOCKS_PER_FILE = 16                           # reference default: 256-token files / 16-token blocks (spec.py:50-85)
MIGRATE_BLOCKS = 2048                          # BASELINE config #4: 32k-token context = 2048 blocks (4.29 GB, 8B shape)
# The file tier (reference arm and our like-for-like arm) runs on tmpfs at single-digit GB/s: its blocks per step are
# bounded so that the whole --steps K --warmup W run stays within a few minutes.  The full 10 000 blocks when the run is
# short enough, never fewer than 2048, and the number REALLY used is what `config.blocks_per_step` reports.
FILE_TIER_BLOCK_BUDGET = 100_000               # blocks moved each way over the whole run, per rank


def file_tier_blocks(steps: int, warmup: int) -> int:
    per_step = FILE_TIER_BLOCK_BUDGET // max(1, steps + warmup)
    n = max(2048, min(N_BLOCKS, per_step)) // BLOCKS_PER_FILE * BLOCKS_PER_FILE
    n = min(n, N_BLOCKS // BLOCKS_PER_FILE * BLOCKS_PER_FILE)
    try:  # and it must fit the tmpfs, with room for every rank of this node
        free = shutil.disk_usage("/dev/shm").free
        world = int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1")))
        fit = int(free * 0.6 / world / BLOCK_BYTES) // BLOCKS_PER_FILE * BLOCKS_PER_FILE
        n = max(BLOCKS_PER_FILE, min(n, fit))
    except Exception:
        pass
    return n


_JSON_FD = None


def emit_json(obj) -> None:
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def env_int(name, d):
    v = os.environ.get(name)
    return int(v) if v else d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_reference_engine():
    """The unmodified reference engine built into oracle/_ref by oracle/ref_build/build_ref.py (or None)."""
    so = os.path.join(ROOT, "oracle", "_ref", "storage_offload_ref.so")
    if not os.path.exists(so):
        return None, "oracle/_ref/storage_offload_ref.so not built"
    try:
        import torch  # noqa: F401  (libtorch must be loaded first)
        spec = importlib.util.spec_from_file_location("storage_offload_ref", so)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod, None
    except Exception as e:
        return None, f"cannot load reference engine: {e}"


def file_groups(ids, bpf=BLOCKS_PER_FILE):
    """worker.py:158-193 grouping: the first file takes the remainder."""
    n_files = (len(ids) + bpf - 1) // bpf
    first = len(ids) % bpf or bpf
    groups, pos, take = [], 0, first
    for _ in range(n_files):
        groups.append([int(x) for x in ids[pos:pos + take]])
        pos += take
        take = bpf
    return groups


def reference_step(mod, tensors, ids, step_tag, io_threads, root="/dev/shm/kvb_ref_bench"):
    """One save+load of `ids` through the reference engine (default memcpy path), files on tmpfs.
    Returns seconds for (store, load)."""
    import torch
    bpf = BLOCKS_PER_FILE
    groups = file_groups(ids, bpf)
    files = [f"{root}/{step_tag}/{i:06d}.bin" for i in range(len(groups))]
    eng = reference_step.engines.get(id(tensors[0]))
    if eng is None:
        eng = mod.StorageOffloadEngine(io_threads, bpf, tensors, max(1, int(io_threads * 0.75)), "disabled", 0.0)
        reference_step.engines[id(tensors[0])] = eng
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.async_store_gpu_blocks(1, files, groups)
    _drain(eng, 1)
    t1 = time.perf_counter()
    eng.async_load_gpu_blocks(2, files, groups)
    _drain(eng, 2)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    shutil.rmtree(f"{root}/{step_tag}", ignore_errors=True)
    return t1 - t0, t2 - t1


reference_step.engines = {}

_drain = bx._drain
barrier_sync = bx.barrier_sync
max_over_ranks = bx.max_over_ranks


def pipelined_save_load(eng, files, groups, files_per_job=25, first_job=1000):
    """Same work as store-all-then-load-all, submitted as many small jobs: file group j is loaded as soon as its own
    store job has finished, while later groups are still being stored — so D2H and H2D are in flight together.
    Works for any engine with the reference's surface.  Returns seconds."""
    jobs = [(files[i:i + files_per_job], groups[i:i + files_per_job]) for i in range(0, len(files), files_per_job)]
    t0 = time.perf_counter()
    for j, (f, g) in enumerate(jobs):
        assert eng.async_store_gpu_blocks(first_job + 2 * j, f, g)
    pending_loads = len(jobs)
    deadline = t0 + 900
    while pending_loads and time.perf_counter() < deadline:
        for jid, ok in eng.get_finished():
            if not ok:
                raise RuntimeError(f"job {jid} failed")
            k = jid - first_job
            if k % 2 == 0:      # a store finished: its files can be loaded back now
                f, g = jobs[k // 2]
                assert eng.async_load_gpu_blocks(jid + 1, f, g)
            else:
                pending_loads -= 1
        time.sleep(0.0002)
    if pending_loads:
        raise TimeoutError("pipelined save+load")
    return time.perf_counter() - t0


def single_file_job_latency(eng, ids, root, jobs=40, first_job=500000, cleanup=None):
    """Median wall time of ONE-file jobs (16 blocks = 32 MiB) issued one at a time: store latency and load latency.
    Small jobs are what a serving engine issues per request; works for any engine with the reference's surface."""
    bpf = BLOCKS_PER_FILE
    st, ld = [], []
    for j in range(jobs):
        grp = [[int(x) for x in ids[(j * bpf) % (len(ids) - bpf):(j * bpf) % (len(ids) - bpf) + bpf]]]
        f = [f"{root}/lat_{j:04d}.bin"]
        t0 = time.perf_counter()
        assert eng.async_store_gpu_blocks(first_job + 2 * j, f, grp)
        _drain(eng, first_job + 2 * j, sleep=0)
        t1 = time.perf_counter()
        assert eng.async_load_gpu_blocks(first_job + 2 * j + 1, f, grp)
        _drain(eng, first_job + 2 * j + 1, sleep=0)
        t2 = time.perf_counter()
        if j >= 5:  # first jobs warm the workers
            st.append(t1 - t0)
            ld.append(t2 - t1)
    if cleanup:
        cleanup()
    return {"store_ms_median": float(np.median(st)) * 1e3, "load_ms_median": float(np.median(ld)) * 1e3,
            "blocks_per_job": bpf, "bytes_per_job": bpf * BLOCK_BYTES, "jobs": len(st)}


def pool_checksum(big) -> int:
    """64-bit wrap-around sum of every 8-byte word of the pool (order independent)."""
    import torch
    return int(big.view(torch.int64).sum().item())


def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


DUMP_SAMPLE = 1 << 22   # values sampled from each dumped output: 2 x 4 Mi float32 = 32 MiB


def dump_outputs(out_dir, packed, big, ids_dev):
    """What the timed path computed in its last step, so that two builds can be compared output for output: the packed
    buffer the gather kernel wrote (packed.npy) and the pool pages the scatter kernel wrote back (pool.npy).  Both are
    ~21 GB, so each is a sample at fixed seeded byte positions, stored as float32 (the bytes are exact in it)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(2024)
    pos = torch.from_numpy(np.sort(rng.integers(0, packed.numel(), DUMP_SAMPLE))).cuda()
    np.save(os.path.join(out_dir, "packed.npy"), packed[pos].float().cpu().numpy())
    t = torch.from_numpy(rng.integers(0, big.shape[0], DUMP_SAMPLE)).cuda()
    k = torch.from_numpy(rng.integers(0, ids_dev.numel(), DUMP_SAMPLE)).cuda()
    b = torch.from_numpy(rng.integers(0, big.shape[2], DUMP_SAMPLE)).cuda()
    np.save(os.path.join(out_dir, "pool.npy"), big[t, ids_dev[k], b].float().cpu().numpy())


def workload_config(n_gpus, blocks_per_step=N_BLOCKS):
    cfg = {"workload": "BASELINE config #2: Llama-3-8B fp16 paged-KV, 16-tok blocks, save+load 10k blocks GPU<->host",
           "tensors": T_TENSORS, "fragment_bytes": FRAG_BYTES, "block_bytes": BLOCK_BYTES, "pool_blocks": POOL_BLOCKS,
           "blocks_per_step": blocks_per_step, "workload_blocks": N_BLOCKS,
           "block_ids": f"rng(1).permutation({POOL_BLOCKS})[:{blocks_per_step}] (non-contiguous, unsorted)",
           "gpu_blocks_per_file": BLOCKS_PER_FILE, "partitioning": f"{n_gpus} independent KV partitions (one per GPU)",
           "l2_policy": f"inputs_exceed_l2 ({blocks_per_step * BLOCK_BYTES / 1e9:.2f} GB per pass vs 126 MB L2)"}
    return cfg


# ---------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The unmodified reference engine, ONE PER RANK on its own GPU (storage_offload.cpp:160-167: the engine takes the
    caller's current device), files under /dev/shm/<rank>; the line reports the aggregate over all ranks with the
    max-over-ranks time, like our own arm."""
    import torch
    rank, world, local, dist = dist_setup(args.gpus)
    mod, why = load_reference_engine()
    n_ref = file_tier_blocks(args.steps, args.warmup)
    ids = np.random.default_rng(1).permutation(POOL_BLOCKS)[:n_ref].astype(np.int64)
    cores = os.cpu_count() or 1
    io_threads = min(64, cores)
    big = torch.empty((T_TENSORS, POOL_BLOCKS, FRAG_BYTES), dtype=torch.int8, device="cuda")
    big.view(torch.uint8).random_(0, 256)
    tensors = list(big.unbind(0))
    payload = n_ref * BLOCK_BYTES
    kind = "reference"
    root = f"/dev/shm/kvb_ref_bench/rank_{rank}"
    if mod is None:
        # oracle port: numpy pack/unpack of the same bytes on the host (single thread)
        kind = "port"
        from oracle import offload_oracle as oo
        host = [t.cpu().numpy().view(np.uint8) for t in tensors]

        def step(tag):
            t0 = time.perf_counter()
            p = oo.pack_blocks(host, ids)
            oo.unpack_blocks(host, ids, p)
            return time.perf_counter() - t0
        io_threads = 1
    else:
        def step(tag):
            a, b = reference_step(mod, tensors, ids, tag, io_threads, root=root)
            return a + b
    for w in range(args.warmup):
        step(f"w{w}")
    barrier_sync(dist)
    # timed region = the store and load phases of every step; deleting the previous step's tmpfs files (several GB of
    # page frees) is housekeeping between steps and is NOT charged to the reference
    dt = 0.0
    for k in range(args.steps):
        barrier_sync(dist)
        dt += step(f"s{k}")
    barrier_sync(dist)
    dt = max_over_ranks(dist, dt)
    shutil.rmtree(root, ignore_errors=True)
    gbs = world * 2 * payload * args.steps / dt / 1e9
    sample = (f"{n_ref} of the workload's {N_BLOCKS} blocks per step (seed-1 permutation prefix) on each of {world} GPU(s), "
              f"save+load per step, {BLOCKS_PER_FILE} blocks/file on /dev/shm, default cudaMemcpyAsync copy path, "
              f"{io_threads} io_threads per engine")
    if rank == 0:
        line = {
            "impl": "reference", "metric": "kv_block_offload_gbps_save_plus_load", "value": gbs, "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world, n_ref),
            "blocks_per_s": world * 2 * n_ref * args.steps / dt,
            "engines": world, "tier": "file (/dev/shm)",
            "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": io_threads * world, "kind": kind, "sample": sample,
                             "host_cores": cores, **({"note": why} if why else {})},
            "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        emit_json(line)
    reference_step.engines.clear()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def pcie_probe(kvb, dist, world, local, huge_pages=False):
    """What a plain cudaMemcpyAsync of one contiguous 2 GiB buffer achieves when the host side is pinned memory placed on
    the GPU's NUMA node (kvb_host_alloc — the same placement the engine's arena uses), all ranks at once: the ceiling
    the e2e number is a fraction of.  Per-rank figures are kept so that a lagging root complex is visible."""
    import torch
    try:
        from cuda.bindings import runtime as cudart
    except Exception:  # older cuda-python
        from cuda import cudart
    probe_n = 2 << 30
    pin = kvb.pool.PinnedBuffer(probe_n, huge_pages=huge_pages)
    dbuf = torch.empty(probe_n, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    out = {}
    for name, (dst, src, kind) in (("d2h_gbs", (pin.ptr, dbuf.data_ptr(), cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)),
                                   ("h2d_gbs", (dbuf.data_ptr(), pin.ptr, cudart.cudaMemcpyKind.cudaMemcpyHostToDevice))):
        cudart.cudaMemcpyAsync(dst, src, probe_n, kind, stream)
        barrier_sync(dist)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            (err,) = cudart.cudaMemcpyAsync(dst, src, probe_n, kind, stream)
            assert int(err) == 0, f"cudaMemcpyAsync: {err}"
        b.record()
        barrier_sync(dist)
        mine = 3 * probe_n / (a.elapsed_time(b) / 1e3) / 1e9
        out[name] = world * 3 * probe_n / (max_over_ranks(dist, a.elapsed_time(b)) / 1e3) / 1e9
        out[name.replace("_gbs", "_gbs_per_gpu")] = [round(x, 2) for x in bx.gather_objects(dist, mine)]
    del dbuf
    pin.free()
    out["what"] = ("contiguous 2 GiB cudaMemcpyAsync, host side pinned on the GPU's NUMA node ("
                   + ("transparent huge pages + cudaHostRegister" if huge_pages else "kvb_host_alloc / cudaHostAlloc")
                   + "), all ranks at once (aggregate GB/s = bytes / max-over-ranks time)")
    return out


def run_file_tier(kvb, dist, rank, world, tensors, n_ref, with_latency):
    """Our engine, tier=file: the reference's on-disk format on the same tmpfs, same blocks per step and file grouping as
    the reference arm — the like-for-like comparison for the storage tier — at every N (one engine per rank)."""
    import torch
    root = f"/dev/shm/kvb_file_bench/rank_{rank}"
    ids = np.random.default_rng(1).permutation(POOL_BLOCKS)[:n_ref].astype(np.int64)
    payload = n_ref * BLOCK_BYTES
    bpf = BLOCKS_PER_FILE
    groups = file_groups(ids, bpf)
    n_files = len(groups)
    threads = min(env_int("KVB_BENCH_FILE_THREADS", 16), os.cpu_count() or 1)
    eng = kvb.engine.StorageOffloadEngine(threads, bpf, tensors, max(1, int(threads * 0.75)), "disabled", 0.0,
                                          tier="file", chunk_bytes=bpf * BLOCK_BYTES)
    res = {}
    try:
        for tag in ("warm", "base"):
            files = [f"{root}/{tag}/{i:06d}.bin" for i in range(n_files)]
            barrier_sync(dist)
            t0 = time.perf_counter()
            assert eng.async_store_gpu_blocks(1, files, groups)
            _drain(eng, 1)
            t1 = time.perf_counter()
            if tag == "warm":   # the warm-up pass doubles as the proof: zero the saved pages before loading them back
                ids_dev = torch.from_numpy(ids).to(tensors[0].device)
                keep = [t[ids_dev[:32]].clone() for t in tensors[::16]]
                for t in tensors:
                    t[ids_dev] = 0
                torch.cuda.synchronize()
            t1b = time.perf_counter()
            assert eng.async_load_gpu_blocks(2, files, groups)
            _drain(eng, 2)
            t2 = time.perf_counter()
            if tag == "warm":
                for t, k in zip(tensors[::16], keep):
                    assert torch.equal(t[ids_dev[:32]], k), "file-tier load did not restore zeroed pages"
            shutil.rmtree(f"{root}/{tag}", ignore_errors=True)
            barrier_sync(dist)
            st, ld = max_over_ranks(dist, t1 - t0), max_over_ranks(dist, t2 - t1b)
            res = {"value": world * 2 * payload / (st + ld) / 1e9, "unit": "GB/s", "store_gbs": world * payload / st / 1e9,
                   "load_gbs": world * payload / ld / 1e9, "io_threads": threads, "tier": "file (/dev/shm)",
                   "blocks_per_step": n_ref, "engines": world, "bit_exact": True,
                   "store_gbs_per_gpu": [round(x, 2) for x in bx.gather_objects(dist, payload / (t1 - t0) / 1e9)],
                   "load_gbs_per_gpu": [round(x, 2) for x in bx.gather_objects(dist, payload / (t2 - t1b) / 1e9)],
                   "sample": f"{n_ref} blocks per rank, {bpf} blocks/file, reference .bin format on /dev/shm "
                             "(same blocks per step and grouping as the --impl reference arm)"}
        if with_latency:
            res["single_file_job_latency"] = single_file_job_latency(eng, ids, f"{root}/lat")
    finally:
        eng.shutdown()
        shutil.rmtree(root, ignore_errors=True)
    return res


def run_ours(args):
    import torch
    rank, world, local, dist = dist_setup(args.gpus)
    kvb = importlib.import_module("llm-d-kv-cache_b200")
    lib = kvb.lib
    peak, peak_src = measured_hbm_peak()
    n_ref = file_tier_blocks(args.steps, args.warmup)

    # ---- data: pool resident in HBM, random bytes, random block table
    big = torch.empty((T_TENSORS, POOL_BLOCKS, FRAG_BYTES), dtype=torch.uint8, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(42 + rank)
    big.random_(0, 256, generator=g)
    tensors = list(big.unbind(0))
    pool = kvb.pool.KVPool(tensors)
    ids_np = np.random.default_rng(1).permutation(POOL_BLOCKS)[:N_BLOCKS].astype(np.int64)
    ids_dev = torch.from_numpy(ids_np).cuda()
    packed = torch.empty(N_BLOCKS * BLOCK_BYTES, dtype=torch.uint8, device="cuda")
    payload = N_BLOCKS * BLOCK_BYTES
    check_ids = ids_dev[:: max(1, N_BLOCKS // 64)]
    check_ref = [t[check_ids].clone() for t in tensors[::8]]

    # ---- device-resident arm: gather + scatter, every launch timed with CUDA events on its own stream
    def dev_step(evs=None):
        if evs is not None:
            evs[0].record()
        pool.gather_dev(ids_dev, packed)
        if evs is not None:
            evs[1].record()
        pool.scatter_dev(ids_dev, packed)
        if evs is not None:
            evs[2].record()

    for _ in range(args.warmup):
        dev_step()
    sampler = ClockSampler(local)
    launches_start = lib.kvb_launch_count()
    barrier_sync(dist)
    if rank == 0:
        sampler.start()
    ev_sets = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for k in range(args.steps):
        dev_step(ev_sets[k])
    stop.record()
    barrier_sync(dist)
    dev_ms = max_over_ranks(dist, start.elapsed_time(stop))
    gather_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in ev_sets]))
    scatter_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in ev_sets]))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, packed, big, ids_dev)
    # untimed proof that the load leg really restores: save, ZERO every saved page, load, compare
    sum0 = pool_checksum(big)
    pool.gather_dev(ids_dev, packed)
    big[:, ids_dev] = 0
    assert pool_checksum(big) != sum0
    pool.scatter_dev(ids_dev, packed)
    assert pool_checksum(big) == sum0, "device-resident save+load did not restore the pool bit-exact"
    for t, r in zip(tensors[::8], check_ref):
        assert torch.equal(t[check_ids], r), "device-resident save+load did not restore the pool bit-exact"
    value = world * 2 * payload * args.steps / (dev_ms / 1e3) / 1e9
    del packed
    torch.cuda.empty_cache()

    # ---- e2e arm: reference-facing engine API, host-arena tier, D2H + H2D inside the timed region
    bpf = BLOCKS_PER_FILE
    n_files = N_BLOCKS // bpf
    groups = [ids_np[i * bpf:(i + 1) * bpf].tolist() for i in range(n_files)]
    eng = kvb.engine.StorageOffloadEngine(env_int("KVB_BENCH_IO_THREADS", 4), bpf, tensors, 3, "disabled", 0.0,
                                          tier="host_arena", host_arena_bytes=payload + (64 << 20),
                                          chunk_bytes=env_int("KVB_BENCH_CHUNK_MB", 64) << 20)
    job = [0]

    def e2e_step(tag):
        files = [f"{tag}/{i:06d}" for i in range(n_files)]
        job[0] += 1
        assert eng.async_store_gpu_blocks(job[0], files, groups)
        _drain(eng, job[0])
        t_mid = time.perf_counter()
        job[0] += 1
        assert eng.async_load_gpu_blocks(job[0], files, groups)
        _drain(eng, job[0])
        eng.arena_clear()
        return t_mid

    for w in range(args.warmup):
        e2e_step(f"w{w}")
    stats0 = eng.stats()
    barrier_sync(dist)
    t0 = time.perf_counter()
    store_s = 0.0
    for k in range(args.steps):
        ts = time.perf_counter()
        store_s += e2e_step(f"s{k}") - ts
    my_e2e_s = time.perf_counter() - t0
    barrier_sync(dist)
    e2e_s = max_over_ranks(dist, time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    stats1 = eng.stats()
    per_gpu = bx.gather_objects(dist, {"store": payload * args.steps / store_s / 1e9,
                                       "load": payload * args.steps / max(my_e2e_s - store_s, 1e-9) / 1e9})
    store_s_max = max_over_ranks(dist, store_s)
    # untimed proof through the engine: store, ZERO every saved page, load, whole-pool checksum + samples
    vfiles = [f"verify/{i:06d}" for i in range(n_files)]
    job[0] += 1
    assert eng.async_store_gpu_blocks(job[0], vfiles, groups)
    _drain(eng, job[0])
    big[:, ids_dev] = 0
    job[0] += 1
    assert eng.async_load_gpu_blocks(job[0], vfiles, groups)
    _drain(eng, job[0])
    eng.arena_clear()
    assert pool_checksum(big) == sum0, "engine save+load did not restore the pool bit-exact"
    for t, r in zip(tensors[::8], check_ref):
        assert torch.equal(t[check_ids], r), "engine save+load did not restore the pool bit-exact"
    e2e_gbs = world * 2 * payload * args.steps / e2e_s / 1e9
    h2d = (stats1["h2d_bytes"] - stats0["h2d_bytes"]) // args.steps
    d2h = (stats1["d2h_bytes"] - stats0["d2h_bytes"]) // args.steps
    # same bytes, submitted as pipelined jobs (loads of group j overlap stores of later groups: full-duplex PCIe)
    pipelined_save_load(eng, [f"pw/{i:06d}" for i in range(n_files)], groups)
    eng.arena_clear()
    barrier_sync(dist)
    t_pipe = pipelined_save_load(eng, [f"pp/{i:06d}" for i in range(n_files)], groups, first_job=100000)
    barrier_sync(dist)
    t_pipe = max_over_ranks(dist, t_pipe)
    for t, r in zip(tensors[::8], check_ref):
        assert torch.equal(t[check_ids], r), "pipelined save+load did not restore the pool bit-exact"
    eng.arena_clear()
    job_latency = single_file_job_latency(eng, ids_np, "lat") if rank == 0 else None
    eng.shutdown()
    # extra: fused variant — the gather / scatter kernels address the pinned arena directly (no staging, no memcpy)
    eng_d = kvb.engine.StorageOffloadEngine(env_int("KVB_BENCH_IO_THREADS", 4), bpf, tensors, 3, "disabled", 0.0,
                                            tier="host_arena", host_arena_bytes=payload + (64 << 20),
                                            chunk_bytes=env_int("KVB_BENCH_CHUNK_MB", 64) << 20, direct_host_io=True)
    t_direct = None
    for tag in ("dw", "dt"):
        dfiles = [f"{tag}/{i:06d}" for i in range(n_files)]
        barrier_sync(dist)
        td0 = time.perf_counter()
        assert eng_d.async_store_gpu_blocks(1, dfiles, groups)
        _drain(eng_d, 1)
        if tag == "dt":
            big[:, ids_dev[:256]] = 0
        assert eng_d.async_load_gpu_blocks(2, dfiles, groups)
        _drain(eng_d, 2)
        barrier_sync(dist)
        t_direct = max_over_ranks(dist, time.perf_counter() - td0)
        eng_d.arena_clear()
    assert pool_checksum(big) == sum0, "direct_host_io save+load did not restore the pool bit-exact"
    eng_d.shutdown()

    probe = pcie_probe(kvb, dist, world, local)
    probe_thp = pcie_probe(kvb, dist, world, local, huge_pages=True)
    # the same e2e arm with the arena on transparent huge pages (A/B of the host side; where several GPUs share a socket
    # the D2H leg is what falls behind): one warm-up step + two timed steps
    thp_arm = None
    if world > 1 or os.environ.get("KVB_BENCH_THP_ARM"):
        eng_t = kvb.engine.StorageOffloadEngine(env_int("KVB_BENCH_IO_THREADS", 4), bpf, tensors, 3, "disabled", 0.0,
                                                tier="host_arena", host_arena_bytes=payload + (64 << 20),
                                                chunk_bytes=env_int("KVB_BENCH_CHUNK_MB", 64) << 20, arena_huge_pages=True)
        jt = [0]

        def thp_step(tag):
            files = [f"{tag}/{i:06d}" for i in range(n_files)]
            jt[0] += 1
            assert eng_t.async_store_gpu_blocks(jt[0], files, groups)
            _drain(eng_t, jt[0])
            t_mid = time.perf_counter()
            jt[0] += 1
            assert eng_t.async_load_gpu_blocks(jt[0], files, groups)
            _drain(eng_t, jt[0])
            eng_t.arena_clear()
            return t_mid
        thp_step("tw")
        barrier_sync(dist)
        tt0 = time.perf_counter()
        st_t = 0.0
        for k in range(2):
            ts = time.perf_counter()
            st_t += thp_step(f"tt{k}") - ts
        mine_t = time.perf_counter() - tt0
        barrier_sync(dist)
        tot_t = max_over_ranks(dist, time.perf_counter() - tt0)
        pg = bx.gather_objects(dist, {"store": payload * 2 / st_t / 1e9, "load": payload * 2 / max(mine_t - st_t, 1e-9) / 1e9})
        eng_t.shutdown()
        assert pool_checksum(big) == sum0, "huge-page arena save+load did not restore the pool bit-exact"
        thp_arm = {"value": world * 2 * payload * 2 / tot_t / 1e9, "unit": "GB/s", "steps": 2,
                   "store_gbs_per_gpu": [round(x["store"], 2) for x in pg], "load_gbs_per_gpu": [round(x["load"], 2) for x in pg],
                   "arena": "transparent huge pages + cudaHostRegister, first-touched on the GPU's NUMA node"}

    # ---- like-for-like storage tier: reference-format files on /dev/shm, every N
    file_tier = run_file_tier(kvb, dist, rank, world, tensors, n_ref, with_latency=(rank == 0 and world == 1))
    for t, r in zip(tensors[::8], check_ref):
        assert torch.equal(t[check_ids], r), "file-tier save+load did not restore the pool bit-exact"

    extras = {}
    if rank == 0 and not args.no_extras:
        extras["manager_lookup"] = bx.run_manager_lookup(kvb)

    # ---- cross-GPU migration over NVLink (only where there is a peer)
    migration = None
    ref_mod, _why = load_reference_engine()
    if world > 1 and not args.no_migration:
        migration = bx.run_migration(kvb, dist, rank, world, local, tensors, pool, POOL_BLOCKS, BLOCK_BYTES,
                                     min(MIGRATE_BLOCKS, POOL_BLOCKS // 4), args.steps, args.warmup,
                                     reference_engine=ref_mod, blocks_per_file=BLOCKS_PER_FILE, shape_name="8B-fp16")

    # ---- cpu baseline (rank 0, N=1 only): the reference engine on the same blocks per step as the file-tier arm
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = run_cpu_baseline(tensors, n_ref)
        for t, r in zip(tensors[::8], check_ref):
            assert torch.equal(t[check_ids], r), "the reference arm disturbed the pool"
    launches_cfg2 = lib.kvb_launch_count() - launches_start

    # ---- extras on their own data: config #3 (every rank, weak scaling), then configs #1 / #5 / ingest (rank 0)
    pool.close()
    del check_ref, tensors, big, ids_dev
    torch.cuda.empty_cache()
    if not args.no_extras:
        c3 = bx.run_config3(kvb, dist, rank, world, local, args.steps, args.warmup, peak, peak_src,
                            migrate=not args.no_migration)
        if rank == 0:
            extras["config3"] = c3
            if "migration_70b" in c3:
                extras["migration_70b"] = c3.pop("migration_70b")
            cfg1, cfg5 = bx.run_index_configs(kvb)
            if cfg5["roofline"]["achieved"] is not None:
                cfg5["roofline"]["peak"], cfg5["roofline"]["peak_source"] = peak, peak_src
                cfg5["roofline"]["frac"] = cfg5["roofline"]["achieved"] / peak
            extras["config1"], extras["config5"] = cfg1, cfg5
            extras["ingest"] = bx.run_ingest(kvb)
        barrier_sync(dist)

    if rank == 0:
        achieved = 2 * payload / (gather_ms / 1e3) / 1e9
        traffic = bx._traffic("gather_traffic.json")
        line = {
            "metric": "kv_block_offload_gbps_save_plus_load", "value": value, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(world),
            "value_note": "device-resident gather+scatter (HBM<->HBM, no host leg): judge it against roofline, not against the "
                          "reference arm; the reference-facing numbers are e2e (host arena) and e2e_file_tier (like-for-like)",
            "blocks_per_s": world * 2 * N_BLOCKS * args.steps / (dev_ms / 1e3),
            "e2e": {"value": e2e_gbs, "unit": "GB/s", "tier": "host_arena (pinned host DRAM, NUMA-local)",
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "blocks_per_s": world * 2 * N_BLOCKS * args.steps / e2e_s, "ms_per_step": e2e_s / args.steps * 1e3,
                    "store_gbs": world * payload * args.steps / store_s_max / 1e9,
                    "load_gbs": world * payload * args.steps / max(e2e_s - store_s_max, 1e-9) / 1e9,
                    "store_gbs_per_gpu": [round(x["store"], 2) for x in per_gpu],
                    "load_gbs_per_gpu": [round(x["load"], 2) for x in per_gpu],
                    "pcie_probe": probe, "pcie_probe_huge_pages": probe_thp, "arena_huge_pages_arm": thp_arm,
                    "frac_of_pcie_probe": e2e_gbs / (2 * probe["d2h_gbs"] * probe["h2d_gbs"] / (probe["d2h_gbs"] + probe["h2d_gbs"])),
                    "pipelined_jobs_gbs": world * 2 * payload / t_pipe / 1e9,
                    "single_file_job_latency": job_latency,
                    "direct_host_io_gbs": world * 2 * payload / t_direct / 1e9,
                    "direct_host_io_note": "extra: fused gather+D2H / H2D+scatter kernels addressing the pinned arena (no HBM staging, no cudaMemcpy)",
                    "pipelined_note": "extra, not the headline: 25-file jobs, each group loaded back as soon as it is stored, so D2H and H2D overlap",
                    "api": "StorageOffloadEngine.async_store_gpu_blocks/async_load_gpu_blocks/get_finished"},
            "e2e_file_tier": file_tier,
            "gpu_launches": int(launches_cfg2),
            "roofline": {"kernel": "paged_copy_bulk_kernel<gather>", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": 2 * payload, "gather_ms": gather_ms, "scatter_ms": scatter_ms,
                         "scatter_achieved": 2 * payload / (scatter_ms / 1e3) / 1e9,
                         "frac_of_nominal_8TBs": achieved / 8000.0},
            "clocks": clocks,
        }
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if migration is not None:
            line["migration"] = migration
        if extras:
            line["extras"] = extras
            line["gpu_launches_total"] = int(lib.kvb_launch_count())
        emit_json(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def run_cpu_baseline(tensors, n_ref):
    """Reference engine (oracle/_ref) on the same blocks per step as e2e_file_tier, same box, same run."""
    import torch
    cores = os.cpu_count() or 1
    ids = np.random.default_rng(1).permutation(POOL_BLOCKS)[:n_ref].astype(np.int64)
    payload = n_ref * BLOCK_BYTES
    mod, why = load_reference_engine()
    sample = (f"{n_ref} of the workload's {N_BLOCKS} blocks, save+load once after one warm-up pass, "
              f"{BLOCKS_PER_FILE} blocks/file on /dev/shm")
    if mod is not None:
        io_threads = min(64, cores)
        i8 = [t.view(torch.int8) for t in tensors]
        try:
            reference_step(mod, i8, ids[:256], "warm", io_threads)
            a, b = reference_step(mod, i8, ids, "base", io_threads)
            ref_eng = reference_step.engines[id(i8[0])]
            root = "/dev/shm/kvb_ref_bench/pipe"
            pg = file_groups(ids[:2048])
            pf = [f"{root}/{i:06d}.bin" for i in range(len(pg))]
            try:
                t_pipe = pipelined_save_load(ref_eng, pf, pg, files_per_job=8)
            except Exception as e:  # the extra must not take the baseline down
                t_pipe = None
                print(f"[bench] reference pipelined pattern failed: {e}", file=sys.stderr)
            shutil.rmtree(root, ignore_errors=True)
            try:
                lat = single_file_job_latency(ref_eng, ids, "/dev/shm/kvb_ref_bench/lat",
                                              cleanup=lambda: shutil.rmtree("/dev/shm/kvb_ref_bench/lat", ignore_errors=True))
            except Exception as e:
                lat = {"error": repr(e)}
            reference_step.engines.clear()
            del ref_eng
            # the reference's opt-in SM-copy path (tensor_copier.cu:41-42 reads the switches when the engine is built).
            # It runs on its OWN scratch pool: that path stages a block at slot `block_id % blocks_per_file`
            # (tensor_copier_kernels.cu:78-80), so a file whose ids collide modulo 16 does not round-trip and would
            # corrupt the workload's pool; whether it round-tripped is reported, not assumed.
            kc = None
            try:
                os.environ["USE_KERNEL_COPY_READ"] = os.environ["USE_KERNEL_COPY_WRITE"] = "1"
                g = torch.Generator(device="cuda").manual_seed(7)
                scratch = [torch.randint(0, 127, (1024, FRAG_BYTES), dtype=torch.int8, device="cuda", generator=g)
                           for _ in range(len(tensors))]
                want = [t.clone() for t in scratch]
                # aligned 16-block runs in random order: the only id pattern that path stores without collisions
                runs = np.random.default_rng(3).permutation(1024 // BLOCKS_PER_FILE)[:512 // BLOCKS_PER_FILE]
                small = (runs[:, None] * BLOCKS_PER_FILE + np.arange(BLOCKS_PER_FILE)[None, :]).reshape(-1).astype(np.int64)
                reference_step(mod, scratch, small[:64], "kwarm", io_threads)
                ka, kb = reference_step(mod, scratch, small, "kcopy", io_threads)
                exact = all(torch.equal(x, y) for x, y in zip(scratch, want))
                kc = {"gbs": 2 * len(small) * BLOCK_BYTES / (ka + kb) / 1e9, "store_gbs": len(small) * BLOCK_BYTES / ka / 1e9,
                      "load_gbs": len(small) * BLOCK_BYTES / kb / 1e9, "roundtrip_bit_exact": bool(exact),
                      "sample": f"{len(small)} blocks of a 1024-block scratch pool as aligned {BLOCKS_PER_FILE}-block runs "
                                "(random ids collide in its id % blocks_per_file staging slots), USE_KERNEL_COPY_READ=WRITE=1"}
                del scratch, want
            except Exception as e:
                kc = {"error": repr(e)}
            finally:
                os.environ.pop("USE_KERNEL_COPY_READ", None)
                os.environ.pop("USE_KERNEL_COPY_WRITE", None)
                reference_step.engines.clear()
            return {"value": 2 * payload / (a + b) / 1e9, "unit": "GB/s", "cores": io_threads, "kind": "reference",
                    "single_file_job_latency": lat, "kernel_copy_path": kc, "blocks_per_step": n_ref,
                    "pipelined_jobs_gbs": (2 * 2048 * BLOCK_BYTES / t_pipe / 1e9) if t_pipe else None,
                    "sample": sample + ", default cudaMemcpyAsync path, io_threads=min(64,nproc)",
                    "store_gbs": payload / a / 1e9, "load_gbs": payload / b / 1e9, "host_cores": cores,
                    "numa_note": "built with numa_set_preferred stubbed (no libnuma in the image): its staging buffers are "
                                 "first-touched by threads it pins to the GPU's node itself (thread_pool.cpp:73-131)"}
        except Exception as e:
            why = f"reference engine failed: {e}"
    from oracle import offload_oracle as oo
    n = 256
    host = [t[:2048].cpu().numpy() for t in tensors]
    sub = np.random.default_rng(1).permutation(2048)[:n].astype(np.int64)
    t0 = time.perf_counter()
    p = oo.pack_blocks(host, sub)
    oo.unpack_blocks(host, sub, p)
    dt = time.perf_counter() - t0
    return {"value": 2 * n * BLOCK_BYTES / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
            "sample": f"{n} blocks of the same shape, numpy pack+unpack (oracle port)", "note": why, "host_cores": cores}


def main():
    # stdout must carry exactly ONE JSON line, but native libraries write there too (NCCL prints its version banner on
    # fd 1).  Keep the real stdout aside for the JSON line and point fd 1 at stderr for everything else.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-migration", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip configs #1/#3/#5, ingest and manager lookup (ncu captures)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a fixed sample of what the last step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
