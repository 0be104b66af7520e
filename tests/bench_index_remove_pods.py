"""Time kvb_index_remove_pods on the config #5 index (10 M keys from 64 pods, as bench_extras.run_index_configs builds
it: 512 shared entry lists of 1..10 (pod, tier) entries, 80 % gpu / 20 % cpu) and print one JSON line.

    python tests/bench_index_remove_pods.py [--reps 20]

  (a) a sweep that removes nothing (an interned pod without entries): the pure read of the table
  (b) one pod per call, 8 different pods: median and spread
  (c) 8 other pods in one call
Every call is timed on the host clock around the whole library call, which ends in a device synchronise (bitmap upload,
sweep kernel, counter read-back).  Bytes the algorithm needs: every bucket read once (64 B), plus 64 B per changed bucket
and 8 B per deleted key's stamp written.  Beside it, in the same run, a plain torch read (sum) of as many bytes as the
table holds.  The table (2 GiB) is far larger than the 126 MB L2, so no cache flush is needed between passes.
Before anything is timed, a purge is checked: len before - keys deleted == len after, and a seeded sample of 65536 keys
looks the same before and after except for the purged pod's entries (order kept, emptied keys absent)."""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_KEYS, N_PODS, N_PATTERNS, PPK = 10_000_000, 64, 512, 10
HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still reported, without its power limit
        q = "unavailable (%s)" % e
    return name, q


def inner_lru(ents):
    """The pod list a key holds after one Add of `ents` (inner LRU of PodCacheSize entries, in_memory.go:205-221)."""
    out = []
    for e in ents:
        if e in out:
            out.remove(e)
        elif len(out) == PPK:
            out.pop(0)
        out.append(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="timed sweeps of (a) and of the torch read")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    torch.cuda.set_device(0)
    kvb = importlib.import_module("llm-d-kv-cache_b200")
    K = kvb.kvblock
    rng = np.random.default_rng(2)

    # ---- the config #5 index (bench_extras.run_index_configs' background keys)
    pods = ["10.0.%d.%d" % (i // 8, i % 8) for i in range(N_PODS)]
    idx = K.Index(expected_keys=N_KEYS + (1 << 16), pod_cache_size=PPK)
    for p in pods:
        idx.pods.get(p)
    bg = rng.integers(1, 1 << 63, N_KEYS, dtype=np.int64).astype(np.uint64)
    pat_of = rng.integers(0, N_PATTERNS, N_KEYS)
    order = np.argsort(pat_of, kind="stable")
    bounds = np.searchsorted(pat_of[order], np.arange(N_PATTERNS + 1))
    lists, per_pat = [], np.zeros(N_PATTERNS, dtype=np.int64)
    for pt in range(N_PATTERNS):
        ks = np.ascontiguousarray(bg[order[bounds[pt]:bounds[pt + 1]]])
        ents = [(pods[int(rng.integers(0, N_PODS))], "gpu" if rng.random() < 0.8 else "cpu")
                for _ in range(int(rng.integers(1, 11)))]
        if ks.size:
            idx.add(None, ks, [K.PodEntry(*e) for e in ents])
        lists.append(inner_lru(ents))
        per_pat[pt] = ks.size
    idx.flush()
    st = idx.stats()
    slots = int(st["table_slots"])
    table_bytes = slots * 64
    n_live = len(idx)

    def expect(gone):
        """changed buckets and deleted keys of removing `gone`, and the pattern lists after it"""
        changed = deleted = 0
        for pt, lst in enumerate(lists):
            kept = [e for e in lst if e[0] not in gone]
            if len(kept) != len(lst):
                changed += int(per_pat[pt])
                deleted += int(per_pat[pt]) if not kept else 0
            lists[pt] = kept
        return changed, deleted

    def timed(pod_names):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = idx.remove_pods(pod_names)
        return time.perf_counter() - t0, r

    # ---- correctness before timing: one pod, checked on a seeded sample
    sample = [int(k) for k in bg[np.random.default_rng(7).choice(N_KEYS, 65536, replace=False)]]
    before = idx.lookup(sample)
    probe = pods[63]
    want_changed, want_deleted = expect({probe})
    _, (removed, deleted) = timed([probe])
    assert deleted == want_deleted and len(idx) == n_live - deleted, (deleted, want_deleted)
    after = idx.lookup(sample)
    want = {k: [e for e in v if e.pod_identifier != probe] for k, v in before.items()}
    assert after == {k: v for k, v in want.items() if v}, "sample differs from the expected purge"
    n_live -= deleted

    # ---- (a) read floor: an interned pod without entries
    idx.pods.get("idle-pod")
    timed(["idle-pod"])  # warm-up
    ta = []
    for _ in range(args.reps):
        dt, r = timed(["idle-pod"])
        assert r == (0, 0)
        ta.append(dt)

    # ---- (b) one pod per call, (c) 8 pods in one call
    tb, b_bytes = [], []
    for p in pods[:8]:
        ch, de = expect({p})
        dt, r = timed([p])
        assert r[1] == de
        tb.append(dt)
        b_bytes.append(table_bytes + 64 * ch + 8 * de)
    group = set(pods[8:16])
    ch, de = expect(group)
    tc, rc = timed(sorted(group))
    assert rc[1] == de
    c_bytes = table_bytes + 64 * ch + 8 * de

    # ---- the same number of bytes read by torch, same run
    x = torch.empty(table_bytes // 4, dtype=torch.float32, device="cuda").uniform_()
    x.sum()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tt = []
    for _ in range(args.reps):
        ev0.record()
        x.sum()
        ev1.record()
        ev1.synchronize()
        tt.append(ev0.elapsed_time(ev1) / 1e3)
    del x

    def rate(nbytes, sec):
        return nbytes / sec / 1e9

    t_torch = float(np.median(tt))
    ma, mb = float(np.median(ta)), float(np.median(tb))
    out = {
        "bench": "index_remove_pods",
        "card": card()[0], "power_limit_and_max_sm_clock": card()[1],
        "keys": n_live, "pods": N_PODS, "table_slots": slots, "table_bytes": table_bytes,
        "l2_note": "table of %.2f GB >> 126 MB L2: no flush between passes" % (table_bytes / 1e9),
        "timing": "host clock around the whole call (ends in a device synchronise)",
        "a_no_match": {"ms": ma * 1e3, "ms_min": min(ta) * 1e3, "ms_max": max(ta) * 1e3,
                       "bytes": table_bytes, "GBps": rate(table_bytes, ma),
                       "share_of_7.7TBps": rate(table_bytes, ma) / (HBM_TBPS * 1e3),
                       "vs_torch_read": t_torch / ma},
        "b_one_pod": {"ms_median": mb * 1e3, "ms_min": min(tb) * 1e3, "ms_max": max(tb) * 1e3,
                      "bytes_median": float(np.median(b_bytes)),
                      "GBps": rate(float(np.median(b_bytes)), mb),
                      "share_of_7.7TBps": rate(float(np.median(b_bytes)), mb) / (HBM_TBPS * 1e3),
                      "vs_torch_read": t_torch * float(np.median(b_bytes)) / table_bytes / mb},
        "c_eight_pods": {"ms": tc * 1e3, "bytes": c_bytes, "entries_removed": rc[0], "keys_deleted": rc[1],
                         "GBps": rate(c_bytes, tc), "share_of_7.7TBps": rate(c_bytes, tc) / (HBM_TBPS * 1e3)},
        "torch_read": {"ms_median": t_torch * 1e3, "bytes": table_bytes, "GBps": rate(table_bytes, t_torch)},
        "target": "(a) and (b) >= 0.7 x the same-run torch read",
        "checked": {"sample_keys": len(sample), "keys_deleted": deleted, "entries_removed": removed},
    }
    idx.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
