"""Pod removal on the real kernels (index_remove_pods_kernel in csrc/index.cu): the scenarios of
tests/test_index_remove_pods_sim.py on libkvb.so, a table large enough for a many-CTA sweep, scoring after a purge,
AllBlocksCleared in event streams, and the C++ mirror."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import kvblock_oracle as o
from oracle import kvevents_oracle as eo
from tests import pod_removal as pr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "llm-d-kv-cache_b200")

pytestmark = pytest.mark.gpu


def test_known_answer(kvb, torch_cuda):
    pr.known_answer(kvb.kvblock, None)


def test_queued_ops_apply_in_call_order(kvb, torch_cuda):
    pr.queue_ordering(kvb.kvblock, None)


def test_recency_is_not_touched(kvb, torch_cuda):
    pr.recency_untouched(kvb.kvblock, None)


@pytest.mark.parametrize("batch", [8, 400])
def test_purge_at_capacity_then_add_batches(kvb, torch_cuda, batch):
    st = pr.purge_at_capacity_then_adds(kvb.kvblock, None, batch=batch)
    assert st["lru_evictions"] > 1000
    assert (st["flushes_planned"] if batch > 16 else st["flushes_sequential"]) > 5


@pytest.mark.parametrize("size,n_keys,max_batch", [(3, 60, 40), (300, 500, 5), (10 ** 8, 6000, 400)])
def test_random_traffic_with_purges(kvb, torch_cuda, size, n_keys, max_batch):
    st = pr.random_traffic(kvb.kvblock, None, seed=size % 1000 + 1, size=size, ppk=3, n_keys=n_keys, steps=500,
                           max_batch=max_batch)
    if size == 10 ** 8:
        assert st["rehashes"] >= 1


def test_large_table_three_pods(kvb, torch_cuda):
    """2^22 slots, 1 M keys from 64 pods (shared entry lists, as the benchmark's index): three pods removed in one call;
    every key read back and the counts equal the oracle's LRU applied to each list."""
    K = kvb.kvblock
    rng = np.random.default_rng(17)
    n_keys, n_pat, ppk = 1 << 20, 256, 10
    idx = K.Index(pod_cache_size=ppk, expected_keys=1_200_000)
    assert idx.stats()["table_slots"] >= 1 << 22
    pods = ["10.0.%d.%d" % (i // 8, i % 8) for i in range(64)]
    keys = np.unique(rng.integers(1, 1 << 63, n_keys + 4096, dtype=np.int64).astype(np.uint64))[:n_keys]
    rng.shuffle(keys)
    pat_of = rng.integers(0, n_pat, keys.size)
    lists = []
    for p in range(n_pat):
        ents = [(pods[int(rng.integers(0, 64))], "gpu" if rng.random() < 0.8 else "cpu", bool(rng.random() < 0.1))
                for _ in range(int(rng.integers(1, 11)))]
        ks = np.ascontiguousarray(keys[pat_of == p])
        if ks.size:
            idx.add(None, ks, [K.PodEntry(*e) for e in ents])
        inner = o.LRU(ppk)                       # what the key holds: the oracle's inner LRU over the list
        for e in ents:
            inner.add(o.PodEntry(*e), None)
        lists.append(inner.keys())
    gone = set(pods[i] for i in rng.choice(64, 3, replace=False))
    n_before = len(idx)
    assert n_before == keys.size
    removed, deleted = idx.remove_pods(sorted(gone))
    kept = [[e for e in lst if e.pod_identifier not in gone] for lst in lists]
    per_pat = np.bincount(pat_of, minlength=n_pat)
    assert removed == int(sum((len(lists[p]) - len(kept[p])) * per_pat[p] for p in range(n_pat)))
    assert deleted == int(sum(per_pat[p] for p in range(n_pat) if not kept[p]))
    assert deleted > 0 and len(idx) == n_before - deleted
    st = idx.stats()
    assert st["live_keys"] == n_before - deleted and st["tombstones"] >= deleted
    # every key, entry order included
    def pack(e):
        return idx.pods.ids[e.pod_identifier] | (idx.tiers.ids[e.device_tier] << 16) | (int(e.speculative) << 24)
    want_cnt = np.array([len(k) if k else -1 for k in kept], dtype=np.int32)
    want_ent = np.zeros((n_pat, 13), dtype=np.uint32)
    for p, k in enumerate(kept):
        want_ent[p, :len(k)] = [pack(e) for e in k]
    counts = np.empty(keys.size, dtype=np.int32)
    ents = np.zeros((keys.size, 13), dtype=np.uint32)
    cut = C.c_int64()
    idx._check(idx._lib.kvb_index_lookup(idx._h, keys.ctypes.data, keys.size, None, 0, counts.ctypes.data,
                                         ents.ctypes.data, C.byref(cut)))
    assert cut.value == keys.size
    assert np.array_equal(counts, want_cnt[pat_of])
    mask = np.arange(13)[None, :] < np.maximum(counts, 0)[:, None]
    assert np.array_equal(np.where(mask, ents, 0), np.where(mask, want_ent[pat_of], 0))
    idx.close()


def test_scoring_after_a_purge(kvb, torch_cuda):
    """score_tokens_batch after remove_pods, with and without touch_lru: bit-exact against the oracle Indexer."""
    K = kvb.kvblock
    rng = np.random.default_rng(5)
    tp, otp = K.ChunkedTokenDatabase(16, ""), o.TokenProcessor(16, "")
    idx, oidx = K.Index(), o.InMemoryIndex()
    prompts = [[int(t) for t in rng.integers(0, 50000, 16 * int(rng.integers(1, 12)))] for _ in range(48)]
    pods = ["pod-%d" % i for i in range(8)]
    for pr_ in prompts:
        keys = otp.tokens_to_kv_block_keys(0, pr_, "m")
        for _ in range(int(rng.integers(1, 5))):
            d = int(rng.integers(1, len(keys) + 1))
            ents = [(pods[int(rng.integers(0, 8))], "gpu" if rng.random() < 0.7 else "cpu")]
            idx.add(None, keys[:d], [K.PodEntry(*e) for e in ents])
            oidx.add(None, keys[:d], [o.PodEntry(*e) for e in ents])
    assert idx.remove_pods(["pod-1", "pod-2"]) == pr.remove_pods(oidx, ["pod-1", "pod-2"])
    assert idx.remove_pods(["pod-3"], ["cpu"]) == pr.remove_pods(oidx, ["pod-3"], ["cpu"])
    oracle = o.Indexer(otp, oidx)
    want = [oracle.score_tokens(p, "m") or {} for p in prompts]
    assert any(want) and not any("pod-1" in w or "pod-2" in w for w in want)
    for touch in (False, True):
        got, _ = idx.score_tokens_batch(tp, prompts, "m", touch_lru=touch)
        assert got == want, touch
    idx.close()


# ------------------------------------------------------------------------------------------------ events
def _stream(rnd, n, base):
    events, known, nxt = [], [], base
    for _ in range(n):
        r = rnd.random()
        if r < 0.6 or not known:
            nb = rnd.randrange(1, 4)
            hashes = list(range(nxt, nxt + nb))
            nxt += nb
            events.append(("S", dict(block_hashes=hashes, tokens=[rnd.randrange(30000) for _ in range(16 * nb + rnd.randrange(5))],
                                     parent_hash=rnd.choice(known) if known and rnd.random() < 0.5 else 0,
                                     device_tier=rnd.choice(["", "GPU", "cpu"]))))
            known.extend(hashes)
        elif r < 0.85:
            events.append(("R", dict(block_hashes=[rnd.choice(known)], device_tier=rnd.choice(["", "GPU", "cpu"]))))
        else:
            events.append(("C", dict(device_tier=rnd.choice(["", "GPU", "cpu"]))))
    return events


def _mk(kind, kw, E, oracle):
    if kind == "S":
        return (eo.BlockStored if oracle else E.BlockStoredEvent)(**kw)
    if kind == "R":
        return (eo.BlockRemoved if oracle else E.BlockRemovedEvent)(**kw)
    return (eo.AllBlocksCleared if oracle else E.AllBlocksClearedEvent)(**kw)


def _assert_same_index(idx, oidx):
    assert len(idx) == len(oidx.data)
    for rk, inner in oidx.data.d.items():
        got = idx.host_peek(rk)
        assert [(g.pod_identifier, g.device_tier, g.speculative) for g in got] == \
               [(p.pod_identifier, p.device_tier, p.speculative) for p in inner.keys()]


@pytest.mark.parametrize("clear", [True, False])
def test_all_blocks_cleared_in_event_streams(kvb, torch_cuda, clear):
    """AllBlocksCleared interleaved with BlockStored / BlockRemoved in 8 pods' streams.  clear_on_all_blocks_cleared:
    both the native ingest and process_many equal the oracle replayed in the native round order, with the pod's
    entries of the event's tier removed at the event.  Default: AllBlocksCleared changes nothing, as in the reference."""
    E, K = kvb.kvevents, kvb.kvblock
    rnd = random.Random(77)
    specs = [("pod-%d" % p, "m", _stream(rnd, 40, 100000 * (p + 1))) for p in range(8)]
    assert sum(k == "C" for _, _, s in specs for k, _ in s) > 10
    oidx, otp = o.InMemoryIndex(), o.TokenProcessor(16, "")
    pr.replay_native_rounds(oidx, otp, [(p, m, [_mk(k, kw, E, True) for k, kw in s]) for p, m, s in specs], clear)
    plain = o.InMemoryIndex()
    for p, m, s in specs:
        eo.process_event_batch(plain, otp, [_mk(k, kw, E, True) for k, kw in s], p, m)
    if clear:
        assert len(oidx.data) < len(plain.data)   # the streams' clears do remove something
    else:
        assert pr.as_tuples({k: v.keys() for k, v in oidx.data.d.items()}) == \
               pr.as_tuples({k: v.keys() for k, v in plain.data.d.items()})
    tp = K.ChunkedTokenDatabase(16, "")
    kwargs = {"clear_on_all_blocks_cleared": True} if clear else {}
    for native in (True, False):
        idx = K.Index()
        proc = E.EventProcessor(idx, tp, **kwargs)
        work = [(p, m, [_mk(k, kw, E, False) for k, kw in s]) for p, m, s in specs]
        if native:
            proc.process_many_native(work)
        else:
            proc.process_many(work)
        _assert_same_index(idx, oidx)
        idx.close()
    # the reference-shaped entry point, pod by pod
    idx = K.Index()
    proc = E.EventProcessor(idx, tp, **kwargs)
    want = o.InMemoryIndex()
    for p, m, s in specs:
        proc.process_event_batch([_mk(k, kw, E, False) for k, kw in s], p, m)
        pr.replay_native_rounds(want, otp, [(p, m, [_mk(k, kw, E, True) for k, kw in s])], clear)
    _assert_same_index(idx, want)
    idx.close()


def test_cpp_mirror_known_answer(kvb, torch_cuda, tmp_path):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    exe = str(tmp_path / "test_remove_pods")
    r = subprocess.run([cxx, "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "cpp", "test_remove_pods.cpp"), "-o", exe, "-L", PKG, "-lkvb",
                        "-Wl,-rpath," + PKG, "-lpthread"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.startswith("OK ")
