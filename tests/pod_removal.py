"""Pod removal (kvb_index_remove_pods / Index.remove_pods): the oracle's restatement of the operation and the scenarios
that drive both the host-simulation build (tests/test_index_remove_pods_sim.py) and libkvb.so
(tests/test_gpu_index_remove_pods.py) against it.

The reference has no such operation (pool.go:388-395 ignores AllBlocksCleared), so its semantics are written down here:
every entry whose pod is in `pods` (and whose tier is in `tiers`, if given; the speculative bit is ignored) leaves every
key; surviving entries keep their inner-LRU order; a key left empty is deleted (evictPodsFromRequestKey,
in_memory.go:281-292); no key's recency moves; the engine-key map is untouched."""
from __future__ import annotations

import numpy as np

from oracle import kvblock_oracle as o
from oracle import kvevents_oracle as eo


def remove_pods(index: o.InMemoryIndex, pods, tiers=None):
    """Oracle of Index.remove_pods on an oracle InMemoryIndex.  Walks the LRU's dicts directly (no `get`), so no
    recency moves.  Returns (entries_removed, keys_deleted)."""
    pods = set(pods)
    tiers = None if tiers is None else set(tiers)
    removed = deleted = 0
    for rk in list(index.data.d.keys()):
        inner = index.data.d[rk]
        for e in list(inner.d.keys()):
            if e.pod_identifier in pods and (tiers is None or e.device_tier in tiers):
                del inner.d[e]
                removed += 1
        if len(inner) == 0:
            del index.data.d[rk]
            deleted += 1
    return removed, deleted


def as_tuples(d):
    return {int(k): [(e.pod_identifier, e.device_tier, bool(e.speculative)) for e in v] for k, v in d.items()}


def state(idx, oidx, keys):
    """(device lookup, oracle lookup) of `keys`, without moving the oracle's recency when the caller does not want to:
    use for final-state checks only (both sides are read the same way, so both move alike)."""
    return as_tuples(idx.lookup(keys)), as_tuples(oidx.lookup(keys))


# ------------------------------------------------------------------------------------------------ scenarios
def known_answer(K, lib):
    idx = K.Index(size=1000, pod_cache_size=4, expected_keys=16, lib=lib)
    p0g, p1g, p0c, p1c = (K.PodEntry("p0", "gpu"), K.PodEntry("p1", "gpu"), K.PodEntry("p0", "cpu"),
                          K.PodEntry("p1", "cpu"))
    idx.add(None, [11], [p0g, p1g, p0c])
    idx.add(None, [22], [p0g])
    idx.add(None, [33], [p1c])
    assert idx.remove_pods(["p0"]) == (3, 1)
    assert idx.lookup([11, 22, 33]) == {11: [p1g], 33: [p1c]}
    assert len(idx) == 2
    assert idx.remove_pods(["p1"], ["cpu"]) == (1, 1)
    assert idx.lookup([11, 22, 33]) == {11: [p1g]}
    n_pods = len(idx.pods.names)
    assert idx.remove_pods(["never-seen"]) == (0, 0)
    assert idx.remove_pods(["p1"], ["never-seen-tier"]) == (0, 0)
    assert idx.remove_pods([]) == (0, 0)
    assert len(idx.pods.names) == n_pods and "never-seen" not in idx.pods.ids   # unknown names are not interned
    assert idx.lookup([11, 22, 33]) == {11: [p1g]}
    # speculative entries of the pod go too; the engine-key map keeps the deleted key's mapping
    idx.add([900, 901], [44, 55], [K.PodEntry("p2", "gpu", True)])
    idx.add(None, [44], [p1g])
    assert idx.remove_pods(["p2"]) == (2, 1)
    assert idx.lookup([44, 55]) == {44: [p1g]}
    assert idx.get_request_key(901) == 55
    st = idx.stats()
    assert st["live_keys"] == 2 and st["tombstones"] >= 3
    idx.close()


def queue_ordering(K, lib):
    """Adds and evicts queued before the call are applied first; adds queued after it land after it."""
    idx = K.Index(size=1000, pod_cache_size=4, expected_keys=16, lib=lib)
    oidx = o.InMemoryIndex(size=1000, pod_cache_size=4)
    ops = [
        ("add", [1, 2, 3], [("a", "gpu"), ("b", "gpu")]),
        ("evict", 2, [("b", "gpu")]),
        ("add", [4], [("a", "cpu")]),
        ("purge", ["a"], None),
        ("add", [1, 5], [("a", "gpu")]),
        ("purge", ["b"], ["gpu"]),
        ("add", [3], [("b", "gpu"), ("c", "cpu")]),
    ]
    for op, x, y in ops:   # nothing in between reads the index: every purge meets a queue of unapplied ops
        if op == "add":
            idx.add(None, x, [K.PodEntry(*e) for e in y])
            oidx.add(None, x, [o.PodEntry(*e) for e in y])
        elif op == "evict":
            idx.evict(x, K.REQUEST_KEY, [K.PodEntry(*e) for e in y])
            oidx.evict(x, o.REQUEST_KEY, [o.PodEntry(*e) for e in y])
        else:
            assert idx.remove_pods(x, y) == remove_pods(oidx, x, y)
    got, want = state(idx, oidx, [1, 2, 3, 4, 5])
    assert got == want == {1: [("a", "gpu", False)], 3: [("b", "gpu", False), ("c", "cpu", False)],
                           5: [("a", "gpu", False)]}
    idx.close()


def recency_untouched(K, lib):
    """Size 300: fill, shuffle recency with lookups, purge, refill past capacity.  Which keys the outer LRU drops
    depends on the stamps the survivors kept: a sweep that re-stamped them would evict different keys."""
    rng = np.random.default_rng(3)
    idx = K.Index(size=300, pod_cache_size=4, expected_keys=16, lib=lib)
    oidx = o.InMemoryIndex(size=300, pod_cache_size=4)
    pods = ["p%d" % i for i in range(6)]
    for k in range(1, 301):
        ents = [(pods[int(i)], "gpu") for i in rng.choice(6, int(rng.integers(1, 3)), replace=False)]
        idx.add(None, [k], [K.PodEntry(*e) for e in ents])
        oidx.add(None, [k], [o.PodEntry(*e) for e in ents])
    for _ in range(20):
        ks = [int(x) for x in rng.integers(1, 301, 10)]
        assert as_tuples(idx.lookup(ks)) == as_tuples(oidx.lookup(ks))
    r = idx.remove_pods(["p0", "p1"])
    assert r == remove_pods(oidx, ["p0", "p1"]) and r[1] > 50
    assert len(idx) == len(oidx.data)
    new = list(range(1000, 1000 + r[1] + 60))   # refills the freed room, then 60 old keys must go: the 60 oldest
    for i in range(0, len(new), 4):              # small batches: the one-thread replay at capacity
        idx.add(None, new[i:i + 4], [K.PodEntry("new", "cpu")])
        oidx.add(None, new[i:i + 4], [o.PodEntry("new", "cpu")])
    got, want = state(idx, oidx, list(range(1, 301)) + new)
    assert got == want and len(idx) == len(oidx.data) == 300
    idx.close()


def purge_at_capacity_then_adds(K, lib, batch):
    """At capacity, a purge deletes about half of the keys; add-only batches refill the index past `Size` again.
    Exact LRU against the oracle, and the eviction plan (large batches) never falls back."""
    rng = np.random.default_rng(batch)
    size = 1500
    idx = K.Index(size=size, pod_cache_size=3, expected_keys=16, lib=lib)
    oidx = o.InMemoryIndex(size=size, pod_cache_size=3)
    nxt = 1
    for _ in range(4):   # 2000 keys into a 1500-key index: at capacity
        ks = list(range(nxt, nxt + 500))
        nxt += 500
        pod = "half-%d" % int(rng.integers(0, 2))
        idx.add(None, ks, [K.PodEntry(pod, "gpu")])
        oidx.add(None, ks, [o.PodEntry(pod, "gpu")])
    ks = [int(x) for x in rng.integers(1, nxt, 300)]
    assert as_tuples(idx.lookup(ks)) == as_tuples(oidx.lookup(ks))
    r = idx.remove_pods(["half-0"])
    assert r == remove_pods(oidx, ["half-0"]) and r[1] > 300, r
    while nxt < 6000:
        n = int(rng.integers(max(1, batch // 2), batch + 1))
        ks = [int(x) for x in rng.integers(1, nxt + n, n)]   # new keys and re-announced old ones
        nxt += n
        idx.add(None, ks, [K.PodEntry("re", "cpu")])
        oidx.add(None, ks, [o.PodEntry("re", "cpu")])
        if rng.random() < 0.2:
            ks = [int(x) for x in rng.integers(1, nxt, 50)]
            assert as_tuples(idx.lookup(ks)) == as_tuples(oidx.lookup(ks))
    got, want = state(idx, oidx, list(range(1, nxt + 1)))
    assert got == want and len(idx) == len(oidx.data) == size
    st = idx.stats()
    idx.close()
    assert st["plan_fallbacks"] == 0, st
    return st


def random_traffic(K, lib, seed, size, ppk, n_keys, steps, max_batch, expected_keys=16):
    """Add / Evict / Lookup / remove_pods at random; every lookup, len, the engine-key map and the final state against
    the oracle."""
    rng = np.random.default_rng(seed)
    idx = K.Index(size=size, pod_cache_size=ppk, expected_keys=expected_keys, lib=lib)
    oidx = o.InMemoryIndex(size=size, pod_cache_size=ppk)
    pods = ["pod-%d" % i for i in range(12)]
    tiers = ["gpu", "cpu", "GPU", "disk"]
    keyspace = [int(x) for x in rng.integers(1, 1 << 63, n_keys)]
    purged = 0
    for step in range(steps):
        op = rng.random()
        if op < 0.5:
            n = int(rng.integers(1, max_batch + 1))
            rks = [keyspace[int(i)] for i in rng.integers(0, len(keyspace), n)]
            eks = None if rng.random() < 0.3 else [int(x) for x in rng.integers(1, 400, n)]
            ents = [(pods[int(rng.integers(0, 12))], tiers[int(rng.integers(0, 4))], bool(rng.integers(0, 2)))
                    for _ in range(int(rng.integers(1, 4)))]
            idx.add(eks, rks, [K.PodEntry(*e) for e in ents])
            oidx.add(eks, rks, [o.PodEntry(*e) for e in ents])
        elif op < 0.65:
            ents = [(pods[int(rng.integers(0, 12))], tiers[int(rng.integers(0, 4))], bool(rng.integers(0, 2)))
                    for _ in range(int(rng.integers(1, 3)))]
            if rng.random() < 0.5:
                k, kt = int(rng.integers(1, 400)), 0
            else:
                k, kt = keyspace[int(rng.integers(0, len(keyspace)))], 1
            idx.evict(k, kt, [K.PodEntry(*e) for e in ents])
            oidx.evict(k, kt, [o.PodEntry(*e) for e in ents])
        elif op < 0.72:
            ps = [pods[int(i)] for i in rng.integers(0, 12, int(rng.integers(1, 3)))] + ["unknown-pod"]
            ts = None if rng.random() < 0.5 else [tiers[int(i)] for i in rng.integers(0, 4, int(rng.integers(1, 3)))]
            r = idx.remove_pods(ps, ts)
            assert r == remove_pods(oidx, ps, ts), step
            purged += r[0]
        else:
            ks = [keyspace[int(i)] for i in rng.integers(0, len(keyspace), int(rng.integers(1, 40)))]
            flt = [] if rng.random() < 0.5 else [pods[int(i)] for i in rng.integers(0, 12, 3)]
            assert as_tuples(idx.lookup(ks, flt)) == as_tuples(oidx.lookup(ks, flt)), step
        if step % 53 == 0:
            assert len(idx) == len(oidx.data), step
            for ek in range(1, 400, 13):   # engine keys of deleted request keys still resolve
                try:
                    want = oidx.get_request_key(ek)
                except KeyError:
                    try:
                        idx.get_request_key(ek)
                    except KeyError:
                        continue
                    raise AssertionError("engine key %d resolves on the device only" % ek)
                assert idx.get_request_key(ek) == want, (step, ek)
    got, want = state(idx, oidx, keyspace)
    assert got == want
    st = idx.stats()
    idx.close()
    assert purged > 0
    return st


# ------------------------------------------------------------------------------------------------ events
def replay_native_rounds(oidx, otp, work, clear: bool):
    """The oracle replayed in kvb_index_ingest_events' order: round r holds the r-th event of every stream; a round's
    BlockRemoved / AllBlocksCleared events go first, in stream order, then its BlockStored events.  AllBlocksCleared
    removes the pod's entries of the event's tier when `clear`, else it is ignored (pool.go:388-395)."""
    n_rounds = max((len(evs) for _, _, evs in work), default=0)
    for r in range(n_rounds):
        stored = []
        for pod, model, evs in work:
            if r >= len(evs):
                continue
            ev = evs[r]
            if isinstance(ev, eo.BlockStored):
                stored.append((pod, model, ev))
            elif isinstance(ev, eo.AllBlocksCleared):
                if clear:
                    remove_pods(oidx, [pod], [ev.device_tier.lower() if ev.device_tier else eo.DEFAULT_TIER])
            else:
                eo.process_event_batch(oidx, otp, [ev], pod, model)
        for pod, model, ev in stored:
            eo.process_event_batch(oidx, otp, [ev], pod, model)
