"""kvevents — the writer side of the index (SURVEY §8f rank 1): vLLM KV-cache events -> Index.Add / Evict.

Mirror of pkg/kvevents (pool.go:253-398 processEventBatch, :206-249 realignExtraFeatures) and of the vLLM adapter
(engineadapter/vllm_adapter.go:64-260, common.go:34-130).  Transport (ZMQ subscribe, pod discovery) stays out of
scope: callers hand in (topic, payload) pairs or decoded events.

B200-first addition: `EventProcessor.process_many` takes the pending batches of MANY pods and hashes one BlockStored
event per pod per round in a single device call (events of one pod stay in order, pods are independent — the
reference runs them on parallel worker shards, pool.go:154-166)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Sequence

import msgpack
import numpy as np

from . import kvblock as K

DEFAULT_EVENT_SOURCE_DEVICE_TIER = "GPU"  # pool.go:32


@dataclass
class BlockStoredEvent:  # events.go:71-79
    block_hashes: list
    tokens: list
    parent_hash: int = 0
    device_tier: str = ""
    lora_id: Optional[int] = None
    lora_name: Optional[str] = None
    extra_keys: Optional[list] = None


@dataclass
class BlockRemovedEvent:  # events.go:87-90
    block_hashes: list
    device_tier: str = ""


@dataclass
class AllBlocksClearedEvent:  # events.go:98-100
    device_tier: str = ""


@dataclass
class EventBatch:  # events.go:37-40
    timestamp: float
    events: list


# ------------------------------------------------------------------------------------------ vLLM adapter
def _hash_u64(raw) -> int:
    """getHashAsUint64 (common.go:50-71)."""
    if isinstance(raw, int) and not isinstance(raw, bool):
        return raw % (1 << 64)
    if isinstance(raw, (bytes, bytearray)):
        if not raw:
            raise ValueError("hash byte slice is empty")
        return int.from_bytes(bytes(raw)[-8:], "big")
    raise ValueError(f"unsupported hash type: {type(raw).__name__}")


def _opt(fields, i):
    return fields[i] if len(fields) > i else None


def _opt_str(fields, i, what):
    v = _opt(fields, i)
    if v is not None and not isinstance(v, str):
        raise ValueError(f"{what} is not a string: {type(v).__name__}")
    return v


class VLLMAdapter:
    """EngineAdapter for vLLM's msgspec array-encoded events (vllm_adapter.go)."""

    @staticmethod
    def parse_topic(topic: str):
        parts = topic.split("@")  # "kv@<pod-id>@<model>" (common.go:34-45)
        return (parts[1], parts[2]) if len(parts) == 3 else (topic, "")

    def sharding_key(self, topic: str) -> str:
        return self.parse_topic(topic)[0]

    def decode_event(self, fields: Sequence):
        if len(fields) < 1:
            raise ValueError("malformed tagged union: no tag")
        tag = fields[0]
        if not isinstance(tag, str):
            raise ValueError(f"event tag is not a string: {type(tag).__name__}")
        if tag == "BlockStored":  # [tag, block_hashes, parent_hash, token_ids, block_size, lora_id?, medium?, lora_name?, extra_keys?]
            if len(fields) < 5:
                raise ValueError(f"BlockStored: need at least 5 fields, got {len(fields)}")
            if not isinstance(fields[1], (list, tuple)):
                raise ValueError("BlockStored: block_hashes is not an array")
            if not isinstance(fields[3], (list, tuple)):
                raise ValueError("token_ids is not an array")
            extra = _opt(fields, 8)
            if extra is not None:
                if not isinstance(extra, (list, tuple)):
                    raise ValueError("BlockStored: extra_keys is not an array")
                for i, k in enumerate(extra):
                    if k is not None and not isinstance(k, (list, tuple)):
                        raise ValueError(f"extra_keys[{i}] has invalid type {type(k).__name__}, expected []any or nil")
                extra = [None if k is None else list(k) for k in extra]
            return BlockStoredEvent(
                block_hashes=[_hash_u64(h) for h in fields[1]],
                tokens=[int(t) % (1 << 32) for t in fields[3]],
                parent_hash=0 if fields[2] is None else _hash_u64(fields[2]),
                device_tier=_opt_str(fields, 6, "BlockStored: medium") or "",
                lora_id=_opt(fields, 5), lora_name=_opt_str(fields, 7, "BlockStored: lora_name"), extra_keys=extra)
        if tag == "BlockRemoved":  # [tag, block_hashes, medium?]
            if len(fields) < 2:
                raise ValueError(f"BlockRemoved: need at least 2 fields, got {len(fields)}")
            if not isinstance(fields[1], (list, tuple)):
                raise ValueError("BlockRemoved: block_hashes is not an array")
            return BlockRemovedEvent([_hash_u64(h) for h in fields[1]], _opt_str(fields, 2, "BlockRemoved: medium") or "")
        if tag == "AllBlocksCleared":
            m = _opt(fields, 1)
            return AllBlocksClearedEvent(m if isinstance(m, str) else "")
        raise ValueError(f"unknown vLLM event tag: {tag}")

    def parse_message(self, topic: str, payload: bytes):
        """ParseMessage (vllm_adapter.go:64-88) -> (pod_id, model_name, EventBatch)."""
        pod, model = self.parse_topic(topic)
        try:
            raw = msgpack.unpackb(payload, raw=False, strict_map_key=False)
        except Exception as e:
            raise ValueError(f"failed to decode vLLM event batch: {e}") from e
        if not isinstance(raw, (list, tuple)) or len(raw) < 2 or not isinstance(raw[1], (list, tuple)):
            raise ValueError("failed to decode vLLM event batch: not [ts, events, ...]")
        return pod, model, EventBatch(float(raw[0]), [self.decode_event(list(e)) for e in raw[1]])


class SGLangAdapter(VLLMAdapter):
    """SGLang publishes the same positional msgpack encoding and may omit trailing optional fields
    (engineadapter/sglang_adapter.go:40-239, padFields); the decoder above already treats absent trailing fields as nil."""


# ------------------------------------------------------------------------------------------ event processing
def realign_extra_features(engine_features, canonical_block_count: int):
    """Per-engine-block features -> per-canonical-block (pool.go:206-249): replicate when the engine block is
    larger, merge (concatenate identifiers) when it is smaller."""
    n = len(engine_features)
    if n == canonical_block_count:
        return engine_features
    if n == 0 or canonical_block_count == 0:
        # the Go code indexes an empty slice here (panic); no canonical block can come out of it either way
        return [None] * canonical_block_count
    if n < canonical_block_count:
        return [engine_features[i * n // canonical_block_count] for i in range(canonical_block_count)]
    merged = [None] * canonical_block_count
    for i, ef in enumerate(engine_features):
        if ef is None:
            continue
        slot = i * canonical_block_count // n
        if merged[slot] is None:
            merged[slot] = K.BlockExtraFeatures(None)  # Go: &BlockExtraFeatures{} — MMHashes is a nil slice ...
        if ef.mm_hashes:  # ... and append(nil, <nothing>...) stays nil, which CBOR-encodes as null (f6), not as [] (80)
            merged[slot].mm_hashes = (merged[slot].mm_hashes or []) + list(ef.mm_hashes)
    return merged


class EventProcessor:
    """Pool.processEventBatch (pool.go:253-398) over a kvblock.Index and a ChunkedTokenDatabase."""

    def __init__(self, index: K.Index, token_processor: K.ChunkedTokenDatabase, clear_on_all_blocks_cleared: bool = False):
        self.index = index
        self.token_processor = token_processor
        self.skipped = 0  # events the reference would log-and-continue on
        # AllBlocksCleared: the reference only logs it (pool.go:388-395), so a pod that reset its prefix cache keeps
        # attracting requests until the outer LRU pushes its entries out.  True: remove the pod's entries of the event's
        # tier from the whole index (Index.remove_pods).
        self.clear_on_all_blocks_cleared = bool(clear_on_all_blocks_cleared)

    # -- helpers -----------------------------------------------------------------------------------------------
    @staticmethod
    def _tier(ev) -> str:
        return ev.device_tier.lower() if ev.device_tier else DEFAULT_EVENT_SOURCE_DEVICE_TIER  # pool.go:265-268

    def _prepare_stored(self, ev: BlockStoredEvent, model: str):
        """Everything before the hash: effective model, parent request key, realigned features.
        Returns None when the reference would `continue`."""
        eff_model = ev.lora_name if ev.lora_name else model  # pool.go:271-274
        parent_rk = K.EMPTY_BLOCK_HASH
        if ev.parent_hash != 0:
            try:
                parent_rk = self.index.get_request_key(ev.parent_hash)  # pool.go:284-294
            except KeyError:
                return None
        feats = K.parse_raw_extra_keys(ev.extra_keys) if ev.extra_keys is not None else None  # pool.go:296-305
        nblk = len(ev.tokens) // self.token_processor.block_size()
        if feats is not None and len(feats) != nblk:
            feats = realign_extra_features(feats, nblk)  # pool.go:310-315
        if nblk == 0:
            return None  # "no request keys produced, skipping" (pool.go:350-355)
        return eff_model, parent_rk, feats

    def _apply_stored(self, ev, pod, request_keys):
        if len(ev.block_hashes) == 0 or len(request_keys) == 0:
            self.skipped += 1
            return
        self.index.add(list(ev.block_hashes), [int(k) for k in request_keys],
                       [K.PodEntry(pod, self._tier(ev))])  # pool.go:360

    def _apply_removed(self, ev, pod):
        entries = [K.PodEntry(pod, self._tier(ev))]
        for h in ev.block_hashes:  # pool.go:379-386
            self.index.evict(int(h), K.ENGINE_KEY, entries)

    def _apply_cleared(self, ev, pod):
        if self.clear_on_all_blocks_cleared:
            self.index.remove_pods([pod], [self._tier(ev)])

    # -- reference-shaped entry point -------------------------------------------------------------------------
    def process_event_batch(self, batch, pod_identifier: str, model_name: str) -> None:
        events = batch.events if isinstance(batch, EventBatch) else batch
        for ev in events:
            if isinstance(ev, BlockStoredEvent):
                prep = self._prepare_stored(ev, model_name)
                if prep is None:
                    self.skipped += 1
                    continue
                eff_model, parent_rk, feats = prep
                keys = self.token_processor.tokens_to_kv_block_keys(parent_rk, ev.tokens, eff_model, feats)
                self._apply_stored(ev, pod_identifier, keys or [])
            elif isinstance(ev, BlockRemovedEvent):
                self._apply_removed(ev, pod_identifier)
            elif isinstance(ev, AllBlocksClearedEvent):
                self._apply_cleared(ev, pod_identifier)  # by default log only, as the reference (pool.go:388-395)

    def process_raw_message(self, adapter: VLLMAdapter, topic: str, payload: bytes) -> None:
        """Pool.processRawMessage (pool.go:196-204): parse failures are logged and dropped."""
        try:
            pod, model, batch = adapter.parse_message(topic, payload)
        except ValueError:
            self.skipped += 1
            return
        self.process_event_batch(batch, pod, model)

    # -- native form: one library call per batch ----------------------------------------------------------------
    def process_many_native(self, work: Sequence) -> int:
        """work: [(pod_identifier, model_name, events)] like ``process_many``, applied by ``kvb_index_ingest_events``:
        parent lookups, hashing (one device launch per round of events), engine-key mapping and the index updates all
        happen inside the library; Python only flattens the batch.  Text-only events (an event with extra_keys makes the
        whole batch fall back to ``process_many``).  Returns the number of events the reference would log and skip."""
        if any(isinstance(ev, BlockStoredEvent) and ev.extra_keys is not None for _, _, evs in work for ev in evs):
            before = self.skipped
            self.process_many(work)
            return self.skipped - before
        batch = self.flatten_events(work)
        return self.ingest_flat(batch) if batch is not None else 0

    def flatten_events(self, work: Sequence):
        """The C-ABI form of a decoded batch: (kvb_kv_event_t[n], uint32 tokens, uint64 engine keys), or None if empty."""
        from . import _lib
        n = sum(len(evs) for _, _, evs in work)
        if n == 0:
            return None
        arr = (_lib.KvEvent * n)()
        tok_parts, ek_parts = [], []
        tok_off = ek_off = i = 0
        idx, tp = self.index, self.token_processor
        for stream, (pod, model, evs) in enumerate(work):
            for ev in evs:
                r = arr[i]
                i += 1
                r.stream = stream
                if isinstance(ev, BlockStoredEvent):
                    r.type = _lib.EVENT_BLOCK_STORED
                    toks = np.asarray(ev.tokens, dtype=np.uint32)
                    r.token_off, r.n_tokens = tok_off, toks.size
                    tok_parts.append(toks)
                    tok_off += toks.size
                    r.parent_engine_key = int(ev.parent_hash)
                    r.root_hash = tp.get_init_hash(ev.lora_name if ev.lora_name else model)  # pool.go:271-274
                elif isinstance(ev, BlockRemovedEvent):
                    r.type = _lib.EVENT_BLOCK_REMOVED
                elif isinstance(ev, AllBlocksClearedEvent) and self.clear_on_all_blocks_cleared:
                    r.type = _lib.EVENT_POD_CLEARED
                    r.entry.pod = idx.pods.get(pod)
                    r.entry.tier = idx._tier_id(self._tier(ev))
                    continue
                else:
                    r.type = _lib.EVENT_OTHER
                    continue
                eks = np.asarray(ev.block_hashes, dtype=np.uint64)
                r.engine_key_off, r.n_engine_keys = ek_off, eks.size
                ek_parts.append(eks)
                ek_off += eks.size
                r.entry.pod = idx.pods.get(pod)
                r.entry.tier = idx._tier_id(self._tier(ev))
                r.entry.speculative = 0
        tokens = np.concatenate(tok_parts) if tok_parts else np.zeros(1, np.uint32)
        eks = np.concatenate(ek_parts) if ek_parts else np.zeros(1, np.uint64)
        return arr, n, tokens, eks

    def ingest_flat(self, batch) -> int:
        """One kvb_index_ingest_events call on a flattened batch; returns the events the reference would skip."""
        import ctypes as C
        arr, n, tokens, eks = batch
        idx = self.index
        skipped = C.c_int32()
        idx._check(idx._lib.kvb_index_ingest_events(idx._h, C.addressof(arr), n, tokens.ctypes.data, eks.ctypes.data,
                                                     self.token_processor.block_size(), C.byref(skipped)))
        self.skipped += int(skipped.value)
        return int(skipped.value)

    # -- data-parallel form ------------------------------------------------------------------------------------
    def process_many(self, work: Sequence) -> None:
        """work: [(pod_identifier, model_name, events)], one entry per pod.  Per-pod order is kept; in every round
        the next BlockStored event of every pod is hashed in ONE device call."""
        cursors = [0] * len(work)
        while True:
            staged = []  # (work idx, event, model, parent, feats)
            progressed = False
            for w, (pod, model, events) in enumerate(work):
                # drain non-hashing events up to (and including) this pod's next BlockStored
                while cursors[w] < len(events):
                    ev = events[cursors[w]]
                    cursors[w] += 1
                    progressed = True
                    if isinstance(ev, BlockRemovedEvent):
                        self._apply_removed(ev, pod)
                        continue
                    if isinstance(ev, AllBlocksClearedEvent):
                        self._apply_cleared(ev, pod)
                        continue
                    if isinstance(ev, BlockStoredEvent):
                        prep = self._prepare_stored(ev, model)
                        if prep is None:
                            self.skipped += 1
                            continue
                        staged.append((w, ev, *prep))
                        break
            if staged:
                keys, off = self.token_processor.tokens_to_kv_block_keys_batch(
                    [s[1].tokens for s in staged], [s[2] for s in staged], [s[3] for s in staged],
                    [s[4] for s in staged] if any(s[4] is not None for s in staged) else None)
                for i, s in enumerate(staged):
                    self._apply_stored(s[1], work[s[0]][0], keys[off[i]:off[i + 1]])
            if not progressed:
                return
