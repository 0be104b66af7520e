"""kvblock — host-side mirror of the Go package pkg/kvcache/kvblock, computing on the GPU via libkvb.so.

    ChunkedTokenDatabase  <- chunkedTokenDatabase / TokenProcessor   (token_processor.go:55-205)
    BlockExtraFeatures, MMHash, PlaceholderRange, compute_block_extra_features, parse_raw_extra_keys
                          <- extra_keys.go:26-163  (host logic: per-block multimodal identifiers)
    Index                 <- kvblock.Index / InMemoryIndex           (index.go:120-149, in_memory.go)
    PodEntry, ENGINE_KEY, REQUEST_KEY, EMPTY_BLOCK_HASH              (index.go:152-183)
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass
from typing import Iterable, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import MAX_PODS_PER_KEY, PodEntryC, check

EMPTY_BLOCK_HASH = 0
ENGINE_KEY = _lib.KEY_ENGINE
REQUEST_KEY = _lib.KEY_REQUEST
DEFAULT_BLOCK_SIZE = 16  # token_processor.go:32


# ------------------------------------------------------------------------------------------ extra keys
@dataclass(frozen=True)
class MMHash:
    hash: str


@dataclass
class BlockExtraFeatures:
    mm_hashes: Optional[list] = None


@dataclass(frozen=True)
class PlaceholderRange:
    offset: int
    length: int


def parse_raw_extra_keys(raw):
    """[][]any from a BlockStored event -> per-block features (extra_keys.go:49-85): strings are
    identifiers, [hash, offset] pairs keep the hash, anything else is skipped; blocks left without an
    identifier stay None."""
    if raw is None:
        return None
    result = []
    for block_keys in raw:
        ids = []
        for entry in (block_keys or ()):
            if isinstance(entry, str):
                ids.append(MMHash(entry))
            elif isinstance(entry, (list, tuple)) and entry and isinstance(entry[0], str):
                ids.append(MMHash(entry[0]))
        result.append(BlockExtraFeatures(ids) if ids else None)
    return result


def compute_block_extra_features(mm_hashes, mm_placeholders, block_size: int, num_tokens: int):
    """Identifiers of the multimodal items overlapping each full block, ordered by item start
    (extra_keys.go:100-163)."""
    if not mm_hashes or block_size <= 0 or num_tokens <= 0:
        return None
    spans = []
    for modality, hashes in mm_hashes.items():
        ranges = (mm_placeholders or {}).get(modality)
        if ranges is None:
            continue
        spans.extend((r.offset, r.offset + r.length, h) for h, r in zip(hashes, ranges))
    if not spans:
        return None
    spans.sort(key=lambda s: s[0])
    out = []
    for b in range(num_tokens // block_size):
        lo, hi = b * block_size, (b + 1) * block_size
        ids = [MMHash(h) for (s, e, h) in spans if e > lo and s < hi]
        out.append(BlockExtraFeatures(ids) if ids else None)
    return out


def _cbor_head(major: int, n: int) -> bytes:
    if n < 24:
        return bytes([major | n])
    for code, width in ((24, 1), (25, 2), (26, 4), (27, 8)):
        if n < 1 << (8 * width):
            return bytes([major | code]) + n.to_bytes(width, "big")
    raise OverflowError(n)


def encode_extra(ef: Optional[BlockExtraFeatures]) -> bytes:
    """Trailing CBOR item of a block payload: nil -> f6; []MMHash -> array of {"Hash": text}
    (token_processor.go:146-148 passes extraFeatures[i].MMHashes; canonical CBOR of the struct)."""
    if ef is None or ef.mm_hashes is None:
        return b"\xf6"
    out = bytearray(_cbor_head(0x80, len(ef.mm_hashes)))
    for m in ef.mm_hashes:
        raw = m.hash.encode("utf-8")
        out += b"\xa1\x64Hash" + _cbor_head(0x60, len(raw)) + raw
    return bytes(out)


# ------------------------------------------------------------------------------------------ token processor
class ChunkedTokenDatabase:
    """TokenProcessor (token_processor.go:55-69) on the GPU."""

    def __init__(self, block_size: int = DEFAULT_BLOCK_SIZE, hash_seed: str = "", device: int = 0):
        if block_size <= 0:
            raise ValueError(f"blockSize must be greater than 0, got {block_size}")  # :86-88
        self._block_size = int(block_size)
        self.hash_seed = hash_seed
        self.device = int(device)
        seed = hash_seed.encode("utf-8")
        buf = C.create_string_buffer(seed, len(seed))
        self.init_hash = int(_lib.load().kvb_fnv64a(buf, len(seed)))  # :90-95
        self._init_cache: dict = {}

    def block_size(self) -> int:
        return self._block_size

    def get_init_hash(self, model_name: str) -> int:
        h = self._init_cache.get(model_name)
        if h is None:
            raw = model_name.encode("utf-8")
            out = C.c_uint64()
            check(_lib.load().kvb_init_hash(self.device, self.init_hash, raw, len(raw), C.byref(out)))
            h = self._init_cache[model_name] = int(out.value)
        return h

    # -- batch form: the data-parallel hot path ------------------------------------------------
    def prepare_batch(self, prompts: Sequence, model_names, parent_keys=None, extra_features=None):
        """Flatten a batch into the arrays the C ABI takes."""
        n = len(prompts)
        if isinstance(model_names, str):
            model_names = [model_names] * n
        lens = np.fromiter((len(p) for p in prompts), dtype=np.int64, count=n)
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        tokens = np.empty(int(off[-1]), dtype=np.uint32)
        for i, p in enumerate(prompts):
            tokens[off[i]:off[i + 1]] = np.asarray(p, dtype=np.uint32)
        parents = np.empty(n, dtype=np.uint64)
        for i in range(n):
            pk = 0 if parent_keys is None else int(parent_keys[i])
            parents[i] = np.uint64(pk if pk != EMPTY_BLOCK_HASH else self.get_init_hash(model_names[i]))  # :181-186
        nblk = lens // self._block_size
        extra = extra_off = None
        if extra_features is not None and any(ef is not None for ef in extra_features):
            chunks = []
            for i, efs in enumerate(extra_features):
                if efs is None:
                    chunks.extend([b""] * int(nblk[i]))
                    continue
                if len(efs) != int(nblk[i]):  # :195-198
                    raise ValueError(
                        f"extraFeatures length {len(efs)} does not match token chunk count {int(nblk[i])} "
                        f"(blockSize={self._block_size}, tokens={int(lens[i])})")
                chunks.extend(b"" if ef is None else encode_extra(ef) for ef in efs)
            extra_off = np.zeros(len(chunks) + 1, dtype=np.int64)
            np.cumsum([len(c) for c in chunks], out=extra_off[1:])
            extra = np.frombuffer(b"".join(chunks) or b"\0", dtype=np.uint8).copy()
        return tokens, off, parents, nblk, extra, extra_off

    def tokens_to_kv_block_keys_batch(self, prompts, model_names, parent_keys=None, extra_features=None, stream=0):
        """Keys of every prompt; returns (flat uint64 keys, int64 key offsets)."""
        tokens, off, parents, nblk, extra, extra_off = self.prepare_batch(prompts, model_names, parent_keys,
                                                                          extra_features)
        n = len(prompts)
        keys = np.empty(max(int(nblk.sum()), 1), dtype=np.uint64)
        key_off = np.zeros(n + 1, dtype=np.int64)
        check(_lib.load().kvb_hash_token_blocks(
            self.device, tokens.ctypes.data, off.ctypes.data, parents.ctypes.data, n, self._block_size,
            None if extra is None else extra.ctypes.data, None if extra_off is None else extra_off.ctypes.data,
            keys.ctypes.data, key_off.ctypes.data, stream))
        return keys[:int(key_off[-1])], key_off

    # -- reference signature -------------------------------------------------------------------
    def tokens_to_kv_block_keys(self, parent_key: int, tokens, model_name: str, extra_features=None):
        """TokensToKVBlockKeys (token_processor.go:177-205); None for "nil, nil" (no full block)."""
        if len(tokens) // self._block_size == 0:
            return None
        keys, _ = self.tokens_to_kv_block_keys_batch([tokens], [model_name], [parent_key],
                                                     None if extra_features is None else [extra_features])
        return [int(k) for k in keys]


# ------------------------------------------------------------------------------------------ index
@dataclass(frozen=True)
class PodEntry:
    """index.go:176-183."""

    pod_identifier: str
    device_tier: str
    speculative: bool = False


class _Interner:
    """name <-> dense id; safe to call from several threads (Index operations are, index.go:119)."""

    def __init__(self, limit: int, what: str):
        self.ids: dict = {}
        self.names: list = []
        self.limit, self.what = limit, what
        self._lock = threading.Lock()

    def get(self, name: str) -> int:
        i = self.ids.get(name)
        if i is None:
            with self._lock:
                i = self.ids.get(name)
                if i is None:
                    if len(self.names) >= self.limit:
                        raise OverflowError(f"too many distinct {self.what} (limit {self.limit})")
                    i = len(self.names)
                    self.names.append(name)
                    self.ids[name] = i
        return i


class Index:
    """kvblock.Index (index.go:120-149) with InMemoryIndex semantics (in_memory.go), reads on the GPU.

    Pod identifiers / device tiers are interned to the dense ids the C ABI carries."""

    def __init__(self, size: int = int(1e8), pod_cache_size: int = 10, device: int = 0, expected_keys: int = 0,
                 medium_weights: Optional[dict] = None, lib=None):
        self.device = int(device)
        self._lib = lib if lib is not None else _lib.load()  # tests hand in the host-simulation build of index.cu
        h = C.c_void_p()
        self._check(self._lib.kvb_index_create(self.device, int(size), int(pod_cache_size), int(expected_keys),
                                               C.byref(h)))
        self._h = h
        self.pods = _Interner(65536, "pod identifiers")
        self.tiers = _Interner(256, "device tiers")
        self._tier_lock = threading.Lock()
        self._weights: dict = {}
        self.set_medium_weights({"gpu": 1.0, "cpu": 0.8} if medium_weights is None else medium_weights)  # backend.go:26-31

    def _check(self, rc: int) -> int:
        if rc < 0:
            raise _lib.KvbError(rc, self._lib.kvb_last_error().decode("utf-8", "replace"))
        return rc

    def close(self):
        if getattr(self, "_h", None):
            self._lib.kvb_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- interning ------------------------------------------------------------------------------
    def set_medium_weights(self, weights: Optional[dict]):
        """LongestPrefixScorer.MediumWeights (kvblock_scorer.go:82-85): unknown tier -> 1.0."""
        with self._tier_lock:  # _tier_id registers new tiers under the same lock
            self._weights = dict(weights or {})
            for name, tid in list(self.tiers.ids.items()):
                self._push_weight(name, tid)

    def _push_weight(self, name: str, tid: int):
        known = name in self._weights
        self._check(self._lib.kvb_index_set_tier_weight(self._h, tid, float(self._weights.get(name, 1.0)), int(known)))

    def _tier_id(self, name: str) -> int:
        tid = self.tiers.ids.get(name)
        if tid is None:
            with self._tier_lock:
                tid = self.tiers.ids.get(name)
                if tid is None:
                    # register the weight BEFORE the id becomes visible to other threads
                    nxt = len(self.tiers.names)
                    known = name in self._weights
                    self._check(self._lib.kvb_index_set_tier_weight(self._h, nxt, float(self._weights.get(name, 1.0)), int(known)))
                    tid = self.tiers.get(name)
        return tid

    def _entries(self, entries: Sequence[PodEntry]):
        arr = (PodEntryC * max(len(entries), 1))()
        for i, e in enumerate(entries):
            arr[i].pod = self.pods.get(e.pod_identifier)
            arr[i].tier = self._tier_id(e.device_tier)
            arr[i].speculative = 1 if e.speculative else 0
        return arr

    def _filter(self, pod_identifiers: Optional[Iterable[str]]):
        """Dense ids of the pod filter; unknown identifiers cannot match anything.
        Returns (array or None, n).  n == 0 means "no filter" (sets.Len()==0, in_memory.go:128)."""
        names = list(dict.fromkeys(pod_identifiers or ()))
        if not names:
            return None, 0
        ids = [self.pods.ids[n] for n in names if n in self.pods.ids]
        if not ids:  # filter present but nothing known: use a never-assigned id so nothing matches
            ids = [self.pods.get("\0__kvb_no_such_pod__")]
        return np.asarray(ids, dtype=np.uint16), len(ids)

    def _entry_from_c(self, c) -> PodEntry:
        return PodEntry(self.pods.names[c.pod], self.tiers.names[c.tier], bool(c.speculative))

    # -- Index interface ------------------------------------------------------------------------
    def add(self, engine_keys: Optional[Sequence[int]], request_keys: Sequence[int], entries: Sequence[PodEntry]):
        if len(request_keys) == 0 or len(entries) == 0:
            raise ValueError("no keys or entries provided for adding to index")  # in_memory.go:155-157
        rk = np.asarray(request_keys, dtype=np.uint64)
        ek = None if engine_keys is None else np.asarray(engine_keys, dtype=np.uint64)
        self._check(self._lib.kvb_index_add(self._h, None if ek is None else ek.ctypes.data,
                                        0 if ek is None else ek.size, int(ek is not None), rk.ctypes.data, rk.size,
                                        self._entries(entries), len(entries)))

    def evict(self, key: int, key_type: int, entries: Sequence[PodEntry]):
        if len(entries) == 0:
            raise ValueError("no entries provided for eviction from index")  # in_memory.go:230-232
        if key_type not in (ENGINE_KEY, REQUEST_KEY):
            raise ValueError(f"unknown key type: {key_type}")
        self._check(self._lib.kvb_index_evict(self._h, int(key), int(key_type), self._entries(entries), len(entries)))

    def remove_pods(self, pod_identifiers: Iterable[str], device_tiers: Optional[Iterable[str]] = None):
        """Remove every entry of these pods (of these tiers; None = every tier) from every key, in one device sweep
        (kvb_index_remove_pods).  Keys left empty are deleted; no key's recency changes; the engine-key map is untouched.
        Names the index has never seen match nothing and are not interned.  Returns (entries_removed, keys_deleted)."""
        pods = [self.pods.ids[n] for n in dict.fromkeys(pod_identifiers) if n in self.pods.ids]
        tiers = None
        if device_tiers is not None:
            tiers = [self.tiers.ids[t] for t in dict.fromkeys(device_tiers) if t in self.tiers.ids]
            if not tiers:
                return 0, 0
        if not pods:
            return 0, 0
        p = np.asarray(pods, dtype=np.uint16)
        t = None if tiers is None else np.asarray(tiers, dtype=np.uint8)
        removed, deleted = C.c_int64(), C.c_int64()
        self._check(self._lib.kvb_index_remove_pods(self._h, p.ctypes.data, p.size, None if t is None else t.ctypes.data,
                                                    0 if t is None else t.size, C.byref(removed), C.byref(deleted)))
        return int(removed.value), int(deleted.value)

    def get_request_key(self, engine_key: int) -> int:
        out = C.c_uint64()
        rc = self._lib.kvb_index_get_request_key(self._h, int(engine_key), C.byref(out))
        if rc == -4:
            raise KeyError(f"engine key not found: {engine_key}")  # in_memory.go:299-302
        self._check(rc)
        return int(out.value)

    def lookup(self, request_keys: Sequence[int], pod_identifier_set: Optional[Iterable[str]] = None) -> dict:
        """Lookup (in_memory.go:107-148): {key: [PodEntry]} for the keys found before the cut."""
        if len(request_keys) == 0:
            raise ValueError("no requestKeys provided for lookup")
        keys = np.asarray(request_keys, dtype=np.uint64)
        filt, nf = self._filter(pod_identifier_set)
        counts = np.empty(keys.size, dtype=np.int32)
        ents = (PodEntryC * (keys.size * MAX_PODS_PER_KEY))()
        cut = C.c_int64()
        self._check(self._lib.kvb_index_lookup(self._h, keys.ctypes.data, keys.size,
                                           None if filt is None else filt.ctypes.data, nf, counts.ctypes.data,
                                           C.addressof(ents), C.byref(cut)))
        out: dict = {}
        for i in range(min(int(cut.value), keys.size)):
            c = int(counts[i])
            if c > 0:
                found = [self._entry_from_c(ents[i * MAX_PODS_PER_KEY + e]) for e in range(c)]
                k = int(keys[i])
                if nf and k in out:
                    out[k].extend(found)  # filtered path APPENDS per occurrence of a repeated key (in_memory.go:131-137)
                else:
                    out[k] = found        # unfiltered path assigns (in_memory.go:128-130)
        return out

    def __len__(self) -> int:
        return int(self._lib.kvb_index_num_keys(self._h))

    def stats(self) -> dict:
        """Counters of the device-resident index (kvb_index_get_stats): live keys, table slots, how many op batches went
        through the parallel / sequential apply kernels, LRU evictions, ..."""
        st = _lib.IndexStats()
        self._check(self._lib.kvb_index_get_stats(self._h, C.byref(st)))
        return {n: getattr(st, n) for n, _ in _lib.IndexStats._fields_}

    def flush(self) -> None:
        """Apply every queued Add / Evict on the device and wait for it."""
        self._check(self._lib.kvb_index_flush(self._h, None))

    def host_peek(self, request_key: int):
        ents = (PodEntryC * MAX_PODS_PER_KEY)()
        n = self._lib.kvb_index_host_peek(self._h, int(request_key), ents, MAX_PODS_PER_KEY)
        return None if n < 0 else [self._entry_from_c(ents[i]) for i in range(n)]

    # -- batched read path ----------------------------------------------------------------------
    def _unpack_scores(self, n_prompts, out_n, out_pods, out_scores):
        res = []
        for p in range(n_prompts):
            k = int(out_n[p])
            base = p * MAX_PODS_PER_KEY
            res.append({self.pods.names[int(out_pods[base + j])]: float(out_scores[base + j]) for j in range(k)})
        return res

    def score_keys_batch(self, keys: np.ndarray, key_off: np.ndarray, pod_identifiers=None, touch_lru: bool = True):
        """Lookup + LongestPrefixScorer.Score for many prompts (kvblock_scorer.go:106-154)."""
        n = len(key_off) - 1
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        key_off = np.ascontiguousarray(key_off, dtype=np.int64)
        filt, nf = self._filter(pod_identifiers)
        out_n = np.zeros(max(n, 1), dtype=np.int32)
        out_pods = np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.uint16)
        out_scores = np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.float64)
        self._check(self._lib.kvb_index_score_batch(
            self._h, keys.ctypes.data if keys.size else None, key_off.ctypes.data, n,
            None if filt is None else filt.ctypes.data, nf, 0 if touch_lru else _lib.SCORE_NO_TOUCH,
            out_n.ctypes.data, out_pods.ctypes.data, out_scores.ctypes.data))
        return self._unpack_scores(n, out_n, out_pods, out_scores)

    def score_tokens_flat(self, block_size: int, tokens: np.ndarray, prompt_off: np.ndarray, parents: np.ndarray,
                          pod_identifiers=None, touch_lru: bool = True, out=None, flags: int = 0):
        """Same fused call on pre-flattened arrays (uint32 tokens, int64 offsets, uint64 parents); returns the raw
        (n, pods, scores) arrays — the zero-copy form a host-language shim would use: token and output buffers from
        ``pool.PinnedBuffer`` are read and written by the kernel in place.  ``flags``: extra KVB_SCORE_* bits (A/B)."""
        n = len(prompt_off) - 1
        filt, nf = self._filter(pod_identifiers)
        if out is None:
            out = (np.zeros(max(n, 1), dtype=np.int32), np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.uint16),
                   np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.float64))
        self._check(self._lib.kvb_index_score_tokens_batch(
            self._h, tokens.ctypes.data, prompt_off.ctypes.data, parents.ctypes.data, n, int(block_size), None, None,
            None if filt is None else filt.ctypes.data, nf, (0 if touch_lru else _lib.SCORE_NO_TOUCH) | int(flags),
            out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data))
        return out

    def score_tokens_batch(self, tp: ChunkedTokenDatabase, prompts, model_names, pod_identifiers=None,
                           extra_features=None, touch_lru: bool = True, raw: bool = False):
        """Fused tokens -> keys -> lookup -> score on the device for a batch of prompts."""
        tokens, off, parents, nblk, extra, extra_off = tp.prepare_batch(prompts, model_names, None, extra_features)
        n = len(prompts)
        filt, nf = self._filter(pod_identifiers)
        out_n = np.zeros(max(n, 1), dtype=np.int32)
        out_pods = np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.uint16)
        out_scores = np.zeros(max(n, 1) * MAX_PODS_PER_KEY, dtype=np.float64)
        self._check(self._lib.kvb_index_score_tokens_batch(
            self._h, tokens.ctypes.data, off.ctypes.data, parents.ctypes.data, n, tp.block_size(),
            None if extra is None else extra.ctypes.data, None if extra_off is None else extra_off.ctypes.data,
            None if filt is None else filt.ctypes.data, nf, 0 if touch_lru else _lib.SCORE_NO_TOUCH,
            out_n.ctypes.data, out_pods.ctypes.data, out_scores.ctypes.data))
        if raw:
            return out_n, out_pods, out_scores, nblk
        return self._unpack_scores(n, out_n, out_pods, out_scores), nblk
