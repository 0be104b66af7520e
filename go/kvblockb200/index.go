package kvblockb200

/*
#include <stdlib.h>
#include "kvb.h"
*/
import "C"

import (
	"context"
	"fmt"
	"sync"
	"unsafe"

	"k8s.io/apimachinery/pkg/util/sets"

	"github.com/llm-d/llm-d-kv-cache/pkg/kvcache/kvblock"
)

// GPUIndexConfig slots into kvblock.IndexConfig next to InMemoryConfig (index.go:32-47); NewIndex gets one more
// `case cfg.GPUConfig != nil` (index.go:68-93).
type GPUIndexConfig struct {
	Size         int `json:"size"`         // InMemoryIndexConfig.Size
	PodCacheSize int `json:"podCacheSize"` // <= 13 (one 64 B device bucket)
	Device       int `json:"device"`
	ExpectedKeys int `json:"expectedKeys"`
}

// Index implements kvblock.Index over kvb_index_*.  Pod identifiers and device tiers are interned to the dense
// ids the C ABI carries; the table of names lives here, on the host side of the boundary.
type Index struct {
	h     *C.kvb_index_t
	mu    sync.Mutex
	pods  map[string]uint16
	podN  []string
	tiers map[string]uint8
	tierN []string
	w     map[string]float64 // LongestPrefixScorer.MediumWeights
}

var _ kvblock.Index = (*Index)(nil)

func NewIndex(cfg *GPUIndexConfig, mediumWeights map[string]float64) (*Index, error) {
	ix := &Index{pods: map[string]uint16{}, tiers: map[string]uint8{}, w: mediumWeights}
	if rc := C.kvb_index_create(C.int(cfg.Device), C.int64_t(cfg.Size), C.int32_t(cfg.PodCacheSize),
		C.int64_t(cfg.ExpectedKeys), &ix.h); rc != 0 {
		return nil, lastError(rc)
	}
	return ix, nil
}

func (ix *Index) Close() { C.kvb_index_destroy(ix.h) }

// The C ABI carries pods as uint16 and tiers as uint8: interning more than that would wrap and alias ids.
const (
	maxPods  = 1 << 16
	maxTiers = 1 << 8
)

func (ix *Index) entries(in []kvblock.PodEntry) ([]C.kvb_pod_entry_t, error) {
	out := make([]C.kvb_pod_entry_t, len(in))
	for i, e := range in {
		p, ok := ix.pods[e.PodIdentifier]
		if !ok {
			if len(ix.podN) >= maxPods {
				return nil, fmt.Errorf("too many distinct pod identifiers (limit %d)", maxPods)
			}
			p = uint16(len(ix.podN))
			ix.pods[e.PodIdentifier] = p
			ix.podN = append(ix.podN, e.PodIdentifier)
		}
		t, ok := ix.tiers[e.DeviceTier]
		if !ok {
			if len(ix.tierN) >= maxTiers {
				return nil, fmt.Errorf("too many distinct device tiers (limit %d)", maxTiers)
			}
			t = uint8(len(ix.tierN))
			ix.tiers[e.DeviceTier] = t
			ix.tierN = append(ix.tierN, e.DeviceTier)
			wt, known := ix.w[e.DeviceTier] // unknown tier scores 1.0 (kvblock_scorer.go:93-98)
			k := C.int(0)
			if known {
				k = 1
			}
			C.kvb_index_set_tier_weight(ix.h, C.uint8_t(t), C.double(wt), k)
		}
		out[i].pod, out[i].tier = C.uint16_t(p), C.uint8_t(t)
		if e.Speculative {
			out[i].speculative = 1
		}
	}
	return out, nil
}

func keysPtr(k []kvblock.BlockHash) *C.uint64_t {
	if len(k) == 0 {
		return nil
	}
	return (*C.uint64_t)(unsafe.Pointer(&k[0]))
}

// Add mirrors InMemoryIndex.Add (in_memory.go:154-224).
func (ix *Index) Add(_ context.Context, engineKeys, requestKeys []kvblock.BlockHash, entries []kvblock.PodEntry) error {
	if len(requestKeys) == 0 || len(entries) == 0 {
		return fmt.Errorf("no keys or entries provided for adding to index")
	}
	ix.mu.Lock()
	defer ix.mu.Unlock()
	e, err := ix.entries(entries)
	if err != nil {
		return err
	}
	has := C.int(0)
	if engineKeys != nil {
		has = 1
	}
	if rc := C.kvb_index_add(ix.h, keysPtr(engineKeys), C.int64_t(len(engineKeys)), has,
		keysPtr(requestKeys), C.int64_t(len(requestKeys)), &e[0], C.int32_t(len(e))); rc != 0 {
		return lastError(rc)
	}
	return nil
}

// Evict mirrors InMemoryIndex.Evict (in_memory.go:229-255).
func (ix *Index) Evict(_ context.Context, key kvblock.BlockHash, keyType kvblock.KeyType, entries []kvblock.PodEntry) error {
	if len(entries) == 0 {
		return fmt.Errorf("no entries provided for eviction from index")
	}
	ix.mu.Lock()
	defer ix.mu.Unlock()
	e, err := ix.entries(entries)
	if err != nil {
		return err
	}
	if rc := C.kvb_index_evict(ix.h, C.uint64_t(key), C.int(keyType), &e[0], C.int32_t(len(e))); rc != 0 {
		return lastError(rc)
	}
	return nil
}

// RemovePods removes every entry of the named pods (of the named tiers; none = every tier) from every key in one device
// sweep (kvb_index_remove_pods).  No reference counterpart: the reference ignores AllBlocksCleared (pool.go:388-395).
// Keys left empty are deleted, no key's recency changes, the engine-key map is untouched.  Names the index has never
// seen match nothing.  Returns (entries removed, keys deleted).
func (ix *Index) RemovePods(_ context.Context, pods []string, tiers []string) (int64, int64, error) {
	ix.mu.Lock()
	defer ix.mu.Unlock()
	var pids []C.uint16_t
	for _, name := range pods {
		if id, ok := ix.pods[name]; ok {
			pids = append(pids, C.uint16_t(id))
		}
	}
	var tids []C.uint8_t
	for _, name := range tiers {
		if id, ok := ix.tiers[name]; ok {
			tids = append(tids, C.uint8_t(id))
		}
	}
	if len(pids) == 0 || (len(tiers) > 0 && len(tids) == 0) {
		return 0, 0, nil
	}
	var tp *C.uint8_t
	if len(tids) > 0 {
		tp = &tids[0]
	}
	var removed, deleted C.int64_t
	if rc := C.kvb_index_remove_pods(ix.h, &pids[0], C.int32_t(len(pids)), tp, C.int32_t(len(tids)), &removed,
		&deleted); rc != 0 {
		return 0, 0, lastError(rc)
	}
	return int64(removed), int64(deleted), nil
}

// GetRequestKey mirrors in_memory.go:298-304.
func (ix *Index) GetRequestKey(_ context.Context, engineKey kvblock.BlockHash) (kvblock.BlockHash, error) {
	var out C.uint64_t
	if rc := C.kvb_index_get_request_key(ix.h, C.uint64_t(engineKey), &out); rc != 0 {
		return kvblock.EmptyBlockHash, fmt.Errorf("engine key not found: %s", engineKey.String())
	}
	return kvblock.BlockHash(out), nil
}

// Lookup mirrors in_memory.go:107-148 (device probe; the host only rebuilds the map).
func (ix *Index) Lookup(_ context.Context, requestKeys []kvblock.BlockHash, podSet sets.Set[string]) (map[kvblock.BlockHash][]kvblock.PodEntry, error) {
	if len(requestKeys) == 0 {
		return nil, fmt.Errorf("no requestKeys provided for lookup")
	}
	ix.mu.Lock()
	defer ix.mu.Unlock()
	var filter []C.uint16_t
	for name := range podSet {
		if id, ok := ix.pods[name]; ok {
			filter = append(filter, C.uint16_t(id))
		}
	}
	if podSet.Len() > 0 && len(filter) == 0 {
		return map[kvblock.BlockHash][]kvblock.PodEntry{}, nil // filter names nobody the index has seen
	}
	n := len(requestKeys)
	counts := make([]C.int32_t, n)
	ents := make([]C.kvb_pod_entry_t, n*C.KVB_INDEX_MAX_PODS_PER_KEY)
	var cut C.int64_t
	var fp *C.uint16_t
	if len(filter) > 0 {
		fp = &filter[0]
	}
	if rc := C.kvb_index_lookup(ix.h, keysPtr(requestKeys), C.int64_t(n), fp, C.int32_t(len(filter)),
		&counts[0], &ents[0], &cut); rc != 0 {
		return nil, lastError(rc)
	}
	out := make(map[kvblock.BlockHash][]kvblock.PodEntry)
	for i := 0; i < int(cut) && i < n; i++ {
		for e := 0; e < int(counts[i]); e++ {
			c := ents[i*C.KVB_INDEX_MAX_PODS_PER_KEY+e]
			pe := kvblock.PodEntry{PodIdentifier: ix.podN[c.pod], DeviceTier: ix.tierN[c.tier], Speculative: c.speculative != 0}
			if len(filter) > 0 {
				out[requestKeys[i]] = append(out[requestKeys[i]], pe) // filtered path appends (in_memory.go:131-137)
			} else if e == 0 {
				out[requestKeys[i]] = []kvblock.PodEntry{pe}
			} else {
				out[requestKeys[i]] = append(out[requestKeys[i]], pe)
			}
		}
	}
	return out, nil
}

// ScoreTokensBatch is the data-parallel form of Indexer.ScoreTokens (pkg/kvcache/indexer.go:239-304): tokens of
// many prompts in, per-prompt pod scores out, hashing + lookup + scoring fused on the device.
func (ix *Index) ScoreTokensBatch(tp *TokenProcessor, prompts [][]uint32, model string, podIdentifiers []string) ([]map[string]float64, error) {
	init, err := tp.getInitHash(model)
	if err != nil {
		return nil, err
	}
	n := len(prompts)
	off := make([]int64, n+1)
	for i, p := range prompts {
		off[i+1] = off[i] + int64(len(p))
	}
	flat := make([]uint32, off[n])
	parents := make([]uint64, n)
	for i, p := range prompts {
		copy(flat[off[i]:], p)
		parents[i] = init
	}
	ix.mu.Lock()
	defer ix.mu.Unlock()
	var filter []C.uint16_t
	for _, name := range podIdentifiers {
		if id, ok := ix.pods[name]; ok {
			filter = append(filter, C.uint16_t(id))
		}
	}
	if len(podIdentifiers) > 0 && len(filter) == 0 {
		// A filter that names only pods the index has never seen matches nothing: Lookup builds
		// sets.New(podIdentifiers...) and finds no entry in it (in_memory.go:131-137).  Passing n_filter = 0 here would
		// mean "no filter" to the C ABI and score every pod.
		res := make([]map[string]float64, n)
		for i := range res {
			if len(prompts[i])/tp.BlockSize() > 0 {
				res[i] = map[string]float64{}
			}
		}
		return res, nil
	}
	var fp *C.uint16_t
	if len(filter) > 0 {
		fp = &filter[0]
	}
	const m = C.KVB_INDEX_MAX_PODS_PER_KEY
	outN := make([]C.int32_t, n)
	outP := make([]C.uint16_t, n*m)
	outS := make([]C.double, n*m)
	var tokp *C.uint32_t
	if len(flat) > 0 {
		tokp = (*C.uint32_t)(unsafe.Pointer(&flat[0]))
	}
	if rc := C.kvb_index_score_tokens_batch(ix.h, tokp, (*C.int64_t)(unsafe.Pointer(&off[0])),
		(*C.uint64_t)(unsafe.Pointer(&parents[0])), C.int32_t(n), C.int32_t(tp.BlockSize()), nil, nil,
		fp, C.int32_t(len(filter)), 0 /* recency refreshed by default */, &outN[0], &outP[0], &outS[0]); rc != 0 {
		return nil, lastError(rc)
	}
	res := make([]map[string]float64, n)
	for i := range res {
		if len(prompts[i])/tp.BlockSize() == 0 {
			continue // "nil, nil" (indexer.go:266-270)
		}
		res[i] = make(map[string]float64, int(outN[i]))
		for j := 0; j < int(outN[i]); j++ {
			res[i][ix.podN[outP[i*m+j]]] = float64(outS[i*m+j])
		}
	}
	return res, nil
}
