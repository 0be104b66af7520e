// kvb_kvblock.hpp — C++17 host-side mirror of the reference's Go interfaces over the C ABI (kvb.h).
//
// The reference's indexer is compiled Go code and the build image has no Go toolchain, so the host side above the
// C ABI is provided in C++ with the SAME names, argument meaning and error behaviour as the Go interfaces:
//
//   kvblock::TokenProcessor   pkg/kvcache/kvblock/token_processor.go:55-69   (TokensToKVBlockKeys, BlockSize)
//   kvblock::Index            pkg/kvcache/kvblock/index.go:120-149           (Lookup, Add, Evict, GetRequestKey; RemovePods)
//   kvblock::PodEntry, BlockHash, KeyType, BlockExtraFeatures, MMHash         index.go:152-183, extra_keys.go:26-34
//   kvcache::Indexer          pkg/kvcache/indexer.go:65-304                   (ScoreTokens, ComputeBlockKeysFromTokens)
//
// Go `error` returns become kvb::Error exceptions carrying the same message text; "nil, nil" becomes an empty
// optional / empty vector.  The cgo shim (go/kvblockb200) and the Python mirror (llm-d-kv-cache_b200/kvblock.py)
// issue the identical C calls.  Header-only; link with -lkvb.
#pragma once
#include <algorithm>
#include <cstdint>
#include <map>
#include <memory>
#include <mutex>
#include <optional>
#include <set>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "kvb.h"

namespace kvb {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
inline void check(int rc) {
  if (rc < 0) throw Error(rc, kvb_last_error());
}

namespace kvblock {

using BlockHash = uint64_t;                 // index.go:164
constexpr BlockHash EmptyBlockHash = 0;     // index.go:168
enum KeyType : int { EngineKey = KVB_KEY_ENGINE, RequestKey = KVB_KEY_REQUEST };  // index.go:152-161

struct PodEntry {  // index.go:176-183
  std::string PodIdentifier;
  std::string DeviceTier;
  bool Speculative = false;
  bool operator==(const PodEntry& o) const {
    return PodIdentifier == o.PodIdentifier && DeviceTier == o.DeviceTier && Speculative == o.Speculative;
  }
};

struct MMHash {  // extra_keys.go:26-28
  std::string Hash;
};
struct BlockExtraFeatures {  // extra_keys.go:32-34; a null pointer in a vector of these means a pure-text block
  std::vector<MMHash> MMHashes;
};
using ExtraFeatures = std::vector<std::shared_ptr<BlockExtraFeatures>>;

struct PlaceholderRange {  // extra_keys.go:38-41
  int Offset = 0;
  int Length = 0;
};

// ComputeBlockExtraFeatures (extra_keys.go:100-163): identifiers of the multimodal items overlapping each full block,
// ordered by item start; nullptr entries are pure-text blocks; an empty result means "nil" (text-only prompt).
inline ExtraFeatures ComputeBlockExtraFeatures(const std::map<std::string, std::vector<std::string>>& mmHashes,
                                               const std::map<std::string, std::vector<PlaceholderRange>>& mmPlaceholders,
                                               int blockSize, int numTokens) {
  ExtraFeatures result;
  if (mmHashes.empty() || blockSize <= 0 || numTokens <= 0) return result;
  struct Item {
    int start, end;
    const std::string* hash;
  };
  std::vector<Item> items;
  for (const auto& kv : mmHashes) {
    auto r = mmPlaceholders.find(kv.first);
    if (r == mmPlaceholders.end()) continue;
    const size_t n = std::min(kv.second.size(), r->second.size());
    for (size_t i = 0; i < n; ++i)
      items.push_back({r->second[i].Offset, r->second[i].Offset + r->second[i].Length, &kv.second[i]});
  }
  if (items.empty()) return result;
  std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.start < b.start; });
  const int nblk = numTokens / blockSize;
  result.resize((size_t)nblk);
  for (int b = 0; b < nblk; ++b) {
    const int lo = b * blockSize, hi = lo + blockSize;
    std::shared_ptr<BlockExtraFeatures> f;
    for (const auto& it : items) {
      if (it.end <= lo) continue;
      if (it.start >= hi) break;
      if (!f) f = std::make_shared<BlockExtraFeatures>();
      f->MMHashes.push_back(MMHash{*it.hash});
    }
    result[(size_t)b] = f;
  }
  return result;
}

struct TokenProcessorConfig {  // token_processor.go:35-43
  int BlockSize = 16;
  std::string HashSeed;
};

namespace detail {
inline void cbor_head(std::vector<uint8_t>& out, uint8_t major, uint64_t n) {
  if (n < 24) {
    out.push_back(major | (uint8_t)n);
  } else if (n < 0x100) {
    out.push_back(major | 24);
    out.push_back((uint8_t)n);
  } else if (n < 0x10000) {
    out.push_back(major | 25);
    out.push_back((uint8_t)(n >> 8));
    out.push_back((uint8_t)n);
  } else if (n < 0x100000000ull) {
    out.push_back(major | 26);
    for (int s = 24; s >= 0; s -= 8) out.push_back((uint8_t)(n >> s));
  } else {
    out.push_back(major | 27);
    for (int s = 56; s >= 0; s -= 8) out.push_back((uint8_t)(n >> s));
  }
}
// trailing CBOR item of one block: nil -> nothing (the kernel folds 0xf6); []MMHash -> array of {"Hash": text}
inline void encode_extra(std::vector<uint8_t>& out, const BlockExtraFeatures* f) {
  if (!f) return;
  cbor_head(out, 0x80, f->MMHashes.size());
  for (const auto& m : f->MMHashes) {
    const uint8_t key[] = {0xa1, 0x64, 'H', 'a', 's', 'h'};
    out.insert(out.end(), key, key + sizeof(key));
    cbor_head(out, 0x60, m.Hash.size());
    out.insert(out.end(), m.Hash.begin(), m.Hash.end());
  }
}
}  // namespace detail

// chunkedTokenDatabase (token_processor.go:72-205) computing on the GPU.
class TokenProcessor {
 public:
  explicit TokenProcessor(const TokenProcessorConfig& cfg = {}, int device = 0) : cfg_(cfg), device_(device) {
    if (cfg.BlockSize <= 0)  // token_processor.go:86-88
      throw Error(KVB_ERR_INVALID, "blockSize must be greater than 0, got " + std::to_string(cfg.BlockSize));
    seed_hash_ = kvb_fnv64a(cfg.HashSeed.data(), cfg.HashSeed.size());  // :90-95
  }
  int BlockSize() const { return cfg_.BlockSize; }
  int Device() const { return device_; }

  uint64_t InitHash(const std::string& model) {  // getInitHash (:109-111), cached
    std::lock_guard<std::mutex> lk(mu_);
    auto it = init_.find(model);
    if (it != init_.end()) return it->second;
    uint64_t h = 0;
    check(kvb_init_hash(device_, seed_hash_, model.data(), model.size(), &h));
    return init_[model] = h;
  }

  // TokensToKVBlockKeys (:177-205).  Empty vector = "nil, nil" (no full block).
  std::vector<BlockHash> TokensToKVBlockKeys(BlockHash parentKey, const std::vector<uint32_t>& tokens,
                                             const std::string& modelName, const ExtraFeatures* extraFeatures = nullptr) {
    const uint64_t parent = parentKey != EmptyBlockHash ? parentKey : InitHash(modelName);
    const size_t nblk = tokens.size() / (size_t)cfg_.BlockSize;
    if (nblk == 0) return {};
    std::vector<uint8_t> extra;
    std::vector<int64_t> extra_off;
    if (extraFeatures) {
      if (extraFeatures->size() != nblk)  // :195-198
        throw Error(KVB_ERR_INVALID, "extraFeatures length " + std::to_string(extraFeatures->size()) +
                                         " does not match token chunk count " + std::to_string(nblk) + " (blockSize=" +
                                         std::to_string(cfg_.BlockSize) + ", tokens=" + std::to_string(tokens.size()) + ")");
      extra_off.assign(nblk + 1, 0);
      for (size_t i = 0; i < nblk; ++i) {
        detail::encode_extra(extra, (*extraFeatures)[i].get());
        extra_off[i + 1] = (int64_t)extra.size();
      }
    }
    const int64_t prompt_off[2] = {0, (int64_t)tokens.size()};
    std::vector<BlockHash> keys(nblk);
    int64_t key_off[2] = {0, 0};
    check(kvb_hash_token_blocks(device_, tokens.data(), prompt_off, &parent, 1, cfg_.BlockSize,
                                extraFeatures && !extra.empty() ? extra.data() : nullptr,
                                extraFeatures ? extra_off.data() : nullptr, keys.data(), key_off, nullptr));
    return keys;
  }

 private:
  TokenProcessorConfig cfg_;
  int device_;
  uint64_t seed_hash_ = 0;
  std::mutex mu_;
  std::unordered_map<std::string, uint64_t> init_;
};

struct IndexConfig {  // InMemoryIndexConfig (in_memory.go:40-45) + device placement
  int64_t Size = 100000000;
  int PodCacheSize = 10;
  int Device = 0;
  int64_t ExpectedKeys = 0;
};

// kvblock.Index with InMemoryIndex semantics (in_memory.go:57-304); reads run on the GPU.
class Index {
 public:
  explicit Index(const IndexConfig& cfg = {}, std::map<std::string, double> mediumWeights = {{"gpu", 1.0}, {"cpu", 0.8}})
      : weights_(std::move(mediumWeights)) {
    check(kvb_index_create(cfg.Device, cfg.Size, cfg.PodCacheSize, cfg.ExpectedKeys, &h_));
  }
  ~Index() { kvb_index_destroy(h_); }
  Index(const Index&) = delete;
  Index& operator=(const Index&) = delete;
  kvb_index_t* handle() const { return h_; }

  // Add (in_memory.go:154-224).  engineKeys == nullptr <=> Go nil (speculative entries without engine keys).
  void Add(const std::vector<BlockHash>* engineKeys, const std::vector<BlockHash>& requestKeys,
           const std::vector<PodEntry>& entries) {
    if (requestKeys.empty() || entries.empty())
      throw Error(KVB_ERR_INVALID, "no keys or entries provided for adding to index");
    std::lock_guard<std::mutex> lk(mu_);
    auto e = intern(entries);
    check(kvb_index_add(h_, engineKeys ? engineKeys->data() : nullptr, engineKeys ? (int64_t)engineKeys->size() : 0,
                        engineKeys != nullptr, requestKeys.data(), (int64_t)requestKeys.size(), e.data(), (int32_t)e.size()));
  }
  // Evict (in_memory.go:229-255)
  void Evict(BlockHash key, KeyType keyType, const std::vector<PodEntry>& entries) {
    if (entries.empty()) throw Error(KVB_ERR_INVALID, "no entries provided for eviction from index");
    std::lock_guard<std::mutex> lk(mu_);
    auto e = intern(entries);
    check(kvb_index_evict(h_, key, (int)keyType, e.data(), (int32_t)e.size()));
  }
  // Every entry of `pods` (of `tiers`; empty = every tier) leaves every key, in one device sweep (kvb_index_remove_pods).
  // No reference counterpart (pool.go:388-395 ignores AllBlocksCleared).  Keys left empty are deleted, no recency
  // changes, the engine-key map is untouched; names the index has never seen match nothing.
  // Returns {entries removed, keys deleted}.
  std::pair<int64_t, int64_t> RemovePods(const std::vector<std::string>& pods, const std::vector<std::string>& tiers = {}) {
    std::lock_guard<std::mutex> lk(mu_);
    std::vector<uint16_t> p;
    for (const auto& name : pods) {
      auto it = pods_.find(name);
      if (it != pods_.end()) p.push_back(it->second);
    }
    std::vector<uint8_t> t;
    for (const auto& name : tiers) {
      auto it = tiers_.find(name);
      if (it != tiers_.end()) t.push_back(it->second);
    }
    if (p.empty() || (!tiers.empty() && t.empty())) return {0, 0};
    int64_t removed = 0, deleted = 0;
    check(kvb_index_remove_pods(h_, p.data(), (int32_t)p.size(), t.empty() ? nullptr : t.data(), (int32_t)t.size(),
                                &removed, &deleted));
    return {removed, deleted};
  }
  // GetRequestKey (in_memory.go:298-304)
  BlockHash GetRequestKey(BlockHash engineKey) {
    uint64_t out = 0;
    int rc = kvb_index_get_request_key(h_, engineKey, &out);
    if (rc == KVB_ERR_NOTFOUND) throw Error(rc, "engine key not found: " + std::to_string(engineKey));
    check(rc);
    return out;
  }
  // Lookup (in_memory.go:107-148): keys found before the cut -> their (filtered) pod entries.
  std::map<BlockHash, std::vector<PodEntry>> Lookup(const std::vector<BlockHash>& requestKeys,
                                                    const std::set<std::string>& podIdentifierSet = {}) {
    if (requestKeys.empty()) throw Error(KVB_ERR_INVALID, "no requestKeys provided for lookup");
    std::lock_guard<std::mutex> lk(mu_);
    std::vector<uint16_t> filter;
    for (const auto& name : podIdentifierSet) {
      auto it = pods_.find(name);
      if (it != pods_.end()) filter.push_back(it->second);
    }
    std::map<BlockHash, std::vector<PodEntry>> out;
    if (!podIdentifierSet.empty() && filter.empty()) return out;  // the filter names nobody the index has seen
    const size_t n = requestKeys.size();
    std::vector<int32_t> counts(n);
    std::vector<kvb_pod_entry_t> ents(n * KVB_INDEX_MAX_PODS_PER_KEY);
    int64_t cut = 0;
    check(kvb_index_lookup(h_, requestKeys.data(), (int64_t)n, filter.empty() ? nullptr : filter.data(),
                           (int32_t)filter.size(), counts.data(), ents.data(), &cut));
    for (int64_t i = 0; i < cut && i < (int64_t)n; ++i) {
      if (counts[i] <= 0) continue;
      std::vector<PodEntry> found;
      for (int e = 0; e < counts[i]; ++e) {
        const auto& c = ents[i * KVB_INDEX_MAX_PODS_PER_KEY + e];
        found.push_back(PodEntry{pod_names_[c.pod], tier_names_[c.tier], c.speculative != 0});
      }
      auto& slot = out[requestKeys[i]];
      if (!filter.empty())
        slot.insert(slot.end(), found.begin(), found.end());  // filtered path appends (in_memory.go:131-137)
      else
        slot = std::move(found);
    }
    return out;
  }

  // data-parallel Indexer.ScoreTokens: tokens of many prompts in, per-prompt pod scores out (fused on the device)
  std::vector<std::map<std::string, double>> ScoreTokensBatch(TokenProcessor& tp, const std::vector<std::vector<uint32_t>>& prompts,
                                                              const std::string& model,
                                                              const std::vector<std::string>& podIdentifiers = {}, bool touchLRU = true) {
    const uint64_t init = tp.InitHash(model);
    const int32_t n = (int32_t)prompts.size();
    std::vector<int64_t> off(n + 1, 0);
    for (int32_t i = 0; i < n; ++i) off[i + 1] = off[i] + (int64_t)prompts[i].size();
    std::vector<uint32_t> flat((size_t)off[n]);
    for (int32_t i = 0; i < n; ++i) std::copy(prompts[i].begin(), prompts[i].end(), flat.begin() + off[i]);
    std::vector<uint64_t> parents(n, init);
    std::lock_guard<std::mutex> lk(mu_);
    std::vector<uint16_t> filter;
    for (const auto& name : podIdentifiers) {
      auto it = pods_.find(name);
      if (it != pods_.end()) filter.push_back(it->second);
    }
    std::vector<std::map<std::string, double>> res(n);
    if (!podIdentifiers.empty() && filter.empty()) return res;
    std::vector<int32_t> out_n(n);
    std::vector<uint16_t> out_p((size_t)n * KVB_INDEX_MAX_PODS_PER_KEY);
    std::vector<double> out_s((size_t)n * KVB_INDEX_MAX_PODS_PER_KEY);
    check(kvb_index_score_tokens_batch(h_, flat.data(), off.data(), parents.data(), n, tp.BlockSize(), nullptr, nullptr,
                                       filter.empty() ? nullptr : filter.data(), (int32_t)filter.size(),
                                       touchLRU ? 0 : KVB_SCORE_NO_TOUCH, out_n.data(), out_p.data(), out_s.data()));
    for (int32_t i = 0; i < n; ++i)
      for (int j = 0; j < out_n[i]; ++j)
        res[i][pod_names_[out_p[(size_t)i * KVB_INDEX_MAX_PODS_PER_KEY + j]]] = out_s[(size_t)i * KVB_INDEX_MAX_PODS_PER_KEY + j];
    return res;
  }

 private:
  std::vector<kvb_pod_entry_t> intern(const std::vector<PodEntry>& in) {
    std::vector<kvb_pod_entry_t> out(in.size());
    for (size_t i = 0; i < in.size(); ++i) {
      auto p = pods_.find(in[i].PodIdentifier);
      if (p == pods_.end()) {
        if (pod_names_.size() >= 65536) throw Error(KVB_ERR_UNSUPPORTED, "too many distinct pod identifiers");
        p = pods_.emplace(in[i].PodIdentifier, (uint16_t)pod_names_.size()).first;
        pod_names_.push_back(in[i].PodIdentifier);
      }
      auto t = tiers_.find(in[i].DeviceTier);
      if (t == tiers_.end()) {
        if (tier_names_.size() >= 256) throw Error(KVB_ERR_UNSUPPORTED, "too many distinct device tiers");
        const uint8_t id = (uint8_t)tier_names_.size();
        auto w = weights_.find(in[i].DeviceTier);  // unknown tier scores 1.0 (kvblock_scorer.go:93-98)
        check(kvb_index_set_tier_weight(h_, id, w != weights_.end() ? w->second : 1.0, w != weights_.end()));
        t = tiers_.emplace(in[i].DeviceTier, id).first;
        tier_names_.push_back(in[i].DeviceTier);
      }
      out[i].pod = p->second;
      out[i].tier = t->second;
      out[i].speculative = in[i].Speculative ? 1 : 0;
    }
    return out;
  }
  kvb_index_t* h_ = nullptr;
  std::mutex mu_;
  std::map<std::string, double> weights_;
  std::unordered_map<std::string, uint16_t> pods_;
  std::vector<std::string> pod_names_;
  std::unordered_map<std::string, uint8_t> tiers_;
  std::vector<std::string> tier_names_;
};

}  // namespace kvblock

namespace kvcache {

// kvcache.Indexer (indexer.go:65-304): tokens -> block keys -> Lookup -> longest-prefix Score.
class Indexer {
 public:
  Indexer(std::shared_ptr<kvblock::TokenProcessor> tokenProcessor, std::shared_ptr<kvblock::Index> index)
      : tp_(std::move(tokenProcessor)), index_(std::move(index)) {
    if (!tp_) throw Error(KVB_ERR_INVALID, "tokenProcessor cannot be nil");  // indexer.go:82-84
    if (!index_) throw Error(KVB_ERR_INVALID, "config cannot be nil");
  }
  kvblock::Index& KVBlockIndex() { return *index_; }
  std::vector<kvblock::BlockHash> ComputeBlockKeysFromTokens(const std::vector<uint32_t>& tokens, const std::string& modelName,
                                                             const kvblock::ExtraFeatures* extra = nullptr) {
    return tp_->TokensToKVBlockKeys(kvblock::EmptyBlockHash, tokens, modelName, extra);
  }
  // ScoreTokens (indexer.go:239-304).  nullopt = "nil, nil" (the prompt has no full block).
  std::optional<std::map<std::string, double>> ScoreTokens(const std::vector<uint32_t>& tokens, const std::string& modelName,
                                                           const std::vector<std::string>& podIdentifiers = {}) {
    if (tokens.size() / (size_t)tp_->BlockSize() == 0) return std::nullopt;
    return index_->ScoreTokensBatch(*tp_, {tokens}, modelName, podIdentifiers)[0];
  }

 private:
  std::shared_ptr<kvblock::TokenProcessor> tp_;
  std::shared_ptr<kvblock::Index> index_;
};

}  // namespace kvcache
}  // namespace kvb
