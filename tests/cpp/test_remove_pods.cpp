// Known answer of kvblock::Index::RemovePods (include/kvb_kvblock.hpp) over libkvb.so.
// Usage: test_remove_pods   (compiled and run by tests/test_gpu_index_remove_pods.py; prints "OK <checks>")
#include <cstdio>
#include <map>
#include <vector>

#include "kvb_kvblock.hpp"

using namespace kvb;
using kvblock::PodEntry;

static int g_checks = 0;
#define CHECK(cond)                                                                   \
  do {                                                                                \
    ++g_checks;                                                                       \
    if (!(cond)) {                                                                    \
      std::fprintf(stderr, "CHECK failed at %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      return 1;                                                                       \
    }                                                                                 \
  } while (0)

int main() {
  try {
    kvblock::IndexConfig cfg;
    cfg.Size = 1000;
    cfg.PodCacheSize = 4;
    kvblock::Index idx(cfg);
    const PodEntry p0g{"p0", "gpu", false}, p1g{"p1", "gpu", false}, p0c{"p0", "cpu", false}, p1c{"p1", "cpu", false};
    const std::vector<kvblock::BlockHash> a{11}, b{22}, c{33}, all{11, 22, 33};
    idx.Add(nullptr, a, {p0g, p1g, p0c});
    idx.Add(nullptr, b, {p0g});
    idx.Add(nullptr, c, {p1c});

    // removing p0 (every tier): A keeps p1/gpu, B is deleted, C is untouched
    auto r = idx.RemovePods({"p0"});
    CHECK(r.first == 3 && r.second == 1);
    auto got = idx.Lookup(all);
    CHECK(got.size() == 2);
    CHECK(got[11] == std::vector<PodEntry>{p1g});
    CHECK(got[33] == std::vector<PodEntry>{p1c});

    // (p1, cpu) only: C goes, A's p1/gpu stays
    r = idx.RemovePods({"p1"}, {"cpu"});
    CHECK(r.first == 1 && r.second == 1);
    got = idx.Lookup(all);
    CHECK(got.size() == 1 && got[11] == std::vector<PodEntry>{p1g});

    // names the index has never seen match nothing
    r = idx.RemovePods({"nobody"});
    CHECK(r.first == 0 && r.second == 0);
    r = idx.RemovePods({"p1"}, {"disk"});
    CHECK(r.first == 0 && r.second == 0);
    CHECK(idx.Lookup(all).size() == 1);

    // speculative entries of the pod go too; the engine-key map is untouched
    const std::vector<kvblock::BlockHash> ek{900};
    idx.Add(&ek, {44}, {PodEntry{"p2", "gpu", true}, p1g});
    r = idx.RemovePods({"p2"});
    CHECK(r.first == 1 && r.second == 0);
    CHECK(idx.Lookup({44})[44] == std::vector<PodEntry>{p1g});
    r = idx.RemovePods({"p1"});
    CHECK(r.first == 2 && r.second == 2);
    CHECK(idx.Lookup({11, 44}).empty());
    CHECK(idx.GetRequestKey(900) == 44);
  } catch (const std::exception& e) {
    std::fprintf(stderr, "exception: %s\n", e.what());
    return 1;
  }
  std::printf("OK %d\n", g_checks);
  return 0;
}
