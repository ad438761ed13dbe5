// Pins xllm_service_b200/host/index_wire.h against what the REFERENCE ITSELF wrote to etcd: the reference's
// etcd_client.cpp + global_kvcache_mgr.cpp + types.h, compiled unmodified, ran a random event history on a master and
// uploaded it (etcd_client.cpp:122-137); tests/golden/make_ref_goldens.py stored the resulting store listing with the
// sets the master held for each key (tests/golden/ref_etcd_listing.bin, format in that script).  Our key / JSON
// readers must read every pair into the sets the reference held, and our writer must emit the same key and — up to
// the order of names inside an array (unordered_set iteration in the reference) — the same JSON.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../xllm_service_b200/host/index_wire.h"

static int fails = 0;
#define EXPECT(c)                                                   \
  do {                                                              \
    if (!(c)) { ++fails; printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); } \
  } while (0)

static std::string sorted_arrays(const std::string& json) {   // canonical form: sort the strings inside each [...]
  std::string out;
  size_t i = 0;
  while (i < json.size()) {
    if (json[i] != '[') { out += json[i++]; continue; }
    size_t j = i + 1;
    std::vector<std::string> items;
    while (json[j] != ']') {
      if (json[j] == ',') { ++j; continue; }
      size_t s = j++;
      while (json[j] != '"' || json[j - 1] == '\\') {
        if (json[j] == '\\' && json[j + 1] == '\\') ++j;   // skip an escaped backslash pair as a unit
        ++j;
      }
      ++j;
      items.push_back(json.substr(s, j - s));
    }
    std::sort(items.begin(), items.end());
    out += '[';
    for (size_t k = 0; k < items.size(); ++k) out += (k ? "," : "") + items[k];
    out += ']';
    i = j + 1;
  }
  return out;
}

struct Reader {   // little-endian u32 / u64 and u32-length-prefixed byte strings
  std::string buf;
  size_t at = 0;
  bool ok = true;
  uint64_t num(size_t width) {
    uint64_t v = 0;
    if (at + width > buf.size()) { ok = false; return 0; }
    memcpy(&v, buf.data() + at, width);
    at += width;
    return v;
  }
  std::string bytes() {
    const size_t n = num(4);
    if (at + n > buf.size()) { ok = false; return std::string(); }
    at += n;
    return buf.substr(at - n, n);
  }
};

int main(int argc, char** argv) {
  using namespace xllm_host;
  if (argc < 2) { printf("usage: %s ref_etcd_listing.bin\n", argv[0]); return 2; }
  Reader in;
  {
    std::ifstream f(argv[1], std::ios::binary);
    in.buf.assign(std::istreambuf_iterator<char>(f), std::istreambuf_iterator<char>());
  }
  std::vector<std::string> names(in.num(4));
  for (auto& n : names) n = in.bytes();
  std::unordered_map<std::string, int> ids;
  for (int i = 0; i < (int)names.size(); ++i) ids[names[i]] = i;
  auto id_of = [&](const std::string& n) { auto it = ids.find(n); return it == ids.end() ? -1 : it->second; };

  const uint32_t n_ns = (uint32_t)in.num(4);
  EXPECT(in.ok && n_ns == 2);
  for (uint32_t s = 0; s < n_ns && in.ok; ++s) {
    const std::string ns = in.bytes();
    const std::string nsp = ns.empty() ? "" : "/" + ns + "/";   // utils.cpp:105-124
    const std::string prefix = nsp + etcd_cache_prefix();
    const uint32_t n = (uint32_t)in.num(4);
    EXPECT(n > 100);
    for (uint32_t i = 0; i < n && in.ok; ++i) {
      const std::string k = in.bytes(), v = in.bytes();
      uint64_t want[3];
      for (auto& w : want) w = in.num(8);
      uint8_t key[16];
      uint64_t m[3] = {~0ull, ~0ull, ~0ull};
      EXPECT(parse_cache_etcd_key(k, prefix.size(), key));
      EXPECT(cache_etcd_key(nsp, key) == k);
      EXPECT(cache_locations_from_json(v, id_of, &m[0], &m[1], &m[2]));
      EXPECT(want[0] == m[0] && want[1] == m[1] && want[2] == m[2]);
      std::string ours;
      EXPECT(cache_locations_to_json(m[0], m[1], m[2], names, &ours));
      EXPECT(ours.size() == v.size() && sorted_arrays(ours) == sorted_arrays(v));
    }
    printf("namespace '%s': %u pairs checked\n", ns.c_str(), n);
  }
  EXPECT(in.ok && in.at == in.buf.size());
  printf(fails ? "FAILED %d\n" : "OK\n", fails);
  return fails ? 1 : 0;
}
