// TEST HARNESS (not product, not oracle): compiles the product's component steps
// image_to_pointcloud_b200/csrc/d2pc_components.h for the host and drives them single-threaded in the launch
// order of d2pc_mesh_components_enqueue, with the (triangle, edge) operations of each concurrent launch visited in a
// seeded random order.  The result must equal the oracle's for every order, and no step may exhaust its bound.
#include <algorithm>
#include <cstdint>
#include <random>
#include <vector>

#include "../../image_to_pointcloud_b200/csrc/d2pc_components.h"

using namespace d2pc;

extern "C" {

// error bits as the device's: 1 bad triangle id, 2 non-finite vertex, 4 bound exhausted.  labels [T], ncount [T],
// carea [T] (first *K in use).  Returns the longest probe + find walk seen, for the bound checks.
long hc_components(const float *xyz, uint32_t V, const int32_t *tri, uint32_t T, uint64_t seed, int32_t *labels,
                   int64_t *ncount, double *carea, uint32_t *K, int32_t *err) {
  std::mt19937_64 rng(seed);
  *err = 0;
  *K = 0;
  for (uint32_t i = 0; i < V; ++i)
    for (int c = 0; c < 3; ++c)
      if (!std::isfinite(xyz[3 * (size_t)i + c])) *err |= 2;
  if (T == 0) return 0;
  if (V == 0) { *err |= 1; return 0; }
  const uint32_t cap = std::max<uint32_t>(1024u, 4u * T);
  std::vector<unsigned long long> keys(cap, kCompNoKey);
  std::vector<uint32_t> vals(cap, kCompNone), eslot(3 * (size_t)T, kCompNone), parent(T), root(T);
  std::vector<double> area(T, 0.0);
  std::vector<bool> ok(T);
  double amax = 0.0;
  for (uint32_t t = 0; t < T; ++t) {
    parent[t] = t;
    const int32_t *v = tri + 3 * (size_t)t;
    ok[t] = v[0] >= 0 && (uint32_t)v[0] < V && v[1] >= 0 && (uint32_t)v[1] < V && v[2] >= 0 && (uint32_t)v[2] < V;
    if (!ok[t]) { *err |= 1; continue; }
    double p[3][3];
    for (int k = 0; k < 3; ++k)
      for (int c = 0; c < 3; ++c) p[k][c] = (double)xyz[3 * (size_t)v[k] + c];
    area[t] = comp_triangle_area(p);
    if (!std::isfinite(area[t])) area[t] = 0.0;
    amax = std::max(amax, area[t]);
  }
  // edge inserts in a random order
  std::vector<uint64_t> ops(3 * (size_t)T);
  for (size_t i = 0; i < ops.size(); ++i) ops[i] = i;
  std::shuffle(ops.begin(), ops.end(), rng);
  for (uint64_t op : ops) {
    const uint32_t t = (uint32_t)(op / 3), k = (uint32_t)(op % 3);
    if (!ok[t]) continue;
    const int32_t *v = tri + 3 * (size_t)t;
    const uint32_t s = comp_edge_insert(keys.data(), vals.data(), cap, comp_edge_key(v[k], v[k == 2 ? 0 : k + 1]), t);
    if (s == kCompFail) *err |= 4;
    else eslot[op] = s;
  }
  // unions in another random order
  std::shuffle(ops.begin(), ops.end(), rng);
  for (uint64_t op : ops) {
    const uint32_t t = (uint32_t)(op / 3), s = eslot[op];
    if (s == kCompNone) continue;
    const uint32_t r = vals[s];
    if (r > t) *err |= 8;   // the table's value is the lowest triangle on the edge
    if (r != t && comp_unite(parent.data(), t, r, T) == kCompFail) *err |= 4;
  }
  // roots in a random order (halving as it goes), then numbering in triangle order
  std::vector<uint32_t> order(T);
  for (uint32_t t = 0; t < T; ++t) order[t] = t;
  std::shuffle(order.begin(), order.end(), rng);
  for (uint32_t t : order) {
    const uint32_t r = comp_find(parent.data(), t, T);
    if (r == kCompFail) *err |= 4;
    root[t] = r == kCompFail ? t : r;
  }
  uint32_t k = 0;
  for (uint32_t t = 0; t < T; ++t)
    if (root[t] == t) labels[t] = (int32_t)k++;
  for (uint32_t t = 0; t < T; ++t) labels[t] = labels[root[t]];
  const double s = comp_area_scale(amax, T);
  std::vector<unsigned long long> acc(k, 0ull);
  std::fill(ncount, ncount + k, 0);
  for (uint32_t t : order) {
    acc[labels[t]] += (unsigned long long)(long long)std::nearbyint(area[t] * s);
    ncount[labels[t]] += 1;
  }
  for (uint32_t c = 0; c < k; ++c) carea[c] = (double)(long long)acc[c] / s;
  *K = *err ? 0u : k;
  return 0;
}

// the bounds themselves: a full table; a chain parent[x] = x - 1 walked with a bound below and at its length
int hc_insert_full(uint32_t cap) {
  std::vector<unsigned long long> keys(cap);
  std::vector<uint32_t> vals(cap, kCompNone);
  for (uint32_t i = 0; i < cap; ++i) keys[i] = i;   // every slot holds another key
  return comp_edge_insert(keys.data(), vals.data(), cap, comp_edge_key(7, 1 << 30), 0) == kCompFail ? 1 : 0;
}

int hc_chain_bounds(uint32_t len) {
  std::vector<uint32_t> parent(len);
  for (uint32_t i = 0; i < len; ++i) parent[i] = i ? i - 1 : 0;
  std::vector<uint32_t> copy = parent;
  const bool short_fails = comp_find(copy.data(), len - 1, 2) == kCompFail &&
                           comp_unite(copy.data(), len - 1, 0, 1) == kCompFail;
  const bool full_ok = comp_find(parent.data(), len - 1, len) == 0 && comp_unite(parent.data(), len - 1, 0, len) == 0;
  return short_fails && full_ok ? 1 : 0;
}

}  // extern "C"
