// d2pc_components.h -- the hazardous steps of row m3 (connected components of a triangle mesh), written once for
// host and device like d2pc_math.h: the probe of the open-addressed edge table, find with path halving, and the
// hook of one root under another.  The sm_100a kernels (d2pc_components.cu) run them concurrently; the host harness
// (tests/hostcomp/) runs the same bodies single-threaded in random orders and checks their bounds.
//
// Invariant: parent[x] <= x for every triangle x.  A hook only writes a smaller id into a root (compare-and-swap
// on the root), path halving only writes an ancestor (which is smaller) into a non-root, so every find strictly
// decreases and ends at the component's lowest triangle whatever the schedule.  Every loop has a bound known at
// launch (the table's capacity, the triangle count); an exhausted bound returns kCompFail instead of spinning.
#ifndef D2PC_COMPONENTS_H_
#define D2PC_COMPONENTS_H_

#include "d2pc_math.h"

namespace d2pc {

constexpr uint32_t kCompNone = 0xFFFFFFFFu;   // empty value slot, and "no slot"
constexpr uint32_t kCompFail = 0xFFFFFFFEu;   // a bound was exhausted
constexpr unsigned long long kCompNoKey = 0xFFFFFFFFFFFFFFFFull;   // empty key slot (no edge has it: ids < 2^31)

// the atomics the steps need: the device's, or plain single-threaded ones on the host
D2PC_HD unsigned long long comp_cas64(unsigned long long *p, unsigned long long cmp, unsigned long long val) {
#if defined(__CUDA_ARCH__)
  return atomicCAS(p, cmp, val);
#else
  const unsigned long long old = *p;
  if (old == cmp) *p = val;
  return old;
#endif
}
D2PC_HD uint32_t comp_cas32(uint32_t *p, uint32_t cmp, uint32_t val) {
#if defined(__CUDA_ARCH__)
  return atomicCAS(p, cmp, val);
#else
  const uint32_t old = *p;
  if (old == cmp) *p = val;
  return old;
#endif
}
D2PC_HD void comp_min32(uint32_t *p, uint32_t val) {
#if defined(__CUDA_ARCH__)
  atomicMin(p, val);
#else
  if (val < *p) *p = val;
#endif
}
// parent links are read and halved with plain (volatile: not cached in L1) accesses; only a root is ever CASed
D2PC_HD uint32_t comp_load(const uint32_t *p) { return *(const volatile uint32_t *)p; }
D2PC_HD void comp_store(uint32_t *p, uint32_t v) { *(volatile uint32_t *)p = v; }

// Open3D's GetTriangleArea in float64: x = p0 - p1, y = p0 - p2, 0.5 * |x cross y| (Eigen's component order, the norm
// summed left to right; no contraction: --fmad=false / -ffp-contract=off)
D2PC_HD double comp_triangle_area(const double p[3][3]) {
  const double x0 = p[0][0] - p[1][0], x1 = p[0][1] - p[1][1], x2 = p[0][2] - p[1][2];
  const double y0 = p[0][0] - p[2][0], y1 = p[0][1] - p[2][1], y2 = p[0][2] - p[2][2];
  const double c0 = x1 * y2 - x2 * y1, c1 = x2 * y0 - x0 * y2, c2 = x0 * y1 - x1 * y0;
  return 0.5 * sqrt(c0 * c0 + c1 * c1 + c2 * c2);
}

// s = 2^(62 - e_a - e_T) with amax < 2^e_a (0 when amax is 0) and T <= 2^e_T: every term rint(a_t s) is below
// 2^(62 - e_T), so a sum of at most T terms stays below 2^62
D2PC_HD double comp_area_scale(double amax, uint32_t T) {
  int ea = 0;
  if (amax > 0.0) frexp(amax, &ea);
  int et = 0;
  while (et < 32 && (1ull << et) < (unsigned long long)T) ++et;
  return ldexp(1.0, 62 - ea - et);
}

// the unordered vertex pair as one key: (min << 32) | max
D2PC_HD unsigned long long comp_edge_key(int32_t a, int32_t b) {
  const uint32_t lo = (uint32_t)(a < b ? a : b), hi = (uint32_t)(a < b ? b : a);
  return ((unsigned long long)lo << 32) | hi;
}

D2PC_HD unsigned long long comp_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}

// Claims (or finds) the slot of `key` in keys[cap] (kCompNoKey = empty) and lowers vals[slot] to t.  Linear probe of
// at most cap steps; returns the slot, or kCompFail when all cap slots hold other keys.
D2PC_HD uint32_t comp_edge_insert(unsigned long long *keys, uint32_t *vals, uint32_t cap, unsigned long long key,
                                  uint32_t t) {
  uint32_t slot = (uint32_t)(((comp_hash(key) >> 32) * (unsigned long long)cap) >> 32);
  for (uint32_t step = 0; step < cap; ++step) {
    const unsigned long long prev = comp_cas64(keys + slot, kCompNoKey, key);
    if (prev == kCompNoKey || prev == key) {
      comp_min32(vals + slot, t);
      return slot;
    }
    slot = slot + 1u == cap ? 0u : slot + 1u;
  }
  return kCompFail;
}

// Root of x (parent[x] <= x), halving the path on the way: at most n steps (n = the triangle count), else kCompFail.
D2PC_HD uint32_t comp_find(uint32_t *parent, uint32_t x, uint32_t n) {
  for (uint32_t step = 0; step < n; ++step) {
    const uint32_t p = comp_load(parent + x);
    if (p == x) return x;
    const uint32_t g = comp_load(parent + p);
    if (g != p) comp_store(parent + x, g);   // g < p < x: still an ancestor of x
    x = g;
  }
  return kCompFail;
}

// Joins the trees of a and b: the larger root is hooked under the smaller with a CAS on the root.  A failed CAS means
// another thread hooked that root meanwhile; its new (smaller) parent is taken and the loop goes on, so the sum of the
// two ids strictly decreases: at most 2n rounds.  Returns 0, or kCompFail when a bound is exhausted.
D2PC_HD uint32_t comp_unite(uint32_t *parent, uint32_t a, uint32_t b, uint32_t n) {
  uint32_t ra = comp_find(parent, a, n), rb = comp_find(parent, b, n);
  for (uint32_t round = 0; round < 2u * n; ++round) {
    if (ra == kCompFail || rb == kCompFail) return kCompFail;
    if (ra == rb) return 0;
    const uint32_t hi = ra > rb ? ra : rb, lo = ra > rb ? rb : ra;
    const uint32_t prev = comp_cas32(parent + hi, hi, lo);
    if (prev == hi) return 0;
    // hi is no longer a root: continue from its new parent (< hi), the other side unchanged
    if (ra == hi) ra = comp_find(parent, prev, n);
    else rb = comp_find(parent, prev, n);
  }
  return kCompFail;
}

}  // namespace d2pc

#endif  // D2PC_COMPONENTS_H_
