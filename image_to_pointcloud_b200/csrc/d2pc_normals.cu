// d2pc_normals.cu -- point normals with Open3D's semantics: PointCloud::EstimateNormals (KDTreeSearchParamKNN(knn)
// or KDTreeSearchParamHybrid(radius, knn), fast_normal_computation = true) followed by
// OrientNormalsTowardsCameraLocation.  Spec restated in oracle/d2pc_oracle.py::estimate_normals (Open3D itself is
// not installed: parity unpinned):
//   neighbours  the k nearest points of i, i itself included, d2 accumulated axis by axis in float64; with a
//               radius only d2 < radius^2 counts; ties ordered by (d2, source row)
//   covariance  ComputeCovariance: cumulants of p and p p^T over the neighbours in ascending (d2, row) order,
//               divided by their number, E[pp^T] - mean mean^T; fewer than 3 neighbours -> identity
//   normal      FastEigen3x3 (Geometric Tools' robust symmetric 3x3 solver) in float64, normalised; a zero
//               result -> (0, 0, 1); oriented so that n . (camera - p) >= 0
//
// The grid is the one statistical outlier removal builds (d2pc_grid.cuh, sor_grid_build).  The query walks it the
// way sor_query_kernel does (own cell, shells of growing Chebyshev radius, x-window in heavy cells, float32
// pre-filter, exactness bound) but keeps (d2, row) pairs, so that the k-th neighbour is defined on ties.
#include <cmath>
#include <stdlib.h>
#include "d2pc_grid.cuh"

namespace d2pc {

constexpr int kNrmThreads = 128;
constexpr int kNrmSharedK = 32;   // [k][kNrmThreads] (d2, row) pairs in shared memory: 12 B * 32 * 128 = 48 KB

// The k best (d2, row) pairs of one query as a binary max-heap (root = the current k-th pair).  STRIDE 1: local
// arrays; STRIDE kNrmThreads: one column of [k][kNrmThreads] arrays in shared memory.
template <int STRIDE>
struct PairHeap {
  double *d;
  uint32_t *r;
  __device__ __forceinline__ double &dist(int t) const { return d[t * STRIDE]; }
  __device__ __forceinline__ uint32_t &row(int t) const { return r[t * STRIDE]; }
};

__device__ __forceinline__ bool pair_less(double a, uint32_t ra, double b, uint32_t rb) {
  return a < b || (a == b && ra < rb);
}

template <class H>
__device__ __forceinline__ void pair_sift(const H &hp, int size, double v, uint32_t vr) {
  int pos = 0;
  while (true) {
    const int l = 2 * pos + 1;
    if (l >= size) break;
    const int r = l + 1;
    int c = l;
    double vc = hp.dist(l);
    uint32_t rc = hp.row(l);
    if (r < size) {
      const double vr2 = hp.dist(r);
      const uint32_t rr2 = hp.row(r);
      if (pair_less(vc, rc, vr2, rr2)) { c = r; vc = vr2; rc = rr2; }
    }
    if (!pair_less(v, vr, vc, rc)) break;
    hp.dist(pos) = vc;
    hp.row(pos) = rc;
    pos = c;
  }
  hp.dist(pos) = v;
  hp.row(pos) = vr;
}

struct Kth {
  double d;
  uint32_t r;
  float thrf;
};

template <class H>
__device__ __forceinline__ void nrm_offer(const H &hp, int k, double d2, uint32_t row, Kth &kth) {
  if (!pair_less(d2, row, kth.d, kth.r)) return;
  pair_sift(hp, k, d2, row);
  kth.d = hp.dist(0);
  kth.r = hp.row(0);
  kth.thrf = sor_filter(kth.d);
}

__device__ __forceinline__ double nrm_d2(const double q[3], const float p[3]) {
  const double dx = q[0] - (double)p[0], dy = q[1] - (double)p[1], dz = q[2] - (double)p[2];
  double d2 = dx * dx;   // nanoflann L2_Simple, axis by axis (no contraction: --fmad=false)
  d2 += dy * dy;
  d2 += dz * dz;
  return d2;
}

// Candidates of one cell; the float32 filter is conservative (d2f <= thrf for every d2 <= kth), so a candidate that
// ties the k-th distance still reaches the exact (d2, row) comparison.
template <class H>
__device__ __forceinline__ void nrm_visit_cell(const SorWs &w, uint32_t cell, const double q[3], const float qf[3],
                                               const H &hp, int k, Kth &kth) {
  const uint32_t s = w.cell_off[cell], e = w.cell_off[cell + 1];
  constexpr int U = 4;
  if (w.cell_cnt[cell] & kSorSortedFlag) {
    uint32_t lo = s, hi = e;
    while (lo < hi) {  // first point with x >= q.x
      const uint32_t mid = lo + ((hi - lo) >> 1);
      if (w.sorted[3 * (size_t)mid] < qf[0]) lo = mid + 1; else hi = mid;
    }
    uint32_t r = lo, l = lo;
    bool go_r = r < e, go_l = l > s;
    while ((go_r || go_l) && kth.d > 0.0) {
      float p[2 * U][3];
      bool ok[2 * U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        ok[u] = go_r && r + (uint32_t)u < e;
        ok[U + u] = go_l && l >= s + 1u + (uint32_t)u;
        const uint32_t jr = ok[u] ? r + (uint32_t)u : s, jl = ok[U + u] ? l - 1u - (uint32_t)u : s;
#pragma unroll
        for (int a = 0; a < 3; ++a) { p[u][a] = w.sorted[3 * (size_t)jr + a]; p[U + u][a] = w.sorted[3 * (size_t)jl + a]; }
      }
#pragma unroll
      for (int u = 0; u < 2 * U; ++u) {
        const bool right = u < U;
        if (!ok[u] || (right ? !go_r : !go_l)) continue;
        const float fx = qf[0] - p[u][0];
        if (fx * fx > kth.thrf) { if (right) go_r = false; else go_l = false; continue; }
        const float fy = qf[1] - p[u][1], fz = qf[2] - p[u][2];
        if (fx * fx + fy * fy + fz * fz <= kth.thrf) {
          const double d2 = nrm_d2(q, p[u]);
          if (d2 <= kth.d) {
            const uint32_t j = right ? r + (uint32_t)u : l - 1u - (uint32_t)(u - U);
            nrm_offer(hp, k, d2, w.sorted_idx[j], kth);
          }
        }
      }
      if (go_r) { r += U; go_r = r < e; }
      if (go_l) { l = l >= s + (uint32_t)U ? l - (uint32_t)U : s; go_l = l > s; }
    }
    return;
  }
  for (uint32_t j0 = s; j0 < e && kth.d > 0.0; j0 += U) {
    float p[U][3], d2f[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint32_t j = min(j0 + (uint32_t)u, e - 1u);
#pragma unroll
      for (int a = 0; a < 3; ++a) p[u][a] = w.sorted[3 * (size_t)j + a];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const float fx = qf[0] - p[u][0], fy = qf[1] - p[u][1], fz = qf[2] - p[u][2];
      d2f[u] = fx * fx + fy * fy + fz * fz;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (j0 + (uint32_t)u >= e || d2f[u] > kth.thrf) continue;
      const double d2 = nrm_d2(q, p[u]);
      if (d2 <= kth.d) nrm_offer(hp, k, d2, w.sorted_idx[j0 + (uint32_t)u], kth);
    }
  }
}

template <class H>
__device__ __forceinline__ void nrm_visit_key(const SorWs &w, unsigned long long key, const double q[3], const float qf[3],
                                              const H &hp, int k, Kth &kth) {
  uint32_t slot;
  if (sor_find(w, key, &slot)) nrm_visit_cell(w, slot, q, qf, hp, k, kth);
}

// ---- Open3D's FastEigen3x3 (Geometric Tools, "A Robust Eigensolver for 3x3 Symmetric Matrices") ----------------
// A = {a00, a01, a02, a11, a12, a22}
struct Vec3 { double x, y, z; };
__device__ __forceinline__ Vec3 cross3(Vec3 a, Vec3 b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__device__ __forceinline__ double dot3(Vec3 a, Vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

__device__ __forceinline__ Vec3 eigenvector0(const double A[6], double eval0) {
  const Vec3 row0{A[0] - eval0, A[1], A[2]}, row1{A[1], A[3] - eval0, A[4]}, row2{A[2], A[4], A[5] - eval0};
  const Vec3 r0xr1 = cross3(row0, row1), r0xr2 = cross3(row0, row2), r1xr2 = cross3(row1, row2);
  const double d0 = dot3(r0xr1, r0xr1), d1 = dot3(r0xr2, r0xr2), d2 = dot3(r1xr2, r1xr2);
  double dmax = d0;
  int imax = 0;
  if (d1 > dmax) { dmax = d1; imax = 1; }
  if (d2 > dmax) imax = 2;
  const Vec3 v = imax == 0 ? r0xr1 : (imax == 1 ? r0xr2 : r1xr2);
  const double s = sqrt(imax == 0 ? d0 : (imax == 1 ? d1 : d2));
  return {v.x / s, v.y / s, v.z / s};
}

__device__ __forceinline__ Vec3 eigenvector1(const double A[6], Vec3 evec0, double eval1) {
  Vec3 U;
  if (fabs(evec0.x) > fabs(evec0.y)) {
    const double inv_length = 1 / sqrt(evec0.x * evec0.x + evec0.z * evec0.z);
    U = {-evec0.z * inv_length, 0, evec0.x * inv_length};
  } else {
    const double inv_length = 1 / sqrt(evec0.y * evec0.y + evec0.z * evec0.z);
    U = {0, evec0.z * inv_length, -evec0.y * inv_length};
  }
  const Vec3 V = cross3(evec0, U);
  const Vec3 AU{A[0] * U.x + A[1] * U.y + A[2] * U.z, A[1] * U.x + A[3] * U.y + A[4] * U.z,
                A[2] * U.x + A[4] * U.y + A[5] * U.z};
  const Vec3 AV{A[0] * V.x + A[1] * V.y + A[2] * V.z, A[1] * V.x + A[3] * V.y + A[4] * V.z,
                A[2] * V.x + A[4] * V.y + A[5] * V.z};
  double m00 = U.x * AU.x + U.y * AU.y + U.z * AU.z - eval1;
  double m01 = U.x * AV.x + U.y * AV.y + U.z * AV.z;
  double m11 = V.x * AV.x + V.y * AV.y + V.z * AV.z - eval1;
  const double absM00 = fabs(m00), absM01 = fabs(m01), absM11 = fabs(m11);
  if (absM00 >= absM11) {
    if ((absM00 < absM01 ? absM01 : absM00) > 0) {
      if (absM00 >= absM01) {
        m01 /= m00;
        m00 = 1 / sqrt(1 + m01 * m01);
        m01 *= m00;
      } else {
        m00 /= m01;
        m01 = 1 / sqrt(1 + m00 * m00);
        m00 *= m01;
      }
      return {m01 * U.x - m00 * V.x, m01 * U.y - m00 * V.y, m01 * U.z - m00 * V.z};
    }
    return U;
  }
  if ((absM11 < absM01 ? absM01 : absM11) > 0) {
    if (absM11 >= absM01) {
      m01 /= m11;
      m11 = 1 / sqrt(1 + m01 * m01);
      m01 *= m11;
    } else {
      m11 /= m01;
      m01 = 1 / sqrt(1 + m11 * m11);
      m11 *= m01;
    }
    return {m11 * U.x - m01 * V.x, m11 * U.y - m01 * V.y, m11 * U.z - m01 * V.z};
  }
  return U;
}

// eigenvector of the smallest eigenvalue of the covariance C (unnormalised; the zero vector when max(C) == 0)
__device__ __forceinline__ Vec3 fast_eigen3x3(const double C[6]) {
  double mx = C[0];
#pragma unroll
  for (int t = 1; t < 6; ++t) mx = C[t] > mx ? C[t] : mx;   // maxCoeff over the 9 entries: the 6 unique ones
  if (mx == 0) return {0, 0, 0};
  double A[6];
#pragma unroll
  for (int t = 0; t < 6; ++t) A[t] = C[t] / mx;
  const double norm = A[1] * A[1] + A[2] * A[2] + A[4] * A[4];
  if (norm > 0) {
    const double q = (A[0] + A[3] + A[5]) / 3;
    const double b00 = A[0] - q, b11 = A[3] - q, b22 = A[5] - q;
    const double p = sqrt((b00 * b00 + b11 * b11 + b22 * b22 + norm * 2) / 6);
    const double c00 = b11 * b22 - A[4] * A[4];
    const double c01 = A[1] * b22 - A[4] * A[2];
    const double c02 = A[1] * A[4] - b11 * A[2];
    const double det = (b00 * c00 - A[1] * c01 + A[2] * c02) / (p * p * p);
    double half_det = det * 0.5;
    half_det = half_det < -1.0 ? -1.0 : half_det;   // std::min(std::max(half_det, -1.0), 1.0)
    half_det = 1.0 < half_det ? 1.0 : half_det;
    const double angle = acos(half_det) / (double)3;
    const double two_thirds_pi = 2.09439510239319549;
    const double beta2 = cos(angle) * 2;
    const double beta0 = cos(angle + two_thirds_pi) * 2;
    const double beta1 = -(beta0 + beta2);
    const double eval0 = q + p * beta0, eval1 = q + p * beta1, eval2 = q + p * beta2;
    if (half_det >= 0) {
      const Vec3 evec2 = eigenvector0(A, eval2);
      if (eval2 < eval0 && eval2 < eval1) return evec2;
      const Vec3 evec1 = eigenvector1(A, evec2, eval1);
      if (eval1 < eval0 && eval1 < eval2) return evec1;
      return cross3(evec1, evec2);
    }
    const Vec3 evec0 = eigenvector0(A, eval0);
    if (eval0 < eval1 && eval0 < eval2) return evec0;
    const Vec3 evec1 = eigenvector1(A, evec0, eval1);
    if (eval1 < eval0 && eval1 < eval2) return evec1;
    return cross3(evec0, evec1);
  }
  const double d0 = A[0] * mx, d1 = A[3] * mx, d2 = A[5] * mx;   // A *= max_coeff, then the diagonal
  if (d0 < d1 && d0 < d2) return {1, 0, 0};
  if (d1 < d0 && d1 < d2) return {0, 1, 0};
  return {0, 0, 1};
}

struct NrmParams {
  double r2;          // radius^2 (radius mode) or +inf (k-NN mode): only d2 < r2 counts
  uint32_t seed_row;  // row of the heap's initial pairs (r2, seed_row)
  int knn;
  int orient;
  double cam[3];
};

template <bool SHARED>
__global__ void __launch_bounds__(kNrmThreads) normals_query_kernel(SorWs w, const float *xyz, NrmParams prm,
                                                                    double *out_normals, double *out_cov) {
  extern __shared__ __align__(16) unsigned char s_heap[];   // SHARED: double [k][T], then uint32 [k][T]
  const SorHeader *h = w.hdr;
  const uint32_t n = h->n;
  const uint32_t j = blockIdx.x * (uint32_t)kNrmThreads + threadIdx.x;
  if (j >= n) return;
  const uint32_t i = w.sorted_idx[j];
  const int k = (int)min((uint32_t)prm.knn, n);
  double loc_d[SHARED ? 1 : kSorMaxK];
  uint32_t loc_r[SHARED ? 1 : kSorMaxK];
  const PairHeap<SHARED ? kNrmThreads : 1> hp{
      SHARED ? reinterpret_cast<double *>(s_heap) + threadIdx.x : loc_d,
      SHARED ? reinterpret_cast<uint32_t *>(s_heap + (size_t)prm.knn * kNrmThreads * sizeof(double)) + threadIdx.x : loc_r};
  for (int t = 0; t < k; ++t) { hp.dist(t) = prm.r2; hp.row(t) = prm.seed_row; }
  Kth kth{prm.r2, prm.seed_row, sor_filter(prm.r2)};
  const float qf[3] = {w.sorted[3 * (size_t)j], w.sorted[3 * (size_t)j + 1], w.sorted[3 * (size_t)j + 2]};
  const double q[3] = {(double)qf[0], (double)qf[1], (double)qf[2]};
  const int32_t nx = h->dim[0], ny = h->dim[1], nz = h->dim[2];
  const uint32_t cell = w.pt_cell[i];
  const unsigned long long ckey = w.keys[cell];
  const int32_t cm = (1 << kSorCoordBits) - 1;
  const int32_t c0 = (int32_t)(ckey >> (2 * kSorCoordBits)) & cm, c1 = (int32_t)(ckey >> kSorCoordBits) & cm,
                c2 = (int32_t)ckey & cm;
  const int32_t c[3] = {c0, c1, c2};
  double dlo[3], dhi[3];
  int32_t rmax = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double lo = h->mn[a] + (double)c[a] * h->h;
    dlo[a] = fmax(q[a] - lo, 0.0);
    dhi[a] = fmax(lo + h->h - q[a], 0.0);
    rmax = max(rmax, max(c[a], h->dim[a] - 1 - c[a]));
  }
  nrm_visit_cell(w, cell, q, qf, hp, k, kth);
  const int32_t dim[3] = {nx, ny, nz};
  for (int32_t R = 1; R <= rmax; ++R) {
    // unvisited points are at least `reach` away; they cannot tie the k-th pair either (strictly farther)
    double reach = __longlong_as_double(0x7FF0000000000000ll);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (c[a] - R >= 0) reach = fmin(reach, (double)(R - 1) * h->h + dlo[a]);
      if (c[a] + R <= dim[a] - 1) reach = fmin(reach, (double)(R - 1) * h->h + dhi[a]);
    }
    reach -= h->slack;
    if ((reach > 0.0 && kth.d <= reach * reach) || kth.d == 0.0) break;  // k coincident points: same cumulants
    const int32_t y0 = max(c1 - R, 0), y1 = min(c1 + R, ny - 1);
    const int32_t z0 = max(c2 - R, 0), z1 = min(c2 + R, nz - 1);
    const int32_t xi0 = max(c0 - R + 1, 0), xi1 = min(c0 + R - 1, nx - 1);
    const int32_t yi0 = max(c1 - R + 1, 0), yi1 = min(c1 + R - 1, ny - 1);
    for (int side = 0; side < 2; ++side) {
      const int32_t a0 = side ? c0 + R : c0 - R;
      if (a0 < 0 || a0 >= nx) continue;
      for (int32_t a1 = y0; a1 <= y1; ++a1)
        for (int32_t a2 = z0; a2 <= z1; ++a2) nrm_visit_key(w, sor_key(a0, a1, a2), q, qf, hp, k, kth);
    }
    for (int side = 0; side < 2; ++side) {
      const int32_t a1 = side ? c1 + R : c1 - R;
      if (a1 < 0 || a1 >= ny) continue;
      for (int32_t a0 = xi0; a0 <= xi1; ++a0)
        for (int32_t a2 = z0; a2 <= z1; ++a2) nrm_visit_key(w, sor_key(a0, a1, a2), q, qf, hp, k, kth);
    }
    for (int side = 0; side < 2; ++side) {
      const int32_t a2 = side ? c2 + R : c2 - R;
      if (a2 < 0 || a2 >= nz) continue;
      for (int32_t a0 = xi0; a0 <= xi1; ++a0)
        for (int32_t a1 = yi0; a1 <= yi1; ++a1) nrm_visit_key(w, sor_key(a0, a1, a2), q, qf, hp, k, kth);
    }
  }
  // heap -> ascending (d2, row) in place
  for (int m = k; m > 1; --m) {
    const double td = hp.dist(0), ld = hp.dist(m - 1);
    const uint32_t tr = hp.row(0), lr = hp.row(m - 1);
    hp.dist(m - 1) = td;
    hp.row(m - 1) = tr;
    pair_sift(hp, m - 1, ld, lr);
  }
  // Open3D ComputeCovariance over the neighbours in that order; the seed pairs (d2 == r2) sort last
  double cu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int cnt = 0;
  for (int t = 0; t < k; ++t) {
    if (!(hp.dist(t) < prm.r2)) break;
    const uint32_t src = hp.row(t);
    const double p0 = (double)__ldg(xyz + 3 * (size_t)src), p1 = (double)__ldg(xyz + 3 * (size_t)src + 1),
                 p2 = (double)__ldg(xyz + 3 * (size_t)src + 2);
    cu[0] += p0; cu[1] += p1; cu[2] += p2;
    cu[3] += p0 * p0; cu[4] += p0 * p1; cu[5] += p0 * p2;
    cu[6] += p1 * p1; cu[7] += p1 * p2; cu[8] += p2 * p2;
    ++cnt;
  }
  double C[6] = {1, 0, 0, 1, 0, 1};  // a00, a01, a02, a11, a12, a22
  if (cnt >= 3) {
#pragma unroll
    for (int t = 0; t < 9; ++t) cu[t] /= (double)cnt;
    C[0] = cu[3] - cu[0] * cu[0];
    C[3] = cu[6] - cu[1] * cu[1];
    C[5] = cu[8] - cu[2] * cu[2];
    C[1] = cu[4] - cu[0] * cu[1];
    C[2] = cu[5] - cu[0] * cu[2];
    C[4] = cu[7] - cu[1] * cu[2];
  }
  if (out_cov) {
#pragma unroll
    for (int t = 0; t < 6; ++t) out_cov[6 * (size_t)i + t] = C[t];
  }
  Vec3 nv = fast_eigen3x3(C);
  const double s = dot3(nv, nv);
  if (s == 0.0) {
    nv = {0.0, 0.0, 1.0};
  } else {
    const double len = sqrt(s);
    nv = {nv.x / len, nv.y / len, nv.z / len};
  }
  if (prm.orient) {
    const Vec3 ref{prm.cam[0] - q[0], prm.cam[1] - q[1], prm.cam[2] - q[2]};
    if (dot3(nv, ref) < 0.0) nv = {nv.x * -1.0, nv.y * -1.0, nv.z * -1.0};
  }
  out_normals[3 * (size_t)i] = nv.x;
  out_normals[3 * (size_t)i + 1] = nv.y;
  out_normals[3 * (size_t)i + 2] = nv.z;
}

}  // namespace d2pc

using namespace d2pc;

extern "C" int d2pc_normals_scratch_bytes(uint32_t capacity_rows, size_t *bytes) {
  if (!bytes || capacity_rows == 0) return D2PC_ERR_INVALID_ARGUMENT;
  *bytes = sor_ws_bytes(capacity_rows);
  return D2PC_OK;
}

extern "C" int d2pc_normals_enqueue(const float *d_xyz, const uint32_t *d_count, uint32_t capacity_rows,
                                    const float *d_bounds, int32_t knn, double radius, int32_t orient,
                                    const double camera[3], void *d_scratch, size_t scratch_bytes,
                                    double *d_out_normals, double *d_out_cov, void *stream) {
  if (!d_xyz || !d_count || !d_bounds || !d_scratch || !d_out_normals) return D2PC_ERR_INVALID_ARGUMENT;
  if (capacity_rows == 0 || knn < 1 || knn > kSorMaxK || radius != radius) return D2PC_ERR_INVALID_ARGUMENT;
  if (orient && (!camera || !std::isfinite(camera[0]) || !std::isfinite(camera[1]) || !std::isfinite(camera[2])))
    return D2PC_ERR_INVALID_ARGUMENT;
  if (((uintptr_t)d_scratch & 255u) != 0) return D2PC_ERR_INVALID_ARGUMENT;
  if (scratch_bytes < sor_ws_bytes(capacity_rows)) return D2PC_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = (cudaStream_t)stream;
  SorWs w = sor_ws(d_scratch, capacity_rows);
  const int rc = sor_grid_build(w, d_xyz, d_count, d_bounds, capacity_rows, st);
  if (rc != D2PC_OK) return rc;
  NrmParams prm;
  const double inf = HUGE_VAL;
  // radius mode: the heap starts full of (radius^2, 0), so only d2 < radius^2 enters and the shell walk stops at
  // the radius; k-NN mode: (inf, ~0u) admits every point
  prm.r2 = radius > 0.0 ? radius * radius : inf;
  prm.seed_row = radius > 0.0 ? 0u : 0xFFFFFFFFu;
  prm.knn = knn;
  prm.orient = orient ? 1 : 0;
  for (int a = 0; a < 3; ++a) prm.cam[a] = orient ? camera[a] : 0.0;
  const uint32_t blocks = (capacity_rows + kNrmThreads - 1) / kNrmThreads;
  const char *heap_env = getenv("D2PC_NORMALS_HEAP");  // measurement aid: "local" forces the local-memory heap
  const bool local = heap_env && heap_env[0] == 'l';
  if (knn <= kNrmSharedK && !local) {
    const size_t smem = (size_t)knn * kNrmThreads * (sizeof(double) + sizeof(uint32_t));   // <= 48 KB
    normals_query_kernel<true><<<blocks, kNrmThreads, smem, st>>>(w, d_xyz, prm, d_out_normals, d_out_cov);
  } else {
    normals_query_kernel<false><<<blocks, kNrmThreads, 0, st>>>(w, d_xyz, prm, d_out_normals, d_out_cov);
  }
  D2PC_CHECK_LAUNCH();
  return D2PC_OK;
}
