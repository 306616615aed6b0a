// d2pc_smooth.h -- the arithmetic of row m4 (mesh smoothing, vertex normals of any mesh), written once for host and
// device like d2pc_components.h: the update of one vertex in one simple or Laplacian pass, and the normal of one
// vertex from its incident triangles.  The sm_100a kernels (d2pc_smooth.cu) run them one thread per vertex; the host
// harness (tests/hostsmooth/) runs the same bodies over the oracle's adjacency, so the order of every sum is checked
// without a GPU.  Compiled without contraction (--fmad=false / -ffp-contract=off): every operation rounds like NumPy.
#ifndef D2PC_SMOOTH_H_
#define D2PC_SMOOTH_H_

#include "d2pc_math.h"

namespace d2pc {

constexpr double kSmoothEps = 1e-12;   // Open3D's eps in w = 1 / (d + eps)

// Where a pass reads the three fields (f = 0 position, 1 normal, 2 colour: bit f of a scope is D2PC_SMOOTH_VERTEX,
// _NORMAL, _COLOR): the float64 state of the previous pass when state[f] is set, else the input (float32 positions
// and colours, float64 normals) widened to float64.
struct SmoothSrc {
  const double *state[3];
  const float *xyz, *rgb;
  const double *nrm;
};

D2PC_HD void smooth_load(const SmoothSrc &s, int f, uint32_t j, double y[3]) {
  const size_t b = 3 * (size_t)j;
  if (s.state[f]) {
    y[0] = s.state[f][b]; y[1] = s.state[f][b + 1]; y[2] = s.state[f][b + 2];
  } else if (f == 1) {
    y[0] = s.nrm[b]; y[1] = s.nrm[b + 1]; y[2] = s.nrm[b + 2];
  } else {
    const float *p = f == 0 ? s.xyz : s.rgb;
    y[0] = (double)p[b]; y[1] = (double)p[b + 1]; y[2] = (double)p[b + 2];
  }
}

// One pass for vertex i whose neighbours are nb[0 .. deg) in ascending id, for the fields in `fields` (bits as
// above).  simple:    out = (x + sum_nb x_nb) / (1 + deg)
// laplacian: w = 1 / (sqrt((dx dx + dy dy) + dz dz) + eps) of p - p_nb, W = sum w, S = sum w x_nb,
//            out = x + lam (S / W - x); a vertex without neighbours keeps x.
// Every sum runs left to right from zero, each weight is computed once and applied to every field.
D2PC_HD void smooth_vertex(const SmoothSrc &src, uint32_t i, const uint32_t *nb, uint32_t deg, bool laplacian,
                           double lam, uint32_t fields, double out[3][3]) {
  double x[3][3], s[3][3];
  for (int f = 0; f < 3; ++f) {
    s[f][0] = s[f][1] = s[f][2] = 0.0;
    if ((fields >> f) & 1u) smooth_load(src, f, i, x[f]);
  }
  double p[3];
  if (laplacian) smooth_load(src, 0, i, p);
  double W = 0.0;
  for (uint32_t k = 0; k < deg; ++k) {
    const uint32_t j = nb[k];
    double w = 1.0;
    if (laplacian) {
      double q[3];
      smooth_load(src, 0, j, q);
      const double dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
      w = 1.0 / (sqrt((dx * dx + dy * dy) + dz * dz) + kSmoothEps);
      W += w;
    }
    for (int f = 0; f < 3; ++f) {
      if (!((fields >> f) & 1u)) continue;
      double y[3];
      smooth_load(src, f, j, y);
      if (laplacian) {
        s[f][0] += w * y[0]; s[f][1] += w * y[1]; s[f][2] += w * y[2];
      } else {
        s[f][0] += y[0]; s[f][1] += y[1]; s[f][2] += y[2];
      }
    }
  }
  for (int f = 0; f < 3; ++f) {
    if (!((fields >> f) & 1u)) continue;
    for (int c = 0; c < 3; ++c) {
      if (!laplacian) out[f][c] = (x[f][c] + s[f][c]) / (double)(1u + deg);
      else out[f][c] = deg == 0 ? x[f][c] : x[f][c] + lam * (s[f][c] / W - x[f][c]);
    }
  }
}

// Unnormalised n = (p1 - p0) x (p2 - p0) of a triangle from its float32 corners as float64 (Eigen's cross)
D2PC_HD void smooth_tri_normal(const float *xyz, int32_t a, int32_t b, int32_t c, double n[3]) {
  double p[3][3];
  const int32_t v[3] = {a, b, c};
  for (int k = 0; k < 3; ++k)
    for (int d = 0; d < 3; ++d) p[k][d] = (double)xyz[3 * (size_t)v[k] + d];
  const double u0 = p[1][0] - p[0][0], u1 = p[1][1] - p[0][1], u2 = p[1][2] - p[0][2];
  const double w0 = p[2][0] - p[0][0], w1 = p[2][1] - p[0][1], w2 = p[2][2] - p[0][2];
  n[0] = u1 * w2 - u2 * w1;
  n[1] = u2 * w0 - u0 * w2;
  n[2] = u0 * w1 - u1 * w0;
}

// Normal of a vertex whose incident triangles are tri[0 .. n) (ascending, once per corner): their normals tn [T][3]
// summed from zero in that order, then v / sqrt(v.v), (0, 0, 1) for a zero sum
D2PC_HD void smooth_vertex_normal(const uint32_t *tri, uint32_t n, const double *tn, double out[3]) {
  double a0 = 0.0, a1 = 0.0, a2 = 0.0;
  for (uint32_t k = 0; k < n; ++k) {
    const size_t b = 3 * (size_t)tri[k];
    a0 += tn[b]; a1 += tn[b + 1]; a2 += tn[b + 2];
  }
  const double ss = a0 * a0 + a1 * a1 + a2 * a2;
  if (ss == 0.0) {
    out[0] = 0.0; out[1] = 0.0; out[2] = 1.0;
    return;
  }
  const double len = sqrt(ss);
  out[0] = a0 / len; out[1] = a1 / len; out[2] = a2 / len;
}

}  // namespace d2pc

#endif  // D2PC_SMOOTH_H_
