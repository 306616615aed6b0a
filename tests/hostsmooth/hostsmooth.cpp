// TEST HARNESS (not product, not oracle): compiles the product's per-vertex arithmetic
// image_to_pointcloud_b200/csrc/d2pc_smooth.h for the host and drives it in the pass order of
// d2pc_mesh_smooth_enqueue (the first pass reads the inputs, every pass writes a fresh float64 state, the last one is
// rounded to the float32 outputs) over an adjacency given by the caller.  The result must equal the oracle's.
#include <cstdint>
#include <vector>

#include "../../image_to_pointcloud_b200/csrc/d2pc_smooth.h"

using namespace d2pc;

extern "C" {

// fields: bit 0 positions, 1 normals, 2 colours (nrm may be NULL without bit 1); lams[passes]: the lambda of every
// pass (laplacian != 0) or ignored (simple).  Outputs are written only for the filtered fields.
void hs_smooth(const float *xyz, const float *rgb, const double *nrm, uint32_t V, const uint32_t *off,
               const uint32_t *nbr, int laplacian, const double *lams, uint32_t passes, uint32_t fields,
               float *oxyz, float *orgb, double *onrm) {
  std::vector<double> st[2][3];
  for (auto &b : st)
    for (auto &f : b) f.assign(3 * (size_t)V, 0.0);
  for (uint32_t p = 0; p < passes; ++p) {
    SmoothSrc src{{nullptr, nullptr, nullptr}, xyz, rgb, nrm};
    for (int f = 0; f < 3; ++f)
      if (p > 0 && ((fields >> f) & 1u)) src.state[f] = st[(p - 1) & 1u][f].data();
    const bool last = p + 1 == passes;
    for (uint32_t i = 0; i < V; ++i) {
      double out[3][3];
      smooth_vertex(src, i, nbr + off[i], off[i + 1] - off[i], laplacian != 0, lams[p], fields, out);
      for (int f = 0; f < 3; ++f) {
        if (!((fields >> f) & 1u)) continue;
        for (int c = 0; c < 3; ++c) {
          const size_t o = 3 * (size_t)i + c;
          if (!last) st[p & 1u][f][o] = out[f][c];
          else if (f == 0) oxyz[o] = (float)out[f][c];
          else if (f == 2) orgb[o] = (float)out[f][c];
          else onrm[o] = out[f][c];
        }
      }
    }
  }
}

// vertex normals over an incidence CSR (off [V + 1], tri: the triangles of every vertex in ascending order)
void hs_normals(const float *xyz, uint32_t V, const int32_t *t, uint32_t T, const uint32_t *off, const uint32_t *tri,
                double *out) {
  std::vector<double> tn(3 * (size_t)T);
  for (uint32_t k = 0; k < T; ++k) smooth_tri_normal(xyz, t[3 * k], t[3 * k + 1], t[3 * k + 2], tn.data() + 3 * k);
  for (uint32_t i = 0; i < V; ++i) smooth_vertex_normal(tri + off[i], off[i + 1] - off[i], tn.data(), out + 3 * i);
}

}  // extern "C"
