/*
 * mc_oracle.c — CPU restatement of batched marching cubes (genre_b200_iso_surface_count / _emit).  TEST
 * INFRASTRUCTURE ONLY: loaded by tests/, __graft_entry__.smoke() and profiles/microbench_mesh.py, never by the
 * product.  Built with -ffp-contract=off, so every fp32 operation rounds once, as the kernels' __f*_rn do.
 *
 * One [D][H][W] volume at a time, with the case table of genre_shapehd_b200/csrc/mc_table.h and the order and
 * rounding of genre_b200_iso_surface_emit (include/genre_b200.h).  A straight per-point / per-cell loop with an
 * index volume (not the kernels' popc prefixes): vertices in C order of their owner point, then by axis; faces in
 * C order of the cell, then by table order.  The table itself is checked separately, by the mesh-property tests
 * of tests/test_iso_surface_cpu.py, so sharing it here does not hide table bugs.
 */
#include <math.h>
#include <stdint.h>

#include "../genre_shapehd_b200/csrc/mc_table.h"

#define ORACLE_API __attribute__((visibility("default")))

static inline int mc_in(const float *vol, long D, long H, long W, long i, long j, long k, float level) {
  (void)D;
  return vol[(i * H + j) * W + k] > level; /* NaN: 0 */
}

static inline int mc_crossed(const float *vol, long D, long H, long W, long i, long j, long k, int a, float level) {
  long q[3] = {i, j, k};
  const long n[3] = {D, H, W};
  if (q[a] + 1 >= n[a]) return 0;
  q[a] += 1;
  return mc_in(vol, D, H, W, i, j, k, level) != mc_in(vol, D, H, W, q[0], q[1], q[2], level);
}

static long mc_cell_case(const float *vol, long D, long H, long W, long i, long j, long k, float level) {
  long cs = 0;
  for (int c = 0; c < 8; ++c)
    cs |= (long)mc_in(vol, D, H, W, i + ((c >> 2) & 1), j + ((c >> 1) & 1), k + (c & 1), level) << c;
  return cs;
}

/* -> number of vertices and of triangles */
ORACLE_API void oracle_iso_surface_count(const float *vol, long D, long H, long W, float level, long *nv, long *nf) {
  long v = 0, f = 0;
  for (long i = 0; i < D; ++i)
    for (long j = 0; j < H; ++j)
      for (long k = 0; k < W; ++k)
        for (int a = 0; a < 3; ++a) v += mc_crossed(vol, D, H, W, i, j, k, a, level);
  for (long i = 0; i + 1 < D; ++i)
    for (long j = 0; j + 1 < H; ++j)
      for (long k = 0; k + 1 < W; ++k) f += mc_ntri[mc_cell_case(vol, D, H, W, i, j, k, level)];
  *nv = v;
  *nf = f;
}

/* verts [nv][3], faces [nf][3] (0-based), values [nv] or NULL; idx: scratch of D*H*W*3 int32 */
ORACLE_API void oracle_iso_surface(const float *vol, long D, long H, long W, float level, const float *spacing,
                                   const float *offset, float *verts, int32_t *faces, float *values, int32_t *idx) {
  int32_t nv = 0;
  long nf = 0;
  for (long i = 0; i < D; ++i)
    for (long j = 0; j < H; ++j)
      for (long k = 0; k < W; ++k)
        for (int a = 0; a < 3; ++a) {
          int32_t *slot = &idx[((i * H + j) * W + k) * 3 + a];
          *slot = -1;
          if (!mc_crossed(vol, D, H, W, i, j, k, a, level)) continue;
          const long p[3] = {i, j, k};
          long q[3] = {i, j, k};
          q[a] += 1;
          const float f0 = vol[(p[0] * H + p[1]) * W + p[2]];
          const float f1 = vol[(q[0] * H + q[1]) * W + q[2]];
          const float num = level - f0, den = f1 - f0;
          const float t = num / den;
          for (int b = 0; b < 3; ++b) {
            float c;
            if (b == a) {
              const float pt = (float)p[b] + t;
              const float ps = pt * spacing[b];
              c = ps + offset[b];
            } else {
              const float ps = (float)p[b] * spacing[b];
              c = ps + offset[b];
            }
            verts[(long)nv * 3 + b] = c;
          }
          if (values) values[nv] = fmaxf(f0, f1);
          *slot = nv++;
        }
  for (long i = 0; i + 1 < D; ++i)
    for (long j = 0; j + 1 < H; ++j)
      for (long k = 0; k + 1 < W; ++k) {
        const long cs = mc_cell_case(vol, D, H, W, i, j, k, level);
        for (int t = 0; t < mc_ntri[cs]; ++t)
          for (int c = 0; c < 3; ++c) {
            /* edge e: axis e / 4, owner offset along the other two axes (in increasing order) = ((e % 4) >> 1, e & 1) */
            const int e = mc_tri[cs][3 * t + c], a = e / 4, r = e % 4;
            long o[3] = {0, 0, 0};
            const int b0 = a == 0 ? 1 : 0, b1 = a == 2 ? 1 : 2;
            o[b0] = r >> 1;
            o[b1] = r & 1;
            faces[(nf + t) * 3 + c] = idx[(((i + o[0]) * H + (j + o[1])) * W + (k + o[2])) * 3 + a];
          }
        nf += mc_ntri[cs];
      }
}
