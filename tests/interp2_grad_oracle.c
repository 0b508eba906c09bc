/* interp2_grad_oracle.c — CPU oracle for the derivatives of scattered interp2 (b200_interp2_scattered_grad and
 * b200_interp2_scattered_adjoint).  TEST INFRASTRUCTURE ONLY, compiled by tests/test_interp2_grad.py with the flags of
 * oracle/Makefile (-ffp-contract=off: every operation rounded once).  It reuses the value oracle's bracket rule and
 * two-pass value (oracle/interp_oracle_impl.inc) and restates the derivative rules of include/b200_interp.h:
 *
 *   gradient  zq = the value oracle's;  a NaN coordinate -> dzdx = dzdy = NaN;  else out of range -> +0, +0;
 *             else dzdx = ((1-wy)*(Z(ay,bx) - Z(ay,ax)) + wy*(Z(by,bx) - Z(by,ax))) / (X[bx] - X[ax]), dzdy mirrored,
 *             with the cell (n-2, n-1) along an axis whose bracket is the last knot (a == b).
 *   adjoint   G(i,j) = +0, then the terms c*g[k] (c00 = (1-wx)(1-wy) at (ay,ax), c10 = (1-wx)wy at (by,ax),
 *             c01 = wx(1-wy) at (ay,bx), c11 = wx wy at (by,bx)) of every query in range, added one at a time in
 *             ascending (cell key ax*ny + ay, k, role) order: here a stable counting sort by cell key. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include "../oracle/oracle.h"

static int oracle_interp2_yfirst = 0;
void grad_oracle_set_order(int y_first) { oracle_interp2_yfirst = y_first ? 1 : 0; }

#define GRAD_BODY                                                                                                   \
  static REAL SUFFIX(slope)(REAL w, REAL a0, REAL a1, REAL b0, REAL b1, REAL k0, REAL k1) {                         \
    REAL omw = (REAL)1 - w;                                                                                         \
    REAL da = a1 - a0, db = b1 - b0;                                                                                \
    REAL pa = omw * da, pb = w * db;                                                                                \
    REAL s = pa + pb;                                                                                               \
    REAL dk = k1 - k0;                                                                                              \
    return s / dk;                                                                                                  \
  }                                                                                                                 \
  int SUFFIX(grad_oracle_scattered)(const REAL* x, size_t nx, const REAL* y, size_t ny, const REAL* z,             \
                                    const REAL* xq, const REAL* yq, size_t nq, REAL* zq, REAL* dzdx, REAL* dzdy,     \
                                    REAL extrap) {                                                                  \
    int rc;                                                                                                         \
    if ((rc = SUFFIX(check_axis)(x, nx))) return rc;                                                                \
    if ((rc = SUFFIX(check_axis)(y, ny))) return rc;                                                                \
    for (size_t k = 0; k < nq; ++k) {                                                                               \
      SUFFIX(bw) bx = SUFFIX(bracket_weight)(x, nx, xq[k]);                                                         \
      SUFFIX(bw) by = SUFFIX(bracket_weight)(y, ny, yq[k]);                                                         \
      zq[k] = SUFFIX(two_pass)(z, ny, bx, by, extrap, oracle_interp2_yfirst);                                       \
      if (bx.is_nan || by.is_nan) { dzdx[k] = dzdy[k] = REAL_NAN; continue; }                                       \
      if (!bx.in_range || !by.in_range) { dzdx[k] = dzdy[k] = (REAL)0; continue; }                                  \
      size_t x0 = bx.a == bx.b ? nx - 2 : bx.a, x1 = x0 + 1;                                                        \
      size_t y0 = by.a == by.b ? ny - 2 : by.a, y1 = y0 + 1;                                                        \
      dzdx[k] = SUFFIX(slope)(by.w, z[x0 * ny + by.a], z[x1 * ny + by.a], z[x0 * ny + by.b], z[x1 * ny + by.b],     \
                              x[x0], x[x1]);                                                                        \
      dzdy[k] = SUFFIX(slope)(bx.w, z[bx.a * ny + y0], z[bx.a * ny + y1], z[bx.b * ny + y0], z[bx.b * ny + y1],     \
                              y[y0], y[y1]);                                                                        \
    }                                                                                                               \
    return 0;                                                                                                       \
  }                                                                                                                 \
  int SUFFIX(grad_oracle_adjoint)(const REAL* x, size_t nx, const REAL* y, size_t ny, const REAL* xq,              \
                                  const REAL* yq, const REAL* g, size_t nq, REAL* G) {                              \
    int rc;                                                                                                         \
    if ((rc = SUFFIX(check_axis)(x, nx))) return rc;                                                                \
    if ((rc = SUFFIX(check_axis)(y, ny))) return rc;                                                                \
    size_t ncells = nx * ny;                                                                                        \
    size_t* key = (size_t*)malloc((nq ? nq : 1) * sizeof(size_t));                                                  \
    size_t* start = (size_t*)calloc(ncells + 1, sizeof(size_t));                                                    \
    size_t* order = (size_t*)malloc((nq ? nq : 1) * sizeof(size_t));                                                \
    if (!key || !start || !order) { free(key); free(start); free(order); return -2; }                               \
    for (size_t k = 0; k < nq; ++k) {                                                                               \
      SUFFIX(bw) bx = SUFFIX(bracket_weight)(x, nx, xq[k]);                                                         \
      SUFFIX(bw) by = SUFFIX(bracket_weight)(y, ny, yq[k]);                                                         \
      key[k] = (bx.in_range && by.in_range) ? bx.a * ny + by.a : ncells;                                            \
      if (key[k] < ncells) start[key[k] + 1]++;                                                                     \
    }                                                                                                               \
    for (size_t c = 0; c < ncells; ++c) start[c + 1] += start[c];                                                   \
    for (size_t k = 0; k < nq; ++k)                                                                                 \
      if (key[k] < ncells) order[start[key[k]]++] = k; /* stable: k ascending within a cell */                      \
    for (size_t i = 0; i < ncells; ++i) G[i] = (REAL)0;                                                             \
    for (size_t s = 0; s < (ncells ? start[ncells - 1] : 0); ++s) {                                                 \
      size_t k = order[s];                                                                                          \
      SUFFIX(bw) bx = SUFFIX(bracket_weight)(x, nx, xq[k]);                                                         \
      SUFFIX(bw) by = SUFFIX(bracket_weight)(y, ny, yq[k]);                                                         \
      REAL omx = (REAL)1 - bx.w, omy = (REAL)1 - by.w;                                                              \
      REAL c00 = omx * omy, c10 = omx * by.w, c01 = bx.w * omy, c11 = bx.w * by.w;                                  \
      REAL t00 = c00 * g[k], t10 = c10 * g[k], t01 = c01 * g[k], t11 = c11 * g[k];                                  \
      /* sorted by cell, so each node receives its terms in (cell key, k, role) order */                            \
      G[bx.a * ny + by.a] += t00;                                                                                   \
      G[bx.a * ny + by.b] += t10;                                                                                   \
      G[bx.b * ny + by.a] += t01;                                                                                   \
      G[bx.b * ny + by.b] += t11;                                                                                   \
    }                                                                                                               \
    free(key); free(start); free(order);                                                                            \
    return 0;                                                                                                       \
  }

#define REAL double
#define SUFFIX(name) name##_f64
#define REAL_NAN ((double)NAN)
#define REAL_INF ((double)INFINITY)
#include "../oracle/interp_oracle_impl.inc"
GRAD_BODY
#undef REAL
#undef SUFFIX
#undef REAL_NAN
#undef REAL_INF

#define REAL float
#define SUFFIX(name) name##_f32
#define REAL_NAN ((float)NAN)
#define REAL_INF ((float)INFINITY)
#include "../oracle/interp_oracle_impl.inc"
GRAD_BODY
#undef REAL
#undef SUFFIX
#undef REAL_NAN
#undef REAL_INF
