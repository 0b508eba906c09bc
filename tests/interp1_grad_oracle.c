/* interp1_grad_oracle.c — CPU oracle for the derivatives of interp1 (b200_interp1_grad and b200_interp1_adjoint).
 * TEST INFRASTRUCTURE ONLY, compiled by tests/test_interp1_grad.py with the flags of oracle/Makefile
 * (-ffp-contract=off: every operation rounded once).  It reuses the value oracle's bracket rule
 * (oracle/interp_oracle_impl.inc) and restates the derivative rules of include/b200_interp.h:
 *
 *   gradient  yi = the value oracle's;  a NaN query -> dydx = NaN;  else out of range -> +0;
 *             else dydx = (Y[b'] - Y[a']) / (X[b'] - X[a']) on (a', b') = (a, a+1), (n-2, n-1) on the last knot.
 *   adjoint   the terms (1-w)*g[k] at node a (role 0) and w*g[k] at node b (role 1) of every query in range, listed
 *             per node in ascending (segment a, k, role) order (here: a stable counting sort by segment), and each
 *             node's list summed by the blocked sum R with B = B200_INTERP1_ADJOINT_BLOCK (blocked_sum below). */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include "../include/b200_interp.h"
#include "../oracle/oracle.h"

#define ADJ_B ((size_t)B200_INTERP1_ADJOINT_BLOCK)

static int oracle_interp2_yfirst = 0;   /* read by the included interp2 value oracle, unused here */

size_t grad1_oracle_block(void) { return ADJ_B; }

#define GRAD1_BODY                                                                                                  \
  int SUFFIX(grad1_oracle)(const REAL* x, const REAL* y, size_t n, const REAL* xi, size_t ni, REAL* yi, REAL* dydx,  \
                           REAL extrap) {                                                                           \
    int rc = SUFFIX(oracle_interp1)(x, y, n, xi, ni, yi, NULL, extrap, 0, 1);                                       \
    if (rc) return rc;                                                                                              \
    for (size_t k = 0; k < ni; ++k) {                                                                               \
      SUFFIX(bw) b = SUFFIX(bracket_weight)(x, n, xi[k]);                                                           \
      if (b.is_nan) { dydx[k] = REAL_NAN; continue; }                                                               \
      if (!b.in_range) { dydx[k] = (REAL)0; continue; }                                                             \
      size_t a0 = b.a == n - 1 ? n - 2 : b.a;                                                                       \
      REAL dy = y[a0 + 1] - y[a0], dx = x[a0 + 1] - x[a0];                                                          \
      dydx[k] = dy / dx;                                                                                            \
    }                                                                                                               \
    return 0;                                                                                                       \
  }                                                                                                                 \
  /* R: at most B items -> +0, then left to right; more -> R of the sums of consecutive blocks of B items */        \
  static REAL SUFFIX(blocked_sum)(const REAL* t, size_t len) {                                                      \
    if (len <= ADJ_B) {                                                                                             \
      REAL acc = (REAL)0;                                                                                           \
      for (size_t i = 0; i < len; ++i) acc = acc + t[i];                                                            \
      return acc;                                                                                                   \
    }                                                                                                               \
    size_t nb = (len + ADJ_B - 1) / ADJ_B;                                                                          \
    REAL* s = (REAL*)malloc(nb * sizeof(REAL));                                                                     \
    for (size_t b = 0; b < nb; ++b)                                                                                 \
      s[b] = SUFFIX(blocked_sum)(t + b * ADJ_B, (b + 1) * ADJ_B <= len ? ADJ_B : len - b * ADJ_B);                   \
    REAL r = SUFFIX(blocked_sum)(s, nb);                                                                            \
    free(s);                                                                                                        \
    return r;                                                                                                       \
  }                                                                                                                 \
  int SUFFIX(adj1_oracle)(const REAL* x, size_t n, const REAL* xi, const REAL* g, size_t ni, REAL* G) {             \
    int rc;                                                                                                         \
    if ((rc = SUFFIX(check_axis)(x, n))) return rc;                                                                 \
    size_t* key = (size_t*)malloc((ni ? ni : 1) * sizeof(size_t));                                                 \
    size_t* start = (size_t*)calloc(n + 1, sizeof(size_t));                                                         \
    size_t* order = (size_t*)malloc((ni ? ni : 1) * sizeof(size_t));                                               \
    size_t* len = (size_t*)calloc(n + 1, sizeof(size_t));                                                           \
    REAL* terms = (REAL*)malloc((2 * ni + 1) * sizeof(REAL));                                                       \
    if (!key || !start || !order || !len || !terms) {                                                               \
      free(key); free(start); free(order); free(len); free(terms); return -2;                                       \
    }                                                                                                               \
    for (size_t k = 0; k < ni; ++k) {                                                                               \
      SUFFIX(bw) b = SUFFIX(bracket_weight)(x, n, xi[k]);                                                           \
      key[k] = b.in_range ? b.a : n;                                                                                \
      if (key[k] < n) { start[key[k] + 1]++; len[b.a]++; len[b.b]++; }                                              \
    }                                                                                                               \
    for (size_t c = 0; c < n; ++c) start[c + 1] += start[c];                                                        \
    for (size_t k = 0; k < ni; ++k)                                                                                 \
      if (key[k] < n) order[start[key[k]]++] = k; /* stable: k ascending within a segment */                        \
    size_t nin = n ? start[n - 1] : 0;                                                                              \
    /* node j's list begins at the sum of the lengths before it; fill in (segment, k, role) order */                \
    size_t* pos = (size_t*)calloc(n + 1, sizeof(size_t));                                                           \
    for (size_t j = 0; j < n; ++j) pos[j + 1] = pos[j] + len[j];                                                    \
    size_t* fill = (size_t*)malloc((n + 1) * sizeof(size_t));                                                       \
    for (size_t j = 0; j <= n; ++j) fill[j] = pos[j];                                                               \
    for (size_t s = 0; s < nin; ++s) {                                                                              \
      size_t k = order[s];                                                                                          \
      SUFFIX(bw) b = SUFFIX(bracket_weight)(x, n, xi[k]);                                                           \
      REAL t0 = ((REAL)1 - b.w) * g[k], t1 = b.w * g[k];                                                            \
      terms[fill[b.a]++] = t0;                                                                                      \
      terms[fill[b.b]++] = t1;                                                                                      \
    }                                                                                                               \
    for (size_t j = 0; j < n; ++j) G[j] = SUFFIX(blocked_sum)(terms + pos[j], len[j]);                              \
    free(key); free(start); free(order); free(len); free(terms); free(pos); free(fill);                             \
    return 0;                                                                                                       \
  }

#define REAL double
#define SUFFIX(name) name##_f64
#define REAL_NAN ((double)NAN)
#define REAL_INF ((double)INFINITY)
#include "../oracle/interp_oracle_impl.inc"
GRAD1_BODY
#undef REAL
#undef SUFFIX
#undef REAL_NAN
#undef REAL_INF

#define REAL float
#define SUFFIX(name) name##_f32
#define REAL_NAN ((float)NAN)
#define REAL_INF ((float)INFINITY)
#include "../oracle/interp_oracle_impl.inc"
GRAD1_BODY
#undef REAL
#undef SUFFIX
#undef REAL_NAN
#undef REAL_INF
