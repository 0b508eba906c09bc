/* b200_interp.h — C-ABI of the batched 1-D / 2-D linear interpolation path.
 *
 * What it replaces.  BASELINE.json configs 1-2 name `arma::interp1` / `arma::interp2`
 * (Armadillo, a third-party dependency of the reference that is NOT vendored under
 * /root/reference and not pinned: Makefile:5 links `-larmadillo`; the author's binary
 * linked libarmadillo.6, Driver.o.dep:554 lists fn_interp1.hpp).  The reference itself
 * has no interp1/interp2 call site; its own "linear interpolation" is the uniform-grid
 * bracket scan of EventDrivenMap.cu:361-372 and the two-point blend of
 * EventDrivenMap.cu:779-783.  The entry points below are what a host program that
 * today calls
 *
 *     arma::interp1(X, Y, XI, YI, "*linear", extrap);        // fn_interp1.hpp
 *     arma::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap);  // fn_interp2.hpp (>= 10.x)
 *
 * binds instead.  Semantics follow Armadillo's published algorithm (restated with
 * citations in oracle/interp_oracle.c): per query, lower bracket a = last knot <= xi,
 * b = min(a+1, n-1), w = |X[a]-xi| / (|X[a]-xi| + |X[b]-xi|) (0 when the query hits a
 * knot), value = (1-w)*Y[a] + w*Y[b] with every operation individually rounded (no FMA
 * contraction); queries outside [X[0], X[n-1]] give `extrap_val`; NaN queries give NaN.
 * Results are bit-identical to that restatement; bracket indices are exact.
 *
 * Knots must be strictly ascending ("*linear": Armadillo's own sort/unique pre-pass of
 * the default "linear" method is not part of the hot path and is not reproduced;
 * B200_ERR_NOT_SORTED is returned instead).  Queries may be in ANY order: the result
 * of each query does not depend on the others, so Armadillo's sort/unsort of XI
 * (fn_interp1.hpp) is a no-op on values and is skipped.
 *
 * Layout: vectors are contiguous; matrices are column-major (arma::mat), Z is
 * ny rows x nx columns, ZI is nyi rows x nxi columns.
 */
#ifndef B200_INTERP_H
#define B200_INTERP_H

#include "b200_common.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { B200_F64 = 0, B200_F32 = 1 } b200_dtype;

typedef struct b200_interp1_plan b200_interp1_plan;   /* grid X,Y resident in HBM */
typedef struct b200_interp2_plan b200_interp2_plan;   /* grid X,Y,Z resident in HBM */

/* ---- one-shot calls, host buffers (the drop-in for the arma:: free functions) ---- */

/* arma::interp1(X,Y,XI,YI,"*linear",extrap) for arma::vec.  idx_out (nullable) receives
 * the lower bracket index a of each query, or -1 where the query is out of range/NaN. */
int b200_interp1_f64(const double* xg, const double* yg, size_t ng,
                     const double* xi, size_t ni, double* yi, int32_t* idx_out,
                     double extrap_val);
/* Same for arma::fvec. */
int b200_interp1_f32(const float* xg, const float* yg, size_t ng,
                     const float* xi, size_t ni, float* yi, int32_t* idx_out,
                     float extrap_val);

/* arma::interp2(X,Y,Z,XI,YI,ZI,"linear",extrap): XI (nxi) and YI (nyi) define a tensor
 * grid; ZI is nyi x nxi column-major.  X.n_elem == Z.n_cols == nx, Y.n_elem == Z.n_rows == ny. */
int b200_interp2_f64(const double* x, size_t nx, const double* y, size_t ny, const double* z,
                     const double* xi, size_t nxi, const double* yi, size_t nyi,
                     double* zi, double extrap_val);
int b200_interp2_f32(const float* x, size_t nx, const float* y, size_t ny, const float* z,
                     const float* xi, size_t nxi, const float* yi, size_t nyi,
                     float* zi, float extrap_val);

/* ---- plans: upload the grid once, interpolate many query batches ---- */

/* dtype selects double/float for every buffer of the plan (void* below). */
int b200_interp1_plan_create(b200_dtype dtype, const void* xg, const void* yg, size_t ng,
                             b200_interp1_plan** plan);
/* Replace the values Y on the same knots (a new coarse profile on an unchanged grid).  Host buffer; runs on the
 * plan's internal stream and returns when the plan holds the new values. */
int b200_interp1_plan_set_values(b200_interp1_plan* plan, const void* yg);
/* Same from device memory (ng contiguous values of the plan's dtype), ordered on `stream`: no allocation, no host
 * synchronisation, graph-capturable.  Work of this plan queued earlier on the same stream sees the old values, later
 * work the new.  As for every call of a plan, the caller must not have work of the same plan in flight on another
 * stream.  Results are bit-identical to those of a plan created with the new values. */
int b200_interp1_plan_set_values_dev(b200_interp1_plan* plan, const void* yg_dev, void* stream);
int b200_interp1_plan_destroy(b200_interp1_plan* plan);

/* Host-buffer execution: H2D of xi, kernel, D2H of yi (and idx) inside the call, chunked
 * and overlapped on internal streams; fastest with b200_host_alloc'ed buffers. */
int b200_interp1_exec(b200_interp1_plan* plan, const void* xi, size_t ni, void* yi,
                      int32_t* idx_out, double extrap_val);
/* Device-buffer execution on `stream` (queries/outputs already resident in HBM). */
int b200_interp1_exec_dev(b200_interp1_plan* plan, const void* xi_dev, size_t ni,
                          void* yi_dev, int32_t* idx_dev, double extrap_val, void* stream);

/* Derivatives of interp1.  Notation: a is the value call's lower bracket, b = min(a+1, n-1), w its weight; every
 * operation is rounded once.
 * Gradient: yi exactly as b200_interp1_exec gives it, plus the slope of the piecewise-linear interpolant,
 *   dydx = (Y[b'] - Y[a']) / (X[b'] - X[a'])  on the segment (a', b') = (a, a+1);
 * on the last knot (a == n-1) the segment is (n-2, n-1), from the left; on an interior knot it is the segment to the
 * right.  A NaN query gives a NaN slope; any other out-of-range query (+-inf included) gives +0.  NaN / inf in Y
 * propagate as IEEE arithmetic gives (the 1-D form of the interp2 rule).
 * The _dev call is ordered on `stream`, allocates nothing and never synchronises the host (graph-capturable); the host
 * call is synchronous. */
int b200_interp1_grad(b200_interp1_plan* plan, const void* xi, size_t ni, void* yi, void* dydx, double extrap_val);
int b200_interp1_grad_dev(b200_interp1_plan* plan, const void* xi_dev, size_t ni, void* yi_dev, void* dydx_dev,
                          double extrap_val, void* stream);
/* Adjoint onto the values: G = W^T g, the gradient of sum_k g[k]*yi[k] with respect to Y.  Only queries inside
 * [X[0], X[n-1]] and not NaN contribute, each with two terms: (1-w)*g[k] at node a (role 0) and w*g[k] at node b
 * (role 1); a zero coefficient still makes a term (0 * inf = NaN).  S_j, the terms of node j in ascending
 * (segment a, query index k, role) order, is summed by the blocked sum R with B = B200_INTERP1_ADJOINT_BLOCK:
 *   R(empty) = +0;  a list of at most B terms: +0, then the terms added left to right;
 *   a longer list: cut into consecutive blocks of B terms counted from its start, each block reduced by R, then R of
 *   the list of block sums.
 * So a node with at most B terms gets exactly the one-at-a-time bits of the interp2 adjoint, and a heavily loaded node
 * (1e8 queries on 1e3 knots) is summed in parallel.  The bits depend only on X, the queries, g and B — not on the
 * launch, the stream or graph replay.  Because the order spans the whole batch, splitting a batch into several calls
 * and summing changes the bits: pass all queries in one call (ni <= 2^31-1).
 * G_dev receives all ng values, contiguous.  Scratch is the caller's `workspace` of at least the queried size, so the
 * _dev call allocates nothing, never synchronises the host and can be captured into a graph.  Cost: a radix sort of the
 * segment keys plus a few streaming passes.  NULL pointers, a short workspace or ni > 2^31-1 give B200_ERR_INVALID_ARG
 * before any device work. */
#define B200_INTERP1_ADJOINT_BLOCK 256
int b200_interp1_adjoint_workspace(const b200_interp1_plan* plan, size_t ni, size_t* bytes);
int b200_interp1_adjoint_dev(b200_interp1_plan* plan, const void* xi_dev, const void* g_dev, size_t ni, void* G_dev,
                             void* workspace, size_t workspace_bytes, void* stream);
/* Host buffers (G: ng values): allocates, runs on the plan's internal stream, synchronous. */
int b200_interp1_adjoint(b200_interp1_plan* plan, const void* xi, const void* g, size_t ni, void* G);

int b200_interp2_plan_create(b200_dtype dtype, const void* x, size_t nx, const void* y,
                             size_t ny, const void* z, b200_interp2_plan** plan);
/* Same, with layout flags.  By default the plan also builds one 2x2 corner record per grid cell
 * (4x the memory of Z) when that pays (records L2 resident, or Z too large for L2 anyway), so
 * that a scattered query costs one 32-byte sector gather instead of 2-4;
 * B200_INTERP2_NO_CELLS keeps only the column-major matrix, B200_INTERP2_FORCE_CELLS always builds them. */
#define B200_INTERP2_NO_CELLS 1u
#define B200_INTERP2_FORCE_CELLS 2u
/* Opt-in L2-banded pipeline: with B200_INTERP2_FORCE_BANDS the plan builds the corner records and every
 * device-buffer scattered call first partitions the queries by column band of the records (<= 32 MiB
 * per band) so that every record gather hits L2 (four streaming passes instead of one 128-byte DRAM line
 * fill per query; same bits).  Grids too narrow for two bands, and plans with B200_INTERP2_NO_BANDS, take
 * the direct kernels.  Its scratch (26 B per query, f64) lives in the plan: as with the grid call, one
 * plan must not run on two streams at once. */
#define B200_INTERP2_NO_BANDS 4u
#define B200_INTERP2_FORCE_BANDS 8u
/* f64 matrices of more than 12 and less than 180 MiB are stored as overlapping 4x4 tiles (stride 3; 16/9
 * the memory of Z) instead of corner records: the four corners of any cell then sit in ONE 128-byte line
 * of a table less than half the size of the corner records, and scattered queries — bounded on B200 by
 * DRAM row activations, one per L2 miss — miss L2 correspondingly less often.  Same bits.  NO_TILES /
 * FORCE_TILES override; NO_CELLS / FORCE_CELLS without FORCE_TILES build no tiles. */
#define B200_INTERP2_NO_TILES 16u
#define B200_INTERP2_FORCE_TILES 32u
/* Order of Armadillo's two separable passes.  Default: along X first (whole columns of Z blended into
 * tmp = Y.n_elem x XI.n_elem), then along Y — fn_interp2.hpp as recalled by two independent readers; Armadillo is
 * not installed, so this is unverified.  B200_INTERP2_ORDER_YX selects the mirrored order (along Y first, then X),
 * which round 1 shipped.  The two differ by rounding only, and in which coordinate decides extrap_val / NaN when
 * one query coordinate is NaN and the other out of range (the LAST pass wins). */
#define B200_INTERP2_ORDER_YX 64u
int b200_interp2_plan_create_ex(b200_dtype dtype, const void* x, size_t nx, const void* y,
                                size_t ny, const void* z, unsigned flags, b200_interp2_plan** plan);
/* Replace Z (ny x nx) on the same axes: a field that changes while its grid stays fixed.  The plan rebuilds its
 * column-major Z and its scattered-query table (corner records or tiles) from the new values; the layout, the axis
 * tables and the pass order chosen at creation stay.  Results are bit-identical to those of a plan created with the
 * new Z (NaN and +-inf values are accepted, as at creation).
 * Host buffer, column-major (arma::mat): synchronous, like plan creation (runs on the plan's internal stream). */
int b200_interp2_plan_set_values(b200_interp2_plan* plan, const void* z);
/* Same from device memory, ordered on `stream`: no allocation, no host synchronisation, graph-capturable; work of
 * this plan queued earlier on the same stream sees the old values, later work the new.  row_major == 0: element
 * (i, j) at j*ld + i, ld >= ny (arma::mat, or a column block of a larger one); row_major != 0: at i*ld + j, ld >= nx
 * (a C-contiguous torch tensor of shape (ny, nx), or a row slice of a larger one).  ld below its minimum gives
 * B200_ERR_INVALID_ARG.  The caller must not have work of the same plan in flight on another stream. */
int b200_interp2_plan_set_values_dev(b200_interp2_plan* plan, const void* z_dev, size_t ld, int row_major,
                                     void* stream);
int b200_interp2_plan_destroy(b200_interp2_plan* plan);

/* Tensor-grid queries (Armadillo's interp2 API shape). */
int b200_interp2_grid(b200_interp2_plan* plan, const void* xi, size_t nxi, const void* yi,
                      size_t nyi, void* zi, double extrap_val);
int b200_interp2_grid_dev(b200_interp2_plan* plan, const void* xi_dev, size_t nxi,
                          const void* yi_dev, size_t nyi, void* zi_dev, double extrap_val,
                          void* stream);

/* Scattered queries (xq[k], yq[k]) -> zq[k]: the per-point restatement of interp2
 * (Y-direction blend at both bracketing columns, then X-direction blend). */
int b200_interp2_scattered(b200_interp2_plan* plan, const void* xq, const void* yq,
                           size_t nq, void* zq, double extrap_val);
int b200_interp2_scattered_dev(b200_interp2_plan* plan, const void* xq_dev,
                               const void* yq_dev, size_t nq, void* zq_dev,
                               double extrap_val, void* stream);

/* Derivatives of scattered queries.  Every operation is rounded once; the rules do not depend on the pass order.
 * Gradient: zq exactly as b200_interp2_scattered gives it, plus dz/dx and dz/dy of the piecewise-bilinear interpolant,
 *   dzdx = ((1-wy)*(Z(ay,bx) - Z(ay,ax)) + wy*(Z(by,bx) - Z(by,ax))) / (X[bx] - X[ax])   (dzdy mirrored).
 * A NaN coordinate gives NaN slopes; otherwise an out-of-range coordinate gives +0 (the output is the constant
 * extrap_val).  On the last knot of an axis the slope along it is that of the last cell (from the left); on an
 * interior knot it is that of the cell to the right.  NaN / inf in Z propagate as IEEE arithmetic gives.
 * The _dev call is ordered on `stream`, allocates nothing and never synchronises the host (graph-capturable); the host
 * call is synchronous.  Served by the plan's direct kernel (the banded pipeline serves value-only calls). */
int b200_interp2_scattered_grad(b200_interp2_plan* plan, const void* xq, const void* yq, size_t nq,
                                void* zq, void* dzdx, void* dzdy, double extrap_val);
int b200_interp2_scattered_grad_dev(b200_interp2_plan* plan, const void* xq_dev, const void* yq_dev, size_t nq,
                                    void* zq_dev, void* dzdx_dev, void* dzdy_dev, double extrap_val, void* stream);
/* Adjoint onto the grid: G = W^T g, where row k of W holds the four bilinear weights of query k (the transpose of the
 * scattered call; the gradient of sum_k g[k]*zq[k] with respect to Z).  Only queries with both coordinates in range
 * contribute, each with c00 = (1-wx)(1-wy) g at (ay,ax), c10 = (1-wx) wy g at (by,ax), c01 = wx (1-wy) g at (ay,bx),
 * c11 = wx wy g at (by,bx); a zero coefficient still makes a term (0 * inf = NaN).  Deterministic: G(i,j) = +0, then its
 * terms added one at a time in ascending (cell key ax*ny + ay, query index k, role 00/10/01/11) order — the same bits on
 * every call, stream and graph replay.  Because that order spans the whole batch, splitting a batch into several calls
 * and summing changes the bits: pass all queries in one call (nq <= 2^31-1).
 * Every G(i,j) is written: at j*ld + i (row_major == 0, ld >= ny) or i*ld + j (row_major != 0, ld >= nx), as for
 * b200_interp2_plan_set_values_dev.  Scratch is the caller's `workspace` of at least the queried size, so the _dev call
 * allocates nothing, never synchronises the host and can be captured into a graph.  Cost: a radix sort of the cell
 * keys plus a few streaming passes; the terms of one node are added serially, so a batch whose queries all fall in
 * one cell is slow (correct).  NULL pointers, a short workspace, ld below its minimum or nq > 2^31-1 give
 * B200_ERR_INVALID_ARG before any device work; grids with nx*ny >= 2^32 give B200_ERR_UNSUPPORTED. */
int b200_interp2_scattered_adjoint_workspace(const b200_interp2_plan* plan, size_t nq, size_t* bytes);
int b200_interp2_scattered_adjoint_dev(b200_interp2_plan* plan, const void* xq_dev, const void* yq_dev,
                                       const void* g_dev, size_t nq, void* G_dev, size_t ld, int row_major,
                                       void* workspace, size_t workspace_bytes, void* stream);
/* Host buffers, G column-major ny x nx (arma::mat): allocates, runs on the plan's internal stream, synchronous. */
int b200_interp2_scattered_adjoint(b200_interp2_plan* plan, const void* xq, const void* yq, const void* g, size_t nq,
                                   void* G);

/* Derivatives of tensor-grid queries.  Take the grid's outputs in column-major order: output (i, j) is query
 * k = j*nyi + i at (XI[j], YI[i]) — the mesh.  Each rule is the scattered rule above, applied to the mesh.
 * Gradient: zi has exactly the bits of b200_interp2_grid (in either pass order); dzdx(i,j) and dzdy(i,j) have exactly the
 * bits b200_interp2_scattered_grad gives for mesh query k: NaN slopes for a NaN coordinate, +0 for any other out-of-range
 * one, the last cell's slope on the last knot of an axis, the slope of the cell to the right on an interior knot.
 * zi, dzdx and dzdy are nyi x nxi, column-major.  Empty axes (nxi == 0 or nyi == 0): nothing is written.  The _dev call
 * uses the plan's scratch for the per-axis brackets, as b200_interp2_grid_dev does: one plan must not run on two streams
 * at once.  nxi or nyi > 2^31-1 gives B200_ERR_UNSUPPORTED. */
int b200_interp2_grid_grad(b200_interp2_plan* plan, const void* xi, size_t nxi, const void* yi, size_t nyi, void* zi,
                           void* dzdx, void* dzdy, double extrap_val);
int b200_interp2_grid_grad_dev(b200_interp2_plan* plan, const void* xi_dev, size_t nxi, const void* yi_dev, size_t nyi,
                               void* zi_dev, void* dzdx_dev, void* dzdy_dev, double extrap_val, void* stream);
/* Adjoint onto the grid: G = W^T g with g an nyi x nxi matrix — the gradient of sum_ij g(i,j)*zi(i,j) with respect to Z.
 * G has exactly the bits of b200_interp2_scattered_adjoint on the mesh with g[k] = g(k % nyi, k / nyi): the same
 * (cell key, k, role) order, the same once-rounded terms mul(mul(omx, omy), g), and a zero coefficient still makes a
 * term (NaN payloads aside: a NaN's payload may come from either operand of an add).  That holds also where nxi*nyi exceeds the scattered call's 2^31-1 limit: the product has no limit here, only
 * nxi, nyi <= 2^31-1 (else B200_ERR_UNSUPPORTED).  The mesh is never formed and no output is sorted: a stable sort of
 * each axis by its bracket gives the order of the whole sum, and one pass over the nodes forms every term from the two
 * axes' weights and g.  Workspace O(nxi + nyi + nx + ny).  The terms of one node are added serially, so a small Z under
 * a large grid is slow (correct).
 * g_dev: element (i,j) at j*ldg + i (g_row_major == 0, ldg >= nyi) or i*ldg + j (g_row_major != 0, ldg >= nxi).
 * G_dev: every G(i,j) written at j*ld + i (row_major == 0, ld >= ny) or i*ld + j (row_major != 0, ld >= nx).
 * Empty axes give an all-+0 G.  The _dev call uses only the caller's `workspace` of at least the queried size: it
 * allocates nothing, never synchronises the host and can be captured into a graph.  NULL pointers, a short workspace or
 * ld / ldg below its minimum give B200_ERR_INVALID_ARG before any device work. */
int b200_interp2_grid_adjoint_workspace(const b200_interp2_plan* plan, size_t nxi, size_t nyi, size_t* bytes);
int b200_interp2_grid_adjoint_dev(b200_interp2_plan* plan, const void* xi_dev, size_t nxi, const void* yi_dev, size_t nyi,
                                  const void* g_dev, size_t ldg, int g_row_major, void* G_dev, size_t ld, int row_major,
                                  void* workspace, size_t workspace_bytes, void* stream);
/* Host buffers, g column-major nyi x nxi, G column-major ny x nx (arma::mat): allocates, runs on the plan's internal
 * stream, synchronous. */
int b200_interp2_grid_adjoint(b200_interp2_plan* plan, const void* xi, size_t nxi, const void* yi, size_t nyi,
                              const void* g, void* G);

/* Introspection for the bench: which bracket-lookup path the plan selected
 * (0 = (quasi-)uniform knots: index arithmetic + knot fix-up on one segment record per query,
 *  1 = bucket table + bounded scan / binary search on segment records,
 *  2 = small grid (<= ~6000 f64 knots): knots, values and bucket table staged in shared memory by
 *      TMA bulk copy; index arithmetic as in 0/1 inside the SM). */
int b200_interp1_plan_lookup_mode(const b200_interp1_plan* plan);

/* Self-test of the branch-free FP64 divide of the headline interp2 kernel (the fast path of the IEEE divide without its
 * range check; interp2.cu: div_rn_fast) against __ddiv_rn on n pseudo-random operand pairs inside its contract:
 * *mismatches receives the number of pairs whose result bits differ (expected 0). */
int b200_selftest_div_fast(unsigned long long n, unsigned long long seed, unsigned long long* mismatches);

#ifdef __cplusplus
}
#endif
#endif /* B200_INTERP_H */
