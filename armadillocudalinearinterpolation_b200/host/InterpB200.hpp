// InterpB200.hpp — Armadillo-facing adaptor of the batched linear-interpolation path (header only).
//
// Same argument order and meaning as the Armadillo free functions the path replaces
// (fn_interp1.hpp / fn_interp2.hpp; the reference links Armadillo un-vendored: Makefile:5,
// Driver.o.dep:554):
//
//     arma::interp1(X, Y, XI, YI, "linear", extrap)          ->  b200::interp1(X, Y, XI, YI, "linear", extrap)
//     arma::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap)   ->  b200::interp2(X, Y, Z, XI, YI, ZI, "linear", extrap)
//
// plus what Armadillo does not have: scattered 2-D queries and plans that keep the grid resident in
// HBM between batches.  Results are bit-identical to the restatement of Armadillo's algorithm in
// oracle/ (bracket = last knot <= xi, w = |X[a]-xi| / (|X[a]-xi| + |X[b]-xi|), (1-w) Y[a] + w Y[b], every
// operation rounded once).  Differences to know about: knots must already be strictly ascending (what
// "*linear" promises; plain "linear" is accepted when it holds, std::runtime_error otherwise — the
// sort/unique pre-pass is not part of the hot path), "nearest"/"*nearest" are not offered, and errors
// surface as std::runtime_error carrying b200_last_error() instead of arma's logic_error.
// Only b200_interp.h crosses into nvcc-compiled code; no Armadillo type does.
#ifndef B200_INTERP_ARMA_HPP
#define B200_INTERP_ARMA_HPP

#include <armadillo>
#include <cstring>
#include <stdexcept>
#include <string>
#include "b200_interp.h"

namespace b200 {

namespace detail {
inline void check_method(const char* method) {
  const char* m = (method && method[0] == '*') ? method + 1 : method;
  if (!m || (std::strcmp(m, "linear") != 0))
    throw std::logic_error(std::string("b200::interp: unsupported interpolation type '") + (method ? method : "") +
                           "' (only \"linear\" / \"*linear\")");
}
inline void check(int status) {
  if (status != B200_OK) throw std::runtime_error(b200_last_error());
}
}  // namespace detail

// arma::interp1(X, Y, XI, YI, method, extrapolation_value)
inline void interp1(const arma::vec& X, const arma::vec& Y, const arma::vec& XI, arma::vec& YI,
                    const char* method = "linear", const double extrapolation_value = arma::datum::nan) {
  detail::check_method(method);
  if (X.n_elem != Y.n_elem) throw std::logic_error("b200::interp1: X and Y must have the same number of elements");
  YI.set_size(XI.n_elem);
  detail::check(b200_interp1_f64(X.memptr(), Y.memptr(), X.n_elem, XI.memptr(), XI.n_elem, YI.memptr(), NULL,
                                 extrapolation_value));
}

// arma::interp2(X, Y, Z, XI, YI, ZI, method, extrapolation_value): XI x YI is a tensor grid, ZI is YI.n_elem x XI.n_elem
inline void interp2(const arma::vec& X, const arma::vec& Y, const arma::mat& Z, const arma::vec& XI,
                    const arma::vec& YI, arma::mat& ZI, const char* method = "linear",
                    const double extrapolation_value = arma::datum::nan) {
  detail::check_method(method);
  if (X.n_elem != Z.n_cols || Y.n_elem != Z.n_rows)
    throw std::logic_error("b200::interp2: X.n_elem must equal Z.n_cols and Y.n_elem must equal Z.n_rows");
  ZI.set_size(YI.n_elem, XI.n_elem);   // arma::mat is column-major: passes through unchanged
  detail::check(b200_interp2_f64(X.memptr(), X.n_elem, Y.memptr(), Y.n_elem, Z.memptr(), XI.memptr(), XI.n_elem,
                                 YI.memptr(), YI.n_elem, ZI.memptr(), extrapolation_value));
}

// arma::fvec / arma::fmat overloads (FP32 arithmetic throughout, same rule)
inline void interp1(const arma::fvec& X, const arma::fvec& Y, const arma::fvec& XI, arma::fvec& YI,
                    const char* method = "linear", const float extrapolation_value = (float)arma::datum::nan) {
  detail::check_method(method);
  if (X.n_elem != Y.n_elem) throw std::logic_error("b200::interp1: X and Y must have the same number of elements");
  YI.set_size(XI.n_elem);
  detail::check(b200_interp1_f32(X.memptr(), Y.memptr(), X.n_elem, XI.memptr(), XI.n_elem, YI.memptr(), NULL,
                                 extrapolation_value));
}
inline void interp2(const arma::fvec& X, const arma::fvec& Y, const arma::fmat& Z, const arma::fvec& XI,
                    const arma::fvec& YI, arma::fmat& ZI, const char* method = "linear",
                    const float extrapolation_value = (float)arma::datum::nan) {
  detail::check_method(method);
  if (X.n_elem != Z.n_cols || Y.n_elem != Z.n_rows)
    throw std::logic_error("b200::interp2: X.n_elem must equal Z.n_cols and Y.n_elem must equal Z.n_rows");
  ZI.set_size(YI.n_elem, XI.n_elem);
  detail::check(b200_interp2_f32(X.memptr(), X.n_elem, Y.memptr(), Y.n_elem, Z.memptr(), XI.memptr(), XI.n_elem,
                                 YI.memptr(), YI.n_elem, ZI.memptr(), extrapolation_value));
}

// Grid resident in HBM: one upload, many query batches (host buffers; pinned ones — b200_host_alloc — overlap best).
class Interp1Plan {
 public:
  Interp1Plan(const arma::vec& X, const arma::vec& Y) : p_(NULL), n_(X.n_elem) {
    if (X.n_elem != Y.n_elem) throw std::logic_error("b200::Interp1Plan: X and Y must have the same number of elements");
    detail::check(b200_interp1_plan_create(B200_F64, X.memptr(), Y.memptr(), X.n_elem, &p_));
  }
  ~Interp1Plan() { b200_interp1_plan_destroy(p_); }
  void SetValues(const arma::vec& Y) { detail::check(b200_interp1_plan_set_values(p_, Y.memptr())); }   // new profile, same knots
  void operator()(const arma::vec& XI, arma::vec& YI, double extrapolation_value = arma::datum::nan) const {
    YI.set_size(XI.n_elem);
    detail::check(b200_interp1_exec(p_, XI.memptr(), XI.n_elem, YI.memptr(), NULL, extrapolation_value));
  }
  // operator() plus the slope DYDX of the piecewise-linear interpolant at each query (rules: b200_interp.h)
  void Grad(const arma::vec& XI, arma::vec& YI, arma::vec& DYDX, double extrapolation_value = arma::datum::nan) const {
    YI.set_size(XI.n_elem);
    DYDX.set_size(XI.n_elem);
    detail::check(b200_interp1_grad(p_, XI.memptr(), XI.n_elem, YI.memptr(), DYDX.memptr(), extrapolation_value));
  }
  // dY = W^T G (one value per knot): the gradient of sum_k G(k) * YI(k) with respect to Y, deterministic
  void Adjoint(const arma::vec& XI, const arma::vec& G, arma::vec& dY) const {
    if (XI.n_elem != G.n_elem) throw std::logic_error("b200::Interp1Plan::Adjoint: XI and G must have the same number of elements");
    dY.set_size(n_);
    detail::check(b200_interp1_adjoint(p_, XI.memptr(), G.memptr(), XI.n_elem, dY.memptr()));
  }
  b200_interp1_plan* handle() const { return p_; }   // for the *_dev entry points

 private:
  Interp1Plan(const Interp1Plan&);
  Interp1Plan& operator=(const Interp1Plan&);
  b200_interp1_plan* p_;
  arma::uword n_;
};

class Interp2Plan {
 public:
  Interp2Plan(const arma::vec& X, const arma::vec& Y, const arma::mat& Z, unsigned flags = 0)
      : p_(NULL), nx_(X.n_elem), ny_(Y.n_elem) {
    CheckShape(Z);
    detail::check(b200_interp2_plan_create_ex(B200_F64, X.memptr(), X.n_elem, Y.memptr(), Y.n_elem, Z.memptr(), flags, &p_));
  }
  ~Interp2Plan() { b200_interp2_plan_destroy(p_); }
  // new Z (Y.n_elem x X.n_elem) on the same axes; same results as a plan created with it
  void SetValues(const arma::mat& Z) {
    CheckShape(Z);
    detail::check(b200_interp2_plan_set_values(p_, Z.memptr()));
  }
  void Grid(const arma::vec& XI, const arma::vec& YI, arma::mat& ZI, double extrapolation_value = arma::datum::nan) const {
    ZI.set_size(YI.n_elem, XI.n_elem);
    detail::check(b200_interp2_grid(p_, XI.memptr(), XI.n_elem, YI.memptr(), YI.n_elem, ZI.memptr(), extrapolation_value));
  }
  // Grid plus the slopes dZ/dX, dZ/dY at every (XI(j), YI(i)), each YI.n_elem x XI.n_elem (rules: b200_interp.h)
  void GridGrad(const arma::vec& XI, const arma::vec& YI, arma::mat& ZI, arma::mat& DZDX, arma::mat& DZDY,
                double extrapolation_value = arma::datum::nan) const {
    ZI.set_size(YI.n_elem, XI.n_elem);
    DZDX.set_size(YI.n_elem, XI.n_elem);
    DZDY.set_size(YI.n_elem, XI.n_elem);
    detail::check(b200_interp2_grid_grad(p_, XI.memptr(), XI.n_elem, YI.memptr(), YI.n_elem, ZI.memptr(), DZDX.memptr(),
                                         DZDY.memptr(), extrapolation_value));
  }
  // dZ = W^T G (Y.n_elem x X.n_elem) with G YI.n_elem x XI.n_elem: the gradient of accu(G % ZI) with respect to Z,
  // deterministic
  void GridAdjoint(const arma::vec& XI, const arma::vec& YI, const arma::mat& G, arma::mat& dZ) const {
    if (G.n_rows != YI.n_elem || G.n_cols != XI.n_elem)
      throw std::logic_error("b200::Interp2Plan::GridAdjoint: G must be YI.n_elem x XI.n_elem");
    dZ.set_size(ny_, nx_);
    detail::check(b200_interp2_grid_adjoint(p_, XI.memptr(), XI.n_elem, YI.memptr(), YI.n_elem, G.memptr(), dZ.memptr()));
  }
  // (XQ(k), YQ(k)) -> ZQ(k): the per-point restatement of interp2
  void Scattered(const arma::vec& XQ, const arma::vec& YQ, arma::vec& ZQ, double extrapolation_value = arma::datum::nan) const {
    if (XQ.n_elem != YQ.n_elem) throw std::logic_error("b200::Interp2Plan::Scattered: XQ and YQ must have the same number of elements");
    ZQ.set_size(XQ.n_elem);
    detail::check(b200_interp2_scattered(p_, XQ.memptr(), YQ.memptr(), XQ.n_elem, ZQ.memptr(), extrapolation_value));
  }
  // Scattered plus the slopes dZ/dX, dZ/dY of the bilinear interpolant at each query (rules: b200_interp.h)
  void ScatteredGrad(const arma::vec& XQ, const arma::vec& YQ, arma::vec& ZQ, arma::vec& DZDX, arma::vec& DZDY,
                     double extrapolation_value = arma::datum::nan) const {
    if (XQ.n_elem != YQ.n_elem) throw std::logic_error("b200::Interp2Plan::ScatteredGrad: XQ and YQ must have the same number of elements");
    ZQ.set_size(XQ.n_elem);
    DZDX.set_size(XQ.n_elem);
    DZDY.set_size(XQ.n_elem);
    detail::check(b200_interp2_scattered_grad(p_, XQ.memptr(), YQ.memptr(), XQ.n_elem, ZQ.memptr(), DZDX.memptr(),
                                              DZDY.memptr(), extrapolation_value));
  }
  // dZ = W^T G (Y.n_elem x X.n_elem): the gradient of sum_k G(k) * ZQ(k) with respect to Z, deterministic
  void ScatteredAdjoint(const arma::vec& XQ, const arma::vec& YQ, const arma::vec& G, arma::mat& dZ) const {
    if (XQ.n_elem != YQ.n_elem || XQ.n_elem != G.n_elem)
      throw std::logic_error("b200::Interp2Plan::ScatteredAdjoint: XQ, YQ and G must have the same number of elements");
    dZ.set_size(ny_, nx_);
    detail::check(b200_interp2_scattered_adjoint(p_, XQ.memptr(), YQ.memptr(), G.memptr(), XQ.n_elem, dZ.memptr()));
  }
  b200_interp2_plan* handle() const { return p_; }

 private:
  Interp2Plan(const Interp2Plan&);
  Interp2Plan& operator=(const Interp2Plan&);
  void CheckShape(const arma::mat& Z) const {
    if (nx_ != Z.n_cols || ny_ != Z.n_rows)
      throw std::logic_error("b200::Interp2Plan: X.n_elem must equal Z.n_cols and Y.n_elem must equal Z.n_rows");
  }
  b200_interp2_plan* p_;
  arma::uword nx_, ny_;
};

}  // namespace b200
#endif
