// stan/gp_lml_stan.hpp -- Stan external C++ function backed by libgpb200.so.
//
// NOT COMPILED IN THE BUILD CONTAINER (no Stan Math / Eigen there).  Usage mirrors the mechanism the
// reference uses for models/cubic_interpolated_gp.hpp (test_interpolate.R:16-23):
//
//   functions { real gp_lml(real[] x, vector y, real alpha, real rho, real sigma); }
//   model     { target += gp_lml(t, y, alpha, rho, sigma); ... priors ... }
//
//   stanc(file, allow_undefined = TRUE)
//   stan_model(stanc_ret = ..., includes = '#include "/abs/path/stan/gp_lml_stan.hpp"')
//   and link with  -L<repo>/gp_b200/lib -lgpb200
//
// It replaces lines 19-25 and 31 of models/fit_hyperparameters.stan (cov_exp_quad, diagonal add,
// cholesky_decompose, multi_normal_cholesky) and their reverse sweep by one GPU call: the value is
// the LML WITH constants and the three partials are injected with precomputed_gradients, the same
// device the reference uses in cubic_interpolated_gp.hpp:28 (precomp_v_vari).
// A non-positive-definite matrix throws std::domain_error, as Stan Math's cholesky_decompose does,
// so NUTS rejects the proposal.
#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

extern "C" {
#include "../include/gpb200.h"
}

namespace gpb200_stan {
inline gpb200_handle_t handle() {
  static thread_local gpb200_handle_t h = nullptr;
  if (!h) {
    if (gpb200_create(&h, 0) != 0) throw std::runtime_error("gpb200: no usable B200 GPU (no CPU fallback)");
  }
  return h;
}
inline void eval(const std::vector<double>& x, const Eigen::VectorXd& y, double alpha, double rho, double sigma,
                 double& lml, double* grad) {
  const double theta[3] = {alpha, rho, sigma};
  const int rc = gpb200_lml_grad(handle(), (int)x.size(), x.data(), y.data(), theta, 0.0, &lml, grad);
  if (rc > 0) throw std::domain_error("gp_lml: covariance is not positive definite (pivot " + std::to_string(rc) + ")");
  if (rc < 0) throw std::runtime_error(std::string("gp_lml: ") + gpb200_last_error(handle()));
}
}  // namespace gpb200_stan

namespace gpb200_stan {
// operands that are `var` contribute a partial; `double` arguments contribute nothing (C++11 overloads,
// no `if constexpr`: the rstan toolchains of the reference's era compile as C++11/14)
inline void add_operand(std::vector<stan::math::var>& ops, std::vector<double>& partials, const stan::math::var& v,
                        double g) {
  ops.push_back(v);
  partials.push_back(g);
}
inline void add_operand(std::vector<stan::math::var>&, std::vector<double>&, double, double) {}
}  // namespace gpb200_stan

// reverse-mode overload: any of alpha, rho, sigma may be var
template <typename T0__, typename T1__, typename T2__>
typename boost::math::tools::promote_args<T0__, T1__, T2__>::type
gp_lml(const std::vector<double>& x, const Eigen::Matrix<double, Eigen::Dynamic, 1>& y, const T0__& alpha,
       const T1__& rho, const T2__& sigma, std::ostream* pstream__) {
  using stan::math::value_of;
  double lml, g[3];
  gpb200_stan::eval(x, y, value_of(alpha), value_of(rho), value_of(sigma), lml, g);
  std::vector<stan::math::var> operands;
  std::vector<double> partials;
  gpb200_stan::add_operand(operands, partials, alpha, g[0]);
  gpb200_stan::add_operand(operands, partials, rho, g[1]);
  gpb200_stan::add_operand(operands, partials, sigma, g[2]);
  return stan::math::precomputed_gradients(lml, operands, partials);
}

// all-double overload (generated quantities / transformed data), like cubic_interpolated_gp.hpp:34-36
inline double gp_lml(const std::vector<double>& x, const Eigen::Matrix<double, Eigen::Dynamic, 1>& y,
                     const double& alpha, const double& rho, const double& sigma, std::ostream* pstream__) {
  double lml;
  gpb200_stan::eval(x, y, alpha, rho, sigma, lml, nullptr);
  return lml;
}

// ---- GP observed through first derivatives only: the model block of the Stan program embedded in
// gpderivs.py:62-83 (Sigma = sf2 * covdd(t_i, t_j, l2) + s2 I; dx ~ multi_normal(zeros, Sigma)) as one
// call, in that program's own (sf2, l2, s2) parametrisation:
//
//   functions { real gp_lml_dd(vector t, vector dx, real sf2, real l2, real s2); }
//   model     { target += gp_lml_dd(t, dx, sf2, l2, s2); ... cauchy priors ... }
namespace gpb200_stan {
inline void eval_dd(const Eigen::VectorXd& t, const Eigen::VectorXd& dx, double sf2, double l2, double s2, double& lml,
                    double* grad3) {
  const double alpha = std::sqrt(sf2), l = std::sqrt(0.5 * l2), sigma = std::sqrt(s2);
  const double theta[3] = {alpha, l, sigma};
  double g[3];
  int info = 0;
  const int rc = gpb200_lml_grad_deriv_batched(handle(), (int)t.size(), /*order0=*/1, /*nblocks=*/1, 1, t.data(), 0,
                                               dx.data(), 0, theta, 0.0, grad3 != nullptr, &lml, g, &info);
  if (rc < 0) throw std::runtime_error(std::string("gp_lml_dd: ") + gpb200_last_error(handle()));
  if (info > 0) throw std::domain_error("gp_lml_dd: covariance is not positive definite (pivot " + std::to_string(info) + ")");
  if (grad3) {  // chain rule to (sf2, l2, s2)
    grad3[0] = g[0] / (2.0 * alpha);
    grad3[1] = g[1] / (4.0 * l);
    grad3[2] = g[2] / (2.0 * sigma);
  }
}
}  // namespace gpb200_stan

template <typename T0__, typename T1__, typename T2__>
typename boost::math::tools::promote_args<T0__, T1__, T2__>::type
gp_lml_dd(const Eigen::Matrix<double, Eigen::Dynamic, 1>& t, const Eigen::Matrix<double, Eigen::Dynamic, 1>& dx,
          const T0__& sf2, const T1__& l2, const T2__& s2, std::ostream* pstream__) {
  using stan::math::value_of;
  double lml, g[3];
  gpb200_stan::eval_dd(t, dx, value_of(sf2), value_of(l2), value_of(s2), lml, g);
  std::vector<stan::math::var> operands;
  std::vector<double> partials;
  gpb200_stan::add_operand(operands, partials, sf2, g[0]);
  gpb200_stan::add_operand(operands, partials, l2, g[1]);
  gpb200_stan::add_operand(operands, partials, s2, g[2]);
  return stan::math::precomputed_gradients(lml, operands, partials);
}

inline double gp_lml_dd(const Eigen::Matrix<double, Eigen::Dynamic, 1>& t, const Eigen::Matrix<double, Eigen::Dynamic, 1>& dx,
                        const double& sf2, const double& l2, const double& s2, std::ostream* pstream__) {
  double lml;
  gpb200_stan::eval_dd(t, dx, sf2, l2, s2, lml, nullptr);
  return lml;
}

// ---- joint derivative observations (design_notes.Rmd:25-46; BASELINE config 2): y_stack = (y, y', y'') on the
// grid t, noise = per-block sd (1 to 3 entries), jitter 1e-6 as in R/ode_gp_library.R:30:
//
//   functions { real gp_lml_joint(vector t, vector y_stack, real alpha, real rho, vector noise); }
//   model     { target += gp_lml_joint(t, append_row(y, append_row(yp, ypp)), alpha, rho, noise); }
namespace gpb200_stan {
inline void eval_joint(const Eigen::VectorXd& t, const Eigen::VectorXd& y, double alpha, double rho, const double* noise,
                       int nblocks, double& lml, double* grad) {
  if (nblocks < 1 || nblocks > 3 || y.size() != t.size() * nblocks)
    throw std::domain_error("gp_lml_joint: y_stack must hold 1 to 3 blocks of length(t) observations");
  double theta[5] = {alpha, rho, 0.0, 0.0, 0.0};
  for (int b = 0; b < nblocks; b++) theta[2 + b] = noise[b];
  double g[5];
  int info = 0;
  const int rc = gpb200_lml_grad_deriv_batched(handle(), (int)t.size(), /*order0=*/0, nblocks, 1, t.data(), 0, y.data(), 0,
                                               theta, 1e-6, grad != nullptr, &lml, g, &info);
  if (rc < 0) throw std::runtime_error(std::string("gp_lml_joint: ") + gpb200_last_error(handle()));
  if (info > 0) throw std::domain_error("gp_lml_joint: covariance is not positive definite (pivot " + std::to_string(info) + ")");
  if (grad) for (int q = 0; q < 2 + nblocks; q++) grad[q] = g[q];
}
}  // namespace gpb200_stan

template <typename T0__, typename T1__, typename T2__>
typename boost::math::tools::promote_args<T0__, T1__, T2__>::type
gp_lml_joint(const Eigen::Matrix<double, Eigen::Dynamic, 1>& t, const Eigen::Matrix<double, Eigen::Dynamic, 1>& y_stack,
             const T0__& alpha, const T1__& rho, const Eigen::Matrix<T2__, Eigen::Dynamic, 1>& noise, std::ostream* pstream__) {
  using stan::math::value_of;
  const int nb = (int)noise.size();
  double nz[3] = {0.0, 0.0, 0.0};
  for (int b = 0; b < nb && b < 3; b++) nz[b] = value_of(noise.data()[b]);
  double lml, g[5];
  gpb200_stan::eval_joint(t, y_stack, value_of(alpha), value_of(rho), nz, nb, lml, g);
  std::vector<stan::math::var> operands;
  std::vector<double> partials;
  gpb200_stan::add_operand(operands, partials, alpha, g[0]);
  gpb200_stan::add_operand(operands, partials, rho, g[1]);
  for (int b = 0; b < nb; b++) gpb200_stan::add_operand(operands, partials, noise.data()[b], g[2 + b]);
  return stan::math::precomputed_gradients(lml, operands, partials);
}

inline double gp_lml_joint(const Eigen::Matrix<double, Eigen::Dynamic, 1>& t,
                           const Eigen::Matrix<double, Eigen::Dynamic, 1>& y_stack, const double& alpha, const double& rho,
                           const Eigen::Matrix<double, Eigen::Dynamic, 1>& noise, std::ostream* pstream__) {
  double lml;
  gpb200_stan::eval_joint(t, y_stack, alpha, rho, noise.data(), (int)noise.size(), lml, nullptr);
  return lml;
}

// ---- one GP per group, groups of different sizes: the per-player GPs of multiple_players.stan:59-63, all groups'
// LMLs and gradients in one call at every leapfrog step.  x and y hold the groups one after the other, sizes[g] >= 1
// points each (sum(sizes) == size(x) == rows(y)); alpha, rho, sigma hold one entry per group:
//
//   functions { real gp_lml_groups(real[] x, vector y, int[] sizes, vector alpha, vector rho, vector sigma); }
//   model     { target += gp_lml_groups(x, y, sizes, alpha, rho, sigma); ... priors ... }
//
// Returns sum_g lml_g (with constants) with a partial for every group's three parameters; a group whose covariance
// is not positive definite throws std::domain_error, so NUTS rejects the proposal.
namespace gpb200_stan {
inline void eval_groups(const std::vector<double>& x, const Eigen::VectorXd& y, const std::vector<int>& sizes,
                        const std::vector<double>& theta, double& total, std::vector<double>* grad) {
  const int G = (int)sizes.size();
  if ((int)theta.size() != 3 * G) throw std::domain_error("gp_lml_groups: alpha, rho and sigma need one entry per group");
  std::vector<long long> off(G + 1, 0);
  for (int g = 0; g < G; g++) {
    if (sizes[g] < 1) throw std::domain_error("gp_lml_groups: every group size must be >= 1");
    off[g + 1] = off[g] + sizes[g];
  }
  if (off[G] != (long long)x.size() || off[G] != (long long)y.size())
    throw std::domain_error("gp_lml_groups: sum(sizes) must equal the length of x and of y");
  total = 0.0;
  if (G == 0) return;
  std::vector<double> lml(G), g3(3 * G);
  std::vector<int> info(G);
  const int rc = gpb200_lml_grad_ragged(handle(), G, off.data(), x.data(), y.data(), theta.data(), 0.0, grad != nullptr,
                                        lml.data(), g3.data(), info.data());
  if (rc < 0) throw std::runtime_error(std::string("gp_lml_groups: ") + gpb200_last_error(handle()));
  for (int g = 0; g < G; g++)
    if (info[g] > 0)
      throw std::domain_error("gp_lml_groups: covariance of group " + std::to_string(g + 1) + " is not positive definite (pivot " +
                              std::to_string(info[g]) + ")");
  for (int g = 0; g < G; g++) total += lml[g];
  if (grad) *grad = g3;
}
}  // namespace gpb200_stan

template <typename T0__, typename T1__, typename T2__>
typename boost::math::tools::promote_args<T0__, T1__, T2__>::type
gp_lml_groups(const std::vector<double>& x, const Eigen::Matrix<double, Eigen::Dynamic, 1>& y, const std::vector<int>& sizes,
              const Eigen::Matrix<T0__, Eigen::Dynamic, 1>& alpha, const Eigen::Matrix<T1__, Eigen::Dynamic, 1>& rho,
              const Eigen::Matrix<T2__, Eigen::Dynamic, 1>& sigma, std::ostream* pstream__) {
  using stan::math::value_of;
  const int G = (int)sizes.size();
  if (alpha.size() != G || rho.size() != G || sigma.size() != G)
    throw std::domain_error("gp_lml_groups: alpha, rho and sigma need one entry per group");
  std::vector<double> theta(3 * G), grad;
  for (int g = 0; g < G; g++) {
    theta[3 * g] = value_of(alpha.data()[g]);
    theta[3 * g + 1] = value_of(rho.data()[g]);
    theta[3 * g + 2] = value_of(sigma.data()[g]);
  }
  double total;
  gpb200_stan::eval_groups(x, y, sizes, theta, total, &grad);
  std::vector<stan::math::var> operands;
  std::vector<double> partials;
  for (int g = 0; g < G; g++) {
    gpb200_stan::add_operand(operands, partials, alpha.data()[g], grad[3 * g]);
    gpb200_stan::add_operand(operands, partials, rho.data()[g], grad[3 * g + 1]);
    gpb200_stan::add_operand(operands, partials, sigma.data()[g], grad[3 * g + 2]);
  }
  return stan::math::precomputed_gradients(total, operands, partials);
}

inline double gp_lml_groups(const std::vector<double>& x, const Eigen::Matrix<double, Eigen::Dynamic, 1>& y,
                            const std::vector<int>& sizes, const Eigen::Matrix<double, Eigen::Dynamic, 1>& alpha,
                            const Eigen::Matrix<double, Eigen::Dynamic, 1>& rho,
                            const Eigen::Matrix<double, Eigen::Dynamic, 1>& sigma, std::ostream* pstream__) {
  const int G = (int)sizes.size();
  if (alpha.size() != G || rho.size() != G || sigma.size() != G)
    throw std::domain_error("gp_lml_groups: alpha, rho and sigma need one entry per group");
  std::vector<double> theta(3 * G);
  for (int g = 0; g < G; g++) {
    theta[3 * g] = alpha.data()[g];
    theta[3 * g + 1] = rho.data()[g];
    theta[3 * g + 2] = sigma.data()[g];
  }
  double total;
  gpb200_stan::eval_groups(x, y, sizes, theta, total, nullptr);
  return total;
}
