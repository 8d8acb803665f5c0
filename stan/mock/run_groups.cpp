// Executes gp_lml_groups of stan/gp_lml_stan.hpp against the functional mock of Stan Math and the real libgpb200.so:
// the all-var overload with its reverse sweep, a mixed overload (only rho a parameter) and the all-double overload on
// groups of different sizes, and the std::domain_error of a singular group.  Values and adjoints are printed as one
// JSON object for tests/test_lml_ragged_cpu.py to compare with the oracle; the inputs are closed forms it rebuilds.
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include "stan/math.hpp"
#include "../gp_lml_stan.hpp"
using stan::math::var;
typedef Eigen::Matrix<var, Eigen::Dynamic, 1> VectorXv;

int main() {
  const std::vector<int> sizes = {1, 7, 130, 300, 64};
  const int G = (int)sizes.size();
  int N = 0;
  for (int s : sizes) N += s;
  std::vector<double> x(N);
  Eigen::VectorXd y(N), a(G), r(G), s(G);
  for (int g = 0, i0 = 0; g < G; i0 += sizes[g], g++) {
    for (int i = 0; i < sizes[g]; i++) {
      x[i0 + i] = 0.05 * i + 0.01 * std::sin(1.7 * i + g);
      y[i0 + i] = std::sin(x[i0 + i]) + 0.3 * std::cos(5.0 * x[i0 + i] + g);
    }
    a[g] = 1.0 + 0.1 * g;
    r[g] = 0.8 + 0.05 * g;
    s[g] = 0.2 + 0.03 * g;
  }
  std::printf("{\n");
  try {
    {
      VectorXv av(G), rv(G), sv(G);
      for (int g = 0; g < G; g++) { av[g] = var(a[g]); rv[g] = var(r[g]); sv[g] = var(s[g]); }
      var lp = gp_lml_groups(x, y, sizes, av, rv, sv, nullptr);
      stan::math::grad(lp);
      std::printf("\"vvv\": {\"value\": %.17g, \"adj\": [", lp.val());
      for (int g = 0; g < G; g++)
        std::printf("[%.17g, %.17g, %.17g]%s", av[g].adj(), rv[g].adj(), sv[g].adj(), g + 1 < G ? ", " : "]},\n");
    }
    {
      VectorXv rv(G);
      for (int g = 0; g < G; g++) rv[g] = var(r[g]);
      var lp = gp_lml_groups(x, y, sizes, a, rv, s, nullptr);
      stan::math::grad(lp);
      std::printf("\"dvd\": {\"value\": %.17g, \"adj_rho\": [", lp.val());
      for (int g = 0; g < G; g++) std::printf("%.17g%s", rv[g].adj(), g + 1 < G ? ", " : "]},\n");
    }
    std::printf("\"ddd\": {\"value\": %.17g},\n", gp_lml_groups(x, y, sizes, a, r, s, nullptr));
    bool threw = false;
    try {
      std::vector<double> xd(x);
      xd[8 + 41] = xd[8 + 40];  // group 3: duplicated input, no noise -- exactly singular
      Eigen::VectorXd s0(s);
      s0[2] = 0.0;
      (void)gp_lml_groups(xd, y, sizes, a, r, s0, nullptr);
    } catch (const std::domain_error &e) {
      threw = std::string(e.what()).find("group 3") != std::string::npos;
    }
    std::printf("\"domain_error_on_singular_group\": %s\n", threw ? "true" : "false");
  } catch (const std::exception &e) {
    std::printf("\"error\": \"%s\"\n}\n", e.what());
    return 1;
  }
  std::printf("}\n");
  return 0;
}
