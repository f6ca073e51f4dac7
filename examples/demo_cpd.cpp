// DemoCPD (examples/DemoCPD.scala:10-26 of the reference) through the C++ host mirror include/gingr.hpp, on a synthetic pair:
// a Fibonacci sphere as reference, the same sphere deformed and moved as target, a Gaussian-kernel GPMM built on the
// device, deterministic CPD.  Build (from the repository root, after python -m gingr_b200.build):
//   g++ -std=c++17 -O2 -Iinclude examples/demo_cpd.cpp -o demo_cpd -Lgingr_b200/lib -lgingr_cuda -Wl,-rpath,$PWD/gingr_b200/lib
// Exit codes: 0 = registration ran and the fit improved; 2 = the library reported an error (e.g. no CUDA device).
#include <cmath>
#include <cstdio>
#include <vector>

#include "gingr.hpp"

static std::vector<double> fibonacci_sphere(int n, double radius) {
  std::vector<double> p(static_cast<size_t>(3) * n);
  const double golden = M_PI * (3.0 - std::sqrt(5.0));
  for (int i = 0; i < n; ++i) {
    const double z = 1.0 - 2.0 * (i + 0.5) / n, rho = std::sqrt(1.0 - z * z), th = golden * i;
    p[3 * i] = radius * rho * std::cos(th);
    p[3 * i + 1] = radius * rho * std::sin(th);
    p[3 * i + 2] = radius * z;
  }
  return p;
}

static double mean_nearest_distance(const std::vector<double>& a, const std::vector<double>& b) {
  double sum = 0.0;
  const size_t na = a.size() / 3, nb = b.size() / 3;
  for (size_t i = 0; i < na; ++i) {
    double best = INFINITY;
    for (size_t j = 0; j < nb; ++j) {
      const double dx = a[3 * i] - b[3 * j], dy = a[3 * i + 1] - b[3 * j + 1], dz = a[3 * i + 2] - b[3 * j + 2];
      best = std::fmin(best, dx * dx + dy * dy + dz * dz);
    }
    sum += std::sqrt(best);
  }
  return sum / static_cast<double>(na);
}

int main() {
  try {
    gingr::Context ctx(0);
    const int M = 400, N = 500;
    const std::vector<double> ref = fibonacci_sphere(M, 100.0);
    std::vector<double> tgt = fibonacci_sphere(N, 100.0);
    for (int j = 0; j < N; ++j) {  // smooth deformation + offset
      const double x = tgt[3 * j], y = tgt[3 * j + 1], z = tgt[3 * j + 2];
      tgt[3 * j] = x + 4.0 * std::sin(y / 50.0) + 5.0;
      tgt[3 * j + 1] = y + 3.0 * std::sin(z / 40.0) - 2.0;
      tgt[3 * j + 2] = z * 1.05 + 2.0 * std::cos(x / 60.0) + 3.0;
    }
    gingr::Model model = gingr::Model::gaussianMixture(ctx, M, ref.data(), nullptr, 0, {70.0}, {50.0}, 0.01);
    gingr::Target target(ctx, N, tgt.data());
    gingr::CpdConfiguration config;
    // On this pair sigma2 keeps shrinking: from the 25th proposal on, some model point has no target point within the
    // reach of exp() and its P1 underflows to 0, so the posterior fails (ModelFlexibilityError, as in the reference).
    config.maxIterations = 20;
    config.w = 0.05;
    gingr::CpdRegistration cpd(ctx, model, target, config);
    gingr::GeneralRegistrationState init = cpd.initializeState(gingr::GlobalTransformationType::RigidTransforms);
    const double before = mean_nearest_distance(init.fit, tgt);
    int states = 0;
    gingr::GeneralRegistrationState best = cpd.run(init, [&](const gingr::GeneralRegistrationState&) { ++states; });
    const double after = mean_nearest_distance(best.fit, tgt);
    std::printf("model: %d points, rank %d; %d states; status %d, sigma2 %.6g -> %.6g; mean distance to target %.4f -> %.4f\n",
                model.points(), model.rank(), states, static_cast<int>(best.status), init.sigma2, best.sigma2, before, after);
    return (best.status != gingr::FittingStatus::ModelFlexibilityError && after < before) ? 0 : 1;
  } catch (const gingr::Error& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return 2;
  }
}
