// tests/cpp/gate_test.cpp -- TargetManager::gatedTargets on managers that hold three model types, each with several dense SPD
// classes made by initBatch(type, Q, R, P0, ...): uniform-acceleration, angular-rates and uniform-velocity ids interleaved, on a
// ShardedTargetManager and on one plain TargetManager.  For every query the result must equal, bit for bit, the merge by (d2, id)
// of one homogeneous manager per model type that holds that type's ids with the same classes and the same records (counts summed),
// and the two mixed managers must agree.  Run by tests/test_gpu_gate.py (needs a GPU).
// Usage: gate_test <models dir> <shards>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <random>
#include <string>
#include <vector>

#include "target_estimation_b200/target_manager.hpp"

using namespace target_estimation_b200;

static int g_checks = 0, g_failed = 0;
#define CHECK(cond)                                                              \
  do {                                                                           \
    ++g_checks;                                                                  \
    if (!(cond)) { ++g_failed; std::printf("FAILED %s:%d  %s\n", __FILE__, __LINE__, #cond); } \
  } while (0)

// a random dense SPD matrix with the diagonal magnitudes of ref, bitwise symmetric
static MatrixXd dense_spd(std::mt19937& rng, const MatrixXd& ref) {
  const int n = ref.rows();
  std::normal_distribution<double> g(0.0, 1.0);
  std::vector<double> a((size_t)n * n), s(n);
  for (double& v : a) v = g(rng);
  double dmax = 0.0;
  for (int i = 0; i < n; ++i) dmax = std::max(dmax, ref(i, i));
  for (int i = 0; i < n; ++i) s[i] = std::sqrt(ref(i, i) > 0.0 ? ref(i, i) : dmax * 1e-6);
  MatrixXd x(n, n);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j <= i; ++j) {
      double v = 0.0;
      for (int k = 0; k < n; ++k) v += a[(size_t)i * n + k] * a[(size_t)j * n + k];
      v = (v / n + (i == j ? 0.5 : 0.0)) * s[i] * s[j];
      x(i, j) = v;
      x(j, i) = v;
    }
  return x;
}

struct Rows {
  std::vector<unsigned> ids;
  std::vector<double> d2;
  std::vector<long long> count;
  long long total = 0;
};

static Rows gated(TargetManager& m, long long q, const double* t1, const double* z, const double* gate, long long k) {
  Rows r;
  r.ids.assign((size_t)(q * k), 0u);
  r.d2.assign((size_t)(q * k), 0.0);
  r.count.assign((size_t)q, 0);
  r.total = m.gatedTargets(q, t1, z, gate, k, r.ids.data(), r.d2.data(), r.count.data());
  return r;
}

static bool same(const Rows& a, const Rows& b) {
  return a.total == b.total && a.count == b.count && a.ids == b.ids && std::memcmp(a.d2.data(), b.d2.data(), 8 * a.d2.size()) == 0;
}

// the k smallest (d2, id) rows over the homogeneous managers' lists, counts summed
static Rows merge(const std::vector<Rows>& parts, long long q, long long k) {
  Rows r;
  r.ids.assign((size_t)(q * k), 0xFFFFFFFFu);
  r.d2.assign((size_t)(q * k), -1.0);
  r.count.assign((size_t)q, 0);
  for (long long j = 0; j < q; ++j) {
    std::vector<std::pair<double, unsigned>> all;
    for (const Rows& p : parts) {
      r.count[j] += p.count[j];
      for (long long i = 0; i < std::min(k, p.count[j]); ++i) all.emplace_back(p.d2[j * k + i], p.ids[j * k + i]);
    }
    std::sort(all.begin(), all.end());
    for (long long i = 0; i < std::min<long long>(k, (long long)all.size()); ++i) {
      r.d2[j * k + i] = all[i].first;
      r.ids[j * k + i] = all[i].second;
    }
    r.total += r.count[j];
  }
  return r;
}

int main(int argc, char** argv) {
  const std::string models = argc > 1 ? argv[1] : "models";
  const int G = argc > 2 ? std::atoi(argv[2]) : 3;
  const double dt = 1.0 / 250.0;
  const std::string ua = models + "/model_uniform_acceleration_params.yaml";
  const TargetManager::target_t types[3] = {TargetManager::UNIFORM_ACCELERATION, TargetManager::ANGULAR_RATES, TargetManager::UNIFORM_VELOCITY};
  const char* files[3] = {"uniform_acceleration", "angular_rates", "uniform_velocity"};
  std::vector<int> devices((size_t)G, 0);
  std::shared_ptr<ShardedTargetManager> sharded(new ShardedTargetManager(ua, G, devices.data()));
  std::shared_ptr<TargetManager> plain(new TargetManager(ua, 0));
  std::vector<std::shared_ptr<TargetManager>> homo;   // one manager per model type
  for (int ty = 0; ty < 3; ++ty) homo.emplace_back(new TargetManager(ua, 0));
  plain->quiet = true;
  // three dense classes per model type
  std::mt19937 rng(5);
  MatrixXd Q[3][3], R[3][3], P0[3][3];
  for (int ty = 0; ty < 3; ++ty) {
    MatrixXd q0, r0, p0;
    TargetManager::target_t type;
    CHECK(plain->loadYamlFile(models + "/model_" + files[ty] + "_params.yaml", q0, r0, p0, type) && type == types[ty]);
    for (int c = 0; c < 3; ++c) {
      Q[ty][c] = dense_spd(rng, q0);
      R[ty][c] = dense_spd(rng, r0);
      P0[ty][c] = dense_spd(rng, p0);
    }
  }
  // id 7 + i: model type i % 3, class (i / 3) % 3
  const unsigned n = 3000;
  std::uniform_real_distribution<double> u(-5.0, 5.0), uv(-2.0, 2.0);
  std::normal_distribution<double> noise(0.0, 0.002);
  std::vector<double> x0(n), y0(n), z0(n), vx(n), vy(n);
  std::vector<unsigned> ids(n);
  for (unsigned i = 0; i < n; ++i) {
    x0[i] = u(rng); y0[i] = u(rng); z0[i] = 20.0 + u(rng); vx[i] = uv(rng); vy[i] = uv(rng);
    ids[i] = 7 + i;
  }
  auto pos = [&](unsigned i, double t) { return Vector3d{x0[i] + vx[i] * t, y0[i] + vy[i] * t, z0[i] - 0.5 * 9.81 * t * t}; };
  for (int ty = 0; ty < 3; ++ty)
    for (int c = 0; c < 3; ++c) {
      std::vector<unsigned> gi;
      std::vector<double> p0, t0;
      for (unsigned i = 0; i < n; ++i) {
        if ((int)(i % 3) != ty || (int)((i / 3) % 3) != c) continue;
        const Vector3d p = pos(i, 0.0);
        const double rec[7] = {p[0], p[1], p[2], 0.0, 0.0, 0.0, 1.0};
        gi.push_back(ids[i]);
        p0.insert(p0.end(), rec, rec + 7);
        t0.push_back(0.0);
      }
      const long long m = (long long)gi.size();
      for (TargetManager* mg : {(TargetManager*)sharded.get(), plain.get(), homo[ty].get()})
        CHECK(mg->initBatch(types[ty], Q[ty][c], R[ty][c], P0[ty][c], m, gi.data(), dt, t0.data(), p0.data()) == m);
    }
  double t = 0.0;
  std::vector<double> meas(7 * (size_t)n);
  for (int k = 0; k < 100; ++k) {
    t += dt;
    for (unsigned i = 0; i < n; ++i) {
      const Vector3d p = pos(i, t);
      const double m[7] = {p[0] + noise(rng), p[1] + noise(rng), p[2] + noise(rng), 0.0, 0.0, 0.0, 1.0};
      std::memcpy(&meas[7 * (size_t)i], m, 56);
    }
    CHECK(sharded->updateBatch(n, ids.data(), dt, meas.data()) == n);
    CHECK(plain->updateBatch(n, ids.data(), dt, meas.data()) == n);
    for (int ty = 0; ty < 3; ++ty) {
      std::vector<unsigned> gi;
      std::vector<double> gm;
      for (unsigned i = ty; i < n; i += 3) {
        gi.push_back(ids[i]);
        gm.insert(gm.end(), &meas[7 * (size_t)i], &meas[7 * (size_t)i] + 7);
      }
      CHECK(homo[ty]->updateBatch((long long)gi.size(), gi.data(), dt, gm.data()) == (long long)gi.size());
    }
  }
  // measured positions a few millimetres from the current estimates of targets of every type
  const long long q = 9;
  std::vector<double> t1(q, t + 0.02), z(3 * q), est(7 * q);
  std::vector<unsigned> near_ids(q);
  for (long long j = 0; j < q; ++j) near_ids[j] = ids[(size_t)(j * 397 % n)];
  plain->getEstimatesBatch(q, near_ids.data(), nullptr, est.data(), nullptr, nullptr, nullptr);
  std::normal_distribution<double> near(0.0, 0.003);
  for (long long j = 0; j < q; ++j)
    for (int e = 0; e < 3; ++e) z[3 * j + e] = est[7 * j + e] + near(rng);
  t1[4] = t;   // a second run of t1
  long long inside_chi2 = 0;
  for (const double* when : {(const double*)t1.data(), (const double*)nullptr})
    for (double g0 : {11.34, 1e4, std::numeric_limits<double>::infinity()}) {
      std::vector<double> gate(q);
      for (long long j = 0; j < q; ++j) gate[j] = g0 * (1.0 + 0.1 * (double)j);
      for (long long k : {0LL, 1LL, 50LL, 400LL, 3100LL}) {
        const Rows a = gated(*sharded, q, when, z.data(), gate.data(), k);
        const Rows b = gated(*plain, q, when, z.data(), gate.data(), k);
        std::vector<Rows> parts;
        for (int ty = 0; ty < 3; ++ty) parts.push_back(gated(*homo[ty], q, when, z.data(), gate.data(), k));
        const Rows ref = merge(parts, q, k);
        CHECK(same(a, b));
        CHECK(same(b, ref));
        if (std::isinf(g0)) CHECK(ref.total == q * (long long)n);
        if (g0 == 11.34 && k == 0) inside_chi2 += ref.total;
        if (k == 3100 && std::isinf(g0)) {   // every pool feeds the merge
          bool seen[3] = {false, false, false};
          for (long long r = 0; r < std::min(k, b.count[0]); ++r) seen[(b.ids[r] - 7) % 3] = true;
          CHECK(seen[0] && seen[1] && seen[2]);
        }
      }
    }
  CHECK(inside_chi2 > 0);
  std::printf("targets inside the chi-square gates %lld\n", inside_chi2);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
