// tests/cpp/nearest_test.cpp -- TargetManager::nearestTargets on managers that hold two model types: uniform-acceleration ids made
// with the YAML's defaults and angular-rates ids made by init(ANGULAR_RATES, ...), on a ShardedTargetManager and on one plain
// TargetManager.  For every query the result must equal, bit for bit, the brute force -- getEstimatesBatch over every id, the
// distance rounded operation by operation in the documented order, ranked by (dist, id) -- and the two managers must agree.  Built
// (with -ffp-contract=off, so that the host distance is not contracted either) and run by tests/test_gpu_nearest.py (needs a GPU).
// Usage: nearest_test <models dir> <shards>
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

// brute force: getEstimatesBatch over every id at t1 (NULL = now), then the targets inside ranked by (dist, id)
static void brute(TargetManager& m, const double* t1, const double* p, double r, long long k, long long& count,
                  std::vector<unsigned>& out_ids, std::vector<double>& out_d) {
  const std::vector<unsigned> ids = m.getAvailableTargets();
  const long long n = (long long)ids.size();
  std::vector<double> when(t1 ? n : 0, t1 ? *t1 : 0.0), pose(7 * (size_t)n), dist(n);
  std::vector<unsigned char> found(n);
  m.getEstimatesBatch(n, ids.data(), t1 ? when.data() : nullptr, pose.data(), nullptr, nullptr, found.data());
  std::vector<long long> in;
  for (long long i = 0; i < n; ++i) {
    CHECK(found[i]);
    const double dx = pose[7 * i] - p[0], dy = pose[7 * i + 1] - p[1], dz = pose[7 * i + 2] - p[2];
    dist[i] = std::sqrt((dx * dx + dy * dy) + dz * dz);
    if (dist[i] <= r) in.push_back(i);
  }
  std::sort(in.begin(), in.end(), [&](long long a, long long b) { return dist[a] < dist[b] || (dist[a] == dist[b] && ids[a] < ids[b]); });
  count = (long long)in.size();
  out_ids.assign(k, 0xFFFFFFFFu);
  out_d.assign(k, -1.0);
  for (long long j = 0; j < std::min(k, count); ++j) { out_ids[j] = ids[in[j]]; out_d[j] = dist[in[j]]; }
}

int main(int argc, char** argv) {
  const std::string models = argc > 1 ? argv[1] : "models";
  const int G = argc > 2 ? std::atoi(argv[2]) : 3;
  const double dt = 1.0 / 250.0;
  const std::string ua = models + "/model_uniform_acceleration_params.yaml";
  std::vector<int> devices((size_t)G, 0);
  std::shared_ptr<ShardedTargetManager> sharded(new ShardedTargetManager(ua, G, devices.data()));
  std::shared_ptr<TargetManager> plain(new TargetManager(ua, 0));
  plain->quiet = true;
  MatrixXd Q, R, P;
  TargetManager::target_t type;
  CHECK(plain->loadYamlFile(models + "/model_angular_rates_params.yaml", Q, R, P, type) && type == TargetManager::ANGULAR_RATES);
  const unsigned n = 4000;   // even ids: uniform acceleration, odd ids: angular rates
  std::mt19937 rng(5);
  std::uniform_real_distribution<double> u(-5.0, 5.0), uv(-2.0, 2.0);
  std::normal_distribution<double> noise(0.0, 0.002);
  std::vector<double> x0(n), y0(n), z0(n), vx(n), vy(n);
  std::vector<unsigned> ids(n);
  for (unsigned i = 0; i < n; ++i) {
    x0[i] = u(rng); y0[i] = u(rng); z0[i] = 20.0 + u(rng); vx[i] = uv(rng); vy[i] = uv(rng);
    ids[i] = 7 + i;
  }
  auto pos = [&](unsigned i, double t) { return Vector3d{x0[i] + vx[i] * t, y0[i] + vy[i] * t, z0[i] - 0.5 * 9.81 * t * t}; };
  for (unsigned i = 0; i < n; ++i) {
    const Vector3d p = pos(i, 0.0);
    const Vector7d p0{p[0], p[1], p[2], 0.0, 0.0, 0.0, 1.0};
    for (TargetManager* m : {(TargetManager*)sharded.get(), plain.get()}) {
      if (ids[i] % 2 == 0) m->init(ids[i], dt, 0.0, p0);
      else m->init(TargetManager::ANGULAR_RATES, ids[i], dt, 0.0, Q, R, P, p0);
    }
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
  }
  const long long q = 9;
  std::vector<double> t1(q, t + 0.02), point(3 * q);
  for (long long j = 0; j < q; ++j) {
    const Vector3d c = pos((unsigned)(j * 397 % n), t);
    std::memcpy(&point[3 * j], c.data(), 24);
  }
  t1[4] = t;   // a second run of t1
  long long total_small = 0;
  for (const double* when : {(const double*)t1.data(), (const double*)nullptr})
    for (double r0 : {1.5, std::numeric_limits<double>::infinity()}) {
      std::vector<double> radius(q);
      for (long long j = 0; j < q; ++j) radius[j] = r0 + 0.1 * (double)j;
      for (long long k : {0LL, 1LL, 50LL, 400LL, 5000LL}) {
        std::vector<unsigned> ia((size_t)(q * k)), ib((size_t)(q * k));
        std::vector<double> da((size_t)(q * k)), db((size_t)(q * k));
        std::vector<long long> ca(q), cb(q);
        const long long ta = sharded->nearestTargets(q, when, point.data(), radius.data(), k, ia.data(), da.data(), ca.data());
        const long long tb = plain->nearestTargets(q, when, point.data(), radius.data(), k, ib.data(), db.data(), cb.data());
        CHECK(ta == tb && ca == cb && ia == ib && std::memcmp(da.data(), db.data(), 8 * da.size()) == 0);
        long long sum = 0;
        for (long long j = 0; j < q; ++j) {
          long long c;
          std::vector<unsigned> ri;
          std::vector<double> rd;
          brute(*plain, when ? when + j : nullptr, &point[3 * j], radius[j], k, c, ri, rd);
          CHECK(ca[j] == c);
          CHECK(std::equal(ri.begin(), ri.end(), ia.begin() + j * k));
          CHECK(std::memcmp(rd.data(), da.data() + j * k, 8 * (size_t)k) == 0);
          sum += c;
          bool ua_in = false, ar_in = false;
          for (long long r = 0; r < std::min(k, c); ++r) (ia[j * k + r] % 2 ? ar_in : ua_in) = true;
          if (k >= 400 && c >= 400) CHECK(ua_in && ar_in);   // both pools feed the merge
        }
        CHECK(ta == sum);
        if (std::isinf(r0)) CHECK(sum == q * (long long)n);
        else total_small = sum;
      }
    }
  CHECK(total_small > 100);
  std::printf("targets inside the small spheres %lld\n", total_small);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
