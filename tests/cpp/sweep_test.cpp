// tests/cpp/sweep_test.cpp -- IntersectionSolver::earliestIntersections on managers that hold two model types: uniform-acceleration
// ids made with the YAML's defaults and angular-rates ids made by init(ANGULAR_RATES, ...), on a ShardedTargetManager and on one
// plain TargetManager.  For every sphere the result must equal, bit for bit, the merge of query()'s times over every id ranked by
// (delta, id), and the two managers must agree.  Built and run by tests/test_gpu_sphere_sweep.py (needs a GPU).
// Usage: sweep_test <models dir> <shards>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
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

// brute force: query() over every id for sphere j, hits ranked by (delta, id)
static void brute(IntersectionSolver& s, const std::vector<unsigned>& ids, double t1, const double* o, double r, long long k,
                  long long& hits, std::vector<unsigned>& out_ids, std::vector<double>& out_d) {
  const long long n = (long long)ids.size();
  std::vector<double> t(n, t1), org(3 * n), rad(n, r), d(n);
  for (long long i = 0; i < n; ++i) std::memcpy(&org[3 * i], o, 24);
  s.query(n, ids.data(), nullptr, t.data(), org.data(), rad.data(), nullptr, nullptr, d.data(), nullptr, nullptr);
  std::vector<long long> hit;
  for (long long i = 0; i < n; ++i)
    if (d[i] >= 0.0) hit.push_back(i);
  std::sort(hit.begin(), hit.end(), [&](long long a, long long b) { return d[a] < d[b] || (d[a] == d[b] && ids[a] < ids[b]); });
  hits = (long long)hit.size();
  out_ids.assign(k, 0xFFFFFFFFu);
  out_d.assign(k, -1.0);
  for (long long j = 0; j < std::min(k, hits); ++j) { out_ids[j] = ids[hit[j]]; out_d[j] = d[hit[j]]; }
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
  for (int k = 0; k < 200; ++k) {
    t += dt;
    for (unsigned i = 0; i < n; ++i) {
      const Vector3d p = pos(i, t);
      const double m[7] = {p[0] + noise(rng), p[1] + noise(rng), p[2] + noise(rng), 0.0, 0.0, 0.0, 1.0};
      std::memcpy(&meas[7 * (size_t)i], m, 56);
    }
    CHECK(sharded->updateBatch(n, ids.data(), dt, meas.data()) == n);
    CHECK(plain->updateBatch(n, ids.data(), dt, meas.data()) == n);
  }
  IntersectionSolver s_sh(sharded, 10), s_pl(plain, 10);
  const long long q = 9;
  std::vector<double> t1(q, t), origin(3 * q), radius(q);
  for (long long j = 0; j < q; ++j) {
    const Vector3d c = pos((unsigned)(j * 397 % n), t + 0.3);
    std::memcpy(&origin[3 * j], c.data(), 24);
    radius[j] = 1.5 + 0.1 * (double)j;
  }
  t1[4] += 0.02;   // a second run of t1
  long long total_hits = 0;
  for (long long k : {0LL, 1LL, 50LL, 400LL, 5000LL}) {
    std::vector<unsigned> ia((size_t)(q * k)), ib((size_t)(q * k));
    std::vector<double> da((size_t)(q * k)), db((size_t)(q * k));
    std::vector<long long> ha(q), hb(q);
    const long long ta = s_sh.earliestIntersections(q, t1.data(), origin.data(), radius.data(), k, ia.data(), da.data(), ha.data());
    const long long tb = s_pl.earliestIntersections(q, t1.data(), origin.data(), radius.data(), k, ib.data(), db.data(), hb.data());
    CHECK(ta == tb && ha == hb && ia == ib && std::memcmp(da.data(), db.data(), 8 * da.size()) == 0);
    long long sum = 0;
    for (long long j = 0; j < q; ++j) {
      long long h;
      std::vector<unsigned> ri;
      std::vector<double> rd;
      brute(s_pl, ids, t1[j], &origin[3 * j], radius[j], k, h, ri, rd);
      CHECK(ha[j] == h);
      CHECK(std::equal(ri.begin(), ri.end(), ia.begin() + j * k));
      CHECK(std::memcmp(rd.data(), da.data() + j * k, 8 * (size_t)k) == 0);
      sum += h;
      bool ua_hit = false, ar_hit = false;
      for (long long r = 0; r < std::min(k, h); ++r) (ia[j * k + r] % 2 ? ar_hit : ua_hit) = true;
      if (k >= 400 && h >= 400) CHECK(ua_hit && ar_hit);   // both pools feed the merge
    }
    CHECK(ta == sum);
    total_hits = sum;
  }
  CHECK(total_hits > 100);
  std::printf("total hits %lld\n", total_hits);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
