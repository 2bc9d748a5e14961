// tests/cpp/associate_test.cpp -- TargetManager::associate on managers that hold three model types, each with several dense SPD
// classes made by initBatch(type, Q, R, P0, ...): uniform-acceleration, angular-rates and uniform-velocity ids interleaved, on a
// ShardedTargetManager and on one plain TargetManager (both take the multi-pool path: every pool's candidate lists merged, the
// matching by te_assign_greedy).  For every frame the assignment must equal, bit for bit, a sequential greedy over the manager's own
// gatedTargets(k = K) rows, the counts must be gatedTargets' counts, and after apply = 1 both managers must hold the same states.
// Run by tests/test_gpu_associate.py (needs a GPU).
// Usage: associate_test <models dir> <shards>
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

// the contract's assignment: the edges of the rows [q][K] (d2 -1 = none) visited by (d2, id, j)
static void greedy(long long q, int K, const std::vector<unsigned>& ids, const std::vector<double>& d2, std::vector<unsigned>& id_out,
                   std::vector<double>& d2_out) {
  struct E { double d2; unsigned id; long long j; };
  std::vector<E> e;
  for (long long j = 0; j < q; ++j)
    for (int r = 0; r < K; ++r)
      if (d2[(size_t)(j * K + r)] >= 0.0) e.push_back({d2[(size_t)(j * K + r)], ids[(size_t)(j * K + r)], j});
  std::sort(e.begin(), e.end(), [](const E& a, const E& b) { return a.d2 != b.d2 ? a.d2 < b.d2 : a.id != b.id ? a.id < b.id : a.j < b.j; });
  id_out.assign((size_t)q, 0xFFFFFFFFu);
  d2_out.assign((size_t)q, -1.0);
  std::vector<unsigned> taken;
  for (const E& x : e) {
    if (id_out[(size_t)x.j] != 0xFFFFFFFFu || std::find(taken.begin(), taken.end(), x.id) != taken.end()) continue;
    id_out[(size_t)x.j] = x.id;
    d2_out[(size_t)x.j] = x.d2;
    taken.push_back(x.id);
  }
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
      for (TargetManager* mg : {(TargetManager*)sharded.get(), plain.get()})
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
  }
  // frames: detections near the estimates at t1 of targets of every type, plus clutter
  std::normal_distribution<double> near(0.0, 0.003);
  long long assigned_total = 0;
  for (int f = 0; f < 3; ++f) {
    const double t1 = t + 0.01 * (f + 1);
    const long long q = 660;
    std::vector<unsigned> src(600);
    for (int j = 0; j < 600; ++j) src[(size_t)j] = ids[(size_t)((j * 7 + f * 131) % n)];
    std::vector<double> when(600, t1), est(7 * 600), det(7 * (size_t)q, 0.0), z(3 * (size_t)q);
    plain->getEstimatesBatch(600, src.data(), when.data(), est.data(), nullptr, nullptr, nullptr);
    for (long long j = 0; j < q; ++j) {
      for (int e = 0; e < 3; ++e) det[7 * j + e] = j < 600 ? est[7 * j + e] + near(rng) : u(rng) + (e == 2 ? 20.0 : 0.0);
      det[7 * j + 6] = 1.0;
      for (int e = 0; e < 3; ++e) z[3 * j + e] = det[7 * j + e];
    }
    for (int K : {1, 8, 32}) {
      for (TargetManager* m : {(TargetManager*)sharded.get(), plain.get()}) {
        std::vector<double> gate((size_t)q, 11.34), t1s((size_t)q, t1);
        const Rows rows = gated(*m, q, t1s.data(), z.data(), gate.data(), K);
        std::vector<unsigned> ref_id, id_out((size_t)q);
        std::vector<double> ref_d2, d2_out((size_t)q);
        std::vector<long long> count((size_t)q);
        greedy(q, K, rows.ids, rows.d2, ref_id, ref_d2);
        const long long a = m->associate(t1, q, det.data(), 11.34, K, 0, id_out.data(), d2_out.data(), count.data());
        CHECK(id_out == ref_id);
        CHECK(std::memcmp(d2_out.data(), ref_d2.data(), 8 * (size_t)q) == 0);
        CHECK(count == rows.count);
        CHECK(a == (long long)std::count_if(ref_id.begin(), ref_id.end(), [](unsigned v) { return v != 0xFFFFFFFFu; }));
        assigned_total += a;
      }
    }
    // apply: both managers take the same updates
    std::vector<unsigned> ia((size_t)q), ib((size_t)q);
    std::vector<double> da((size_t)q), db((size_t)q);
    CHECK(sharded->associate(t1, q, det.data(), 11.34, 8, 1, ia.data(), da.data(), nullptr) ==
          plain->associate(t1, q, det.data(), 11.34, 8, 1, ib.data(), db.data(), nullptr));
    CHECK(ia == ib);
    std::vector<double> ea(7 * (size_t)n), eb(7 * (size_t)n);
    sharded->getEstimatesBatch(n, ids.data(), nullptr, ea.data(), nullptr, nullptr, nullptr);
    plain->getEstimatesBatch(n, ids.data(), nullptr, eb.data(), nullptr, nullptr, nullptr);
    CHECK(std::memcmp(ea.data(), eb.data(), 8 * ea.size()) == 0);
    for (unsigned i = 0; i < n; i += 97) {
      const auto sa = sharded->getTarget(ids[i]), sb = plain->getTarget(ids[i]);
      CHECK(sa->getTime() == sb->getTime() && sa->getNumberMeasurements() == sb->getNumberMeasurements());
    }
  }
  CHECK(assigned_total > 0);
  std::printf("assigned %lld\n", assigned_total);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
