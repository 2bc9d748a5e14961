// tests/cpp/isolver_sharded_test.cpp -- the C++ IntersectionSolver on a ShardedTargetManager: one solver object (stream 0, the
// reference's per-id methods) queries ids of every shard in turn, and a second one uses the batched query() with a stream per id
// and a repeated stream.  Every result must equal, bit for bit, that of the same solver on one plain TargetManager fed the same
// calls.  Built and run by tests/test_gpu_isolver_handles.py (needs a GPU).  Usage: isolver_sharded_test <models dir> <shards>
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

static bool same(const void* a, const void* b, size_t bytes) { return std::memcmp(a, b, bytes) == 0; }

int main(int argc, char** argv) {
  const std::string models = argc > 1 ? argv[1] : "models";
  const int G = argc > 2 ? std::atoi(argv[2]) : 3;
  const double dt = 1.0 / 250.0;
  const std::string ua = models + "/model_uniform_acceleration_params.yaml";
  std::vector<int> devices((size_t)G, 0);
  std::shared_ptr<ShardedTargetManager> sharded(new ShardedTargetManager(ua, G, devices.data()));
  std::shared_ptr<TargetManager> plain(new TargetManager(ua, 0));
  plain->quiet = true;
  const unsigned n = 12;
  std::mt19937 rng(3);
  std::uniform_real_distribution<double> u(-3.0, 3.0);
  std::normal_distribution<double> noise(0.0, 0.002);
  std::vector<double> x0(n), y0(n), vx(n);
  for (unsigned i = 0; i < n; ++i) {
    x0[i] = u(rng); y0[i] = u(rng); vx[i] = u(rng) / 2;
  }
  auto pose_at = [&](unsigned i, double t) {   // thrown sideways from 20 m, falling
    return Vector7d{x0[i] + vx[i] * t + noise(rng), y0[i] + noise(rng), 20.0 - 0.5 * 9.81 * t * t + noise(rng), 0.0, 0.0, 0.0, 1.0};
  };
  for (unsigned i = 0; i < n; ++i) {
    const Vector7d p = pose_at(i, 0.0);
    sharded->init(i, dt, 0.0, p);
    plain->init(i, dt, 0.0, p);
  }
  IntersectionSolver one_sh(sharded, 10), one_pl(plain, 10);
  IntersectionSolver batch_sh(sharded, 10, n), batch_pl(plain, 10, n);
  double t = 0.0;
  int n_hit = 0;
  for (unsigned k = 0; k < 300; ++k) {
    t += dt;
    for (unsigned i = 0; i < n; ++i) {
      const Vector7d m = pose_at(i, t);
      CHECK(sharded->update(i, dt, m));
      CHECK(plain->update(i, dt, m));
    }
    if (k < 200) continue;
    for (unsigned j = 0; j < n; ++j) {   // per id, every shard in turn, one solver state
      const unsigned id = (j * 5 + k) % n;
      const Vector3d origin{x0[id] + vx[id] * (t + 0.3), y0[id], 20.0 - 0.5 * 9.81 * (t + 0.3) * (t + 0.3)};
      const double da = one_sh.getIntersectionTimeWithSphere(id, t, origin, 0.5), db = one_pl.getIntersectionTimeWithSphere(id, t, origin, 0.5);
      CHECK(same(&da, &db, 8));
      n_hit += da >= 0.0;
      Vector7d pa, pb;
      const bool ca = one_sh.getIntersectionPoseWithSphere(id, t, 0.05, 0.1, origin, 0.5, pa);
      const bool cb = one_pl.getIntersectionPoseWithSphere(id, t, 0.05, 0.1, origin, 0.5, pb);
      CHECK(ca == cb && same(pa.data(), pb.data(), 56));
    }
    // batched: stream j for query j, ids rotated every tick (the states change shard), stream 0 repeated at the end; one unknown id
    std::vector<unsigned> ids(n + 2);
    std::vector<int> stream(n + 2);
    std::vector<double> t1(n + 2, t), origin(3 * (n + 2)), radius(n + 2, 0.6), th(n + 2, 0.5);
    for (unsigned j = 0; j < n + 2; ++j) {
      ids[j] = j < n ? (j + k) % n : (j == n ? 1000u : k % n);
      stream[j] = j < n ? (int)j : 0;
      const unsigned i = ids[j] % n;
      origin[3 * j] = x0[i] + vx[i] * (t + 0.3);
      origin[3 * j + 1] = y0[i];
      origin[3 * j + 2] = 20.0 - 0.5 * 9.81 * (t + 0.3) * (t + 0.3);
    }
    std::vector<double> da(n + 2), db(n + 2), pa(7 * (n + 2)), pb(7 * (n + 2));
    std::vector<unsigned char> ca(n + 2), cb(n + 2);
    const long long fa = batch_sh.query(n + 2, ids.data(), stream.data(), t1.data(), origin.data(), radius.data(), th.data(), th.data(),
                                        da.data(), pa.data(), ca.data());
    const long long fb = batch_pl.query(n + 2, ids.data(), stream.data(), t1.data(), origin.data(), radius.data(), th.data(), th.data(),
                                        db.data(), pb.data(), cb.data());
    CHECK(fa == (long long)n + 1 && fb == fa);
    CHECK(same(da.data(), db.data(), 8 * da.size()) && same(pa.data(), pb.data(), 8 * pa.size()) && ca == cb);
    CHECK(da[n] == -1.0 && ca[n] == 0 && pa[7 * n + 6] == 1.0);
  }
  CHECK(n_hit > 500);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
