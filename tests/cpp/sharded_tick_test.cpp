// tests/cpp/sharded_tick_test.cpp -- ShardedTickTargetManager with ids the shards know under ANOTHER model type than the tick's
// (created by hand through the typed init): those shards keep host mailboxes, so every message takes the host route (the router
// threads, then each shard's measurementCallBackIds).  Every observable -- erased lists, ids, mailbox count, clock, the published
// poses, n_meas and the filter state of every target -- must equal, bit for bit, that of one TickTargetManager fed the same
// messages.  Built and run by tests/test_gpu_sharded_tick.py (needs a GPU).  Usage: sharded_tick_test <models dir> <shards>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
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

int main(int argc, char** argv) {
  const std::string models = argc > 1 ? argv[1] : "models";
  const int G = argc > 2 ? std::atoi(argv[2]) : 3;
  const double dt = 1.0 / 250.0;
  const std::string ua = models + "/model_uniform_acceleration_params.yaml";
  std::vector<int> devices((size_t)G, 0);
  ShardedTickTargetManager sharded(ua, G, devices.data());
  TickTargetManager one(ua, 0);
  one.quiet = true;
  sharded.setExpirationTime(6 * dt);
  one.setExpirationTime(6 * dt);
  MatrixXd Q, R, P;
  TargetManager::target_t uv;
  CHECK(one.loadYamlFile(models + "/model_uniform_velocity_params.yaml", Q, R, P, uv));
  const unsigned foreign[3] = {5, 11, 32};   // all owned by shard 2 of three: the other shards' mailboxes stay on the device
  for (unsigned id : foreign) {
    const Vector7d p0{0.1 * id, 0.2, 0.3, 0.0, 0.0, 0.0, 1.0};
    sharded.init(uv, id, dt, 0.0, Q, R, P, p0);
    one.init(uv, id, dt, 0.0, Q, R, P, p0);
  }
  std::mt19937 rng(7);
  std::normal_distribution<double> noise(0.0, 0.01);
  const unsigned n_ids = 60;
  long long total_erased = 0;
  for (unsigned k = 0; k < 40; ++k) {
    const uint32_t sec = 1000 + k / 250, nsec = (k % 250) * 4000000u;
    std::vector<unsigned> ids;
    std::vector<uint32_t> s, ns;
    std::vector<double> poses;
    for (unsigned i = 0; i < n_ids; ++i) {
      if (i % 7 == 0 && k > 12 + i % 5 && !(i == 14 && k > 30)) continue;   // silent, then expired; 14 comes back
      const bool stale = i % 4 == 1 && k % 3 == 0 && k > 0;
      ids.push_back(i);
      s.push_back(sec);
      ns.push_back(stale ? nsec - 4000000u : nsec);
      const double v[7] = {0.1 * i + 0.01 * k + noise(rng), -0.005 * k + noise(rng), 0.3 + noise(rng), 0.0, 0.0, 0.0, 1.0};
      poses.insert(poses.end(), v, v + 7);
    }
    std::shuffle(ids.begin(), ids.end(), rng);   // (stamps and poses stay put: any record order is a valid message)
    sharded.measurementCallBackIds((long long)ids.size(), ids.data(), s.data(), ns.data(), poses.data());
    one.measurementCallBackIds((long long)ids.size(), ids.data(), s.data(), ns.data(), poses.data());
    std::vector<unsigned> er_a, er_b;
    sharded.tick(dt, sec, nsec, &er_a);
    one.tick(dt, sec, nsec, &er_b);
    CHECK(er_a == er_b);
    total_erased += (long long)er_b.size();
    const std::vector<unsigned> ids_b = one.getAvailableTargets();
    CHECK(sharded.getAvailableTargets() == ids_b);
    CHECK(sharded.mailboxCount() == one.mailboxCount());
    CHECK(sharded.time() == one.time());
    // published: shard-major on the sharded manager, ascending on the single one -- the same poses per id, bit for bit
    const std::vector<unsigned>& pa = sharded.publishedIds();
    const std::vector<unsigned>& pb = one.publishedIds();
    CHECK(pa.size() == pb.size());
    std::map<unsigned, size_t> row;
    for (size_t j = 0; j < pb.size(); ++j) row[pb[j]] = j;
    for (size_t j = 0; j < pa.size(); ++j) {
      CHECK(j == 0 || sharded.owner(pa[j - 1]) < sharded.owner(pa[j]) || pa[j - 1] < pa[j]);
      auto it = row.find(pa[j]);
      CHECK(it != row.end() && std::memcmp(&sharded.publishedPoses()[7 * j], &one.publishedPoses()[7 * it->second], 56) == 0);
    }
    for (unsigned id : ids_b) {
      CHECK(sharded.getNumberMeasurements(id) == one.getNumberMeasurements(id));
      const VectorXd xa = sharded.getTarget(id)->getEstimator()->getState(), xb = one.getTarget(id)->getEstimator()->getState();
      CHECK(xa.size() == xb.size() && std::memcmp(xa.data(), xb.data(), xa.size() * sizeof(double)) == 0);
    }
  }
  CHECK(total_erased >= 6);
  for (unsigned id : foreign) {
    int type = -1;
    CHECK(sharded.shard(sharded.owner(id)).typeOf(id, type) && type == (int)uv);
  }
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
