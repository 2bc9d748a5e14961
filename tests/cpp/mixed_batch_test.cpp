// tests/cpp/mixed_batch_test.cpp -- the batched calls of managers that hold three model types: uniform acceleration from the YAML's
// defaults, angular rates and uniform velocity made by init(type, ...), ids interleaved so that every shard of three holds two types.
// One plain TargetManager and one ShardedTargetManager hold the same targets; the reference is one homogeneous plain TargetManager
// per model type that receives exactly the records of its ids, in call order.  A target's arithmetic does not depend on the pool
// or manager that holds it, so every comparison is bit for bit.  Built and run by tests/test_gpu_mixed_batches.py (needs a GPU).
// Usage: mixed_batch_test <models dir> <shards> [checks | nomeas | <targets>]
//   checks (default)  updateBatch / getEstimatesBatch / initBatch / eraseBatch / log / IntersectionSolver::query / nearestTargets /
//                     earliestIntersections over some 50 ticks
//   nomeas            updateBatch without measurements: update ops raise std::invalid_argument before any pool is stepped
//   <targets>         host wall time of the batched calls of both mixed managers at that many targets (no checks)
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <numeric>
#include <random>
#include <stdexcept>
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

static const double DT = 1.0 / 250.0;
static const char* YAML[3] = {"uniform_acceleration", "angular_rates", "uniform_velocity"};
static const TargetManager::target_t TYPE[3] = {TargetManager::UNIFORM_ACCELERATION, TargetManager::ANGULAR_RATES,
                                                TargetManager::UNIFORM_VELOCITY};
static const unsigned UNKNOWN[3] = {1, 13, 100001};   // ids no manager ever holds (every target id is even)

template <class T> static bool sameBits(const std::vector<T>& a, const std::vector<T>& b) {
  return a.size() == b.size() && std::memcmp(a.data(), b.data(), sizeof(T) * a.size()) == 0;
}

struct World {
  std::string models;
  int G = 1;
  MatrixXd Q[3], R[3], P[3];
  std::shared_ptr<TargetManager> plain;
  std::shared_ptr<ShardedTargetManager> sharded;
  std::shared_ptr<TargetManager> ref[3];
  std::vector<unsigned> ids;   // every target ever made, ascending
  std::vector<int> type_of;    // [id] index into TYPE, -1 = no target
  std::vector<double> x0, y0, z0, vx, vy;
  std::mt19937 rng{11};

  TargetManager* mixed(int w) { return w == 0 ? plain.get() : (TargetManager*)sharded.get(); }
  int typeOf(unsigned id) const { return id < type_of.size() ? type_of[id] : -1; }
  void pose(unsigned id, double t, double* p7) {
    const double m[7] = {x0[id] + vx[id] * t, y0[id] + vy[id] * t, z0[id] - 0.5 * 9.81 * t * t, 0.0, 0.0, 0.0, 1.0};
    std::memcpy(p7, m, 56);
  }
  // id -> (type, position of the record among the records of that type): what a reference manager receives
  void split(const std::vector<unsigned>& b, std::vector<long long> rows[3]) const {
    for (int t = 0; t < 3; ++t) rows[t].clear();
    for (size_t k = 0; k < b.size(); ++k)
      if (typeOf(b[k]) >= 0) rows[typeOf(b[k])].push_back((long long)k);
  }

  void setup(const std::string& dir, int shards, unsigned n, bool per_id) {
    models = dir;
    G = shards;
    const std::string ua = models + "/model_uniform_acceleration_params.yaml";
    std::vector<int> devices((size_t)G, 0);
    plain.reset(new TargetManager(ua, 0));
    plain->quiet = true;
    sharded.reset(new ShardedTargetManager(ua, G, devices.data()));
    for (int t = 0; t < 3; ++t) {
      ref[t].reset(new TargetManager(ua, 0));
      ref[t]->quiet = true;
      TargetManager::target_t ty;
      CHECK(plain->loadYamlFile(models + "/model_" + YAML[t] + "_params.yaml", Q[t], R[t], P[t], ty) && ty == TYPE[t]);
    }
    // ids 10, 12, 14, ...: model type (k / 2) % 3 of the k-th id, so that owner (id mod 3) and type are independent
    std::vector<unsigned> of_type[3];
    for (unsigned k = 0; k < n; ++k) {
      ids.push_back(10 + 2 * k);
      of_type[(k / 2) % 3].push_back(10 + 2 * k);
    }
    grow(ids.back() + 1000);
    for (unsigned k = 0; k < n; ++k) type_of[ids[k]] = (int)((k / 2) % 3);
    std::vector<TargetManager*> all = {plain.get(), sharded.get()};
    for (int t = 0; t < 3; ++t) all.push_back(ref[t].get());
    for (int t = 0; t < 3; ++t) {
      const std::vector<unsigned>& v = of_type[t];
      std::vector<double> p0(7 * v.size()), t0(v.size(), 0.0);
      for (size_t k = 0; k < v.size(); ++k) pose(v[k], 0.0, &p0[7 * k]);
      for (TargetManager* m : all) {
        if (m == ref[(t + 1) % 3].get() || m == ref[(t + 2) % 3].get()) continue;
        if (t == 0) {
          CHECK(m->initBatch((long long)v.size(), v.data(), DT, t0.data(), p0.data()) == (long long)v.size());
        } else if (per_id) {
          for (size_t k = 0; k < v.size(); ++k) {
            Vector7d p;
            std::memcpy(p.data(), &p0[7 * k], 56);
            m->init(TYPE[t], v[k], DT, 0.0, Q[t], R[t], P[t], p);
          }
        } else {
          CHECK(m->initBatch(TYPE[t], Q[t], R[t], P[t], (long long)v.size(), v.data(), DT, t0.data(), p0.data()) == (long long)v.size());
        }
      }
    }
  }
  void grow(size_t n) {
    std::uniform_real_distribution<double> u(-5.0, 5.0), uv(-2.0, 2.0);
    for (size_t i = type_of.size(); i < n; ++i) {
      type_of.push_back(-1);
      x0.push_back(u(rng)); y0.push_back(u(rng)); z0.push_back(20.0 + u(rng)); vx.push_back(uv(rng)); vy.push_back(uv(rng));
    }
  }
  std::vector<unsigned> live() const {
    std::vector<unsigned> v;
    for (unsigned id : ids)
      if (typeOf(id) >= 0) v.push_back(id);
    return v;
  }
};

// ---- updateBatch: the mixed managers against the references fed the records of their ids -----------------------------------------
static void updateAndCompare(World& w, const std::vector<unsigned>& b, const double* meas, const unsigned char* act) {
  std::vector<long long> rows[3];
  w.split(b, rows);
  long long want = 0;
  for (int t = 0; t < 3; ++t) {
    std::vector<unsigned> s_ids;
    std::vector<double> s_meas;
    std::vector<unsigned char> s_act;
    for (long long k : rows[t]) {
      s_ids.push_back(b[(size_t)k]);
      if (meas) s_meas.insert(s_meas.end(), meas + 7 * k, meas + 7 * k + 7);
      if (act) s_act.push_back(act[k]);
    }
    if (!s_ids.empty())
      want += w.ref[t]->updateBatch((long long)s_ids.size(), s_ids.data(), DT, meas ? s_meas.data() : nullptr, act ? s_act.data() : nullptr);
  }
  for (int m = 0; m < 2; ++m) CHECK(w.mixed(m)->updateBatch((long long)b.size(), b.data(), DT, meas, act) == want);
}

// ---- getEstimatesBatch: per-row t1 (or NULL), all four outputs, unknown ids; outputs pre-filled with a sentinel -----------------
static void estimatesAndCompare(World& w, double t, bool with_t1) {
  std::vector<unsigned> b = w.live();
  b.insert(b.begin() + (long)(b.size() / 3), UNKNOWN[0]);
  b.push_back(UNKNOWN[2]);
  std::shuffle(b.begin(), b.end(), w.rng);
  const size_t n = b.size();
  std::vector<double> t1(n);
  for (size_t k = 0; k < n; ++k) t1[k] = t + 0.001 * (double)(k % 7);
  const double SENTINEL = -12345.678;
  std::vector<double> pose[2], twist[2], acc[2];
  std::vector<unsigned char> found[2];
  for (int m = 0; m < 2; ++m) {
    pose[m].assign(7 * n, SENTINEL); twist[m].assign(6 * n, SENTINEL); acc[m].assign(6 * n, SENTINEL); found[m].assign(n, 7);
    w.mixed(m)->getEstimatesBatch((long long)n, b.data(), with_t1 ? t1.data() : nullptr, pose[m].data(), twist[m].data(), acc[m].data(),
                                  found[m].data());
  }
  std::vector<double> e_pose(7 * n), e_twist(6 * n), e_acc(6 * n);
  std::vector<unsigned char> e_found(n, 0);
  std::vector<long long> rows[3];
  w.split(b, rows);
  for (int t = 0; t < 3; ++t) {
    const size_t m = rows[t].size();
    if (!m) continue;
    std::vector<unsigned> s_ids;
    std::vector<double> s_t1, po(7 * m), tw(6 * m), ac(6 * m);
    std::vector<unsigned char> fo(m);
    for (long long k : rows[t]) { s_ids.push_back(b[(size_t)k]); s_t1.push_back(t1[(size_t)k]); }
    w.ref[t]->getEstimatesBatch((long long)m, s_ids.data(), with_t1 ? s_t1.data() : nullptr, po.data(), tw.data(), ac.data(), fo.data());
    for (size_t i = 0; i < m; ++i) {
      const size_t k = (size_t)rows[t][i];
      std::memcpy(&e_pose[7 * k], &po[7 * i], 56);
      std::memcpy(&e_twist[6 * k], &tw[6 * i], 48);
      std::memcpy(&e_acc[6 * k], &ac[6 * i], 48);
      e_found[k] = fo[i];
      CHECK(fo[i] == 1);
    }
  }
  for (int m = 0; m < 2; ++m) {
    // rows of unknown ids: the plain manager (and a sharded one of one shard, which hands the call to it) leaves them as they were,
    // a sharded one of several shards copies them from zeroed buffers
    const double unknown = (m == 0 || w.G == 1) ? SENTINEL : 0.0;
    std::vector<double> ep = e_pose, et = e_twist, ea = e_acc;
    for (size_t k = 0; k < n; ++k)
      if (w.typeOf(b[k]) < 0) {
        std::fill(&ep[7 * k], &ep[7 * k + 7], unknown);
        std::fill(&et[6 * k], &et[6 * k + 6], unknown);
        std::fill(&ea[6 * k], &ea[6 * k + 6], unknown);
      }
    CHECK(sameBits(pose[m], ep));
    CHECK(sameBits(twist[m], et));
    CHECK(sameBits(acc[m], ea));
    CHECK(found[m] == e_found);
  }
}

// one tick's measurements of the batch b (every record its own noise)
static std::vector<double> measOf(World& w, const std::vector<unsigned>& b, double t) {
  std::normal_distribution<double> noise(0.0, 0.002);
  std::vector<double> m(7 * b.size());
  for (size_t k = 0; k < b.size(); ++k) {
    w.pose(b[k] < w.x0.size() ? b[k] : 0, t, &m[7 * k]);
    for (int c = 0; c < 3; ++c) m[7 * k + c] += noise(w.rng);
  }
  return m;
}

// the batch of tick `tick`: ascending, shuffled, with repeats, with unknown ids; action NULL or a mix of UPDATE / PREDICT / NONE
static void tickBatch(World& w, int tick, double t) {
  std::vector<unsigned> b = w.live();
  const int kind = tick % 5;
  if (kind == 1 || kind == 3)   // unknown ids, in ascending place
    for (unsigned id : {UNKNOWN[0], UNKNOWN[1]}) b.insert(std::lower_bound(b.begin(), b.end(), id), id);
  if (kind == 2 || kind == 4) {   // a quarter of the ids two or three more times
    const std::vector<unsigned> base = b;
    for (size_t k = 0; k < base.size(); k += 4) {
      b.push_back(base[k]);
      if (k % 8 == 0) b.push_back(base[k]);
    }
  }
  if (kind != 0 && kind != 3) std::shuffle(b.begin(), b.end(), w.rng);
  const std::vector<double> meas = measOf(w, b, t);
  std::vector<unsigned char> act(b.size());
  for (size_t k = 0; k < b.size(); ++k) act[k] = (unsigned char)(w.rng() % 5 == 0 ? TE_ACT_PREDICT : (w.rng() % 7 == 0 ? TE_ACT_NONE : TE_ACT_UPDATE));
  updateAndCompare(w, b, meas.data(), (kind == 0 || kind == 4) ? nullptr : act.data());
}

// ---- initBatch of the default type over ids that live under another type (skipped; the registry keeps the type) + fresh ids ----
static void initOverOtherTypes(World& w, double t) {
  std::vector<unsigned> b, fresh;
  const std::vector<unsigned> live = w.live();
  for (size_t k = 0; k < live.size(); k += 5) b.push_back(live[k]);
  for (unsigned k = 0; k < 12; ++k) fresh.push_back(w.ids.back() + 2 + 2 * k);
  b.insert(b.end(), fresh.begin(), fresh.end());
  std::shuffle(b.begin(), b.end(), w.rng);
  const std::vector<double> p0 = measOf(w, b, t);
  std::vector<double> t0(b.size(), t);
  std::vector<int> before(b.size());
  for (size_t k = 0; k < b.size(); ++k) before[k] = w.typeOf(b[k]);
  // the reference of the default type receives the ids no other reference holds
  std::vector<unsigned> r_ids;
  std::vector<double> r_p0, r_t0;
  for (size_t k = 0; k < b.size(); ++k)
    if (before[k] <= 0) { r_ids.push_back(b[k]); r_p0.insert(r_p0.end(), &p0[7 * k], &p0[7 * k + 7]); r_t0.push_back(t); }
  const long long want = w.ref[0]->initBatch((long long)r_ids.size(), r_ids.data(), DT, r_t0.data(), r_p0.data());
  CHECK(want == (long long)fresh.size());
  for (int m = 0; m < 2; ++m) CHECK(w.mixed(m)->initBatch((long long)b.size(), b.data(), DT, t0.data(), p0.data()) == want);
  for (unsigned id : fresh) {
    w.ids.push_back(id);
    w.type_of[id] = 0;
  }
  for (size_t k = 0; k < b.size(); ++k) {
    int ty = -1;
    CHECK(w.plain->typeOf(b[k], ty) && ty == (int)TYPE[std::max(before[k], 0)]);
    ty = -1;
    CHECK(w.sharded->shard(w.sharded->owner(b[k])).typeOf(b[k], ty) && ty == (int)TYPE[std::max(before[k], 0)]);
  }
}

// ---- eraseBatch with unknown and repeated ids ------------------------------------------------------------------------------------
static void eraseSome(World& w) {
  std::vector<unsigned> b;
  const std::vector<unsigned> live = w.live();
  for (size_t k = 3; k < live.size(); k += 9) {
    b.push_back(live[k]);
    if (k % 2) b.push_back(live[k]);
  }
  b.push_back(UNKNOWN[1]);
  b.push_back(b.front());
  std::shuffle(b.begin(), b.end(), w.rng);
  std::vector<long long> rows[3];
  w.split(b, rows);
  long long want = 0;
  for (int t = 0; t < 3; ++t) {
    std::vector<unsigned> s;
    for (long long k : rows[t]) s.push_back(b[(size_t)k]);
    if (!s.empty()) want += w.ref[t]->eraseBatch((long long)s.size(), s.data());
  }
  std::vector<unsigned> distinct = b;
  std::sort(distinct.begin(), distinct.end());
  distinct.erase(std::unique(distinct.begin(), distinct.end()), distinct.end());
  CHECK(want == (long long)distinct.size() - 1);
  for (int m = 0; m < 2; ++m) CHECK(w.mixed(m)->eraseBatch((long long)b.size(), b.data()) == want);
  for (unsigned id : b)
    if (w.typeOf(id) >= 0) w.type_of[id] = -1;
  std::vector<unsigned> all;
  for (int t = 0; t < 3; ++t) {
    const std::vector<unsigned> v = w.ref[t]->getAvailableTargets();
    all.insert(all.end(), v.begin(), v.end());
  }
  std::sort(all.begin(), all.end());
  CHECK(all == w.live());
  for (int m = 0; m < 2; ++m) CHECK(w.mixed(m)->getAvailableTargets() == all);
}

// ---- IntersectionSolver::query: times only and with pose, several streams, a repeated stream --------------------------------------
struct Solvers {
  std::unique_ptr<IntersectionSolver> mixed[2], ref[3];
  explicit Solvers(World& w) {
    mixed[0].reset(new IntersectionSolver(w.plain, 20, 4));
    mixed[1].reset(new IntersectionSolver(w.sharded, 20, 4));
    for (int t = 0; t < 3; ++t) ref[t].reset(new IntersectionSolver(w.ref[t], 20, 4));
  }
};

static void queryAndCompare(World& w, Solvers& s, double t, bool with_pose) {
  const std::vector<unsigned> live = w.live();
  std::vector<unsigned> b;
  std::vector<int> st;
  for (int j = 0; j < 9; ++j) {
    b.push_back(live[(size_t)(j * 37 + (int)(t * 1000)) % live.size()]);
    st.push_back(j % 4);   // streams 0 .. 3, each more than once
  }
  b.insert(b.begin() + 4, UNKNOWN[2]);
  st.insert(st.begin() + 4, 2);
  const size_t n = b.size();
  std::vector<double> t1(n, t), origin(3 * n), radius(n), pth(n, 0.05), ath(n, 0.05);
  for (size_t k = 0; k < n; ++k) {
    double p[7];
    w.pose(b[k] < w.x0.size() ? b[k] : 0, t + 0.3, p);
    std::memcpy(&origin[3 * k], p, 24);
    radius[k] = 0.5 + 0.1 * (double)k;
    t1[k] = t + 0.0005 * (double)(k % 3);
  }
  std::vector<double> d[2], p[2];
  std::vector<unsigned char> c[2];
  long long found[2];
  for (int m = 0; m < 2; ++m) {
    d[m].assign(n, 9.0); p[m].assign(with_pose ? 7 * n : 0, 9.0); c[m].assign(n, 9);
    found[m] = s.mixed[m]->query((long long)n, b.data(), with_pose ? st.data() : nullptr, t1.data(), origin.data(), radius.data(),
                                 pth.data(), ath.data(), d[m].data(), with_pose ? p[m].data() : nullptr, c[m].data());
  }
  static const double init_pose[7] = {0, 0, 0, 0, 0, 0, 1};
  std::vector<double> ed(n, -1.0), ep(with_pose ? 7 * n : 0);
  std::vector<unsigned char> ec(n, 0);
  for (size_t k = 0; k < ep.size() / 7; ++k) std::memcpy(&ep[7 * k], init_pose, 56);
  std::vector<long long> rows[3];
  w.split(b, rows);
  long long want = 0;
  for (int ty = 0; ty < 3; ++ty) {
    const size_t m = rows[ty].size();
    if (!m) continue;
    std::vector<unsigned> s_ids;
    std::vector<int> s_st;
    std::vector<double> s_t1, s_o, s_r, s_pth, s_ath, sd(m), sp(7 * m);
    std::vector<unsigned char> sc(m);
    for (long long k : rows[ty]) {
      s_ids.push_back(b[(size_t)k]); s_st.push_back(st[(size_t)k]); s_t1.push_back(t1[(size_t)k]);
      s_o.insert(s_o.end(), &origin[3 * k], &origin[3 * k + 3]); s_r.push_back(radius[(size_t)k]);
      s_pth.push_back(pth[(size_t)k]); s_ath.push_back(ath[(size_t)k]);
    }
    want += s.ref[ty]->query((long long)m, s_ids.data(), with_pose ? s_st.data() : nullptr, s_t1.data(), s_o.data(), s_r.data(), s_pth.data(),
                             s_ath.data(), sd.data(), with_pose ? sp.data() : nullptr, sc.data());
    for (size_t i = 0; i < m; ++i) {
      const size_t k = (size_t)rows[ty][i];
      ed[k] = sd[i];
      if (with_pose) { std::memcpy(&ep[7 * k], &sp[7 * i], 56); ec[k] = sc[i]; }
    }
  }
  CHECK(want == (long long)n - 1);
  for (int m = 0; m < 2; ++m) {
    CHECK(found[m] == want);
    CHECK(sameBits(d[m], ed));
    if (with_pose) {
      CHECK(sameBits(p[m], ep));
      CHECK(c[m] == ec);
    }
  }
}

// ---- nearestTargets / earliestIntersections: the mixed rows are the merge of the references' rows -------------------------------
static void mergeRefs(const std::vector<unsigned>* ids, const std::vector<double>* val, const std::vector<long long>* cnt, long long q,
                      long long k, std::vector<unsigned>& m_ids, std::vector<double>& m_val, std::vector<long long>& m_cnt) {
  m_ids.assign((size_t)(q * k), 0xFFFFFFFFu);
  m_val.assign((size_t)(q * k), -1.0);
  m_cnt.assign((size_t)q, 0);
  for (long long j = 0; j < q; ++j) {
    std::vector<std::pair<double, unsigned>> rows;
    for (int t = 0; t < 3; ++t) {
      m_cnt[(size_t)j] += cnt[t][(size_t)j];
      for (long long r = 0; r < std::min(k, cnt[t][(size_t)j]); ++r) rows.emplace_back(val[t][(size_t)(j * k + r)], ids[t][(size_t)(j * k + r)]);
    }
    std::sort(rows.begin(), rows.end(), [](const std::pair<double, unsigned>& a, const std::pair<double, unsigned>& b) {
      return a.first < b.first || (a.first == b.first && a.second < b.second);
    });
    for (long long r = 0; r < std::min(k, (long long)rows.size()); ++r) {
      m_val[(size_t)(j * k + r)] = rows[(size_t)r].first;
      m_ids[(size_t)(j * k + r)] = rows[(size_t)r].second;
    }
  }
}

static void rowQueries(World& w, Solvers& s, double t) {
  const long long q = 5, k = 40;
  std::vector<double> t1(q, t + 0.02), point(3 * q), radius(q);
  const std::vector<unsigned> live = w.live();
  for (long long j = 0; j < q; ++j) {
    double p[7];
    w.pose(live[(size_t)(j * 53) % live.size()], t + 0.2, p);
    std::memcpy(&point[3 * j], p, 24);
    radius[j] = 2.0 + 0.5 * (double)j;
  }
  for (int which = 0; which < 2; ++which) {
    std::vector<unsigned> r_ids[3];
    std::vector<double> r_val[3];
    std::vector<long long> r_cnt[3];
    auto run = [&](int m, int ref, std::vector<unsigned>& ids, std::vector<double>& val, std::vector<long long>& cnt) {
      ids.assign((size_t)(q * k), 0); val.assign((size_t)(q * k), 0.0); cnt.assign((size_t)q, 0);
      if (which == 0) {
        TargetManager* mgr = ref >= 0 ? w.ref[ref].get() : w.mixed(m);
        return mgr->nearestTargets(q, t1.data(), point.data(), radius.data(), k, ids.data(), val.data(), cnt.data());
      }
      IntersectionSolver* sv = ref >= 0 ? s.ref[ref].get() : s.mixed[m].get();
      return sv->earliestIntersections(q, t1.data(), point.data(), radius.data(), k, ids.data(), val.data(), cnt.data());
    };
    long long want = 0;
    for (int t = 0; t < 3; ++t) want += run(0, t, r_ids[t], r_val[t], r_cnt[t]);
    std::vector<unsigned> e_ids;
    std::vector<double> e_val;
    std::vector<long long> e_cnt;
    mergeRefs(r_ids, r_val, r_cnt, q, k, e_ids, e_val, e_cnt);
    CHECK(want > 0);
    for (int m = 0; m < 2; ++m) {
      std::vector<unsigned> ids;
      std::vector<double> val;
      std::vector<long long> cnt;
      CHECK(run(m, -1, ids, val, cnt) == want);
      CHECK(ids == e_ids && sameBits(val, e_val) && cnt == e_cnt);
    }
  }
}

// ---- sampled logging over ids of all three types and an unknown id ----------------------------------------------------------------
// (wtype[j]: model type of watched[j] when the watch began, -1 = unknown id)
static void compareLogs(World& w, const std::vector<unsigned>& watched, const std::vector<int>& wtype) {
  const size_t S = w.plain->logSamples();
  CHECK(S > 0);
  for (size_t j = 0; j < watched.size(); ++j) {
    const unsigned id = watched[j];
    const int ty = wtype[j];
    size_t jr = 0, js = 0;   // the place of watched[j] in the lists its reference and its shard were given
    for (size_t i = 0; i < j; ++i) {
      if (ty >= 0 && wtype[i] == ty) ++jr;
      if (w.sharded->owner(watched[i]) == w.sharded->owner(id)) ++js;
    }
    TargetManager& sh = w.sharded->shard(w.sharded->owner(id));
    CHECK(sh.logSamples() == S);
    for (size_t k = 0; k < S; ++k) {
      std::vector<double> row[3], P[3];
      int ns[3] = {-1, -1, -1};
      bool ok[3];
      for (int m = 0; m < 3; ++m) { row[m].assign(26, 5.0); P[m].assign(324, 5.0); }
      ok[0] = w.plain->logSample(k, j, row[0].data(), P[0].data(), &ns[0]);
      ok[1] = sh.logSample(k, js, row[1].data(), P[1].data(), &ns[1]);
      if (ty >= 0) {
        ok[2] = w.ref[ty]->logSample(k, jr, row[2].data(), P[2].data(), &ns[2]);
      } else {   // an id no manager holds
        ok[2] = false;
        ns[2] = 0;
        row[2] = row[0];
        P[2] = P[0];
      }
      for (int m = 0; m < 2; ++m) CHECK(ok[m] == ok[2] && ns[m] == ns[2] && sameBits(row[m], row[2]) && sameBits(P[m], P[2]));
    }
  }
}

static void checks(World& w) {
  std::vector<unsigned> watched;
  std::vector<int> wtype;
  {
    const std::vector<unsigned> live = w.live();
    for (size_t k = 0; k < 24; ++k) watched.push_back(live[k * 23 + 1]);   // some of them are erased on the way
    watched.insert(watched.begin() + 5, UNKNOWN[0]);
    for (unsigned id : watched) wtype.push_back(w.typeOf(id));
    for (int m = 0; m < 2; ++m) w.mixed(m)->watch((long long)watched.size(), watched.data(), 1000);
    for (int t = 0; t < 3; ++t) {
      std::vector<unsigned> mine;
      for (unsigned id : watched)
        if (w.typeOf(id) == t) mine.push_back(id);
      w.ref[t]->watch((long long)mine.size(), mine.data(), 1000);
    }
  }
  Solvers s(w);
  double t = 0.0;
  for (int tick = 0; tick < 50; ++tick) {
    t += DT;
    tickBatch(w, tick, t);
    if (tick == 20) initOverOtherTypes(w, t);
    if (tick == 30) eraseSome(w);
    if (tick % 4 == 3) estimatesAndCompare(w, t, tick % 8 == 3);
    if (tick >= 10 && tick % 3 == 0) queryAndCompare(w, s, t, tick % 6 != 0);
    if (tick % 5 == 4) {
      w.plain->log();
      w.sharded->log();
      for (int ty = 0; ty < 3; ++ty) w.ref[ty]->log();
    }
  }
  estimatesAndCompare(w, t, true);
  rowQueries(w, s, t);
  compareLogs(w, watched, wtype);
}

// ---- updateBatch without measurements -------------------------------------------------------------------------------------------
static void noMeasurements(World& w) {
  double t = 0.0;
  for (int tick = 0; tick < 5; ++tick) {
    t += DT;
    tickBatch(w, tick, t);
  }
  std::vector<unsigned> b = w.live();
  std::shuffle(b.begin(), b.end(), w.rng);
  std::vector<unsigned char> predict(b.size(), TE_ACT_PREDICT), one_update(b.size(), TE_ACT_PREDICT);
  one_update[b.size() / 2] = TE_ACT_UPDATE;
  for (int m = 0; m < 2; ++m)
    for (const unsigned char* act : {(const unsigned char*)nullptr, (const unsigned char*)one_update.data()}) {
      bool raised = false;
      try {
        w.mixed(m)->updateBatch((long long)b.size(), b.data(), DT, nullptr, act);
      } catch (const std::invalid_argument& e) {
        raised = std::string(e.what()) == "update ops without measurements";
      }
      CHECK(raised);
    }
  // nothing was stepped, and prediction-only batches need no measurements
  t += DT;
  updateAndCompare(w, b, nullptr, predict.data());
  estimatesAndCompare(w, t, false);
}

static void timing(World& w, unsigned n) {
  typedef std::chrono::steady_clock clk;
  auto ms = [](clk::time_point a) { return std::chrono::duration<double, std::milli>(clk::now() - a).count(); };
  std::vector<unsigned> b = w.live();
  std::shuffle(b.begin(), b.end(), w.rng);
  const std::vector<double> meas = measOf(w, b, DT);
  std::vector<double> pose(7 * b.size()), twist(6 * b.size()), acc(6 * b.size());
  std::vector<unsigned char> found(b.size());
  std::vector<unsigned> again(b.begin(), b.begin() + (long)(b.size() / 10));
  const std::vector<double> p0 = measOf(w, again, DT);
  std::vector<double> t0(again.size(), DT);
  const char* name[2] = {"plain", "sharded"};
  for (int m = 0; m < 2; ++m) {
    TargetManager* mgr = w.mixed(m);
    for (int rep = 0; rep < 3; ++rep) {
      clk::time_point a = clk::now();
      mgr->updateBatch((long long)b.size(), b.data(), DT, meas.data());
      const double upd = ms(a);
      a = clk::now();
      mgr->getEstimatesBatch((long long)b.size(), b.data(), nullptr, pose.data(), twist.data(), acc.data(), found.data());
      const double est = ms(a);
      a = clk::now();
      const long long erased = mgr->eraseBatch((long long)again.size(), again.data());
      const double era = ms(a);
      a = clk::now();
      const long long added = mgr->initBatch((long long)again.size(), again.data(), DT, t0.data(), p0.data());
      const double ini = ms(a);
      CHECK(erased == (long long)again.size() && added == erased);
      std::printf("timing %s G=%d targets=%u rep=%d: updateBatch(shuffled) %.2f ms, getEstimatesBatch(shuffled) %.2f ms, eraseBatch(%zu) %.2f ms, "
                  "initBatch(%zu) %.2f ms\n", name[m], w.G, n, rep, upd, est, again.size(), era, again.size(), ini);
    }
  }
}

int main(int argc, char** argv) {
  const std::string models = argc > 1 ? argv[1] : "models";
  const int G = argc > 2 ? std::atoi(argv[2]) : 3;
  const std::string mode = argc > 3 ? argv[3] : "checks";
  World w;
  const bool sized = mode != "checks" && mode != "nomeas";
  const unsigned n = sized ? (unsigned)std::atol(mode.c_str()) : 600;
  w.setup(models, G, n, !sized);
  if (mode == "checks") checks(w);
  else if (mode == "nomeas") noMeasurements(w);
  else timing(w, n);
  std::printf("%s: %d checks, %d failed\n", g_failed ? "FAILED" : "ok", g_checks, g_failed);
  return g_failed ? 1 : 0;
}
