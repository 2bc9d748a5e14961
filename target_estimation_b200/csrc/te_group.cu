// te_group.cu -- several pools on several devices of one box: the optional NCCL all-gather of estimate records
// (SURVEY.md 8(e); BASELINE.json north_star: "NCCL over NVLink is used only for the optional all-gather of estimates / intercepts
// to the publishing rank") and the routing of /tf messages to the shards that own their ids (te_group_route_records: upload by
// position, stable partition by owner on every device, point-to-point exchange).  The step itself has no collective: every
// shard steps its own pool on its own device and stream.
//
// One process drives all devices (the host surface is the C++ ShardedTargetManager of host/sharded_manager.cpp), so the
// communicators come from ncclCommInitAll and every collective is issued for all ranks inside one ncclGroupStart / ncclGroupEnd.
// NCCL is loaded with dlopen on first use: libte_pool.so carries no link-time dependency on it, and a process that already
// holds a libnccl.so.2 (PyTorch's) shares that copy.
#include <dlfcn.h>
#include <nccl.h>

#include <cub/device/device_scan.cuh>

#include "te_pool_internal.cuh"

using namespace tehost;

namespace {

struct NcclApi {
  void* h = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

NcclApi& nccl() {
  static NcclApi api;
  if (api.h) return api;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) throw std::runtime_error(std::string("NCCL is required for a multi-device group: ") + dlerror());
  auto sym = [&](const char* name) {
    void* s = dlsym(h, name);
    if (!s) throw std::runtime_error(std::string("libnccl.so.2 lacks ") + name);
    return s;
  };
  api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
  api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
  api.GroupStart = (decltype(api.GroupStart))sym("ncclGroupStart");
  api.GroupEnd = (decltype(api.GroupEnd))sym("ncclGroupEnd");
  api.AllGather = (decltype(api.AllGather))sym("ncclAllGather");
  api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
  api.Send = (decltype(api.Send))sym("ncclSend");
  api.Recv = (decltype(api.Recv))sym("ncclRecv");
  api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
  api.h = h;
  return api;
}

#define NCK(call)                                                                                                        \
  do {                                                                                                                   \
    ncclResult_t r__ = (call);                                                                                           \
    if (r__ != ncclSuccess) throw std::runtime_error(std::string(#call) + ": " + nccl().GetErrorString(r__));            \
  } while (0)

struct Shard {
  int device = 0;
  cudaStream_t own_stream = nullptr;   // used when the shard has no pool in a gather
  cudaStream_t stream = nullptr;       // the stream of the running gather on this device
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double* rec = nullptr;               // this shard's records [count][13]
  size_t rec_cap = 0;
  double* out = nullptr;               // all shards' records [total][13]
  uint32_t* out_ids = nullptr;
  size_t out_cap = 0;
};

// records of a /tf message in SoA form inside one device block of `cap` records: poses [cap][7] | ids | sec | nsec
constexpr size_t REC_BYTES = 68;
struct Recs {
  double* pose;
  uint32_t *ids, *sec, *nsec;
};
inline Recs recs(char* base, size_t cap) {
  double* pose = (double*)base;
  uint32_t* ids = (uint32_t*)(pose + 7 * cap);
  return Recs{pose, ids, ids + cap, ids + 2 * cap};
}

// per shard: the grow-only device buffers of te_group_route_records on the shard's device
struct Route {
  cudaStream_t stream = nullptr;   // the stream of the shard's pool
  cudaEvent_t done = nullptr;      // recorded after the shard's part of the exchange
  char* in = nullptr;              // chunk of the message uploaded to this device
  char* part = nullptr;            // the same chunk partitioned by owner
  char* out = nullptr;             // this shard's records of every chunk, chunk order
  size_t in_cap = 0, part_cap = 0, out_cap = 0;   // records
  char* work = nullptr;            // owner histogram [G][blocks], its scan, the owner counts [G], scan scratch
  size_t work_cap = 0;             // bytes
  long long n_out = 0;
};

}  // namespace

struct te_group {
  std::vector<Shard> sh;
  std::vector<ncclComm_t> comms;
  bool use_nccl = false;
  std::vector<long long> counts;
  long long total = 0;
  bool timed = false;
  std::vector<Route> route;     // created on the first te_group_route_records
  int* h_route_counts = nullptr;   // page-locked [chunk][owner]
  bool routed = false;
};

// ---- routing kernels: stable partition of one chunk of a /tf message by owner = id mod G ----------------------------------------
namespace te_route {

// id mod G without a division: a mask for powers of two, else Lemire's multiply-shift remainder (exact for 32-bit operands; the
// FastMod of host/sharded_manager.cpp)
struct OwnerOf {
  unsigned d;
  bool pow2;
  unsigned long long m;
  __device__ __forceinline__ unsigned operator()(unsigned a) const {
    if (pow2) return a & (d - 1);
    return (unsigned)__umul64hi(m * (unsigned long long)a, (unsigned long long)d);
  }
};
constexpr int WARPS = 8, ITEMS = 4, TILE = WARPS * 32 * ITEMS;   // records per block; warp w of a block owns the w-th quarter-kilo run
constexpr int MAX_OWNERS = 1024;                                   // shared memory: WARPS * G cursors

// hist[r * blocks + b] = records of block b owned by r (owner-major: its exclusive scan is every (owner, block) run's place)
__global__ void __launch_bounds__(WARPS * 32) route_histogram_kernel(const uint32_t* __restrict__ ids, int m, OwnerOf owner, int* __restrict__ hist) {
  extern __shared__ int cnt[];
  const int G = (int)owner.d;
  for (int r = threadIdx.x; r < G; r += blockDim.x) cnt[r] = 0;
  __syncthreads();
  const int lo = blockIdx.x * TILE, hi = min(lo + TILE, m);
  for (int k = lo + threadIdx.x; k < hi; k += blockDim.x) atomicAdd(&cnt[owner(ids[k])], 1);
  __syncthreads();
  for (int r = threadIdx.x; r < G; r += blockDim.x) hist[(size_t)r * gridDim.x + blockIdx.x] = cnt[r];
}

// counts[r] = records owned by r, from the scanned histogram
__global__ void route_counts_kernel(const int* __restrict__ base, int blocks, int G, int m, int* __restrict__ counts) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < G) counts[r] = (r + 1 < G ? base[(size_t)(r + 1) * blocks] : m) - base[(size_t)r * blocks];
}

// Stable scatter: every record goes to base[owner][block] + (records of the same owner before it in the block).  Warp w walks its
// run of the block 32 records at a time, in order; the lanes of one step that share an owner (match.any) take consecutive places in
// lane order, so arrival order is kept inside every owner's run.  Poses move as whole 56-byte rows.
__global__ void __launch_bounds__(WARPS * 32) te_route_partition_kernel(const uint32_t* __restrict__ ids, const uint32_t* __restrict__ sec,
                                                                        const uint32_t* __restrict__ nsec, const double* __restrict__ pose, int m,
                                                                        OwnerOf owner, const int* __restrict__ base, uint32_t* __restrict__ o_ids,
                                                                        uint32_t* __restrict__ o_sec, uint32_t* __restrict__ o_nsec,
                                                                        double* __restrict__ o_pose) {
  extern __shared__ int cur[];   // [WARPS][G]
  const int G = (int)owner.d;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < WARPS * G; i += blockDim.x) cur[i] = 0;
  __syncthreads();
  int* my = cur + warp * G;
  const int w_lo = blockIdx.x * TILE + warp * 32 * ITEMS;
  for (int s = 0; s < ITEMS; ++s) {   // 1. per-warp owner counts
    const int k = w_lo + s * 32 + lane;
    if (k < m) atomicAdd(&my[owner(ids[k])], 1);
  }
  __syncthreads();
  for (int r = threadIdx.x; r < G; r += blockDim.x) {   // 2. cursors: the block's place in owner r's run + earlier warps' records
    int at = base[(size_t)r * gridDim.x + blockIdx.x];
    for (int w = 0; w < WARPS; ++w) {
      const int c = cur[w * G + r];
      cur[w * G + r] = at;
      at += c;
    }
  }
  __syncthreads();
  for (int s = 0; s < ITEMS; ++s) {   // 3. the records, in order
    const int k = w_lo + s * 32 + lane;
    const bool on = k < m;
    const unsigned active = __ballot_sync(0xffffffffu, on);
    if (on) {
      const unsigned id = ids[k];
      const unsigned r = owner(id);
      const unsigned peers = __match_any_sync(active, r);
      const int rank = __popc(peers & ((1u << lane) - 1u));
      const int dst = my[r] + rank;
      o_ids[dst] = id;
      o_sec[dst] = sec[k];
      o_nsec[dst] = nsec[k];
      const double* src = pose + 7 * (size_t)k;
      double* d = o_pose + 7 * (size_t)dst;
#pragma unroll
      for (int j = 0; j < 7; ++j) d[j] = src[j];
      __syncwarp(active);   // every lane has read my[r] before the first lane of its owner group advances it
      if (rank == 0) my[r] += __popc(peers);
    }
    __syncwarp();
  }
}

}  // namespace te_route

namespace {

void grow(te_group* g, int r, size_t n_rec, size_t n_total) {
  Shard& s = g->sh[r];
  if (n_rec > s.rec_cap) {
    CK(cudaStreamSynchronize(s.stream));
    cudaFree(s.rec);
    s.rec = nullptr;
    const size_t cap = n_rec + n_rec / 8 + 32;
    CK(cudaMalloc(&s.rec, cap * 13 * sizeof(double)));
    s.rec_cap = cap;
  }
  if (n_total > s.out_cap) {
    CK(cudaStreamSynchronize(s.stream));
    cudaFree(s.out);
    cudaFree(s.out_ids);
    s.out = nullptr;
    s.out_ids = nullptr;
    const size_t cap = n_total + n_total / 8 + 32;
    CK(cudaMalloc(&s.out, cap * 13 * sizeof(double)));
    CK(cudaMalloc(&s.out_ids, cap * sizeof(uint32_t)));
    s.out_cap = cap;
  }
}

template <class F> long long group_guard(te_group* g, F&& f) {
  int prev = 0;
  cudaGetDevice(&prev);
  long long rc = -1;
  try {
    if (!g) throw std::invalid_argument("null group");
    rc = f();
  } catch (const std::exception& e) {
    last_error() = e.what();
    rc = -1;
  }
  cudaSetDevice(prev);
  return rc;
}

}  // namespace

extern "C" {

te_group* te_group_create(int n, const int* devices) {
  te_group* g = nullptr;
  int prev = 0;
  cudaGetDevice(&prev);
  try {
    if (n <= 0 || !devices) throw std::invalid_argument("a group needs at least one device");
    int n_dev = 0;
    CK(cudaGetDeviceCount(&n_dev));
    g = new te_group();
    g->sh.resize((size_t)n);
    bool distinct = true;
    for (int r = 0; r < n; ++r) {
      if (devices[r] < 0 || devices[r] >= n_dev) throw std::invalid_argument("no such CUDA device: " + std::to_string(devices[r]));
      for (int q = 0; q < r; ++q) distinct = distinct && devices[q] != devices[r];
      Shard& s = g->sh[r];
      s.device = devices[r];
      CK(cudaSetDevice(s.device));
      CK(cudaStreamCreateWithFlags(&s.own_stream, cudaStreamNonBlocking));
      s.stream = s.own_stream;
      CK(cudaEventCreate(&s.ev0));
      CK(cudaEventCreate(&s.ev1));
    }
    g->counts.assign((size_t)n, 0);
    g->use_nccl = distinct && n > 1;
    if (g->use_nccl) {
      g->comms.resize((size_t)n);
      NCK(nccl().CommInitAll(g->comms.data(), n, devices));
    }
  } catch (const std::exception& e) {
    last_error() = e.what();
    if (g) te_group_destroy(g);
    g = nullptr;
  }
  cudaSetDevice(prev);
  return g;
}

void te_group_destroy(te_group* g) {
  if (!g) return;
  int prev = 0;
  cudaGetDevice(&prev);
  for (auto c : g->comms)
    if (c) nccl().CommDestroy(c);
  for (size_t r = 0; r < g->route.size(); ++r) {
    Route& rt = g->route[r];
    cudaSetDevice(g->sh[r].device);
    if (rt.stream) cudaStreamSynchronize(rt.stream);
    cudaFree(rt.in);
    cudaFree(rt.part);
    cudaFree(rt.out);
    cudaFree(rt.work);
    if (rt.done) cudaEventDestroy(rt.done);
  }
  if (g->h_route_counts) cudaFreeHost(g->h_route_counts);
  for (Shard& s : g->sh) {
    cudaSetDevice(s.device);
    if (s.stream) cudaStreamSynchronize(s.stream);
    cudaFree(s.rec);
    cudaFree(s.out);
    cudaFree(s.out_ids);
    if (s.ev0) cudaEventDestroy(s.ev0);
    if (s.ev1) cudaEventDestroy(s.ev1);
    if (s.own_stream) cudaStreamDestroy(s.own_stream);
  }
  cudaSetDevice(prev);
  delete g;
}

int te_group_size(te_group* g) { return g ? (int)g->sh.size() : -1; }
int te_group_uses_nccl(te_group* g) { return g ? (g->use_nccl ? 1 : 0) : -1; }

long long te_group_allgather_estimates(te_group* g, te_pool* const* pools, long long* counts_out) {
  return group_guard(g, [&]() -> long long {
    const int G = (int)g->sh.size();
    if (!pools) throw std::invalid_argument("null pool list");
    long long total = 0;
    bool equal = true;
    for (int r = 0; r < G; ++r) {
      te_pool* p = pools[r];
      if (p && p->device != g->sh[r].device) throw std::invalid_argument("pool of shard " + std::to_string(r) + " lives on another device");
      g->counts[r] = p ? p->n : 0;
      g->sh[r].stream = p ? p->stream : g->sh[r].own_stream;
      total += g->counts[r];
      equal = equal && g->counts[r] == g->counts[0];
      if (counts_out) counts_out[r] = g->counts[r];
    }
    g->total = total;
    g->timed = false;
    if (total == 0) return 0;
    // 1. every shard's records on its own device and stream
    for (int r = 0; r < G; ++r) {
      Shard& s = g->sh[r];
      CK(cudaSetDevice(s.device));
      grow(g, r, (size_t)g->counts[r], (size_t)total);
      if (g->counts[r] > 0 && te_pool_estimates_dev(pools[r], s.rec) < 0) throw std::runtime_error(last_error());
      CK(cudaEventRecord(s.ev0, s.stream));
    }
    // 2. the exchange
    if (g->use_nccl) {
      NCK(nccl().GroupStart());
      if (equal) {
        for (int d = 0; d < G; ++d) {
          Shard& s = g->sh[d];
          NCK(nccl().AllGather(s.rec, s.out, (size_t)g->counts[d] * 13, ncclDouble, g->comms[d], s.stream));
          NCK(nccl().AllGather(pools[d]->buf[pools[d]->cur].cold.ids, s.out_ids, (size_t)g->counts[d], ncclUint32, g->comms[d], s.stream));
        }
      } else {
        long long off = 0;
        for (int r = 0; r < G; ++r) {   // root r sends its block to everyone (ragged all-gather)
          if (g->counts[r] > 0) {
            for (int d = 0; d < G; ++d) {
              Shard& s = g->sh[d];
              const void* src = d == r ? (const void*)s.rec : (const void*)(s.out + off * 13);
              const void* src_ids = d == r ? (const void*)pools[r]->buf[pools[r]->cur].cold.ids : (const void*)(s.out_ids + off);
              NCK(nccl().Broadcast(src, s.out + off * 13, (size_t)g->counts[r] * 13, ncclDouble, r, g->comms[d], s.stream));
              NCK(nccl().Broadcast(src_ids, s.out_ids + off, (size_t)g->counts[r], ncclUint32, r, g->comms[d], s.stream));
            }
          }
          off += g->counts[r];
        }
      }
      NCK(nccl().GroupEnd());
    } else {
      // shards that share a device (one-GPU test of the sharded host logic) or a single shard: plain copies, ordered after the
      // producers through events
      for (int d = 0; d < G; ++d) {
        Shard& s = g->sh[d];
        CK(cudaSetDevice(s.device));
        long long off = 0;
        for (int r = 0; r < G; ++r) {
          if (g->counts[r] > 0) {
            if (r != d) CK(cudaStreamWaitEvent(s.stream, g->sh[r].ev0, 0));
            CK(cudaMemcpyPeerAsync(s.out + off * 13, s.device, g->sh[r].rec, g->sh[r].device, (size_t)g->counts[r] * 13 * sizeof(double), s.stream));
            CK(cudaMemcpyPeerAsync(s.out_ids + off, s.device, pools[r]->buf[pools[r]->cur].cold.ids, g->sh[r].device,
                                   (size_t)g->counts[r] * sizeof(uint32_t), s.stream));
          }
          off += g->counts[r];
        }
      }
    }
    for (int d = 0; d < G; ++d) {
      Shard& s = g->sh[d];
      CK(cudaSetDevice(s.device));
      CK(cudaEventRecord(s.ev1, s.stream));
    }
    g->timed = true;
    return total;
  });
}

int te_group_sync(te_group* g) {
  return (int)group_guard(g, [&]() -> long long {
    for (Shard& s : g->sh) {
      CK(cudaSetDevice(s.device));
      CK(cudaStreamSynchronize(s.stream));
    }
    return 0;
  });
}

const double* te_group_dev_records(te_group* g, int r) { return (g && r >= 0 && r < (int)g->sh.size()) ? g->sh[r].out : nullptr; }
const uint32_t* te_group_dev_ids(te_group* g, int r) { return (g && r >= 0 && r < (int)g->sh.size()) ? g->sh[r].out_ids : nullptr; }

long long te_group_fetch(te_group* g, int root, double* records_out, uint32_t* ids_out, long long cap) {
  return group_guard(g, [&]() -> long long {
    if (root < 0 || root >= (int)g->sh.size()) throw std::invalid_argument("no such shard");
    Shard& s = g->sh[root];
    const long long k = std::min(cap, g->total);
    CK(cudaSetDevice(s.device));
    if (k > 0 && records_out) CK(cudaMemcpyAsync(records_out, s.out, (size_t)k * 13 * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
    if (k > 0 && ids_out) CK(cudaMemcpyAsync(ids_out, s.out_ids, (size_t)k * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.stream));
    CK(cudaStreamSynchronize(s.stream));
    return g->total;
  });
}

double te_group_last_gather_ms(te_group* g) {
  double worst = -1.0;
  group_guard(g, [&]() -> long long {
    if (!g->timed) return 0;
    for (Shard& s : g->sh) {
      CK(cudaSetDevice(s.device));
      CK(cudaEventSynchronize(s.ev1));
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, s.ev0, s.ev1));
      worst = std::max(worst, (double)ms);
    }
    return 0;
  });
  return worst;
}

long long te_group_route_records(te_group* g, te_pool* const* pools, long long n, const uint32_t* ids, const uint32_t* sec,
                                 const uint32_t* nsec, const double* poses, long long* counts_out) {
  return group_guard(g, [&]() -> long long {
    const int G = (int)g->sh.size();
    if (!pools) throw std::invalid_argument("null pool list");
    if (n < 0 || n > 0x7FFFFFFF) throw std::invalid_argument("bad record count");
    if (n > 0 && (!ids || !sec || !nsec || !poses)) throw std::invalid_argument("null record arrays");
    if (G > te_route::MAX_OWNERS) throw std::invalid_argument("at most 1024 shards can route records");
    for (int r = 0; r < G; ++r) {
      if (!pools[r]) throw std::invalid_argument("routing needs the pool of every shard");
      if (pools[r]->device != g->sh[r].device) throw std::invalid_argument("pool of shard " + std::to_string(r) + " lives on another device");
    }
    if (g->route.empty()) {
      g->route.resize((size_t)G);
      for (int r = 0; r < G; ++r) {
        CK(cudaSetDevice(g->sh[r].device));
        CK(cudaEventCreateWithFlags(&g->route[r].done, cudaEventDisableTiming));
      }
      CK(cudaHostAlloc((void**)&g->h_route_counts, (size_t)G * G * sizeof(int), cudaHostAllocPortable));
    }
    for (int r = 0; r < G; ++r) g->route[r].stream = pools[r]->stream;
    // a buffer grows only while no stream of the group uses it (the exchange reads other shards' partitioned chunks)
    auto quiesce = [&]() {
      for (int r = 0; r < G; ++r) {
        CK(cudaSetDevice(g->sh[r].device));
        CK(cudaStreamSynchronize(g->route[r].stream));
      }
    };
    auto grow = [&](int r, char*& buf, size_t& cap, size_t need, size_t unit) {   // cap, need in units of `unit` bytes
      if (need <= cap) return;
      quiesce();
      CK(cudaSetDevice(g->sh[r].device));
      cudaFree(buf);
      buf = nullptr;
      cap = 0;
      const size_t want = need + need / 8 + 1024;
      CK(cudaMalloc((void**)&buf, want * unit));
      cap = want;
    };
    // the previous message's exchange may still read a chunk that this message is about to overwrite
    if (g->routed)
      for (int c = 0; c < G; ++c) {
        CK(cudaSetDevice(g->sh[c].device));
        for (int r = 0; r < G; ++r)
          if (r != c) CK(cudaStreamWaitEvent(g->route[c].stream, g->route[r].done, 0));
      }
    // 1. chunk c (records [n c / G, n (c + 1) / G) of the message) goes to shard c's device -- the links of the G devices copy at
    //    once -- and 2. is partitioned there by owner
    const te_route::OwnerOf owner{(unsigned)G, (G & (G - 1)) == 0, ~0ull / (unsigned long long)G + 1};
    std::vector<long long> lo((size_t)G + 1);
    for (int c = 0; c <= G; ++c) lo[(size_t)c] = (long long)((__int128)n * c / G);
    for (int c = 0; c < G; ++c) {
      Route& rt = g->route[(size_t)c];
      const int m = (int)(lo[(size_t)c + 1] - lo[(size_t)c]);
      int* h_cnt = g->h_route_counts + (size_t)c * G;
      if (m == 0) {
        std::fill(h_cnt, h_cnt + G, 0);
        continue;
      }
      const int blocks = cdiv(m, te_route::TILE);
      const size_t cells = (size_t)G * blocks;
      size_t scan_bytes = 0;
      CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int*)nullptr, (int*)nullptr, (int)cells));
      const size_t off_scan = (cells * sizeof(int) + 255) & ~(size_t)255;
      const size_t off_cnt = off_scan + off_scan;
      const size_t off_tmp = off_cnt + (((size_t)G * sizeof(int) + 255) & ~(size_t)255);
      grow(c, rt.in, rt.in_cap, (size_t)m, REC_BYTES);
      grow(c, rt.part, rt.part_cap, (size_t)m, REC_BYTES);
      grow(c, rt.work, rt.work_cap, off_tmp + scan_bytes, 1);
      CK(cudaSetDevice(g->sh[c].device));
      const Recs in = recs(rt.in, rt.in_cap), part = recs(rt.part, rt.part_cap);
      const long long o = lo[(size_t)c];
      // ids first: the histogram needs nothing else
      CK(cudaMemcpyAsync(in.ids, ids + o, (size_t)m * 4, cudaMemcpyHostToDevice, rt.stream));
      CK(cudaMemcpyAsync(in.sec, sec + o, (size_t)m * 4, cudaMemcpyHostToDevice, rt.stream));
      CK(cudaMemcpyAsync(in.nsec, nsec + o, (size_t)m * 4, cudaMemcpyHostToDevice, rt.stream));
      CK(cudaMemcpyAsync(in.pose, poses + 7 * o, (size_t)m * 56, cudaMemcpyHostToDevice, rt.stream));
      int* hist = (int*)rt.work;
      int* base = (int*)(rt.work + off_scan);
      int* cnt = (int*)(rt.work + off_cnt);
      te_route::route_histogram_kernel<<<blocks, te_route::WARPS * 32, G * sizeof(int), rt.stream>>>(in.ids, m, owner, hist);
      CK(cudaGetLastError());
      CK(cub::DeviceScan::ExclusiveSum(rt.work + off_tmp, scan_bytes, hist, base, (int)cells, rt.stream));
      te_route::route_counts_kernel<<<cdiv(G, 256), 256, 0, rt.stream>>>(base, blocks, G, m, cnt);
      te_route::te_route_partition_kernel<<<blocks, te_route::WARPS * 32, te_route::WARPS * G * sizeof(int), rt.stream>>>(
          in.ids, in.sec, in.nsec, in.pose, m, owner, base, part.ids, part.sec, part.nsec, part.pose);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(h_cnt, cnt, (size_t)G * sizeof(int), cudaMemcpyDeviceToHost, rt.stream));
    }
    for (int c = 0; c < G; ++c)
      if (lo[(size_t)c + 1] > lo[(size_t)c]) {
        CK(cudaSetDevice(g->sh[c].device));
        CK(cudaStreamSynchronize(g->route[(size_t)c].stream));
      }
    // 3. the exchange: shard r receives [its run of chunk 0 | its run of chunk 1 | ...] -- arrival order per id
    const int* cnt = g->h_route_counts;
    std::vector<long long> src_off((size_t)G * G), dst_off((size_t)G * G);   // [c][r]
    for (int c = 0; c < G; ++c) {
      long long a = 0;
      for (int r = 0; r < G; ++r) {
        src_off[(size_t)c * G + r] = a;
        a += cnt[(size_t)c * G + r];
      }
    }
    for (int r = 0; r < G; ++r) {
      long long a = 0;
      for (int c = 0; c < G; ++c) {
        dst_off[(size_t)c * G + r] = a;
        a += cnt[(size_t)c * G + r];
      }
      Route& rt = g->route[(size_t)r];
      rt.n_out = a;
      if (counts_out) counts_out[r] = a;
      grow(r, rt.out, rt.out_cap, (size_t)a, REC_BYTES);
    }
    auto piece = [&](int c, int r, auto&& f) {   // f(src, dst, count) for the run of chunk c that shard r owns
      const long long k = cnt[(size_t)c * G + r];
      if (k == 0) return;
      const Route& from = g->route[(size_t)c];
      const Route& to = g->route[(size_t)r];
      const Recs s = recs(from.part, from.part_cap), d = recs(to.out, to.out_cap);
      const long long so = src_off[(size_t)c * G + r], dof = dst_off[(size_t)c * G + r];
      f(Recs{s.pose + 7 * so, s.ids + so, s.sec + so, s.nsec + so}, Recs{d.pose + 7 * dof, d.ids + dof, d.sec + dof, d.nsec + dof}, (size_t)k);
    };
    auto copy = [&](int c, int r) {
      piece(c, r, [&](const Recs& s, const Recs& d, size_t k) {
        const int sd = g->sh[c].device, dd = g->sh[r].device;
        cudaStream_t st = g->route[(size_t)r].stream;
        CK(cudaMemcpyPeerAsync(d.ids, dd, s.ids, sd, k * 4, st));
        CK(cudaMemcpyPeerAsync(d.sec, dd, s.sec, sd, k * 4, st));
        CK(cudaMemcpyPeerAsync(d.nsec, dd, s.nsec, sd, k * 4, st));
        CK(cudaMemcpyPeerAsync(d.pose, dd, s.pose, sd, k * 56, st));
      });
    };
    for (int r = 0; r < G; ++r) {
      CK(cudaSetDevice(g->sh[r].device));
      if (g->use_nccl) copy(r, r);
      else
        for (int c = 0; c < G; ++c) copy(c, r);
    }
    if (g->use_nccl) {   // distinct devices: every (chunk, owner) run as grouped point-to-point transfers, all ranks in one group
      NCK(nccl().GroupStart());
      for (int c = 0; c < G; ++c)
        for (int r = 0; r < G; ++r) {
          if (r == c) continue;
          piece(c, r, [&](const Recs& s, const Recs& d, size_t k) {
            const Route& from = g->route[(size_t)c];
            const Route& to = g->route[(size_t)r];
            NCK(nccl().Send(s.ids, k, ncclUint32, r, g->comms[(size_t)c], from.stream));
            NCK(nccl().Send(s.sec, k, ncclUint32, r, g->comms[(size_t)c], from.stream));
            NCK(nccl().Send(s.nsec, k, ncclUint32, r, g->comms[(size_t)c], from.stream));
            NCK(nccl().Send(s.pose, k * 7, ncclDouble, r, g->comms[(size_t)c], from.stream));
            NCK(nccl().Recv(d.ids, k, ncclUint32, c, g->comms[(size_t)r], to.stream));
            NCK(nccl().Recv(d.sec, k, ncclUint32, c, g->comms[(size_t)r], to.stream));
            NCK(nccl().Recv(d.nsec, k, ncclUint32, c, g->comms[(size_t)r], to.stream));
            NCK(nccl().Recv(d.pose, k * 7, ncclDouble, c, g->comms[(size_t)r], to.stream));
          });
        }
      NCK(nccl().GroupEnd());
    }
    for (int r = 0; r < G; ++r) {
      CK(cudaSetDevice(g->sh[r].device));
      CK(cudaEventRecord(g->route[(size_t)r].done, g->route[(size_t)r].stream));
    }
    g->routed = true;
    return n;
  });
}

int te_group_routed(te_group* g, int r, long long* n, const uint32_t** dev_ids, const uint32_t** dev_sec, const uint32_t** dev_nsec,
                    const double** dev_poses) {
  return (int)group_guard(g, [&]() -> long long {
    if (r < 0 || r >= (int)g->sh.size()) throw std::invalid_argument("no such shard");
    Recs d{nullptr, nullptr, nullptr, nullptr};
    long long k = 0;
    if (!g->route.empty() && g->route[(size_t)r].out) {
      const Route& rt = g->route[(size_t)r];
      d = recs(rt.out, rt.out_cap);
      k = rt.n_out;
    }
    if (n) *n = k;
    if (dev_ids) *dev_ids = d.ids;
    if (dev_sec) *dev_sec = d.sec;
    if (dev_nsec) *dev_nsec = d.nsec;
    if (dev_poses) *dev_poses = d.pose;
    return 0;
  });
}

}  // extern "C"
