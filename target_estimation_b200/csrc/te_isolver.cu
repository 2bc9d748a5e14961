// te_isolver.cu -- batched IntersectionSolver (/root/reference/src/intersection_solver.cpp:42-124): te_isolver_* of
// include/te_pool.h over isolver_kernel (te_kernels.cuh) and the quartic root finder (te_quartic.h).
#include "te_pool_internal.cuh"

using namespace tehost;
#define g_err (tehost::last_error())

extern "C" {

// ---- batched IntersectionSolver -------------------------------------------------------------
te_isolver* te_isolver_create(te_pool* p, long long n_streams, unsigned filters_length) {
  te_isolver* s = nullptr;
  try {
    if (!p || n_streams <= 0 || filters_length == 0) throw std::invalid_argument("bad isolver arguments");
    DeviceGuard g(p->device);
    s = new te_isolver();
    s->pool = p;
    s->st.n_streams = n_streams;
    s->st.L = filters_length;
    CK(cudaMalloc(&s->st.prev_pose, (size_t)n_streams * 7 * 8));
    CK(cudaMalloc(&s->st.pos_win, (size_t)n_streams * filters_length * 8));
    CK(cudaMalloc(&s->st.ang_win, (size_t)n_streams * filters_length * 8));
    CK(cudaMalloc(&s->st.pos_sum, (size_t)n_streams * 8));
    CK(cudaMalloc(&s->st.ang_sum, (size_t)n_streams * 8));
    CK(cudaMalloc(&s->st.idx, (size_t)n_streams * 4));
    CK(cudaMalloc(&s->st.complete, (size_t)n_streams));
    CK(cudaMalloc(&s->d_found, sizeof(unsigned long long)));
    CK(cudaMemsetAsync(s->st.pos_win, 0, (size_t)n_streams * filters_length * 8, p->stream));
    CK(cudaMemsetAsync(s->st.ang_win, 0, (size_t)n_streams * filters_length * 8, p->stream));
    CK(cudaMemsetAsync(s->st.pos_sum, 0, (size_t)n_streams * 8, p->stream));
    CK(cudaMemsetAsync(s->st.ang_sum, 0, (size_t)n_streams * 8, p->stream));
    CK(cudaMemsetAsync(s->st.idx, 0, (size_t)n_streams * 4, p->stream));
    CK(cudaMemsetAsync(s->st.complete, 0, (size_t)n_streams, p->stream));
    te::init_pose_kernel<<<cdiv(n_streams, 256), 256, 0, p->stream>>>(s->st.prev_pose, n_streams);   // initPose (:39)
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(p->stream));
    return s;
  } catch (const std::exception& e) {
    g_err = e.what();
    if (s) te_isolver_destroy(s);
    return nullptr;
  }
}

void te_isolver_destroy(te_isolver* s) {
  if (!s) return;
  cudaFree(s->st.prev_pose); cudaFree(s->st.pos_win); cudaFree(s->st.ang_win); cudaFree(s->st.pos_sum);
  cudaFree(s->st.ang_sum); cudaFree(s->st.idx); cudaFree(s->st.complete);
  cudaFree(s->d_found); cudaFree(s->move_block); cudaFree(s->move_streams);
  delete s;
}

int te_isolver_query(te_isolver* s, long long n, const uint32_t* ids, const int32_t* stream, const double* t1, const double* origin,
                     const double* radius, const double* pos_th, const double* ang_th, double* delta_t, double* pose7, uint8_t* converged) {
  if (!s) { g_err = "null isolver"; return -1; }
  te_pool* p = s->pool;
  return guarded(p, [&] {
    if (n <= 0) return 0;
    if (!ids || !t1 || !origin || !radius) throw std::invalid_argument("ids, t1, origin and radius are required");
    if (pose7 && (!pos_th || !ang_th)) throw std::invalid_argument("thresholds are required with pose7");
    if (pose7 && !stream && n > s->st.n_streams) throw std::invalid_argument("more queries than solver streams");
    if (stream) for (long long k = 0; k < n; ++k) if (stream[k] < 0 || stream[k] >= s->st.n_streams) throw std::invalid_argument("bad stream index");
    int* slots = p->n ? lookup_slots(p, to_dev(p, ids, n), n) : nullptr;
    if (!slots) {
      slots = p->arena.get_n<int>((size_t)n);
      CK(cudaMemsetAsync(slots, 0xff, (size_t)n * sizeof(int), p->stream));
    }
    const int* d_stream = to_dev(p, stream, n);
    const double* d_t1 = to_dev(p, t1, n);
    const double* d_origin = to_dev(p, origin, n * 3);
    const double* d_radius = to_dev(p, radius, n);
    const double* d_pth = to_dev(p, pos_th, n);
    const double* d_ath = to_dev(p, ang_th, n);
    double* d_delta = delta_t ? p->arena.get_n<double>((size_t)n) : nullptr;
    double* d_pose = pose7 ? p->arena.get_n<double>((size_t)n * 7) : nullptr;
    uint8_t* d_conv = converged ? p->arena.get_n<uint8_t>((size_t)n) : nullptr;
    Buf& b = p->buf[p->cur];
    const int g = cdiv(n, 128);
    unsigned long long found = 0;
    CK(cudaMemsetAsync(s->d_found, 0, sizeof(found), p->stream));
    te::isolver_count_found_kernel<<<g, 128, 0, p->stream>>>(slots, n, s->d_found);
    switch (p->model) {
      case te::UNIFORM_VELOCITY: te::isolver_kernel<te::UNIFORM_VELOCITY><<<g, 128, 0, p->stream>>>(b.tiles, slots, d_stream, n, d_t1, d_origin, d_radius, d_pth, d_ath, s->st, d_delta, d_pose, d_conv); break;
      case te::UNIFORM_ACCELERATION: te::isolver_kernel<te::UNIFORM_ACCELERATION><<<g, 128, 0, p->stream>>>(b.tiles, slots, d_stream, n, d_t1, d_origin, d_radius, d_pth, d_ath, s->st, d_delta, d_pose, d_conv); break;
      case te::ANGULAR_VELOCITIES: te::isolver_kernel<te::ANGULAR_VELOCITIES><<<g, 128, 0, p->stream>>>(b.tiles, slots, d_stream, n, d_t1, d_origin, d_radius, d_pth, d_ath, s->st, d_delta, d_pose, d_conv); break;
      default: te::isolver_kernel<te::ANGULAR_RATES><<<g, 128, 0, p->stream>>>(b.tiles, slots, d_stream, n, d_t1, d_origin, d_radius, d_pth, d_ath, s->st, d_delta, d_pose, d_conv); break;
    }
    CK(cudaGetLastError());
    if (delta_t) CK(cudaMemcpyAsync(delta_t, d_delta, (size_t)n * 8, cudaMemcpyDeviceToHost, p->stream));
    if (pose7) CK(cudaMemcpyAsync(pose7, d_pose, (size_t)n * 56, cudaMemcpyDeviceToHost, p->stream));
    if (converged) CK(cudaMemcpyAsync(converged, d_conv, (size_t)n, cudaMemcpyDeviceToHost, p->stream));
    CK(cudaMemcpyAsync(&found, s->d_found, sizeof(found), cudaMemcpyDeviceToHost, p->stream));
    CK(cudaStreamSynchronize(p->stream));
    return (int)found;
  });
}

namespace {
// the staging of a move on solver s's device: room for n streams (grow-only)
void move_reserve(te_isolver* s, long long n) {
  if ((size_t)n <= s->move_cap) return;
  cudaFree(s->move_block);
  cudaFree(s->move_streams);
  s->move_block = nullptr;
  s->move_streams = nullptr;
  s->move_cap = 0;
  CK(cudaMalloc(&s->move_block, (size_t)n * te::isolver_rows(s->st.L) * sizeof(double)));
  CK(cudaMalloc(&s->move_streams, (size_t)n * sizeof(int)));
  s->move_cap = (size_t)n;
}
int move_grid(long long total) { return (int)std::min<long long>(cdiv(total, 256), 148 * 8); }
}  // namespace

int te_isolver_move_streams(te_isolver* src, te_isolver* dst, long long n, const int32_t* streams) {
  try {
    if (!src || !dst) throw std::invalid_argument("null isolver");
    if (src == dst) throw std::invalid_argument("source and destination are the same solver");
    if (src->pool->model != dst->pool->model || src->st.L != dst->st.L)
      throw std::invalid_argument("solvers of different model types or filter lengths");
    if (src->pool->live.active || dst->pool->live.active) throw std::logic_error("the pool is held by a live launch: call te_pool_live_end first");
    if (n <= 0) return 0;
    if (!streams) throw std::invalid_argument("streams are required");
    const long long lim = std::min(src->st.n_streams, dst->st.n_streams);
    for (long long k = 0; k < n; ++k)
      if (streams[k] < 0 || streams[k] >= lim) throw std::invalid_argument("bad stream index");
    const size_t bytes = (size_t)n * te::isolver_rows(src->st.L) * sizeof(double);
    const long long total = te::isolver_rows(src->st.L) * n;
    te_pool* ps = src->pool;
    te_pool* pd = dst->pool;
    {   // gather the listed streams into src's staging
      DeviceGuard g(ps->device);
      move_reserve(src, n);
      CK(cudaMemcpyAsync(src->move_streams, streams, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ps->stream));
      te::isolver_pack_streams_kernel<<<move_grid(total), 256, 0, ps->stream>>>(src->st, src->move_streams, n, src->move_block);
      CK(cudaGetLastError());
      CK(cudaStreamSynchronize(ps->stream));
    }
    DeviceGuard g(pd->device);   // one copy into dst's staging, then scatter
    move_reserve(dst, n);
    CK(cudaMemcpyAsync(dst->move_streams, streams, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, pd->stream));
    if (ps->device == pd->device) CK(cudaMemcpyAsync(dst->move_block, src->move_block, bytes, cudaMemcpyDeviceToDevice, pd->stream));
    else CK(cudaMemcpyPeerAsync(dst->move_block, pd->device, src->move_block, ps->device, bytes, pd->stream));
    te::isolver_unpack_streams_kernel<<<move_grid(total), 256, 0, pd->stream>>>(dst->st, dst->move_streams, n, dst->move_block);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(pd->stream));
    return 0;
  } catch (const std::exception& e) {
    g_err = e.what();
    return -1;
  }
}

int te_isolver_query_dense(te_isolver* s, const double* dev_t1, const double* dev_origin, const double* dev_radius, double pos_th,
                           double ang_th, double* dev_delta, double* dev_pose7, uint8_t* dev_converged) {
  if (!s) { g_err = "null isolver"; return -1; }
  te_pool* p = s->pool;
  return guarded(p, [&] {
    const long long n = p->n;
    if (n == 0) return 0;
    if (!dev_origin || !dev_radius) throw std::invalid_argument("origin and radius are required");
    if (n > s->st.n_streams) throw std::invalid_argument("more targets than solver streams");
    te::IsolverState st = s->st;
    st.pos_th_all = pos_th;
    st.ang_th_all = ang_th;
    Buf& b = p->buf[p->cur];
    const int g = cdiv(n, 128);
    switch (p->model) {
      case te::UNIFORM_VELOCITY: te::isolver_kernel<te::UNIFORM_VELOCITY><<<g, 128, 0, p->stream>>>(b.tiles, nullptr, nullptr, n, dev_t1, dev_origin, dev_radius, nullptr, nullptr, st, dev_delta, dev_pose7, dev_converged); break;
      case te::UNIFORM_ACCELERATION: te::isolver_kernel<te::UNIFORM_ACCELERATION><<<g, 128, 0, p->stream>>>(b.tiles, nullptr, nullptr, n, dev_t1, dev_origin, dev_radius, nullptr, nullptr, st, dev_delta, dev_pose7, dev_converged); break;
      case te::ANGULAR_VELOCITIES: te::isolver_kernel<te::ANGULAR_VELOCITIES><<<g, 128, 0, p->stream>>>(b.tiles, nullptr, nullptr, n, dev_t1, dev_origin, dev_radius, nullptr, nullptr, st, dev_delta, dev_pose7, dev_converged); break;
      default: te::isolver_kernel<te::ANGULAR_RATES><<<g, 128, 0, p->stream>>>(b.tiles, nullptr, nullptr, n, dev_t1, dev_origin, dev_radius, nullptr, nullptr, st, dev_delta, dev_pose7, dev_converged); break;
    }
    CK(cudaGetLastError());
    return 0;
  });
}

}  // extern "C"
