// C-ABI entry points (include/truss_b200.h).  Device variants enqueue on the caller's stream;
// *_host variants stage host buffers through a grow-only device arena owned by the plan (or a
// process-wide one for ragged batches), run the same device path, and copy the results back.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "tb_common.cuh"
#include "tb_ts.cuh"

namespace {

size_t ws_cap_bytes() {
  static size_t cap = [] {
    const char* s = getenv("TB_WORKSPACE_MAX_GB");
    double gb = s ? atof(s) : 64.0;
    if (gb < 0.25) gb = 0.25;
    return (size_t)(gb * (1ull << 30));
  }();
  return cap;
}

int have_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    (void)cudaGetLastError();
    return 0;
  }
  return 1;
}

int check_batch_in(const tb_plan* p, const tb_batch_in* in) {
  if (!p || !in) return TB_ERR_NULL;
  if (p->device < 0) return TB_ERR_NO_DEVICE;
  if (in->batch < 0) return TB_ERR_SIZE;
  if (in->batch == 0) return TB_OK;
  if (!in->joint_xyz || !in->force) return TB_ERR_NULL;
  if (!in->member_aed && !(in->gene && in->type_table && in->n_type > 0)) return TB_ERR_NULL;
  return TB_OK;
}

// Compact outputs (tb_batch_out.u_free / react): gathered from the dense rows of the same systems
__global__ void __launch_bounds__(256) k_compact_out(const double* __restrict__ u, const double* __restrict__ ext,
                                                      double* __restrict__ u_free, double* __restrict__ react,
                                                      const int32_t* __restrict__ free_ref, const int32_t* __restrict__ sup_idx,
                                                      int N, int n, int s, int nb) {
  for (int b = blockIdx.x; b < nb; b += gridDim.x) {
    if (u_free)
      for (int r = threadIdx.x; r < n; r += 256) u_free[(int64_t)b * n + r] = u[(int64_t)b * N + free_ref[r]];
    if (react)
      for (int r = threadIdx.x; r < s; r += 256) react[(int64_t)b * s + r] = ext[(int64_t)b * N + sup_idx[r]];
  }
}

// dense temporaries of a call that wants the compact outputs without the dense ones (call before the ranges are enqueued)
int ensure_compact_tmp(tb_plan* p, const tb_batch_out* out, int batch, cudaStream_t st) {
  if (!out || p->path != 0) return TB_OK;      // (the blocked pipelines' recovery kernel writes the compact outputs itself)
  auto grow = [&](double** buf, size_t* cap) -> int {
    if (*cap >= (size_t)batch) return TB_OK;
    if (*buf) {
      TB_CUDA(cudaStreamSynchronize(st));
      TB_CUDA(cudaDeviceSynchronize());
      TB_CUDA(cudaFree(*buf));
      *buf = nullptr;
      *cap = 0;
    }
    TB_CUDA(cudaMalloc((void**)buf, (size_t)batch * p->N * sizeof(double)));
    *cap = (size_t)batch;
    return TB_OK;
  };
  if (out->u_free && !out->u) {
    const int rc = grow(&p->compact_u, &p->compact_cap_u);
    if (rc) return rc;
  }
  if (out->react && !out->ext) {
    const int rc = grow(&p->compact_ext, &p->compact_cap_ext);
    if (rc) return rc;
  }
  return TB_OK;
}

int run_plan_range_dense(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                         double allow_d, cudaStream_t st, int b0, int nb, void* ws, int shared_k);

// Systems [b0, b0 + nb) of a uniform batch on stream st; the blocked pipelines use the workspace slice `ws`.
int run_plan_range(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                   double allow_d, cudaStream_t st, int b0, int nb, void* ws, int shared_k = 0) {
  if (!out->u_free && !out->react) return run_plan_range_dense(p, in, out, fit, allow_s, allow_d, st, b0, nb, ws, shared_k);
  if (p->path != 0) return run_plan_range_dense(p, in, out, fit, allow_s, allow_d, st, b0, nb, ws, shared_k);   // the recovery kernel writes them itself
  tb_batch_out eff = *out;
  if (out->u_free && !eff.u) eff.u = p->compact_u;          // (ensure_compact_tmp sized them for the whole batch)
  if (out->react && !eff.ext) eff.ext = p->compact_ext;
  if ((out->u_free && !eff.u) || (out->react && !eff.ext)) return TB_ERR_ALLOC;
  const int rc = run_plan_range_dense(p, in, &eff, fit, allow_s, allow_d, st, b0, nb, ws, shared_k);
  if (rc) return rc;
  const int grid = nb < 148 * 8 ? nb : 148 * 8;
  k_compact_out<<<grid, 256, 0, st>>>(eff.u ? eff.u + (int64_t)b0 * p->N : nullptr, eff.ext ? eff.ext + (int64_t)b0 * p->N : nullptr,
                                      out->u_free ? out->u_free + (int64_t)b0 * p->n : nullptr,
                                      out->react ? out->react + (int64_t)b0 * p->s : nullptr, p->d_free_ref, p->d_sup_idx, p->N,
                                      p->n, p->s, nb);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int run_plan_range_dense(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                         double allow_d, cudaStream_t st, int b0, int nb, void* ws, int shared_k) {
  const int fitness_mode = fit ? 1 : 0;
  int32_t* info = fit && fit->info ? fit->info : out->info;
  if (p->path == 0) {
    SmallArgs a;
    memset(&a, 0, sizeof(a));
    a.batch = nb;
    a.nJ = p->nJ;
    a.M = p->M;
    a.xyz = in->joint_xyz + (int64_t)b0 * in->joint_stride;
    a.xyz_stride = in->joint_stride;
    a.support = p->d_support;
    a.support_stride = 0;
    a.conn = p->d_conn;
    a.conn_stride = 0;
    a.aed = in->member_aed ? in->member_aed + (int64_t)b0 * in->member_stride : nullptr;
    a.aed_stride = in->member_stride;
    a.gene = in->member_aed ? nullptr : in->gene + (int64_t)b0 * in->gene_stride;
    a.gene_stride = in->gene_stride;
    a.type_table = in->type_table;
    a.n_type = in->n_type;
    a.force = in->force + (int64_t)b0 * in->force_stride;
    a.force_stride = in->force_stride;
    // the fused kernels address their outputs by (system index) * (row length)
    a.u = out->u ? out->u + (int64_t)b0 * p->N : nullptr;
    a.ext = out->ext ? out->ext + (int64_t)b0 * p->N : nullptr;
    a.axial = out->axial ? out->axial + (int64_t)b0 * p->M : nullptr;
    a.weight = out->weight ? out->weight + b0 : nullptr;
    a.info = info ? info + b0 : nullptr;
    a.fitness = fit && fit->fitness ? fit->fitness + b0 : nullptr;
    a.flags = fit && fit->flags ? fit->flags + 2 * (int64_t)b0 : nullptr;
    a.allow_stress = allow_s;
    a.allow_displace = allow_d;
    a.fitness_mode = fitness_mode;
    a.max_n = p->n;
    return tb_launch_small(a, p->dim, st);
  }
  LargeArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = nb;
  a.dim = p->dim;
  a.nJ = p->nJ;
  a.M = p->M;
  a.N = p->N;
  a.n = p->n;
  a.n_pad = p->n_pad;
  a.nt = p->nt;
  a.s = p->s;
  a.xyz = in->joint_xyz + (int64_t)b0 * in->joint_stride;
  a.xyz_stride = in->joint_stride;
  a.aed = in->member_aed ? in->member_aed + (int64_t)b0 * in->member_stride : nullptr;
  a.aed_stride = in->member_stride;
  a.gene = in->member_aed ? nullptr : in->gene + (int64_t)b0 * in->gene_stride;
  a.gene_stride = in->gene_stride;
  a.type_table = in->type_table;
  a.n_type = in->n_type;
  a.force = in->force + (int64_t)b0 * in->force_stride;
  a.force_stride = in->force_stride;
  a.conn = p->d_conn;
  a.free_idx = p->d_free_idx;
  a.dof2free = p->d_dof2free;
  a.sup_idx = p->d_sup_idx;
  a.ent_row = p->d_ent_row;
  a.ent_col = p->d_ent_col;
  a.ent_ptr = p->d_ent_ptr;
  a.ctr_member = p->d_ctr_member;
  a.ctr_local = p->d_ctr_local;
  a.tile_ent_ptr = p->d_tile_ent_ptr;
  a.tile_ent = p->d_tile_ent;
  a.tile_pos = p->d_tile_pos;
  a.nnz = (int64_t)p->ent_row.size();
  a.q_ptr = p->path == 2 ? p->d_bq_ptr : p->d_q_ptr;
  a.q_pack = p->path == 2 ? p->d_bq_pack : p->d_q_pack;
  a.q_first = p->path == 2 ? p->d_bq_first : p->d_q_first;
  a.q_multi = p->path == 2 ? p->d_bq_multi : p->d_q_multi;
  a.n_multi = (int)(p->path == 2 ? p->bq_multi.size() : p->q_multi.size());
  a.nb16 = p->nb16;
  a.NB = p->NB;
  a.b16_ptr = p->d_b16_ptr;
  a.b16_pos = p->d_b16_pos;
  a.b16_nz = p->d_b16_nz;
  if (p->path == 2) a.n_pad = p->nb16 * 16;
  a.tile_nz = p->d_tile_nz;
  a.prod_ptr = p->d_prod_ptr;
  a.prod_k = p->d_prod_k;
  a.inc_ptr = p->d_inc_ptr;
  a.inc_mem = p->d_inc_mem;
  tb_large_carve(a, ws, p->path);
  a.u = out->u ? out->u + (int64_t)b0 * p->N : nullptr;
  a.ext = out->ext ? out->ext + (int64_t)b0 * p->N : nullptr;
  a.axial = out->axial ? out->axial + (int64_t)b0 * p->M : nullptr;
  a.weight = out->weight ? out->weight + b0 : nullptr;
  a.info = info ? info + b0 : nullptr;
  a.u_free = out->u_free ? out->u_free + (int64_t)b0 * p->n : nullptr;
  a.react = out->react ? out->react + (int64_t)b0 * p->s : nullptr;
  a.free_ref = p->d_free_ref;
  a.fitness = fit && fit->fitness ? fit->fitness + b0 : nullptr;
  a.flags = fit && fit->flags ? fit->flags + 2 * (int64_t)b0 : nullptr;
  a.allow_stress = allow_s;
  a.allow_displace = allow_d;
  a.fitness_mode = fitness_mode;
  a.plan_stable = p->stable;
  a.shared_k = shared_k;
  if (p->path == 2 && p->ts && p->ts->ok) {      // fused two-sided band kernel: its slice follows the 16x16 pipeline's
    a.ts = p->ts;
    a.ts_b0 = 0;
    a.ts_total = nb;
    a.ts_ws = (char*)ws + ((tb_large_workspace_bytes(nb, p->dim, p->M, p->n_pad, a.nnz, p->path, p->nb16, p->NB) + 255) & ~(size_t)255);
  }
  return tb_launch_large(a, p->num_sm, st, p->path);
}

size_t plan_ws_bytes(const tb_plan* p, int batch) {
  if (p->path == 0) return 0;
  size_t need = tb_large_workspace_bytes(batch, p->dim, p->M, p->n_pad, (int64_t)p->ent_row.size(), p->path, p->nb16, p->NB);
  if (p->path == 2 && p->ts) need = ((need + 255) & ~(size_t)255) + tb_ts_workspace_bytes(p, batch);
  return need;
}

int ensure_ws(tb_plan* p, size_t need, cudaStream_t st) {
  if (p->ws_bytes >= need) return TB_OK;
  if (p->ws) {
    TB_CUDA(cudaStreamSynchronize(st));
    TB_CUDA(cudaDeviceSynchronize());
    TB_CUDA(cudaFree(p->ws));
    p->ws = nullptr;
    p->ws_bytes = 0;
  }
  TB_CUDA(cudaMalloc(&p->ws, need));
  p->ws_bytes = need;
  return TB_OK;
}

// The plan belongs to the device it was created on (its maps and workspace live there)
int check_device(const tb_plan* p) {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return TB_ERR_NO_DEVICE;
  return dev == p->device ? TB_OK : TB_ERR_WRONG_DEVICE;
}

// Workspace ordering across streams: the previous call's kernels may still be running on another stream
int ws_acquire(tb_plan* p, cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) (void)cudaGetLastError();
  if (cap != cudaStreamCaptureStatusNone) return TB_OK;          // a captured step is single-stream by contract
  if (p->ws_used && p->ws_stream != st && p->ws_event) TB_CUDA(cudaStreamWaitEvent(st, p->ws_event, 0));
  return TB_OK;
}
int ws_release(tb_plan* p, cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) (void)cudaGetLastError();
  if (cap != cudaStreamCaptureStatusNone) return TB_OK;
  if (!p->ws_event) TB_CUDA(cudaEventCreateWithFlags(&p->ws_event, cudaEventDisableTiming));
  TB_CUDA(cudaEventRecord(p->ws_event, st));
  p->ws_stream = st;
  p->ws_used = true;
  return TB_OK;
}

int run_plan_unlocked(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                      double allow_d, cudaStream_t st, int shared_k);

// Device entry points: one call at a time per plan (the plan owns ONE workspace), ordered across streams by an event
int run_plan(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
             double allow_d, cudaStream_t st, int shared_k = 0) {
  int rc = check_device(p);
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(p->mu);
  if (p->path != 0) {
    rc = ws_acquire(p, st);
    if (rc) return rc;
  }
  rc = run_plan_unlocked(p, in, out, fit, allow_s, allow_d, st, shared_k);
  if (!rc && p->path != 0) rc = ws_release(p, st);
  return rc;
}

int run_plan_unlocked(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                      double allow_d, cudaStream_t st, int shared_k) {
  static const tb_batch_out none = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (!out) out = &none;
  {
    const int rc0 = ensure_compact_tmp(p, out, in->batch, st);
    if (rc0) return rc0;
  }
  if (p->path == 0) {
    int rc = run_plan_range(p, in, out, fit, allow_s, allow_d, st, 0, in->batch, nullptr);
    if (rc) return rc;
  } else {
    // blocked paths: process the batch in chunks that fit the workspace cap
    const size_t per_sys = plan_ws_bytes(p, 1);
    int chunk = (int)std::min<size_t>((size_t)in->batch, std::max<size_t>(1, ws_cap_bytes() / per_sys));
    int rc = ensure_ws(p, plan_ws_bytes(p, chunk), st);
    if (rc) return rc;
    for (int b0 = 0; b0 < in->batch; b0 += chunk) {
      rc = run_plan_range(p, in, out, fit, allow_s, allow_d, st, b0, std::min(chunk, in->batch - b0), p->ws, shared_k);
      if (rc) return rc;
    }
  }
  if (fit && fit->info && out->info) {
    TB_CUDA(cudaMemcpyAsync(out->info, fit->info, sizeof(int32_t) * in->batch, cudaMemcpyDeviceToDevice, st));
  }
  return TB_OK;
}

// ---- bump allocator over a grow-only device arena -------------------------------------------
struct Arena {
  void** base;
  size_t* cap;
  size_t used = 0;
  Arena(void** b, size_t* c) : base(b), cap(c) {}
  static size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
};

int arena_reserve(void** base, size_t* cap, size_t need) {
  if (*cap >= need) return 0;
  if (*base) {
    TB_CUDA(cudaDeviceSynchronize());
    TB_CUDA(cudaFree(*base));
    *base = nullptr;
    *cap = 0;
  }
  need += need / 8;
  TB_CUDA(cudaMalloc(base, need));
  *cap = need;
  return 0;
}

template <typename Tp>
Tp* take(char*& cur, size_t count) {
  Tp* p = (Tp*)cur;
  cur += Arena::al(count * sizeof(Tp));
  return p;
}

// Helper streams and events of the *_host entry points: one set per device (streams and events belong to the device that
// was current when they were created), made on first use under the pipe mutex.
constexpr int TB_HOST_STREAMS = 8;
constexpr int TB_MAX_DEVICES = 64;
struct HostPipe {
  bool ready = false;
  cudaStream_t comp = nullptr;
  cudaStream_t ain = nullptr, aout = nullptr;  // H2D / D2H streams of the pipelined calls (tb_solve_host_async)
  cudaStream_t copy[TB_HOST_STREAMS] = {};
  cudaEvent_t ev_in[TB_HOST_STREAMS] = {}, ev_out[TB_HOST_STREAMS] = {};
};
HostPipe g_pipes[TB_MAX_DEVICES];
std::mutex g_pipe_mu;                          // one *_host call at a time per process (the pipes and arenas are shared)

HostPipe* host_pipe() {                        // call with g_pipe_mu held
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  HostPipe& hp = g_pipes[dev & (TB_MAX_DEVICES - 1)];
  if (!hp.ready) {
    if (cudaStreamCreateWithFlags(&hp.comp, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&hp.ain, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaStreamCreateWithFlags(&hp.aout, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    for (int i = 0; i < TB_HOST_STREAMS; ++i) {
      if (cudaStreamCreateWithFlags(&hp.copy[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&hp.ev_in[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&hp.ev_out[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    hp.ready = true;
  }
  return &hp;
}
void host_pipe_drain(HostPipe* hp) {           // after an error: nothing of the call may still touch the caller's buffers
  if (!hp) return;
  cudaStreamSynchronize(hp->comp);
  cudaStreamSynchronize(hp->ain);
  cudaStreamSynchronize(hp->aout);
  for (int i = 0; i < TB_HOST_STREAMS; ++i) cudaStreamSynchronize(hp->copy[i]);
  (void)cudaGetLastError();
}
int stride_ok(int64_t stride, int64_t row) { return stride == 0 || stride == row; }

int run_plan_host_locked(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                         double allow_d, int shared_k, HostPipe* hp, int async_slot = -1);

// every pipelined call of this plan has completed (its results are in the caller's buffers)
int async_drain(tb_plan* p) {
  while (p->async_completed < p->async_submitted) {
    TB_CUDA(cudaEventSynchronize(p->async_done[p->async_completed % TB_ASYNC_SLOTS]));
    p->async_completed++;
  }
  return TB_OK;
}

// Host entry points: serialised per process (g_pipe_mu: helper streams, events) and per plan (p->mu: staging arena,
// workspace); on an error the helper streams are drained before the code is returned.
int run_plan_host(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                  double allow_d, int shared_k = 0) {
  int rc = check_batch_in(p, in);
  if (rc) return rc;
  rc = check_device(p);
  if (rc) return rc;
  std::lock_guard<std::mutex> pipe_lock(g_pipe_mu);
  std::lock_guard<std::mutex> plan_lock(p->mu);
  HostPipe* hp = host_pipe();
  if (!hp) return TB_ERR_ALLOC;
  rc = async_drain(p);                          // (the blocking calls share the compute stream and the workspace with the pipelined ones)
  if (rc) return rc;
  if (p->path != 0) {
    rc = ws_acquire(p, hp->comp);
    if (rc) return rc;
  }
  rc = run_plan_host_locked(p, in, out, fit, allow_s, allow_d, shared_k, hp);
  if (rc) host_pipe_drain(hp);
  else if (p->path != 0) rc = ws_release(p, hp->comp);
  return rc;
}

// Pipelined host call: enqueue H2D (stream ain) -> kernels (comp) -> D2H (aout) and return; consecutive calls use the
// async staging arenas in turn, so the copies of one call overlap the kernels of its neighbours.  At most TB_ASYNC_SLOTS
// calls are in flight (one uploading, one computing, one downloading): a further submission first waits for the oldest.
int run_plan_host_async(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, uint64_t* ticket) {
  int rc = check_batch_in(p, in);
  if (rc) return rc;
  rc = check_device(p);
  if (rc) return rc;
  std::lock_guard<std::mutex> pipe_lock(g_pipe_mu);
  std::lock_guard<std::mutex> plan_lock(p->mu);
  HostPipe* hp = host_pipe();
  if (!hp) return TB_ERR_ALLOC;
  const int slot = (int)(p->async_submitted % TB_ASYNC_SLOTS);
  if (p->async_submitted - p->async_completed >= (uint64_t)TB_ASYNC_SLOTS) {      // the slot's previous call
    TB_CUDA(cudaEventSynchronize(p->async_done[p->async_completed % TB_ASYNC_SLOTS]));
    p->async_completed++;
  }
  for (cudaEvent_t* e : {&p->async_in[slot], &p->async_k[slot], &p->async_done[slot]})
    if (!*e) TB_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  if (p->path != 0) {
    rc = ws_acquire(p, hp->comp);
    if (rc) return rc;
  }
  rc = in->batch == 0 ? TB_OK : run_plan_host_locked(p, in, out, nullptr, 0.0, 0.0, 0, hp, slot);
  if (rc) {
    host_pipe_drain(hp);
    p->async_completed = p->async_submitted;
    return rc;
  }
  if (p->path != 0) rc = ws_release(p, hp->comp);
  TB_CUDA(cudaEventRecord(p->async_done[slot], hp->aout));
  if (ticket) *ticket = p->async_submitted;
  p->async_submitted++;
  return rc;
}

int run_plan_host_locked(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                         double allow_d, int shared_k, HostPipe* hp, int async_slot) {
  int rc = 0;
  const bool async = async_slot >= 0;
  const int B = in->batch;
  if (B == 0) return TB_OK;
  const int64_t rowJ = (int64_t)p->nJ * p->dim, rowM3 = (int64_t)p->M * 3, rowM = p->M, rowN = p->N;
  if (!stride_ok(in->joint_stride, rowJ) || !stride_ok(in->force_stride, rowN)) return TB_ERR_SIZE;
  if (in->member_aed && !stride_ok(in->member_stride, rowM3)) return TB_ERR_SIZE;
  if (!in->member_aed && !stride_ok(in->gene_stride, rowM)) return TB_ERR_SIZE;
  auto cnt = [&](int64_t stride, int64_t row) { return (size_t)(stride == 0 ? row : row * B); };
  const size_t nxyz = cnt(in->joint_stride, rowJ), nf = cnt(in->force_stride, rowN);
  const size_t naed = in->member_aed ? cnt(in->member_stride, rowM3) : 0;
  const size_t ngene = in->member_aed ? 0 : cnt(in->gene_stride, rowM);
  const size_t ntab = in->member_aed ? 0 : (size_t)in->n_type * 3;
  static const tb_batch_out none = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (!out) out = &none;

  size_t need = 0;
  auto add = [&](size_t bytes) { need += Arena::al(bytes); };
  add(nxyz * 8); add(nf * 8); add(naed * 8); add(ngene * 4); add(ntab * 8);
  add(out->u ? (size_t)B * rowN * 8 : 0); add(out->ext ? (size_t)B * rowN * 8 : 0);
  add(out->axial ? (size_t)B * rowM * 8 : 0); add(out->weight ? (size_t)B * 8 : 0);
  add((size_t)B * 4); add(fit ? (size_t)B * 8 : 0); add(fit ? (size_t)B * 2 : 0);
  add(out->u_free ? (size_t)B * p->n * 8 : 0); add(out->react ? (size_t)B * p->s * 8 : 0);
  void** arena = async ? &p->stage_async[async_slot] : &p->stage_dev;
  size_t* arena_bytes = async ? &p->stage_async_bytes[async_slot] : &p->stage_dev_bytes;
  rc = arena_reserve(arena, arena_bytes, need + 4096);
  if (rc) return rc;

  cudaStream_t st = hp->comp;
  char* cur = (char*)*arena;
  tb_batch_in din = *in;
  double* dxyz = take<double>(cur, nxyz);
  double* df = take<double>(cur, nf);
  double* daed = take<double>(cur, naed);
  int32_t* dgene = take<int32_t>(cur, ngene);
  double* dtab = take<double>(cur, ntab);
  din.joint_xyz = dxyz;
  din.force = df;
  if (in->member_aed) {
    din.member_aed = daed;
    din.gene = nullptr;
  } else {
    din.gene = dgene;
    din.type_table = dtab;
  }
  tb_batch_out dout;
  dout.u = out->u ? take<double>(cur, (size_t)B * rowN) : nullptr;
  dout.ext = out->ext ? take<double>(cur, (size_t)B * rowN) : nullptr;
  dout.axial = out->axial ? take<double>(cur, (size_t)B * rowM) : nullptr;
  dout.weight = out->weight ? take<double>(cur, (size_t)B) : nullptr;
  dout.info = take<int32_t>(cur, (size_t)B);
  dout.u_free = out->u_free ? take<double>(cur, (size_t)B * p->n) : nullptr;
  dout.react = out->react ? take<double>(cur, (size_t)B * p->s) : nullptr;
  rc = ensure_compact_tmp(p, &dout, B, hp->comp);
  if (rc) return rc;
  tb_fit_out dfit = {nullptr, nullptr, nullptr};
  if (fit) {
    dfit.fitness = take<double>(cur, (size_t)B);
    dfit.flags = take<uint8_t>(cur, (size_t)B * 2);
    dfit.info = dout.info;
    dout.info = nullptr;
  }
  int32_t* dinfo = fit ? dfit.info : dout.info;

  // The batch is cut into chunks.  All kernels run on ONE compute stream, chunk after chunk; every chunk has its own
  // copy stream: its inputs travel (H2D) while the previous chunk is being solved and its results travel back (D2H)
  // while the next chunk is being solved -- PCIe is full duplex, so the two directions overlap as well.  (Chunks on
  // concurrent compute streams all finish together, and nothing can be copied back before that: measured 0.87 ms per
  // 1024 bar-942 systems against 0.75 ms this way.)  Mid-size systems are latency-bound per wave, so a chunk is never
  // smaller than a few systems per SM; arrays shared by the whole batch (stride 0) are copied once, first.
  const size_t per_sys = plan_ws_bytes(p, 1);
  int nch = 1;
  {
    static const int want = [] { const char* s = getenv("TB_HOST_CHUNKS"); int v = s ? atoi(s) : 0; return v < 0 ? 0 : (v > TB_HOST_STREAMS - 1 ? TB_HOST_STREAMS - 1 : v); }();
    const int sms = p->num_sm > 0 ? p->num_sm : 148;
    const int min_chunk = p->path == 0 ? 16 * sms : 3 * sms;
    int fit_ = B / min_chunk;
    if (fit_ > 4) fit_ = 4;
    nch = want > 0 ? want : (fit_ < 1 ? 1 : fit_);
    if (nch > B) nch = B;
    if (p->path != 0 && per_sys * (size_t)B > ws_cap_bytes()) nch = 1;   // run_plan cuts the batch to the workspace cap itself
    // chunking a blocked path only pays through the D2H it hides (each chunk is a latency-bound wave of its own):
    // with little to copy back (fitness only, weights only) one launch over the whole batch is faster
    const size_t d2h_bytes = ((out->u ? rowN : 0) + (out->ext ? rowN : 0) + (out->axial ? rowM : 0) + (out->u_free ? p->n : 0) +
                              (out->react ? p->s : 0)) * (size_t)B * 8;
    if (want == 0 && p->path != 0 && d2h_bytes < ((size_t)4 << 20)) nch = 1;
    if (async) nch = 1;                        // a pipelined call is one chunk: its neighbours hide its copies
  }
  // chunk boundaries: equal parts (a 3:1 split, to shrink the D2H of the last chunk that nothing hides, measured slower:
  // 0.89 ms against 0.82 ms for 1024 bar-942 systems -- the larger first wave costs more than the copy saves)
  int cb[TB_HOST_STREAMS + 1];
  for (int j = 0; j <= nch; ++j) cb[j] = (int)((int64_t)B * j / nch);
  int csz = 0;
  for (int j = 0; j < nch; ++j) csz = std::max(csz, cb[j + 1] - cb[j]);
  if (p->path != 0 && nch > 1) {
    rc = ensure_ws(p, per_sys * (size_t)csz + 4096, st);       // chunks run one after the other: one workspace slice
    if (rc) return rc;
  }
  cudaStream_t comp = st;                      // compute stream
  cudaStream_t* cps = hp->copy;                // copy streams, one per chunk
  cudaStream_t cin = async ? hp->ain : comp;   // where a one-chunk call's inputs / results travel
  cudaStream_t cout = async ? hp->aout : comp;
  cudaEvent_t* ev_in = hp->ev_in;
  cudaEvent_t* ev_out = hp->ev_out;
  const bool sx = in->joint_stride == 0, sf = in->force_stride == 0;
  const bool sm_ = in->member_aed ? in->member_stride == 0 : in->gene_stride == 0;
  // shared inputs first, on the compute stream
  if (sx) TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, nxyz * 8, cudaMemcpyHostToDevice, cin));
  if (sf) TB_CUDA(cudaMemcpyAsync(df, in->force, nf * 8, cudaMemcpyHostToDevice, cin));
  if (in->member_aed) {
    if (sm_) TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, naed * 8, cudaMemcpyHostToDevice, cin));
  } else {
    if (sm_) TB_CUDA(cudaMemcpyAsync(dgene, in->gene, ngene * 4, cudaMemcpyHostToDevice, cin));
    TB_CUDA(cudaMemcpyAsync(dtab, in->type_table, ntab * 8, cudaMemcpyHostToDevice, cin));
  }
  for (int j = 0; j < nch; ++j) {              // every chunk's inputs are queued at once, each on its copy stream
    const int b0 = cb[j], nb = cb[j + 1] - cb[j];
    if (nb <= 0) continue;
    cudaStream_t sj = nch == 1 ? cin : cps[j];
    if (!sx) TB_CUDA(cudaMemcpyAsync(dxyz + (size_t)b0 * rowJ, in->joint_xyz + (size_t)b0 * rowJ, (size_t)nb * rowJ * 8, cudaMemcpyHostToDevice, sj));
    if (!sf) TB_CUDA(cudaMemcpyAsync(df + (size_t)b0 * rowN, in->force + (size_t)b0 * rowN, (size_t)nb * rowN * 8, cudaMemcpyHostToDevice, sj));
    if (in->member_aed) {
      if (!sm_) TB_CUDA(cudaMemcpyAsync(daed + (size_t)b0 * rowM3, in->member_aed + (size_t)b0 * rowM3, (size_t)nb * rowM3 * 8, cudaMemcpyHostToDevice, sj));
    } else {
      if (!sm_) TB_CUDA(cudaMemcpyAsync(dgene + (size_t)b0 * rowM, in->gene + (size_t)b0 * rowM, (size_t)nb * rowM * 4, cudaMemcpyHostToDevice, sj));
    }
    if (nch > 1) TB_CUDA(cudaEventRecord(ev_in[j], sj));
  }
  if (async) {
    TB_CUDA(cudaEventRecord(p->async_in[async_slot], cin));
    TB_CUDA(cudaStreamWaitEvent(comp, p->async_in[async_slot], 0));
  }
  for (int j = 0; j < nch; ++j) {
    const int b0 = cb[j], nb = cb[j + 1] - cb[j];
    if (nb <= 0) continue;
    cudaStream_t sj = nch == 1 ? cout : cps[j];
    if (nch > 1) TB_CUDA(cudaStreamWaitEvent(comp, ev_in[j], 0));
    if (nch == 1 && p->path != 0) {
      rc = run_plan_unlocked(p, &din, &dout, fit ? &dfit : nullptr, allow_s, allow_d, comp, shared_k);   // handles the workspace cap itself
    } else {
      rc = run_plan_range(p, &din, &dout, fit ? &dfit : nullptr, allow_s, allow_d, comp, b0, nb, p->ws, shared_k);
    }
    if (rc) return rc;
    if (nch > 1) {
      TB_CUDA(cudaEventRecord(ev_out[j], comp));
      TB_CUDA(cudaStreamWaitEvent(sj, ev_out[j], 0));
    }
    if (async) {
      TB_CUDA(cudaEventRecord(p->async_k[async_slot], comp));
      TB_CUDA(cudaStreamWaitEvent(cout, p->async_k[async_slot], 0));
    }
    if (out->u) TB_CUDA(cudaMemcpyAsync(out->u + (size_t)b0 * rowN, dout.u + (size_t)b0 * rowN, (size_t)nb * rowN * 8, cudaMemcpyDeviceToHost, sj));
    if (out->ext) TB_CUDA(cudaMemcpyAsync(out->ext + (size_t)b0 * rowN, dout.ext + (size_t)b0 * rowN, (size_t)nb * rowN * 8, cudaMemcpyDeviceToHost, sj));
    if (out->axial) TB_CUDA(cudaMemcpyAsync(out->axial + (size_t)b0 * rowM, dout.axial + (size_t)b0 * rowM, (size_t)nb * rowM * 8, cudaMemcpyDeviceToHost, sj));
    if (out->weight) TB_CUDA(cudaMemcpyAsync(out->weight + b0, dout.weight + b0, (size_t)nb * 8, cudaMemcpyDeviceToHost, sj));
    if (out->u_free) TB_CUDA(cudaMemcpyAsync(out->u_free + (size_t)b0 * p->n, dout.u_free + (size_t)b0 * p->n, (size_t)nb * p->n * 8, cudaMemcpyDeviceToHost, sj));
    if (out->react && p->s > 0) TB_CUDA(cudaMemcpyAsync(out->react + (size_t)b0 * p->s, dout.react + (size_t)b0 * p->s, (size_t)nb * p->s * 8, cudaMemcpyDeviceToHost, sj));
    if (out->info) TB_CUDA(cudaMemcpyAsync(out->info + b0, dinfo + b0, (size_t)nb * 4, cudaMemcpyDeviceToHost, sj));
    if (fit) {
      if (fit->fitness) TB_CUDA(cudaMemcpyAsync(fit->fitness + b0, dfit.fitness + b0, (size_t)nb * 8, cudaMemcpyDeviceToHost, sj));
      if (fit->flags) TB_CUDA(cudaMemcpyAsync(fit->flags + 2 * (size_t)b0, dfit.flags + 2 * (size_t)b0, (size_t)nb * 2, cudaMemcpyDeviceToHost, sj));
      if (fit->info) TB_CUDA(cudaMemcpyAsync(fit->info + b0, dinfo + b0, (size_t)nb * 4, cudaMemcpyDeviceToHost, sj));
    }
  }
  if (async) return TB_OK;                     // completion: the event the caller records on `cout`
  TB_CUDA(cudaStreamSynchronize(comp));
  if (nch > 1)
    for (int j = 0; j < nch; ++j) TB_CUDA(cudaStreamSynchronize(cps[j]));
  return TB_OK;
}

int check_ragged(const tb_ragged_in* in) {
  if (!in) return TB_ERR_NULL;
  if (in->dim != 2 && in->dim != 3) return TB_ERR_DIM;
  if (in->batch < 0 || in->max_joint < 0 || in->max_member < 0) return TB_ERR_SIZE;
  if (in->batch == 0) return TB_OK;
  if (!in->joint_off || !in->member_off || !in->joint_xyz || !in->support || !in->conn || !in->member_aed || !in->force)
    return TB_ERR_NULL;
  if (!tb_small_fits(in->dim, in->max_joint, in->max_member, in->max_joint * in->dim)) return TB_ERR_TOO_LARGE;
  return TB_OK;
}

int run_ragged(const tb_ragged_in* in, const tb_batch_out* out, cudaStream_t st) {
  SmallArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch;
  a.nJ = in->max_joint;
  a.M = in->max_member;
  a.joint_off = in->joint_off;
  a.member_off = in->member_off;
  a.xyz = in->joint_xyz;
  a.support = in->support;
  a.conn = in->conn;
  a.aed = in->member_aed;
  a.force = in->force;
  a.u = out->u;
  a.ext = out->ext;
  a.axial = out->axial;
  a.weight = out->weight;
  a.info = out->info;
  a.max_n = in->max_joint * in->dim;
  return tb_launch_small(a, in->dim, st);
}

// staging arena of the ragged host entry point: one per device (device memory), used under g_pipe_mu
void* g_rag_dev[TB_MAX_DEVICES] = {};
size_t g_rag_dev_bytes[TB_MAX_DEVICES] = {};

// Argument checks of the ragged forward entry points: as check_ragged, up to the envelope kernel's limits
int check_ragged_fwd(const tb_ragged_in* in) {
  if (!in) return TB_ERR_NULL;
  if (in->dim != 2 && in->dim != 3) return TB_ERR_DIM;
  if (in->batch < 0 || in->max_joint < 0 || in->max_member < 0) return TB_ERR_SIZE;
  if (in->batch == 0) return TB_OK;
  if (!in->joint_off || !in->member_off || !in->joint_xyz || !in->support || !in->conn || !in->member_aed || !in->force)
    return TB_ERR_NULL;
  if ((int64_t)in->max_joint * in->dim > TB_RAGGED_MAX_DOF || in->max_member > TB_RAGGED_MAX_MEMBER) return TB_ERR_TOO_LARGE;
  return TB_OK;
}

bool ragged_fits_fused(const tb_ragged_in* in) {
  return tb_small_fits(in->dim, in->max_joint, in->max_member, in->max_joint * in->dim);
}

// Scratch of the envelope kernel: one grow-only arena per device (one slot per CTA of the persistent grid), grown
// stream-ordered on the caller's stream.  `mu` serialises the calls on the device; `ev` orders the arena's use across
// streams (recorded after a call's kernel; a call on another stream waits for it first).
struct EnvScratch {
  std::mutex mu;
  void* buf = nullptr;
  size_t bytes = 0;
  cudaEvent_t ev = nullptr;
  cudaStream_t last = nullptr;
  bool used = false;
};
EnvScratch g_env[TB_MAX_DEVICES];

// Envelope kernel over a batch: every truss (route = false), only the trusses above the fused launch's sizes (route:
// those run first, in one fused launch of the batch), or the ordering mode (order != null).  Inside a stream capture
// the arena is never grown: TB_ERR_ALLOC with nothing enqueued.
int run_env(const tb_ragged_in* in, const tb_batch_out* out, bool route, int32_t* order, int64_t* envelope, cudaStream_t st) {
  const int d = in->dim;
  int dev = 0;
  TB_CUDA(cudaGetDevice(&dev));
  EnvScratch& S = g_env[dev & (TB_MAX_DEVICES - 1)];
  std::lock_guard<std::mutex> lock(S.mu);       // (also keeps the kernel's shared-memory attribute until the launch)
  int grid = 0, smem = 0, env_smem = 0;
  int rc = tb_rag_env_config(d, in->max_joint, in->max_member, in->batch, &grid, &smem, &env_smem);
  if (rc) return rc;
  const size_t slot = tb_rag_env_slot_bytes(d, in->max_joint, in->max_member);
  const size_t need = slot * (size_t)grid;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) (void)cudaGetLastError();
  const bool capturing = cap != cudaStreamCaptureStatusNone;
  if (S.bytes < need && capturing) return TB_ERR_ALLOC;          // (a warm-up call outside the capture grows it)
  if (!capturing && S.used && S.last != st && S.ev) TB_CUDA(cudaStreamWaitEvent(st, S.ev, 0));
  if (S.bytes < need) {                                          // stream-ordered: the previous call is ahead on st
    if (S.buf) TB_CUDA(cudaFreeAsync(S.buf, st));
    S.buf = nullptr;
    S.bytes = 0;
    TB_CUDA(cudaMallocAsync(&S.buf, need, st));
    S.bytes = need;
  }
  const int rj = d == 3 ? TB_RAGGED_ROUTE_J3 : TB_RAGGED_ROUTE_J2, rm = d == 3 ? TB_RAGGED_ROUTE_M3 : TB_RAGGED_ROUTE_M2;
  if (route) {                                   // the fused kernels first, sized at the routing limits (k_dense16)
    tb_ragged_in fin = *in;
    fin.max_joint = std::min(in->max_joint, rj);
    fin.max_member = std::min(in->max_member, rm);
    rc = run_ragged(&fin, out, st);
    if (rc) return rc;
  }
  RagEnvArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.dim = d; a.max_joint = in->max_joint; a.max_member = in->max_member;
  a.route_joint = route ? rj : 0;
  a.route_member = route ? rm : 0;
  a.joint_off = in->joint_off; a.member_off = in->member_off;
  a.xyz = in->joint_xyz; a.support = in->support; a.conn = in->conn; a.aed = in->member_aed; a.force = in->force;
  if (out) { a.u = out->u; a.ext = out->ext; a.axial = out->axial; a.weight = out->weight; a.info = out->info; }
  a.order = order;
  a.envelope = envelope;
  a.scratch = S.buf;
  a.slot_bytes = slot;
  a.env_smem = env_smem;
  rc = tb_launch_rag_env(a, grid, smem, st);
  if (rc) return rc;
  if (!capturing) {
    if (!S.ev) TB_CUDA(cudaEventCreateWithFlags(&S.ev, cudaEventDisableTiming));
    TB_CUDA(cudaEventRecord(S.ev, st));
    S.last = st;
    S.used = true;
  }
  return TB_OK;
}

// The forward of a ragged batch: today's fused launch when the whole batch fits the fused kernels, else split by truss
int run_ragged_fwd(const tb_ragged_in* in, const tb_batch_out* out, cudaStream_t st) {
  if (ragged_fits_fused(in)) return run_ragged(in, out, st);
  return run_env(in, out, true, nullptr, nullptr, st);
}

}  // namespace

extern "C" int tb_solve(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, void* cuda_stream) {
  int rc = check_batch_in(plan, in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  return run_plan(plan, in, out, nullptr, 0.0, 0.0, (cudaStream_t)cuda_stream);
}

extern "C" int tb_solve_host(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out) {
  return run_plan_host(plan, in, out, nullptr, 0.0, 0.0);
}

extern "C" int tb_solve_host_async(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, uint64_t* ticket) {
  return run_plan_host_async(plan, in, out, ticket);
}

extern "C" int tb_host_wait(tb_plan* plan, uint64_t ticket) {
  if (!plan) return TB_ERR_NULL;
  std::lock_guard<std::mutex> plan_lock(plan->mu);
  if (ticket >= plan->async_submitted) return TB_ERR_SIZE;
  while (plan->async_completed <= ticket) {
    TB_CUDA(cudaEventSynchronize(plan->async_done[plan->async_completed % TB_ASYNC_SLOTS]));
    plan->async_completed++;
  }
  return TB_OK;
}

namespace {
// load cases of one truss: geometry and member properties must be shared by the whole batch
int check_loadcases(const tb_batch_in* in) {
  if (in->joint_stride != 0) return TB_ERR_SIZE;
  if (in->member_aed ? in->member_stride != 0 : in->gene_stride != 0) return TB_ERR_SIZE;
  return TB_OK;
}
}  // namespace

extern "C" int tb_solve_loadcases(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, void* cuda_stream) {
  int rc = check_batch_in(plan, in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_loadcases(in);
  if (rc) return rc;
  return run_plan(plan, in, out, nullptr, 0.0, 0.0, (cudaStream_t)cuda_stream, 1);
}

extern "C" int tb_solve_loadcases_host(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out) {
  int rc = check_batch_in(plan, in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_loadcases(in);
  if (rc) return rc;
  return run_plan_host(plan, in, out, nullptr, 0.0, 0.0, 1);
}

extern "C" int tb_fitness(tb_plan* plan, const tb_batch_in* in, double allow_stress, double allow_displace,
                          const tb_fit_out* fit, const tb_batch_out* full, void* cuda_stream) {
  int rc = check_batch_in(plan, in);
  if (rc) return rc;
  if (!fit) return TB_ERR_NULL;
  if (in->batch == 0) return TB_OK;
  return run_plan(plan, in, full, fit, allow_stress, allow_displace, (cudaStream_t)cuda_stream);
}

extern "C" int tb_fitness_host(tb_plan* plan, const tb_batch_in* in, double allow_stress, double allow_displace,
                               const tb_fit_out* fit, const tb_batch_out* full) {
  if (!fit) return TB_ERR_NULL;
  return run_plan_host(plan, in, full, fit, allow_stress, allow_displace);
}

extern "C" int tb_solve_ragged(const tb_ragged_in* in, const tb_batch_out* out, void* cuda_stream) {
  if (out && (out->u_free || out->react)) return TB_ERR_SIZE;   // (the compact layout needs one n and s for the whole batch)
  int rc = check_ragged_fwd(in);
  if (rc) return rc;
  if (!out) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  if (in->batch == 0) return TB_OK;
  return run_ragged_fwd(in, out, (cudaStream_t)cuda_stream);
}

extern "C" int tb_solve_ragged_env(const tb_ragged_in* in, const tb_batch_out* out, void* cuda_stream) {
  if (out && (out->u_free || out->react)) return TB_ERR_SIZE;
  int rc = check_ragged_fwd(in);
  if (rc) return rc;
  if (!out) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  if (in->batch == 0) return TB_OK;
  return run_env(in, out, false, nullptr, nullptr, (cudaStream_t)cuda_stream);
}

extern "C" int tb_ragged_env_order(const tb_ragged_in* in, int32_t* order, int64_t* envelope, void* cuda_stream) {
  int rc = check_ragged_fwd(in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  if (!order || !envelope) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  return run_env(in, nullptr, false, order, envelope, (cudaStream_t)cuda_stream);
}

extern "C" int tb_ragged_limits(int32_t dim, int32_t* max_joint, int32_t* max_member) {
  if (dim != 2 && dim != 3) return TB_ERR_DIM;
  if (!max_joint || !max_member) return TB_ERR_NULL;
  *max_joint = TB_RAGGED_MAX_DOF / dim;
  *max_member = TB_RAGGED_MAX_MEMBER;
  return TB_OK;
}

extern "C" int tb_solve_ragged_host(const tb_ragged_in* in, const tb_batch_out* out) {
  if (out && (out->u_free || out->react)) return TB_ERR_SIZE;
  int rc = check_ragged_fwd(in);
  if (rc) return rc;
  if (!out) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  const int B = in->batch, d = in->dim;
  if (B == 0) return TB_OK;
  // host-side validation of the offsets (they are host pointers here)
  if (in->joint_off[0] != 0 || in->member_off[0] != 0) return TB_ERR_SIZE;
  for (int b = 0; b < B; ++b) {
    const int64_t nj = in->joint_off[b + 1] - in->joint_off[b], nm = in->member_off[b + 1] - in->member_off[b];
    if (nj < 0 || nm < 0) return TB_ERR_SIZE;
    if (nj > in->max_joint || nm > in->max_member) return TB_ERR_TOO_LARGE;
  }
  const size_t SJ = (size_t)in->joint_off[B], SM = (size_t)in->member_off[B];
  std::lock_guard<std::mutex> lock(g_pipe_mu);
  HostPipe* hp = host_pipe();
  if (!hp) return TB_ERR_ALLOC;
  int dev = 0;
  TB_CUDA(cudaGetDevice(&dev));
  void*& rag_dev = g_rag_dev[dev & (TB_MAX_DEVICES - 1)];
  size_t& rag_bytes = g_rag_dev_bytes[dev & (TB_MAX_DEVICES - 1)];
  auto body = [&]() -> int {
  size_t need = 0;
  auto add = [&](size_t bytes) { need += Arena::al(bytes); };
  add((B + 1) * 8); add((B + 1) * 8); add(SJ * d * 8); add(SJ); add(SM * 8); add(SM * 24); add(SJ * d * 8);
  add(out->u ? SJ * d * 8 : 0); add(out->ext ? SJ * d * 8 : 0); add(out->axial ? SM * 8 : 0);
  add(out->weight ? (size_t)B * 8 : 0); add((size_t)B * 4);
  int rc = arena_reserve(&rag_dev, &rag_bytes, need + 4096);
  if (rc) return rc;
  cudaStream_t st = hp->comp;
  char* cur = (char*)rag_dev;
  tb_ragged_in din = *in;
  int64_t* djo = take<int64_t>(cur, B + 1);
  int64_t* dmo = take<int64_t>(cur, B + 1);
  double* dxyz = take<double>(cur, SJ * d);
  uint8_t* dsup = take<uint8_t>(cur, SJ);
  int32_t* dconn = take<int32_t>(cur, SM * 2);
  double* daed = take<double>(cur, SM * 3);
  double* df = take<double>(cur, SJ * d);
  TB_CUDA(cudaMemcpyAsync(djo, in->joint_off, (B + 1) * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dmo, in->member_off, (B + 1) * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, SJ * d * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dsup, in->support, SJ, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dconn, in->conn, SM * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, SM * 24, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(df, in->force, SJ * d * 8, cudaMemcpyHostToDevice, st));
  din.joint_off = djo; din.member_off = dmo; din.joint_xyz = dxyz; din.support = dsup;
  din.conn = dconn; din.member_aed = daed; din.force = df;
  tb_batch_out dout;
  dout.u_free = dout.react = nullptr;
  dout.u = out->u ? take<double>(cur, SJ * d) : nullptr;
  dout.ext = out->ext ? take<double>(cur, SJ * d) : nullptr;
  dout.axial = out->axial ? take<double>(cur, SM) : nullptr;
  dout.weight = out->weight ? take<double>(cur, (size_t)B) : nullptr;
  dout.info = take<int32_t>(cur, (size_t)B);
  rc = run_ragged_fwd(&din, &dout, st);
  if (rc) return rc;
  if (out->u) TB_CUDA(cudaMemcpyAsync(out->u, dout.u, SJ * d * 8, cudaMemcpyDeviceToHost, st));
  if (out->ext) TB_CUDA(cudaMemcpyAsync(out->ext, dout.ext, SJ * d * 8, cudaMemcpyDeviceToHost, st));
  if (out->axial) TB_CUDA(cudaMemcpyAsync(out->axial, dout.axial, SM * 8, cudaMemcpyDeviceToHost, st));
  if (out->weight) TB_CUDA(cudaMemcpyAsync(out->weight, dout.weight, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
  if (out->info) TB_CUDA(cudaMemcpyAsync(out->info, dout.info, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  TB_CUDA(cudaStreamSynchronize(st));
  return TB_OK;
  };
  rc = body();
  if (rc) host_pipe_drain(hp);                 // nothing of a failed call may still be copying into the caller's buffers
  return rc;
}

// Debug export: the K_ff values the device assembles (the band path's program-order lists when the plan has the two-sided
// program, else the tile-order lists), returned in the order of tb_plan_get_scatter.  Host pointers; uniform batch.
extern "C" int tb_debug_assemble_host(tb_plan* p, const tb_batch_in* in, double* kv_out) {
  int rc = check_batch_in(p, in);
  if (rc) return rc;
  if (!kv_out) return TB_ERR_NULL;
  rc = check_device(p);
  if (rc) return rc;
  const int B = in->batch;
  if (B == 0) return TB_OK;
  if (!in->member_aed) return TB_ERR_NULL;                       // (explicit member properties only)
  const bool ts = p->ts && p->ts->ok;
  const size_t nnz_map = p->ent_row.size();                      // scatter-map entries (the output's order)
  const size_t nnz = ts ? p->ts->epos.size() : nnz_map;          // device order: the band program's schedule has holes
  const int64_t rowJ = (int64_t)p->nJ * p->dim, rowM3 = (int64_t)p->M * 3;
  if (!stride_ok(in->joint_stride, rowJ) || !stride_ok(in->member_stride, rowM3)) return TB_ERR_SIZE;
  std::lock_guard<std::mutex> pipe_lock(g_pipe_mu);
  std::lock_guard<std::mutex> plan_lock(p->mu);
  HostPipe* hp = host_pipe();
  if (!hp) return TB_ERR_ALLOC;
  cudaStream_t st = hp->comp;
  const size_t nxyz = (size_t)(in->joint_stride == 0 ? rowJ : rowJ * B), naed = (size_t)(in->member_stride == 0 ? rowM3 : rowM3 * B);
  const int nv = p->dim * (p->dim + 1) / 2;
  double *dxyz = nullptr, *daed = nullptr, *dkv = nullptr, *dscr = nullptr;
  int32_t* dstat = nullptr;
  std::vector<double> host((size_t)B * nnz);
  auto body = [&]() -> int {
    TB_CUDA(cudaMalloc(&dxyz, nxyz * 8));
    TB_CUDA(cudaMalloc(&daed, naed * 8));
    TB_CUDA(cudaMalloc(&dkv, (size_t)B * nnz * 8));
    TB_CUDA(cudaMalloc(&dscr, (size_t)B * p->M * (2 + p->dim + nv) * 8));     // k_geom arrays (only used for very many members)
    TB_CUDA(cudaMalloc(&dstat, (size_t)B * 4));
    TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, nxyz * 8, cudaMemcpyHostToDevice, st));
    TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, naed * 8, cudaMemcpyHostToDevice, st));
    LargeArgs a;
    memset(&a, 0, sizeof(a));
    a.batch = B; a.dim = p->dim; a.nJ = p->nJ; a.M = p->M; a.N = p->N; a.n = p->n;
    a.xyz = dxyz; a.xyz_stride = in->joint_stride;
    a.aed = daed; a.aed_stride = in->member_stride;
    a.conn = p->d_conn;
    a.nnz = (int64_t)nnz;
    a.q_first = ts ? p->ts->d_tq_first : p->d_q_first;
    a.q_multi = ts ? p->ts->d_tq_multi : p->d_q_multi;
    a.q_ptr = ts ? p->ts->d_tq_ptr : p->d_q_ptr;
    a.q_pack = ts ? p->ts->d_tq_pack : p->d_q_pack;
    a.n_multi = (int)(ts ? p->ts->tq_multi.size() : p->q_multi.size());
    a.kv = dkv;
    a.status = dstat;
    double* q = dscr;
    a.mk = q; q += (size_t)B * p->M;
    a.mc = q; q += (size_t)B * p->M * p->dim;
    a.mw = q; q += (size_t)B * p->M;
    a.mkc = q;
    int r2 = tb_launch_assemble_only(a, p->num_sm, st);
    if (r2) return r2;
    TB_CUDA(cudaMemcpyAsync(host.data(), dkv, (size_t)B * nnz * 8, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  };
  rc = body();
  if (rc) host_pipe_drain(hp);
  cudaFree(dxyz); cudaFree(daed); cudaFree(dkv); cudaFree(dscr); cudaFree(dstat);
  if (rc) return rc;
  const std::vector<int32_t>& src = ts ? p->ts->ent_src : p->tile_ent;      // device order -> scatter-map entry
  for (int b = 0; b < B; ++b)
    for (size_t q2 = 0; q2 < nnz; ++q2)
      if (src[q2] >= 0) kv_out[(size_t)b * nnz_map + src[q2]] = host[(size_t)b * nnz + q2];
  return TB_OK;
}

// Reverse mode of tb_solve (DESIGN.md section 9): adjoint load, the adjoint solve through the plan's own pipeline
// (K is symmetric: the forward system with force := r), sensitivities.  Everything on the caller's stream.
extern "C" int tb_adjoint(tb_plan* p, const tb_batch_in* in, const double* u, const tb_adj_in* grad, const tb_adj_out* out,
                          int32_t shared_factor, void* cuda_stream) {
  if (!p || !in) return TB_ERR_NULL;
  if (in->batch > 0 && !in->member_aed) return TB_ERR_NULL;      // (no gradients with respect to a type table)
  int rc = check_batch_in(p, in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  if (!u || !grad || !out || !out->member_aed) return TB_ERR_NULL;
  if (shared_factor) {
    rc = check_loadcases(in);
    if (rc) return rc;
  }
  rc = check_device(p);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const int B = in->batch;
  std::lock_guard<std::mutex> lock(p->mu);
  rc = ws_acquire(p, st);
  if (rc) return rc;
  const bool smem = tb_adjoint_vec_in_smem(p->dim, p->M);
  const size_t rowN = (size_t)B * p->N * 8, nvec = smem ? 0 : (size_t)B * p->M * p->dim * 8;
  const size_t need = 2 * Arena::al(rowN) + Arena::al((size_t)B * 4) + nvec;
  if (p->adj_bytes < need) {                    // stream-ordered: the previous call's kernels are ahead on this stream
    if (p->adj_buf) TB_CUDA(cudaFreeAsync(p->adj_buf, st));
    p->adj_buf = nullptr;
    p->adj_bytes = 0;
    TB_CUDA(cudaMallocAsync(&p->adj_buf, need, st));
    p->adj_bytes = need;
  }
  char* cur = (char*)p->adj_buf;
  double* r = take<double>(cur, (size_t)B * p->N);
  double* lam = take<double>(cur, (size_t)B * p->N);
  int32_t* info_tmp = take<int32_t>(cur, (size_t)B);
  TbAdjArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = B; a.dim = p->dim; a.nJ = p->nJ; a.M = p->M; a.N = p->N;
  a.xyz = in->joint_xyz; a.xyz_stride = in->joint_stride;
  a.aed = in->member_aed; a.aed_stride = in->member_stride;
  a.conn = p->d_conn; a.dof2free = p->d_dof2free; a.inc_ptr = p->d_inc_ptr; a.inc_mem = p->d_inc_mem;
  a.g_u = grad->u; a.g_ext = grad->ext; a.g_axial = grad->axial; a.g_w = grad->weight;
  a.r = r;
  a.u = u;
  a.lam = lam;
  a.info = out->info ? out->info : info_tmp;
  a.vec = smem ? nullptr : (double*)cur;
  a.g_xyz = out->joint_xyz; a.g_aed = out->member_aed; a.g_force = out->force;
  const int num_sm = p->num_sm > 0 ? p->num_sm : 148;
  rc = tb_launch_adj_rhs(a, num_sm, st);
  if (rc) return rc;
  tb_batch_in ain = *in;                        // same systems, load := r (its supported rows are ignored)
  ain.force = r;
  ain.force_stride = p->N;
  const tb_batch_out aout = {lam, nullptr, nullptr, nullptr, const_cast<int32_t*>(a.info), nullptr, nullptr};
  rc = run_plan_unlocked(p, &ain, &aout, nullptr, 0.0, 0.0, st, shared_factor ? 1 : 0);
  if (rc) return rc;
  rc = tb_launch_sens(a, num_sm, st);
  if (rc) return rc;
  return ws_release(p, st);
}

// Reverse mode of tb_solve_ragged: adjoint load, the adjoint solve through run_ragged (the same kernel as the forward of
// the batch; K is symmetric: force := r), sensitivities.  The adjoint solution overwrites the load in `work`: every solve
// kernel stages a truss's load rows before it writes that truss's displacement rows, and a truss's rows belong to one
// warp (or CTA), so the host never needs the device-resident total joint count to place a second array.
extern "C" int tb_adjoint_ragged(const tb_ragged_in* in, const double* u, const tb_adj_in* grad, const tb_adj_out* out,
                                 double* work, void* cuda_stream) {
  int rc = check_ragged(in);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  if (!u || !grad || !out || !out->member_aed || !out->info || !work) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  TbAdjRaggedArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.dim = in->dim; a.max_joint = in->max_joint; a.max_member = in->max_member;
  a.joint_off = in->joint_off; a.member_off = in->member_off;
  a.xyz = in->joint_xyz; a.support = in->support; a.conn = in->conn; a.aed = in->member_aed;
  a.g_u = grad->u; a.g_ext = grad->ext; a.g_axial = grad->axial; a.g_w = grad->weight;
  a.r = work;
  a.u = u;
  a.lam = work;
  a.info = out->info;
  a.g_xyz = out->joint_xyz; a.g_aed = out->member_aed; a.g_force = out->force;
  rc = tb_launch_adj_rhs_ragged(a, st);
  if (rc) return rc;
  tb_ragged_in ain = *in;                       // same trusses, load := r (its supported rows are ignored)
  ain.force = work;
  const tb_batch_out aout = {work, nullptr, nullptr, nullptr, out->info, nullptr, nullptr};
  rc = run_ragged(&ain, &aout, st);
  if (rc) return rc;
  return tb_launch_sens_ragged(a, st);
}

// pinned host buffers for callers that want full-speed H2D/D2H through the *_host entry points
extern "C" int tb_pinned_alloc(void** ptr, size_t bytes) {
  if (!ptr) return TB_ERR_NULL;
  if (!have_device()) return TB_ERR_NO_DEVICE;
  TB_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
  return TB_OK;
}
extern "C" int tb_pinned_free(void* ptr) {
  if (ptr) TB_CUDA(cudaFreeHost(ptr));
  return TB_OK;
}
