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

// ---- grow-only device buffers ----------------------------------------------------------------------------------------
// Grown after the whole device is idle (the workspace, the compact temporaries, the staging arenas), to need + slack bytes
int reserve_sync(DevBuf& b, size_t need, size_t slack) {
  if (b.bytes >= need) return TB_OK;
  if (b.ptr) {
    TB_CUDA(cudaDeviceSynchronize());
    TB_CUDA(cudaFree(b.ptr));
    b = DevBuf();
  }
  TB_CUDA(cudaMalloc(&b.ptr, need + slack));
  b.bytes = need + slack;
  return TB_OK;
}

// the staging arenas of the *_host calls: 4 KB of margin, and an eighth more when they grow
int reserve_stage(DevBuf& b, size_t need) { return reserve_sync(b, need + 4096, (need + 4096) / 8); }

// Grown stream-ordered on `st` (the scratch of tb_adjoint, the modal and the envelope kernels): the previous call's
// kernels are ahead on st, StreamOrder::acquire put them there
int reserve_async(DevBuf& b, size_t need, cudaStream_t st) {
  if (b.bytes >= need) return TB_OK;
  if (b.ptr) TB_CUDA(cudaFreeAsync(b.ptr, st));
  b = DevBuf();
  TB_CUDA(cudaMallocAsync(&b.ptr, need, st));
  b.bytes = need;
  return TB_OK;
}

bool capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) (void)cudaGetLastError();
  return cap != cudaStreamCaptureStatusNone;
}

}  // namespace

// The previous call's kernels may still be running on another stream.  A captured step is single-stream by contract.
int StreamOrder::acquire(cudaStream_t st) {
  if (!capturing(st) && used && last != st && ev) TB_CUDA(cudaStreamWaitEvent(st, ev, 0));
  return TB_OK;
}
int StreamOrder::release(cudaStream_t st) {
  if (capturing(st)) return TB_OK;
  if (!ev) TB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  TB_CUDA(cudaEventRecord(ev, st));
  last = st;
  used = true;
  return TB_OK;
}

namespace {

// Scratch of a call on `st` that kernels of earlier calls on other streams may still use: waits for them (ord), then grows
// stream-ordered; the caller launches, then ord.release.  Inside a stream capture it is never grown: TB_ERR_ALLOC with
// nothing enqueued (a warm-up call outside the capture grows it).
int acquire_scratch(StreamOrder& ord, DevBuf& buf, size_t need, cudaStream_t st) {
  if (buf.bytes < need && capturing(st)) return TB_ERR_ALLOC;
  const int rc = ord.acquire(st);
  if (rc) return rc;
  return reserve_async(buf, need, st);
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
int ensure_compact_tmp(tb_plan* p, const tb_batch_out* out, int batch) {
  if (!out || p->path != 0) return TB_OK;      // (the blocked pipelines' recovery kernel writes the compact outputs itself)
  const size_t bytes = (size_t)batch * p->N * sizeof(double);
  if (out->u_free && !out->u) {
    const int rc = reserve_sync(p->compact_u, bytes, 0);
    if (rc) return rc;
  }
  if (out->react && !out->ext) return reserve_sync(p->compact_ext, bytes, 0);
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
  if (out->u_free && !eff.u) eff.u = (double*)p->compact_u.ptr;          // (ensure_compact_tmp sized them for the whole batch)
  if (out->react && !eff.ext) eff.ext = (double*)p->compact_ext.ptr;
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

// The plan belongs to the device it was created on (its maps and workspace live there)
int check_device(const tb_plan* p) {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) return TB_ERR_NO_DEVICE;
  return dev == p->device ? TB_OK : TB_ERR_WRONG_DEVICE;
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
    rc = p->ws_order.acquire(st);
    if (rc) return rc;
  }
  rc = run_plan_unlocked(p, in, out, fit, allow_s, allow_d, st, shared_k);
  if (!rc && p->path != 0) rc = p->ws_order.release(st);
  return rc;
}

int run_plan_unlocked(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                      double allow_d, cudaStream_t st, int shared_k) {
  static const tb_batch_out none = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (!out) out = &none;
  {
    const int rc0 = ensure_compact_tmp(p, out, in->batch);
    if (rc0) return rc0;
  }
  if (p->path == 0) {
    int rc = run_plan_range(p, in, out, fit, allow_s, allow_d, st, 0, in->batch, nullptr);
    if (rc) return rc;
  } else {
    // blocked paths: process the batch in chunks that fit the workspace cap
    const size_t per_sys = plan_ws_bytes(p, 1);
    int chunk = (int)std::min<size_t>((size_t)in->batch, std::max<size_t>(1, ws_cap_bytes() / per_sys));
    int rc = reserve_sync(p->ws, plan_ws_bytes(p, chunk), 0);
    if (rc) return rc;
    for (int b0 = 0; b0 < in->batch; b0 += chunk) {
      rc = run_plan_range(p, in, out, fit, allow_s, allow_d, st, b0, std::min(chunk, in->batch - b0), p->ws.ptr, shared_k);
      if (rc) return rc;
    }
  }
  if (fit && fit->info && out->info) {
    TB_CUDA(cudaMemcpyAsync(out->info, fit->info, sizeof(int32_t) * in->batch, cudaMemcpyDeviceToDevice, st));
  }
  return TB_OK;
}

// ---- bump allocation over a grow-only device arena: 256-byte aligned pieces ------------------------------------------
struct Arena {
  static size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
  static size_t sum(std::initializer_list<size_t> bytes) {
    size_t s = 0;
    for (size_t b : bytes) s += al(b);
    return s;
  }
};

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
size_t rows(int64_t stride, int64_t row, int B) { return (size_t)(stride == 0 ? row : row * B); }   // elements to stage

// The strides of a uniform batch's geometry and member inputs on the host: 0 (shared by the batch) or one system's row
int check_in_strides(const tb_plan* p, const tb_batch_in* in) {
  if (!stride_ok(in->joint_stride, (int64_t)p->nJ * p->dim)) return TB_ERR_SIZE;
  if (in->member_aed ? !stride_ok(in->member_stride, (int64_t)p->M * 3) : !stride_ok(in->gene_stride, p->M)) return TB_ERR_SIZE;
  return TB_OK;
}

// Elements of those inputs to stage
struct InCounts {
  size_t xyz, aed, gene, tab;
  InCounts(const tb_plan* p, const tb_batch_in* in)
      : xyz(rows(in->joint_stride, (int64_t)p->nJ * p->dim, in->batch)),
        aed(in->member_aed ? rows(in->member_stride, (int64_t)p->M * 3, in->batch) : 0),
        gene(in->member_aed ? 0 : rows(in->gene_stride, p->M, in->batch)),
        tab(in->member_aed ? 0 : (size_t)in->n_type * 3) {}
};

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

// The blocking host entry points run body(hp): serialised per process (g_pipe_mu: helper streams, events, the ragged
// arenas) and per plan (p->mu: staging arena, workspace), after every pipelined call of the plan (they share the compute
// stream and the workspace); on an error the helper streams are drained before the code is returned, so nothing of the
// call may still be copying into the caller's buffers.  p: null for the ragged calls.
template <class F>
int host_call(tb_plan* p, F body) {
  std::lock_guard<std::mutex> pipe_lock(g_pipe_mu);
  std::unique_lock<std::mutex> plan_lock;
  if (p) plan_lock = std::unique_lock<std::mutex>(p->mu);
  HostPipe* hp = host_pipe();
  if (!hp) return TB_ERR_ALLOC;
  int rc = p ? async_drain(p) : TB_OK;
  if (rc) return rc;
  rc = body(hp);
  if (rc) host_pipe_drain(hp);
  return rc;
}

// Stages a uniform batch's geometry and member inputs (strides checked) at the start of the plan's staging arena, grown
// to hold `extra` bytes more, with plain copies on `st`.  *din: the device-side batch (no load); *cur: the arena past them.
int stage_in(tb_plan* p, const tb_batch_in* in, size_t extra, cudaStream_t st, tb_batch_in* din, char** cur) {
  const InCounts c(p, in);
  const int rc = reserve_stage(p->stage_dev, Arena::sum({c.xyz * 8, c.aed * 8, c.gene * 4, c.tab * 8}) + extra);
  if (rc) return rc;
  *cur = (char*)p->stage_dev.ptr;
  *din = *in;
  din->force = nullptr;
  double* dxyz = take<double>(*cur, c.xyz);
  TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, c.xyz * 8, cudaMemcpyHostToDevice, st));
  din->joint_xyz = dxyz;
  if (in->member_aed) {
    double* daed = take<double>(*cur, c.aed);
    TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, c.aed * 8, cudaMemcpyHostToDevice, st));
    din->member_aed = daed;
    din->gene = nullptr;
  } else {
    int32_t* dgene = take<int32_t>(*cur, c.gene);
    double* dtab = take<double>(*cur, c.tab);
    TB_CUDA(cudaMemcpyAsync(dgene, in->gene, c.gene * 4, cudaMemcpyHostToDevice, st));
    TB_CUDA(cudaMemcpyAsync(dtab, in->type_table, c.tab * 8, cudaMemcpyHostToDevice, st));
    din->gene = dgene;
    din->type_table = dtab;
  }
  return TB_OK;
}

int run_plan_host(tb_plan* p, const tb_batch_in* in, const tb_batch_out* out, const tb_fit_out* fit, double allow_s,
                  double allow_d, int shared_k = 0) {
  int rc = check_batch_in(p, in);
  if (rc) return rc;
  rc = check_device(p);
  if (rc) return rc;
  return host_call(p, [&](HostPipe* hp) -> int {
    if (p->path != 0) {
      const int r2 = p->ws_order.acquire(hp->comp);
      if (r2) return r2;
    }
    const int r2 = run_plan_host_locked(p, in, out, fit, allow_s, allow_d, shared_k, hp);
    return r2 || p->path == 0 ? r2 : p->ws_order.release(hp->comp);
  });
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
    rc = p->ws_order.acquire(hp->comp);
    if (rc) return rc;
  }
  rc = in->batch == 0 ? TB_OK : run_plan_host_locked(p, in, out, nullptr, 0.0, 0.0, 0, hp, slot);
  if (rc) {
    host_pipe_drain(hp);
    p->async_completed = p->async_submitted;
    return rc;
  }
  if (p->path != 0) rc = p->ws_order.release(hp->comp);
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
  if (check_in_strides(p, in) || !stride_ok(in->force_stride, rowN)) return TB_ERR_SIZE;
  const InCounts c(p, in);
  const size_t nf = rows(in->force_stride, rowN, B);
  static const tb_batch_out none = {nullptr, nullptr, nullptr, nullptr, nullptr};
  if (!out) out = &none;

  const size_t need = Arena::sum({c.xyz * 8, nf * 8, c.aed * 8, c.gene * 4, c.tab * 8,
                                  out->u ? (size_t)B * rowN * 8 : 0, out->ext ? (size_t)B * rowN * 8 : 0,
                                  out->axial ? (size_t)B * rowM * 8 : 0, out->weight ? (size_t)B * 8 : 0,
                                  (size_t)B * 4, fit ? (size_t)B * 8 : 0, fit ? (size_t)B * 2 : 0,
                                  out->u_free ? (size_t)B * p->n * 8 : 0, out->react ? (size_t)B * p->s * 8 : 0});
  DevBuf& arena = async ? p->stage_async[async_slot] : p->stage_dev;
  rc = reserve_stage(arena, need);
  if (rc) return rc;

  cudaStream_t st = hp->comp;
  char* cur = (char*)arena.ptr;
  tb_batch_in din = *in;
  double* dxyz = take<double>(cur, c.xyz);
  double* df = take<double>(cur, nf);
  double* daed = take<double>(cur, c.aed);
  int32_t* dgene = take<int32_t>(cur, c.gene);
  double* dtab = take<double>(cur, c.tab);
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
  rc = ensure_compact_tmp(p, &dout, B);
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
    rc = reserve_sync(p->ws, per_sys * (size_t)csz + 4096, 0);   // chunks run one after the other: one workspace slice
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
  if (sx) TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, c.xyz * 8, cudaMemcpyHostToDevice, cin));
  if (sf) TB_CUDA(cudaMemcpyAsync(df, in->force, nf * 8, cudaMemcpyHostToDevice, cin));
  if (in->member_aed) {
    if (sm_) TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, c.aed * 8, cudaMemcpyHostToDevice, cin));
  } else {
    if (sm_) TB_CUDA(cudaMemcpyAsync(dgene, in->gene, c.gene * 4, cudaMemcpyHostToDevice, cin));
    TB_CUDA(cudaMemcpyAsync(dtab, in->type_table, c.tab * 8, cudaMemcpyHostToDevice, cin));
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
      rc = run_plan_range(p, &din, &dout, fit ? &dfit : nullptr, allow_s, allow_d, comp, b0, nb, p->ws.ptr, shared_k);
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

bool ragged_fits_fused(const tb_ragged_in* in) {
  return tb_small_fits(in->dim, in->max_joint, in->max_member, in->max_joint * in->dim);
}

// the launch's free-DOF bound of a modal ragged call: max_free, or every DOF of the largest truss up to the kernel's limit
int modes_ragged_bound(const tb_ragged_in* in, const tb_modes_ragged_in* m) {
  return m->max_free ? m->max_free : std::min(in->dim * in->max_joint, TB_SMALL_MAX_DOF);
}

// Argument checks of the ragged entry points, in this order: the layout and sizes; the modal arguments (m != null);
// then, for a non-empty batch, the packed arrays (the load too, unless modal) and the size limit: the fused kernels'
// (`fused`: tb_adjoint_ragged, whose solve runs on them) or the envelope kernel's
int check_ragged(const tb_ragged_in* in, const tb_modes_ragged_in* m, bool fused) {
  if (!in) return TB_ERR_NULL;
  if (in->dim != 2 && in->dim != 3) return TB_ERR_DIM;
  if (in->batch < 0 || in->max_joint < 0 || in->max_member < 0) return TB_ERR_SIZE;
  if (m) {
    if (m->consistent != 0 && m->consistent != 1) return TB_ERR_SIZE;
    if (m->max_free < 0 || m->max_free > TB_SMALL_MAX_DOF || m->n_modes < 1) return TB_ERR_SIZE;
    if (in->batch > 0 && m->n_modes > modes_ragged_bound(in, m)) return TB_ERR_SIZE;
  }
  if (in->batch == 0) return TB_OK;
  if (!in->joint_off || !in->member_off || !in->joint_xyz || !in->support || !in->conn || !in->member_aed || (!m && !in->force))
    return TB_ERR_NULL;
  if (fused) return ragged_fits_fused(in) ? TB_OK : TB_ERR_TOO_LARGE;
  if ((int64_t)in->max_joint * in->dim > TB_RAGGED_MAX_DOF || in->max_member > TB_RAGGED_MAX_MEMBER) return TB_ERR_TOO_LARGE;
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

// Argument checks of tb_solve_ragged, tb_solve_ragged_env and tb_solve_ragged_host: no compact outputs (they need one n
// and s for the whole batch), check_ragged's, the outputs, then the device
int check_ragged_fwd(const tb_ragged_in* in, const tb_batch_out* out) {
  if (out && (out->u_free || out->react)) return TB_ERR_SIZE;
  const int rc = check_ragged(in, nullptr, false);
  if (rc) return rc;
  if (!out) return TB_ERR_NULL;
  return have_device() ? TB_OK : TB_ERR_NO_DEVICE;
}

// staging arena of the ragged host entry points: one per device (device memory), used under g_pipe_mu
DevBuf g_rag_dev[TB_MAX_DEVICES];

// The offsets of a ragged batch on the host (the *_host entry points; batch > 0)
int check_ragged_offsets_host(const tb_ragged_in* in) {
  if (in->joint_off[0] != 0 || in->member_off[0] != 0) return TB_ERR_SIZE;
  for (int b = 0; b < in->batch; ++b) {
    const int64_t nj = in->joint_off[b + 1] - in->joint_off[b], nm = in->member_off[b + 1] - in->member_off[b];
    if (nj < 0 || nm < 0) return TB_ERR_SIZE;
    if (nj > in->max_joint || nm > in->max_member) return TB_ERR_TOO_LARGE;
  }
  return TB_OK;
}

// Stages the six packed arrays of a ragged batch (offsets checked) at the start of the device's ragged arena, grown to hold
// `extra` bytes more, with plain copies on `st`.  *din: the device-side batch (no load); *cur: the arena past them.
int stage_ragged_in(const tb_ragged_in* in, size_t extra, cudaStream_t st, tb_ragged_in* din, char** cur) {
  const int B = in->batch, d = in->dim;
  const size_t SJ = (size_t)in->joint_off[B], SM = (size_t)in->member_off[B];
  int dev = 0;
  TB_CUDA(cudaGetDevice(&dev));
  DevBuf& arena = g_rag_dev[dev & (TB_MAX_DEVICES - 1)];
  const int rc = reserve_stage(arena, Arena::sum({(size_t)(B + 1) * 8, (size_t)(B + 1) * 8, SJ * d * 8, SJ, SM * 8, SM * 24}) + extra);
  if (rc) return rc;
  *cur = (char*)arena.ptr;
  int64_t* djo = take<int64_t>(*cur, B + 1);
  int64_t* dmo = take<int64_t>(*cur, B + 1);
  double* dxyz = take<double>(*cur, SJ * d);
  uint8_t* dsup = take<uint8_t>(*cur, SJ);
  int32_t* dconn = take<int32_t>(*cur, SM * 2);
  double* daed = take<double>(*cur, SM * 3);
  TB_CUDA(cudaMemcpyAsync(djo, in->joint_off, (B + 1) * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dmo, in->member_off, (B + 1) * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dxyz, in->joint_xyz, SJ * d * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dsup, in->support, SJ, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(dconn, in->conn, SM * 8, cudaMemcpyHostToDevice, st));
  TB_CUDA(cudaMemcpyAsync(daed, in->member_aed, SM * 24, cudaMemcpyHostToDevice, st));
  *din = *in;
  din->joint_off = djo; din->member_off = dmo; din->joint_xyz = dxyz; din->support = dsup;
  din->conn = dconn; din->member_aed = daed; din->force = nullptr;
  return TB_OK;
}

// Scratch of the envelope kernel: one grow-only arena per device (one slot per CTA of the persistent grid), grown
// stream-ordered on the caller's stream.  `mu` serialises the calls on the device; `order` orders the arena's use across
// streams.
struct EnvScratch {
  std::mutex mu;
  DevBuf buf;
  StreamOrder order;
};
EnvScratch g_env[TB_MAX_DEVICES];

// Envelope kernel over a batch: every truss (route = false), only the trusses above the fused launch's sizes (route:
// those run first, in one fused launch of the batch), or the ordering mode (order != null).
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
  rc = acquire_scratch(S.order, S.buf, slot * (size_t)grid, st);
  if (rc) return rc;
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
  a.scratch = S.buf.ptr;
  a.slot_bytes = slot;
  a.env_smem = env_smem;
  rc = tb_launch_rag_env(a, grid, smem, st);
  if (rc) return rc;
  return S.order.release(st);
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
  int rc = check_ragged_fwd(in, out);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  return run_ragged_fwd(in, out, (cudaStream_t)cuda_stream);
}

extern "C" int tb_solve_ragged_env(const tb_ragged_in* in, const tb_batch_out* out, void* cuda_stream) {
  int rc = check_ragged_fwd(in, out);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  return run_env(in, out, false, nullptr, nullptr, (cudaStream_t)cuda_stream);
}

extern "C" int tb_ragged_env_order(const tb_ragged_in* in, int32_t* order, int64_t* envelope, void* cuda_stream) {
  int rc = check_ragged(in, nullptr, false);
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
  int rc = check_ragged_fwd(in, out);
  if (rc) return rc;
  const int B = in->batch, d = in->dim;
  if (B == 0) return TB_OK;
  rc = check_ragged_offsets_host(in);
  if (rc) return rc;
  const size_t SJ = (size_t)in->joint_off[B], SM = (size_t)in->member_off[B];
  return host_call(nullptr, [&](HostPipe* hp) -> int {
    cudaStream_t st = hp->comp;
    tb_ragged_in din;
    char* cur = nullptr;
    int r2 = stage_ragged_in(in, Arena::sum({SJ * d * 8, out->u ? SJ * d * 8 : 0, out->ext ? SJ * d * 8 : 0, out->axial ? SM * 8 : 0,
                                             out->weight ? (size_t)B * 8 : 0, (size_t)B * 4}), st, &din, &cur);
    if (r2) return r2;
    double* df = take<double>(cur, SJ * d);
    TB_CUDA(cudaMemcpyAsync(df, in->force, SJ * d * 8, cudaMemcpyHostToDevice, st));
    din.force = df;
    tb_batch_out dout;
    dout.u_free = dout.react = nullptr;
    dout.u = out->u ? take<double>(cur, SJ * d) : nullptr;
    dout.ext = out->ext ? take<double>(cur, SJ * d) : nullptr;
    dout.axial = out->axial ? take<double>(cur, SM) : nullptr;
    dout.weight = out->weight ? take<double>(cur, (size_t)B) : nullptr;
    dout.info = take<int32_t>(cur, (size_t)B);
    r2 = run_ragged_fwd(&din, &dout, st);
    if (r2) return r2;
    if (out->u) TB_CUDA(cudaMemcpyAsync(out->u, dout.u, SJ * d * 8, cudaMemcpyDeviceToHost, st));
    if (out->ext) TB_CUDA(cudaMemcpyAsync(out->ext, dout.ext, SJ * d * 8, cudaMemcpyDeviceToHost, st));
    if (out->axial) TB_CUDA(cudaMemcpyAsync(out->axial, dout.axial, SM * 8, cudaMemcpyDeviceToHost, st));
    if (out->weight) TB_CUDA(cudaMemcpyAsync(out->weight, dout.weight, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
    if (out->info) TB_CUDA(cudaMemcpyAsync(out->info, dout.info, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  });
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
  rc = check_in_strides(p, in);
  if (rc) return rc;
  const size_t nkv = (size_t)B * nnz, nscr = (size_t)B * p->M * (2 + p->dim + p->dim * (p->dim + 1) / 2);
  std::vector<double> host(nkv);
  rc = host_call(p, [&](HostPipe* hp) -> int {
    cudaStream_t st = hp->comp;
    tb_batch_in din;
    char* cur = nullptr;
    int r2 = stage_in(p, in, Arena::sum({nkv * 8, nscr * 8, (size_t)B * 4}), st, &din, &cur);
    if (r2) return r2;
    LargeArgs a;
    memset(&a, 0, sizeof(a));
    a.batch = B; a.dim = p->dim; a.nJ = p->nJ; a.M = p->M; a.N = p->N; a.n = p->n;
    a.xyz = din.joint_xyz; a.xyz_stride = in->joint_stride;
    a.aed = din.member_aed; a.aed_stride = in->member_stride;
    a.conn = p->d_conn;
    a.nnz = (int64_t)nnz;
    a.q_first = ts ? p->ts->d_tq_first : p->d_q_first;
    a.q_multi = ts ? p->ts->d_tq_multi : p->d_q_multi;
    a.q_ptr = ts ? p->ts->d_tq_ptr : p->d_q_ptr;
    a.q_pack = ts ? p->ts->d_tq_pack : p->d_q_pack;
    a.n_multi = (int)(ts ? p->ts->tq_multi.size() : p->q_multi.size());
    a.kv = take<double>(cur, nkv);
    double* q = take<double>(cur, nscr);     // k_geom arrays (only used for very many members)
    a.status = take<int32_t>(cur, (size_t)B);
    a.mk = q; q += (size_t)B * p->M;
    a.mc = q; q += (size_t)B * p->M * p->dim;
    a.mw = q; q += (size_t)B * p->M;
    a.mkc = q;
    r2 = tb_launch_assemble_only(a, p->num_sm, st);
    if (r2) return r2;
    TB_CUDA(cudaMemcpyAsync(host.data(), a.kv, nkv * 8, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  });
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
  rc = p->ws_order.acquire(st);
  if (rc) return rc;
  const bool smem = tb_adjoint_vec_in_smem(p->dim, p->M);
  const size_t rowN = (size_t)B * p->N * 8, nvec = smem ? 0 : (size_t)B * p->M * p->dim * 8;
  const size_t need = 2 * Arena::al(rowN) + Arena::al((size_t)B * 4) + nvec;
  rc = reserve_async(p->adj_buf, need, st);
  if (rc) return rc;
  char* cur = (char*)p->adj_buf.ptr;
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
  return p->ws_order.release(st);
}

// Reverse mode of tb_solve_ragged: adjoint load, the adjoint solve through run_ragged (the same kernel as the forward of
// the batch; K is symmetric: force := r), sensitivities.  The adjoint solution overwrites the load in `work`: every solve
// kernel stages a truss's load rows before it writes that truss's displacement rows, and a truss's rows belong to one
// warp (or CTA), so the host never needs the device-resident total joint count to place a second array.
extern "C" int tb_adjoint_ragged(const tb_ragged_in* in, const double* u, const tb_adj_in* grad, const tb_adj_out* out,
                                 double* work, void* cuda_stream) {
  int rc = check_ragged(in, nullptr, true);
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

// ---- modal analysis (DESIGN.md section 11) ---------------------------------------------------------------------------
namespace {

// Argument checks shared by tb_modes, tb_modes_host and tb_modes_adjoint (p, in, m non-null): sizes, the free-DOF
// limit, the inputs, then the device
int check_modes_args(const tb_plan* p, const tb_batch_in* in, const tb_modes_in* m) {
  if (in->batch < 0 || m->n_modes < 1 || m->n_modes > p->n) return TB_ERR_SIZE;
  if (m->consistent != 0 && m->consistent != 1) return TB_ERR_SIZE;
  if (p->n > TB_SMALL_MAX_DOF) return TB_ERR_TOO_LARGE;
  if (in->batch > 0) {
    if (!in->joint_xyz) return TB_ERR_NULL;
    if (!in->member_aed && !(in->gene && in->type_table && in->n_type > 0)) return TB_ERR_NULL;
  }
  if (p->device < 0 || !have_device()) return TB_ERR_NO_DEVICE;
  return TB_OK;
}

// Argument checks of tb_modes / tb_modes_host: every argument error before the device checks
int check_modes(const tb_plan* p, const tb_batch_in* in, const tb_modes_in* m, const tb_modes_out* out) {
  if (!p || !in || !m || !out) return TB_ERR_NULL;
  if (!out->eigval || !out->info) return TB_ERR_NULL;
  if (m->joint_mass_stride < 0) return TB_ERR_SIZE;
  return check_modes_args(p, in, m);
}

// The batch and plan fields of a k_modes / k_buckling launch
void modes_args(const tb_plan* p, const tb_batch_in* in, ModesArgs& a) {
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.nJ = p->nJ; a.M = p->M; a.N = p->N; a.n = p->n;
  a.plan_stable = p->stable; a.n_type = in->n_type;
  a.xyz = in->joint_xyz; a.xyz_stride = in->joint_stride;
  a.aed = in->member_aed; a.aed_stride = in->member_stride;
  a.gene = in->member_aed ? nullptr : in->gene; a.gene_stride = in->gene_stride;
  a.type_table = in->type_table;
  a.conn = p->d_conn; a.free_ref = p->d_free_ref; a.dof2free = p->d_dof2free;
  a.ent_row = p->d_ent_row; a.ent_col = p->d_ent_col; a.ent_ptr = p->d_ent_ptr; a.nnz = (int64_t)p->ent_row.size();
  a.ctr_member = p->d_ctr_member; a.ctr_local = p->d_ctr_local;
  a.inc_ptr = p->d_inc_ptr; a.inc_mem = p->d_inc_mem;
}

// One k_modes launch over the batch (device pointers), with the plan lock held
int run_modes(tb_plan* p, const tb_batch_in* in, const tb_modes_in* m, const tb_modes_out* out, cudaStream_t st) {
  int threads = 0, smem = 0, per_sm = 0;
  int rc = tb_modes_config(p->dim, p->n, &threads, &smem, &per_sm);
  if (rc) return rc;
  const int sms = p->num_sm > 0 ? p->num_sm : 148;
  const int grid = (int)std::min<int64_t>(in->batch, (int64_t)sms * per_sm);
  if (m->consistent) {                           // the consistent mass's slots: one n x n slot per CTA
    rc = acquire_scratch(p->ws_order, p->modes_buf, (size_t)grid * p->n * p->n * sizeof(double), st);
    if (rc) return rc;
  }
  ModesArgs a;
  modes_args(p, in, a);
  a.n_modes = m->n_modes; a.consistent = m->consistent;
  a.jmass = m->joint_mass; a.jmass_stride = m->joint_mass_stride;
  a.eigval = out->eigval; a.modes = out->modes; a.info = out->info;
  a.slot = m->consistent ? (double*)p->modes_buf.ptr : nullptr;
  rc = tb_launch_modes(a, p->dim, grid, threads, smem, st);
  if (rc) return rc;
  return m->consistent ? p->ws_order.release(st) : TB_OK;
}

}  // namespace

extern "C" int tb_modes(tb_plan* p, const tb_batch_in* in, const tb_modes_in* m, const tb_modes_out* out, void* cuda_stream) {
  int rc = check_modes(p, in, m, out);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_device(p);
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(p->mu);
  return run_modes(p, in, m, out, (cudaStream_t)cuda_stream);
}

// Reverse mode of tb_modes: one k_modes_sens launch, no scratch (so no plan lock and always capturable)
extern "C" int tb_modes_adjoint(tb_plan* p, const tb_batch_in* in, const tb_modes_in* m, const tb_modes_adj_in* g,
                                const tb_modes_adj_out* out, void* cuda_stream) {
  if (!p || !in || !m || !g || !out) return TB_ERR_NULL;
  if (!g->eigval || !g->modes || !g->info || !g->g_eigval) return TB_ERR_NULL;
  if (in->batch > 0 && !in->member_aed) return TB_ERR_NULL;      // (no gradients with respect to a type table)
  int rc = check_modes_args(p, in, m);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_device(p);
  if (rc) return rc;
  ModesSensArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.nJ = p->nJ; a.M = p->M; a.N = p->N; a.n_modes = m->n_modes; a.consistent = m->consistent;
  a.xyz = in->joint_xyz; a.xyz_stride = in->joint_stride;
  a.aed = in->member_aed; a.aed_stride = in->member_stride;
  a.conn = p->d_conn; a.dof2free = p->d_dof2free; a.inc_ptr = p->d_inc_ptr; a.inc_mem = p->d_inc_mem;
  a.eigval = g->eigval; a.modes = g->modes; a.info = g->info; a.g_eigval = g->g_eigval;
  a.g_xyz = out->joint_xyz; a.g_aed = out->member_aed; a.g_jmass = out->joint_mass;
  return tb_launch_modes_sens(a, p->dim, (cudaStream_t)cuda_stream);
}

// Host buffers: staged through the plan's arena like the other *_host calls (plain cudaMemcpyAsync on the compute stream)
extern "C" int tb_modes_host(tb_plan* p, const tb_batch_in* in, const tb_modes_in* m, const tb_modes_out* out) {
  int rc = check_modes(p, in, m, out);
  if (rc) return rc;
  const int B = in->batch;
  if (B == 0) return TB_OK;
  if (check_in_strides(p, in) || (m->joint_mass && !stride_ok(m->joint_mass_stride, p->nJ))) return TB_ERR_SIZE;
  rc = check_device(p);
  if (rc) return rc;
  const size_t njm = m->joint_mass ? rows(m->joint_mass_stride, p->nJ, B) : 0;
  const size_t nval = (size_t)B * m->n_modes, nmode = out->modes ? nval * p->N : 0;
  return host_call(p, [&](HostPipe* hp) -> int {
    cudaStream_t st = hp->comp;
    tb_batch_in din;
    char* cur = nullptr;
    int r2 = stage_in(p, in, Arena::sum({njm * 8, nval * 8, nmode * 8, (size_t)B * 4}), st, &din, &cur);
    if (r2) return r2;
    tb_modes_in dm = *m;
    if (m->joint_mass) {
      double* djm = take<double>(cur, njm);
      TB_CUDA(cudaMemcpyAsync(djm, m->joint_mass, njm * 8, cudaMemcpyHostToDevice, st));
      dm.joint_mass = djm;
    }
    tb_modes_out dout = {take<double>(cur, nval), out->modes ? take<double>(cur, nmode) : nullptr, take<int32_t>(cur, (size_t)B)};
    r2 = run_modes(p, &din, &dm, &dout, st);
    if (r2) return r2;
    TB_CUDA(cudaMemcpyAsync(out->eigval, dout.eigval, nval * 8, cudaMemcpyDeviceToHost, st));
    if (out->modes) TB_CUDA(cudaMemcpyAsync(out->modes, dout.modes, nmode * 8, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->info, dout.info, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  });
}

// ---- linear buckling (DESIGN.md section 12) ---------------------------------------------------------------------------
namespace {

// Argument checks of tb_buckling / tb_buckling_host: the pointers, the axial stride, then tb_modes' checks (sizes, the
// free-DOF limit, the inputs, the device)
int check_buckling(const tb_plan* p, const tb_batch_in* in, const tb_buckling_in* bk, const tb_buckling_out* out) {
  if (!p || !in || !bk || !out) return TB_ERR_NULL;
  if (!bk->axial || !out->factor || !out->info) return TB_ERR_NULL;
  if (bk->axial_stride < 0) return TB_ERR_SIZE;
  const tb_modes_in m = {bk->n_modes, 0, nullptr, 0};
  return check_modes_args(p, in, &m);
}

// One k_buckling launch over the batch (device pointers), with the plan lock held: K_ff and its factor take one slot
// of the modal arena per CTA on every call
int run_buckling(tb_plan* p, const tb_batch_in* in, const tb_buckling_in* bk, const tb_buckling_out* out, cudaStream_t st) {
  int threads = 0, smem = 0, per_sm = 0;
  int rc = tb_buckling_config(p->dim, p->n, &threads, &smem, &per_sm);
  if (rc) return rc;
  const int sms = p->num_sm > 0 ? p->num_sm : 148;
  const int grid = (int)std::min<int64_t>(in->batch, (int64_t)sms * per_sm);
  rc = acquire_scratch(p->ws_order, p->modes_buf, (size_t)grid * p->n * p->n * sizeof(double), st);
  if (rc) return rc;
  BucklingArgs a;
  memset(&a, 0, sizeof(a));
  modes_args(p, in, a.base);
  a.base.n_modes = bk->n_modes; a.base.consistent = 1;
  a.base.eigval = out->factor; a.base.modes = out->modes; a.base.info = out->info;
  a.base.slot = (double*)p->modes_buf.ptr;
  a.axial = bk->axial; a.axial_stride = bk->axial_stride;
  rc = tb_launch_buckling(a, p->dim, grid, threads, smem, st);
  if (rc) return rc;
  return p->ws_order.release(st);
}

}  // namespace

extern "C" int tb_buckling(tb_plan* p, const tb_batch_in* in, const tb_buckling_in* bk, const tb_buckling_out* out,
                           void* cuda_stream) {
  int rc = check_buckling(p, in, bk, out);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_device(p);
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(p->mu);
  return run_buckling(p, in, bk, out, (cudaStream_t)cuda_stream);
}

// Reverse mode of tb_buckling: one k_buckling_sens launch, no scratch (so no plan lock and always capturable).  Argument
// errors in check_buckling's order: the pointers (a gene batch has no member gradient), the axial stride, tb_modes' checks
extern "C" int tb_buckling_adjoint(tb_plan* p, const tb_batch_in* in, const tb_buckling_in* bk, const tb_modes_adj_in* g,
                                   const tb_buckling_adj_out* out, void* cuda_stream) {
  if (!p || !in || !bk || !g || !out) return TB_ERR_NULL;
  if (!bk->axial || !g->eigval || !g->modes || !g->info || !g->g_eigval) return TB_ERR_NULL;
  if (in->batch > 0 && !in->member_aed) return TB_ERR_NULL;      // (no gradients with respect to a type table)
  if (bk->axial_stride < 0) return TB_ERR_SIZE;
  const tb_modes_in m = {bk->n_modes, 0, nullptr, 0};
  int rc = check_modes_args(p, in, &m);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  rc = check_device(p);
  if (rc) return rc;
  BucklingSensArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.nJ = p->nJ; a.M = p->M; a.N = p->N; a.n_modes = bk->n_modes;
  a.xyz = in->joint_xyz; a.xyz_stride = in->joint_stride;
  a.aed = in->member_aed; a.aed_stride = in->member_stride;
  a.axial = bk->axial; a.axial_stride = bk->axial_stride;
  a.conn = p->d_conn; a.dof2free = p->d_dof2free; a.inc_ptr = p->d_inc_ptr; a.inc_mem = p->d_inc_mem;
  a.factor = g->eigval; a.modes = g->modes; a.info = g->info; a.g_factor = g->g_eigval;
  a.g_xyz = out->joint_xyz; a.g_aed = out->member_aed; a.g_axial = out->axial;
  return tb_launch_buckling_sens(a, p->dim, (cudaStream_t)cuda_stream);
}

// Host buffers: staged through the plan's arena like tb_modes_host (plain cudaMemcpyAsync on the compute stream)
extern "C" int tb_buckling_host(tb_plan* p, const tb_batch_in* in, const tb_buckling_in* bk, const tb_buckling_out* out) {
  int rc = check_buckling(p, in, bk, out);
  if (rc) return rc;
  const int B = in->batch;
  if (B == 0) return TB_OK;
  if (check_in_strides(p, in) || !stride_ok(bk->axial_stride, p->M)) return TB_ERR_SIZE;
  rc = check_device(p);
  if (rc) return rc;
  const size_t nax = rows(bk->axial_stride, p->M, B);
  const size_t nval = (size_t)B * bk->n_modes, nmode = out->modes ? nval * p->N : 0;
  return host_call(p, [&](HostPipe* hp) -> int {
    cudaStream_t st = hp->comp;
    tb_batch_in din;
    char* cur = nullptr;
    int r2 = stage_in(p, in, Arena::sum({nax * 8, nval * 8, nmode * 8, (size_t)B * 4}), st, &din, &cur);
    if (r2) return r2;
    tb_buckling_in dbk = *bk;
    double* dax = take<double>(cur, nax);
    TB_CUDA(cudaMemcpyAsync(dax, bk->axial, nax * 8, cudaMemcpyHostToDevice, st));
    dbk.axial = dax;
    tb_buckling_out dout = {take<double>(cur, nval), out->modes ? take<double>(cur, nmode) : nullptr,
                            take<int32_t>(cur, (size_t)B)};
    r2 = run_buckling(p, &din, &dbk, &dout, st);
    if (r2) return r2;
    TB_CUDA(cudaMemcpyAsync(out->factor, dout.factor, nval * 8, cudaMemcpyDeviceToHost, st));
    if (out->modes) TB_CUDA(cudaMemcpyAsync(out->modes, dout.modes, nmode * 8, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->info, dout.info, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  });
}

// ---- modal analysis of ragged batches ---------------------------------------------------------------------------------
namespace {

// Argument checks shared by tb_modes_ragged, tb_modes_ragged_host and tb_modes_adjoint_ragged (in, m non-null):
// check_ragged's, then the device (as tb_solve_ragged, also for B = 0)
int check_modes_ragged_args(const tb_ragged_in* in, const tb_modes_ragged_in* m) {
  const int rc = check_ragged(in, m, false);
  if (rc) return rc;
  return have_device() ? TB_OK : TB_ERR_NO_DEVICE;
}

int check_modes_ragged(const tb_ragged_in* in, const tb_modes_ragged_in* m, const tb_modes_ragged_out* out) {
  if (!in || !m || !out) return TB_ERR_NULL;
  if (!out->eigval || !out->info) return TB_ERR_NULL;
  return check_modes_ragged_args(in, m);
}

// One k_modes_ragged launch over the batch (device pointers).  Consistent mass: one bound x bound slot per CTA in the
// device's envelope arena (g_env: its lock, event and capture rule)
int run_modes_ragged(const tb_ragged_in* in, const tb_modes_ragged_in* m, const tb_modes_ragged_out* out, cudaStream_t st) {
  const int bound = modes_ragged_bound(in, m);
  int threads = 0, smem = 0, per_sm = 0, dev = 0, sms = 0;
  int rc = tb_modes_ragged_config(in->dim, bound, &threads, &smem, &per_sm);
  if (rc) return rc;
  TB_CUDA(cudaGetDevice(&dev));
  TB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = (int)std::min<int64_t>(in->batch, (int64_t)sms * per_sm);
  ModesRagArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.max_joint = in->max_joint; a.max_member = in->max_member; a.max_free = bound;
  a.n_modes = m->n_modes; a.consistent = m->consistent;
  a.joint_off = in->joint_off; a.member_off = in->member_off;
  a.xyz = in->joint_xyz; a.support = in->support; a.conn = in->conn; a.aed = in->member_aed;
  a.jmass = m->joint_mass;
  a.eigval = out->eigval; a.modes = out->modes; a.n_free = out->n_free; a.info = out->info;
  if (!m->consistent) return tb_launch_modes_ragged(a, in->dim, grid, threads, smem, st);
  EnvScratch& S = g_env[dev & (TB_MAX_DEVICES - 1)];
  std::lock_guard<std::mutex> lock(S.mu);
  rc = acquire_scratch(S.order, S.buf, (size_t)grid * bound * bound * sizeof(double), st);
  if (rc) return rc;
  a.slot = (double*)S.buf.ptr;
  rc = tb_launch_modes_ragged(a, in->dim, grid, threads, smem, st);
  if (rc) return rc;
  return S.order.release(st);
}

}  // namespace

extern "C" int tb_modes_ragged(const tb_ragged_in* in, const tb_modes_ragged_in* m, const tb_modes_ragged_out* out,
                               void* cuda_stream) {
  int rc = check_modes_ragged(in, m, out);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  return run_modes_ragged(in, m, out, (cudaStream_t)cuda_stream);
}

// Host buffers: the offsets are validated on the host, then staged through the ragged staging arena on the host pipe's
// compute stream (plain cudaMemcpyAsync), as tb_solve_ragged_host
extern "C" int tb_modes_ragged_host(const tb_ragged_in* in, const tb_modes_ragged_in* m, const tb_modes_ragged_out* out) {
  int rc = check_modes_ragged(in, m, out);
  if (rc) return rc;
  const int B = in->batch, d = in->dim;
  if (B == 0) return TB_OK;
  rc = check_ragged_offsets_host(in);
  if (rc) return rc;
  const size_t SJ = (size_t)in->joint_off[B], nm = (size_t)m->n_modes;
  return host_call(nullptr, [&](HostPipe* hp) -> int {
    cudaStream_t st = hp->comp;
    tb_ragged_in din;
    char* cur = nullptr;
    int r2 = stage_ragged_in(in, Arena::sum({m->joint_mass ? SJ * 8 : 0, (size_t)B * nm * 8, out->modes ? nm * d * SJ * 8 : 0,
                                             (size_t)B * 4, (size_t)B * 4}), st, &din, &cur);
    if (r2) return r2;
    tb_modes_ragged_in dm = *m;
    if (m->joint_mass) {
      double* djm = take<double>(cur, SJ);
      TB_CUDA(cudaMemcpyAsync(djm, m->joint_mass, SJ * 8, cudaMemcpyHostToDevice, st));
      dm.joint_mass = djm;
    }
    tb_modes_ragged_out dout;
    dout.eigval = take<double>(cur, (size_t)B * nm);
    dout.modes = out->modes ? take<double>(cur, nm * d * SJ) : nullptr;
    dout.n_free = take<int32_t>(cur, (size_t)B);
    dout.info = take<int32_t>(cur, (size_t)B);
    r2 = run_modes_ragged(&din, &dm, &dout, st);
    if (r2) return r2;
    TB_CUDA(cudaMemcpyAsync(out->eigval, dout.eigval, (size_t)B * nm * 8, cudaMemcpyDeviceToHost, st));
    if (out->modes) TB_CUDA(cudaMemcpyAsync(out->modes, dout.modes, nm * d * SJ * 8, cudaMemcpyDeviceToHost, st));
    if (out->n_free) TB_CUDA(cudaMemcpyAsync(out->n_free, dout.n_free, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaMemcpyAsync(out->info, dout.info, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    TB_CUDA(cudaStreamSynchronize(st));
    return TB_OK;
  });
}

// Reverse mode of tb_modes_ragged: one k_modes_sens_ragged launch, no scratch (always capturable)
extern "C" int tb_modes_adjoint_ragged(const tb_ragged_in* in, const tb_modes_ragged_in* m, const tb_modes_adj_in* g,
                                       const tb_modes_adj_out* out, void* cuda_stream) {
  if (!in || !m || !g || !out) return TB_ERR_NULL;
  if (!g->eigval || !g->modes || !g->info || !g->g_eigval) return TB_ERR_NULL;
  int rc = check_modes_ragged_args(in, m);
  if (rc) return rc;
  if (in->batch == 0) return TB_OK;
  ModesSensRagArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = in->batch; a.max_joint = in->max_joint; a.max_member = in->max_member;
  a.n_modes = m->n_modes; a.consistent = m->consistent;
  a.joint_off = in->joint_off; a.member_off = in->member_off;
  a.xyz = in->joint_xyz; a.support = in->support; a.conn = in->conn; a.aed = in->member_aed;
  a.eigval = g->eigval; a.modes = g->modes; a.info = g->info; a.g_eigval = g->g_eigval;
  a.g_xyz = out->joint_xyz; a.g_aed = out->member_aed; a.g_jmass = out->joint_mass;
  return tb_launch_modes_sens_ragged(a, in->dim, (cudaStream_t)cuda_stream);
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
