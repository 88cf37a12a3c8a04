// Reverse mode of the solve (tb_adjoint, DESIGN.md section 9).  K is symmetric, so the adjoint system is the forward
// system with another right-hand side: the entry point in tb_api.cu runs
//
//   k_adj_rhs   adjoint load r = g_u + sum_m N^_m k_m (+c at j1, -c at j0),  N^ = g_axial + c.dz (z = g_ext at supports)
//   (solve)     K_ff lambda = r_ff through the plan's own pipeline (fused, band or tiled)
//   k_sens      dL/d(a, e, density) per member, dL/dxyz per joint, dL/df per DOF
//
// One CTA per system.  Per-member vectors (d doubles) live in shared memory when they fit, else in the caller's HBM
// scratch; the per-DOF / per-joint sums gather them over the plan's joint -> member incidence lists in ascending member
// order, so the results do not depend on the batch size or the launch shape (no atomics).
//
// Ragged batches (tb_adjoint_ragged) run k_adj_rhs_ragged / k_sens_ragged: the same member bodies (adj_rhs_member,
// sens_member), one warp per truss and several trusses per CTA, the per-member vectors in the warp's shared memory.  A
// ragged truss has no plan, so the per-joint sums scan the truss's members in ascending order (rag_gather) and the free
// DOFs come from the support codes (tb_dof_free).
#include "tb_common.cuh"

namespace {

constexpr size_t ADJ_SMEM_MAX = 96 * 1024;

// (+) at the member's joint 1, (-) at its joint 0, summed over the incidence list of joint J, component ax
template <int DIM>
__device__ __forceinline__ double gather_joint(const TbAdjArgs& a, const double* vec, int J, int ax) {
  double v = 0.0;
  for (int p = a.inc_ptr[J]; p < a.inc_ptr[J + 1]; ++p) {
    const int me = a.inc_mem[p], m = me >> 1;
    v += (me & 1) ? vec[m * DIM + ax] : -vec[m * DIM + ax];
  }
  return v;
}

// Per-member body of the adjoint load: vec = N^ k c with N^ = g_axial + c.(z1 - z0), z = g_ext at restrained DOFs.
// xyz / gext are the system's own rows, f0 / f1 the free flags of the member's two joints.  Shared by the uniform and
// the ragged kernels (same operations in the same order: the same bits).
template <int DIM>
__device__ __forceinline__ void adj_rhs_member(const double* xyz, const double* aed_m, const double* gext, int j0, int j1,
                                               const bool f0[DIM], const bool f1[DIM], double g, double* vec_m) {
  double dx[DIM], c[DIM], k, w;
  const double len = tb_member_geom<DIM>(xyz, j0, j1, aed_m[0], aed_m[1], aed_m[2], dx, c, k, w);
  double nh = g;
  if (gext)
#pragma unroll
    for (int i = 0; i < DIM; ++i) {
      const int d1 = j1 * DIM + i, d0 = j0 * DIM + i;
      const double z1 = !f1[i] ? gext[d1] : 0.0, z0 = !f0[i] ? gext[d0] : 0.0;
      nh = fma(c[i], z1 - z0, nh);
    }
  const bool ok = len > 0.0;                 // (a zero-length member fails its system: keep NaN out of the solve)
#pragma unroll
  for (int i = 0; i < DIM; ++i) vec_m[i] = ok ? nh * k * c[i] : 0.0;
}

// Per-member body of the sensitivities: the dL/d(a, e, density) row and the geometry vector (gathered per joint)
template <int DIM>
__device__ __forceinline__ void sens_member(const double* xyz, const double* aed_m, const double* u, const double* lam,
                                            const double* gext, int j0, int j1, const bool f0[DIM], const bool f1[DIM],
                                            double g, double gw, double* ga_m, double* vec_m) {
  const double ar = aed_m[0], e = aed_m[1], rho = aed_m[2];
  double dx[DIM], c[DIM], k, w;
  const double len = tb_member_geom<DIM>(xyz, j0, j1, ar, e, rho, dx, c, k, w);
  double du[DIM], dw[DIM], tu = 0.0, tz = 0.0, tl = 0.0;
#pragma unroll
  for (int i = 0; i < DIM; ++i) {
    const int d1 = j1 * DIM + i, d0 = j0 * DIM + i;
    du[i] = (f1[i] ? u[d1] : 0.0) - (f0[i] ? u[d0] : 0.0);
    const double dl = (f1[i] ? lam[d1] : 0.0) - (f0[i] ? lam[d0] : 0.0);
    const double dz = gext ? (f1[i] ? 0.0 : gext[d1]) - (f0[i] ? 0.0 : gext[d0]) : 0.0;
    dw[i] = dz - dl;
    tu = fma(c[i], du[i], tu);
    tz = fma(c[i], dz, tz);
    tl = fma(c[i], dl, tl);
  }
  const double q = g + tz - tl;              // N^ - c.d(lambda)
  const double tw = tz - tl;                 // c.dw, dw = dz - d(lambda)
  const double kl = k / len;
  ga_m[0] = fma(e / len * tu, q, gw * len * rho);
  ga_m[1] = ar / len * tu * q;
  ga_m[2] = gw * ar * len;
  // d/dd of EA [g (d.du)/L^2 + (d.dw)(d.du)/L^3] + g_w a rho L, written with c = d/L
  const double war = gw * ar * rho;
#pragma unroll
  for (int i = 0; i < DIM; ++i)
    vec_m[i] = kl * (g * (du[i] - 2.0 * tu * c[i]) + dw[i] * tu + du[i] * tw - 3.0 * tu * tw * c[i]) + war * c[i];
}

template <int DIM>
__global__ void __launch_bounds__(256) k_adj_rhs(const TbAdjArgs a) {
  extern __shared__ __align__(16) double sVec[];
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    double* vec = a.vec ? a.vec + (int64_t)b * a.M * DIM : sVec;
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed + b * a.aed_stride;
    const double* gext = a.g_ext ? a.g_ext + (int64_t)b * a.N : nullptr;
    const double* gax = a.g_axial ? a.g_axial + (int64_t)b * a.M : nullptr;
    for (int m = tid; m < a.M; m += 256) {
      const int j0 = a.conn[2 * m], j1 = a.conn[2 * m + 1];
      bool f0[DIM], f1[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        f0[i] = a.dof2free[j0 * DIM + i] >= 0;
        f1[i] = a.dof2free[j1 * DIM + i] >= 0;
      }
      adj_rhs_member<DIM>(xyz, aed + 3 * m, gext, j0, j1, f0, f1, gax ? gax[m] : 0.0, vec + m * DIM);
    }
    __syncthreads();
    double* r = a.r + (int64_t)b * a.N;
    const double* gu = a.g_u ? a.g_u + (int64_t)b * a.N : nullptr;
    for (int dof = tid; dof < a.N; dof += 256) {
      double v = 0.0;
      if (a.dof2free[dof] >= 0) {                // (only the free rows enter the solve)
        const int J = dof / DIM;
        v = (gu ? gu[dof] : 0.0) + gather_joint<DIM>(a, vec, J, dof - J * DIM);
      }
      r[dof] = v;
    }
    __syncthreads();
  }
}

template <int DIM>
__global__ void __launch_bounds__(256) k_sens(const TbAdjArgs a) {
  extern __shared__ __align__(16) double sVec[];
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    double* gx = a.g_xyz ? a.g_xyz + (int64_t)b * a.N : nullptr;
    double* ga = a.g_aed + (int64_t)b * a.M * 3;
    double* gf = a.g_force ? a.g_force + (int64_t)b * a.N : nullptr;
    if (a.info[b] != 0) {                        // failed system: zero gradients, never NaN
      for (int i = tid; i < a.N; i += 256) {
        if (gx) gx[i] = 0.0;
        if (gf) gf[i] = 0.0;
      }
      for (int i = tid; i < 3 * a.M; i += 256) ga[i] = 0.0;
      continue;
    }
    double* vec = a.vec ? a.vec + (int64_t)b * a.M * DIM : sVec;
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed + b * a.aed_stride;
    const double* u = a.u + (int64_t)b * a.N;
    const double* lam = a.lam + (int64_t)b * a.N;
    const double* gext = a.g_ext ? a.g_ext + (int64_t)b * a.N : nullptr;
    const double* gax = a.g_axial ? a.g_axial + (int64_t)b * a.M : nullptr;
    const double gw = a.g_w ? a.g_w[b] : 0.0;
    for (int m = tid; m < a.M; m += 256) {
      const int j0 = a.conn[2 * m], j1 = a.conn[2 * m + 1];
      bool f0[DIM], f1[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        f0[i] = a.dof2free[j0 * DIM + i] >= 0;
        f1[i] = a.dof2free[j1 * DIM + i] >= 0;
      }
      sens_member<DIM>(xyz, aed + 3 * m, u, lam, gext, j0, j1, f0, f1, gax ? gax[m] : 0.0, gw, ga + 3 * m, vec + m * DIM);
    }
    __syncthreads();
    for (int dof = tid; dof < a.N; dof += 256) {
      const int J = dof / DIM;
      if (gx) gx[dof] = gather_joint<DIM>(a, vec, J, dof - J * DIM);
      if (gf) gf[dof] = a.dof2free[dof] >= 0 ? lam[dof] + (gext ? gext[dof] : 0.0) : 0.0;
    }
    __syncthreads();
  }
}

template <typename K>
int launch(K kern, const TbAdjArgs& a, int num_sm, cudaStream_t st) {
  const size_t smem = a.vec ? 0 : (size_t)a.M * a.dim * 8;
  if (smem > 48 * 1024) TB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ADJ_SMEM_MAX));
  const int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
  kern<<<grid, 256, smem, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

// ---- ragged batches: one warp per truss, several trusses per CTA ---------------------------------------------------
// Per warp in shared memory: the per-member vectors [max_member][d] doubles, then the truss's conn [max_member][2] int32.
__host__ __device__ inline int rag_warp_doubles(int dim, int max_member) { return max_member * dim + max_member; }

struct RagTruss {
  int64_t jo, mo;
  int nJ, M;
  bool ok;     // sizes within the batch maxima: the solve ran this truss (else it reported TB_INFO_BAD_INDEX)
  bool rows;   // its rows lie inside the packed arrays: safe to write (zeros) even when !ok
};

__device__ __forceinline__ RagTruss rag_truss(const TbAdjRaggedArgs& a, int b) {
  RagTruss t;
  t.jo = a.joint_off[b];
  t.mo = a.member_off[b];
  const int64_t nj = a.joint_off[b + 1] - t.jo, nm = a.member_off[b + 1] - t.mo;
  t.rows = nj >= 0 && nm >= 0 && t.jo >= 0 && t.mo >= 0 && t.jo + nj <= a.joint_off[a.batch] && t.mo + nm <= a.member_off[a.batch];
  t.ok = t.rows && nj <= a.max_joint && nm <= a.max_member;     // (the forward's `oversize` guard, plus the range check)
  t.nJ = t.rows ? (int)nj : 0;
  t.M = t.rows ? (int)nm : 0;
  return t;
}

// Per-joint sums of a ragged truss, lane per joint: every member in ascending order, (-) at its joint 0 then (+) at its
// joint 1 -- the order of the uniform kernels' incidence lists, so the same bits.  Ids outside [0, nJ) match no joint.
template <int DIM>
__device__ __forceinline__ void rag_gather(const int* sConn, const double* vec, int M, int J, double v[DIM]) {
#pragma unroll
  for (int i = 0; i < DIM; ++i) v[i] = 0.0;
  for (int m = 0; m < M; ++m) {
    const int2 e = reinterpret_cast<const int2*>(sConn)[m];   // (every lane reads the same word: a broadcast)
    if (e.x == J)
#pragma unroll
      for (int i = 0; i < DIM; ++i) v[i] += -vec[m * DIM + i];
    if (e.y == J)
#pragma unroll
      for (int i = 0; i < DIM; ++i) v[i] += vec[m * DIM + i];
  }
}

template <int DIM>
__global__ void __launch_bounds__(256) k_adj_rhs_ragged(const TbAdjRaggedArgs a, const int nwarp) {
  extern __shared__ __align__(16) double sRag[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* vec = sRag + (size_t)wid * rag_warp_doubles(DIM, a.max_member);
  int* sConn = (int*)(vec + a.max_member * DIM);
  for (int b = blockIdx.x * nwarp + wid; b < a.batch; b += gridDim.x * nwarp) {
    const RagTruss t = rag_truss(a, b);
    if (!t.ok) continue;                       // the solve skips it; k_sens_ragged zeroes its gradients
    const int nJ = t.nJ, M = t.M;
    const double* xyz = a.xyz + t.jo * DIM;
    const uint8_t* sup = a.support + t.jo;
    const double* aed = a.aed + t.mo * 3;
    const double* gext = a.g_ext ? a.g_ext + t.jo * DIM : nullptr;
    const double* gax = a.g_axial ? a.g_axial + t.mo : nullptr;
    for (int i = lane; i < 2 * M; i += 32) sConn[i] = a.conn[t.mo * 2 + i];
    __syncwarp();
    for (int m = lane; m < M; m += 32) {
      const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
      if ((unsigned)j0 >= (unsigned)nJ || (unsigned)j1 >= (unsigned)nJ) {   // the solve fails the truss (TB_INFO_BAD_INDEX)
#pragma unroll
        for (int i = 0; i < DIM; ++i) vec[m * DIM + i] = 0.0;
        continue;
      }
      const int s0 = sup[j0], s1 = sup[j1];
      bool f0[DIM], f1[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        f0[i] = tb_dof_free(s0, i);
        f1[i] = tb_dof_free(s1, i);
      }
      adj_rhs_member<DIM>(xyz, aed + 3 * m, gext, j0, j1, f0, f1, gax ? gax[m] : 0.0, vec + m * DIM);
    }
    __syncwarp();
    double* r = a.r + t.jo * DIM;
    const double* gu = a.g_u ? a.g_u + t.jo * DIM : nullptr;
    for (int J = lane; J < nJ; J += 32) {
      double v[DIM];
      rag_gather<DIM>(sConn, vec, M, J, v);
      const int s = sup[J];
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        const int dof = J * DIM + i;
        r[dof] = tb_dof_free(s, i) ? (gu ? gu[dof] : 0.0) + v[i] : 0.0;   // (only the free rows enter the solve)
      }
    }
    __syncwarp();                              // shared arrays are reused by the warp's next truss
  }
}

template <int DIM>
__global__ void __launch_bounds__(256) k_sens_ragged(const TbAdjRaggedArgs a, const int nwarp) {
  extern __shared__ __align__(16) double sRag[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* vec = sRag + (size_t)wid * rag_warp_doubles(DIM, a.max_member);
  int* sConn = (int*)(vec + a.max_member * DIM);
  for (int b = blockIdx.x * nwarp + wid; b < a.batch; b += gridDim.x * nwarp) {
    const RagTruss t = rag_truss(a, b);
    const int nJ = t.nJ, M = t.M, N = nJ * DIM;
    double* gx = a.g_xyz ? a.g_xyz + t.jo * DIM : nullptr;
    double* ga = a.g_aed + t.mo * 3;
    double* gf = a.g_force ? a.g_force + t.jo * DIM : nullptr;
    if (!t.ok || a.info[b] != 0) {             // failed truss: zero gradients, never NaN (nothing when its rows are not valid)
      for (int i = lane; i < N; i += 32) {
        if (gx) gx[i] = 0.0;
        if (gf) gf[i] = 0.0;
      }
      for (int i = lane; i < 3 * M; i += 32) ga[i] = 0.0;
      continue;
    }
    const double* xyz = a.xyz + t.jo * DIM;
    const uint8_t* sup = a.support + t.jo;
    const double* aed = a.aed + t.mo * 3;
    const double* u = a.u + t.jo * DIM;
    const double* lam = a.lam + t.jo * DIM;
    const double* gext = a.g_ext ? a.g_ext + t.jo * DIM : nullptr;
    const double* gax = a.g_axial ? a.g_axial + t.mo : nullptr;
    const double gw = a.g_w ? a.g_w[b] : 0.0;
    for (int i = lane; i < 2 * M; i += 32) sConn[i] = a.conn[t.mo * 2 + i];
    __syncwarp();
    for (int m = lane; m < M; m += 32) {
      const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
      if ((unsigned)j0 >= (unsigned)nJ || (unsigned)j1 >= (unsigned)nJ) {   // (info == 0 rules this out; never read out of range)
#pragma unroll
        for (int i = 0; i < DIM; ++i) vec[m * DIM + i] = 0.0;
        ga[3 * m] = ga[3 * m + 1] = ga[3 * m + 2] = 0.0;
        continue;
      }
      const int s0 = sup[j0], s1 = sup[j1];
      bool f0[DIM], f1[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        f0[i] = tb_dof_free(s0, i);
        f1[i] = tb_dof_free(s1, i);
      }
      sens_member<DIM>(xyz, aed + 3 * m, u, lam, gext, j0, j1, f0, f1, gax ? gax[m] : 0.0, gw, ga + 3 * m, vec + m * DIM);
    }
    __syncwarp();
    for (int J = lane; J < nJ; J += 32) {
      const int s = sup[J];
      double v[DIM];
      if (gx) rag_gather<DIM>(sConn, vec, M, J, v);
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        const int dof = J * DIM + i;
        if (gx) gx[dof] = v[i];
        if (gf) gf[dof] = tb_dof_free(s, i) ? lam[dof] + (gext ? gext[dof] : 0.0) : 0.0;
      }
    }
    __syncwarp();
  }
}

// Warps per CTA: whatever puts the most warps (= trusses in flight) on an SM, as tb_launch_dense16 chooses.  The queries
// cost more than the launch, so the choice is cached per device and kernel for the last RAG_SHAPES per-warp sizes (a
// caller alternating batches of a few different max_member values queries each once).  Grid: persistent, at most
// (resident CTAs per SM) x SMs.
constexpr int RAG_SHAPES = 8;

template <typename K>
int launch_ragged(K kern, int which, const TbAdjRaggedArgs& a, cudaStream_t st) {
  const size_t per = (size_t)rag_warp_doubles(a.dim, a.max_member) * 8;
  constexpr size_t SMEM_MAX = 227 * 1024;
  if (per > SMEM_MAX) return (int)cudaErrorInvalidValue;      // (check_ragged bounds max_member far below this)
  struct Choice { size_t per = ~(size_t)0; int nwarp = 0, per_sm = 0, sms = 0; };
  struct Slot { Choice c[RAG_SHAPES]; int next = 0; bool attr = false; };
  static Slot cache[64][4];
  static std::mutex cache_mu;
  int dev = 0;
  TB_CUDA(cudaGetDevice(&dev));
  Choice ch;
  {
    std::lock_guard<std::mutex> lock(cache_mu);
    Slot& sl = cache[dev & 63][which];
    int hit = -1;
    for (int i = 0; i < RAG_SHAPES; ++i)
      if (sl.c[i].per == per) hit = i;
    if (hit < 0) {
      if (!sl.attr) {
        TB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_MAX));
        sl.attr = true;
      }
      Choice best;
      for (int nw = 8; nw >= 1; --nw) {
        if (per * nw > SMEM_MAX) continue;
        int q = 0;
        TB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, 32 * nw, per * nw));
        if (q * nw > best.per_sm * best.nwarp) { best.nwarp = nw; best.per_sm = q; }
      }
      if (best.nwarp == 0) return (int)cudaErrorInvalidConfiguration;
      TB_CUDA(cudaDeviceGetAttribute(&best.sms, cudaDevAttrMultiProcessorCount, dev));
      best.per = per;
      hit = sl.next;
      sl.next = (sl.next + 1) % RAG_SHAPES;
      sl.c[hit] = best;
    }
    ch = sl.c[hit];
  }
  long long grid = (long long)ch.sms * ch.per_sm;
  const long long need = (a.batch + ch.nwarp - 1) / ch.nwarp;
  if (grid > need) grid = need;
  kern<<<(unsigned)grid, 32 * ch.nwarp, per * ch.nwarp, st>>>(a, ch.nwarp);
  tb_count_launch();
  return (int)cudaGetLastError();
}

}  // namespace

bool tb_adjoint_vec_in_smem(int dim, int M) { return (size_t)M * dim * 8 <= ADJ_SMEM_MAX; }

int tb_launch_adj_rhs(const TbAdjArgs& a, int num_sm, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  return a.dim == 3 ? launch(k_adj_rhs<3>, a, num_sm, st) : launch(k_adj_rhs<2>, a, num_sm, st);
}

int tb_launch_sens(const TbAdjArgs& a, int num_sm, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  return a.dim == 3 ? launch(k_sens<3>, a, num_sm, st) : launch(k_sens<2>, a, num_sm, st);
}

int tb_launch_adj_rhs_ragged(const TbAdjRaggedArgs& a, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  return a.dim == 3 ? launch_ragged(k_adj_rhs_ragged<3>, 0, a, st) : launch_ragged(k_adj_rhs_ragged<2>, 1, a, st);
}

int tb_launch_sens_ragged(const TbAdjRaggedArgs& a, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  return a.dim == 3 ? launch_ragged(k_sens_ragged<3>, 2, a, st) : launch_ragged(k_sens_ragged<2>, 3, a, st);
}
