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
      double dx[DIM], c[DIM], k, w;
      const double len = tb_member_geom<DIM>(xyz, j0, j1, aed[3 * m], aed[3 * m + 1], aed[3 * m + 2], dx, c, k, w);
      double nh = gax ? gax[m] : 0.0;
      if (gext)
#pragma unroll
        for (int i = 0; i < DIM; ++i) {
          const int d1 = j1 * DIM + i, d0 = j0 * DIM + i;
          const double z1 = a.dof2free[d1] < 0 ? gext[d1] : 0.0, z0 = a.dof2free[d0] < 0 ? gext[d0] : 0.0;
          nh = fma(c[i], z1 - z0, nh);
        }
      const bool ok = len > 0.0;                 // (a zero-length member fails its system: keep NaN out of the solve)
#pragma unroll
      for (int i = 0; i < DIM; ++i) vec[m * DIM + i] = ok ? nh * k * c[i] : 0.0;
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
      const double ar = aed[3 * m], e = aed[3 * m + 1], rho = aed[3 * m + 2];
      double dx[DIM], c[DIM], k, w;
      const double len = tb_member_geom<DIM>(xyz, j0, j1, ar, e, rho, dx, c, k, w);
      double du[DIM], dw[DIM], tu = 0.0, tz = 0.0, tl = 0.0;
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        const int d1 = j1 * DIM + i, d0 = j0 * DIM + i;
        const bool f1 = a.dof2free[d1] >= 0, f0 = a.dof2free[d0] >= 0;
        du[i] = (f1 ? u[d1] : 0.0) - (f0 ? u[d0] : 0.0);
        const double dl = (f1 ? lam[d1] : 0.0) - (f0 ? lam[d0] : 0.0);
        const double dz = gext ? (f1 ? 0.0 : gext[d1]) - (f0 ? 0.0 : gext[d0]) : 0.0;
        dw[i] = dz - dl;
        tu = fma(c[i], du[i], tu);
        tz = fma(c[i], dz, tz);
        tl = fma(c[i], dl, tl);
      }
      const double g = gax ? gax[m] : 0.0;
      const double q = g + tz - tl;              // N^ - c.d(lambda)
      const double tw = tz - tl;                 // c.dw, dw = dz - d(lambda)
      const double kl = k / len;
      ga[3 * m] = fma(e / len * tu, q, gw * len * rho);
      ga[3 * m + 1] = ar / len * tu * q;
      ga[3 * m + 2] = gw * ar * len;
      // d/dd of EA [g (d.du)/L^2 + (d.dw)(d.du)/L^3] + g_w a rho L, written with c = d/L
      const double war = gw * ar * rho;
#pragma unroll
      for (int i = 0; i < DIM; ++i)
        vec[m * DIM + i] = kl * (g * (du[i] - 2.0 * tu * c[i]) + dw[i] * tu + du[i] * tw - 3.0 * tu * tw * c[i]) + war * c[i];
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
