// Fused shared-memory path: one CTA per truss, everything between the inputs and the results
// stays on chip (HBM sees only the per-truss inputs and outputs).
//
//   stage                          replaces (slientruss3d)
//   DOF map (ballot scan)          Truss.GetDisplacementUnknownMask   truss.py:319-326, type.py:48-74
//   stability counting rule        Truss.isStable                     truss.py:154-164
//   member geometry                Member.length/k/cosines            truss.py:19,56-63
//   row-owner assembly of K_ff     Member.matK + Truss.GetKMatrix     truss.py:65-86,307-316  (+ mask slicing :343)
//   Cholesky + fwd/back solve      np.linalg.solve (LAPACK dgesv)     truss.py:343
//   axial forces                   internal-force loop                truss.py:353-361
//   reactions / ext                matK[~mask] @ vecD                 truss.py:347-351
//   weight, GA fitness             Truss.weight, GA.GetFitness        truss.py:166-168,429-462; ga.py:139-149
//
// Assembly is deterministic without atomics: thread r owns row r of K_ff and visits the members in
// ascending id, so every entry is summed in the reference's order (truss.py:310).  The right-hand
// side rides along as row n of the factorisation (L y = f falls out of the same column loop).
#include <math.h>
#include <stdlib.h>

#include "tb_common.cuh"

namespace {

constexpr int SMALL_MAX_THREADS = 192;

__device__ __forceinline__ double block_sum(double v, double* sRed, int tid, int nthreads) {
  // fixed-shape tree: shuffle-down inside each warp, then warp 0 adds the partials in order
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(full, v, o);
  const int lane = tid & 31, warp = tid >> 5, nw = (nthreads + 31) >> 5;
  __syncthreads();
  if (lane == 0) sRed[warp] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < nw; ++w) t += sRed[w];
  return t;
}

template <int DIM>
__global__ void __launch_bounds__(SMALL_MAX_THREADS) k_small(const SmallArgs a) {
  extern __shared__ __align__(16) double smem[];
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int NJmax = a.nJ, Mmax = a.M, Nmax = NJmax * DIM, nmax = a.max_n;
  const int ldmax = (nmax + 1) | 1;

  double* sK = smem;                         // (n+1) x n, column-major, odd leading dimension
  double* sXyz = sK + (size_t)ldmax * nmax;  // [N]
  double* sF = sXyz + Nmax;                  // [N]
  double* sU = sF + Nmax;                    // [N]
  double* sUf = sU + Nmax;                   // [n]
  double* sDinv = sUf + nmax;                // [n]   1 / L_kk
  double* sMk = sDinv + nmax;                // [M]   EA/L
  double* sMc = sMk + Mmax;                  // [M][d] cosines
  double* sAx = sMc + (size_t)Mmax * DIM;    // [M]   axial force
  double* sArea = sAx + Mmax;                // [M]
  double* sMw = sArea + Mmax;                // [M]   a*L*rho
  double* sRed = sMw + Mmax;                 // [8]
  int* sConn = (int*)(sRed + 8);             // [M][2]
  int* sD2F = sConn + 2 * Mmax;              // [N]
  int* sFree = sD2F + Nmax;                  // [N]
  int* sMeta = sFree + Nmax;                 // [0] n   [1] status
  uint8_t* sSup = (uint8_t*)(sMeta + 4);     // [nJ]

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    int nJ, M;
    int64_t jo, mo;
    const double *xyz, *aed, *force;
    const uint8_t* sup;
    const int32_t *conn, *gene = nullptr;
    if (a.joint_off) {
      jo = a.joint_off[b];
      nJ = (int)(a.joint_off[b + 1] - jo);
      mo = a.member_off[b];
      M = (int)(a.member_off[b + 1] - mo);
      xyz = a.xyz + jo * DIM;
      sup = a.support + jo;
      conn = a.conn + mo * 2;
      aed = a.aed + mo * 3;
      force = a.force + jo * DIM;
    } else {
      nJ = a.nJ;
      M = a.M;
      jo = (int64_t)b * nJ;
      mo = (int64_t)b * M;
      xyz = a.xyz + b * a.xyz_stride;
      sup = a.support + b * a.support_stride;
      conn = a.conn + b * a.conn_stride;
      aed = a.aed ? a.aed + b * a.aed_stride : nullptr;
      gene = a.gene ? a.gene + b * a.gene_stride : nullptr;
      force = a.force + b * a.force_stride;
    }
    const bool oversize = (nJ > NJmax) || (M > Mmax) || (nJ < 0) || (M < 0);
    if (oversize) { nJ = 0; M = 0; }
    const int N = nJ * DIM;

    // ---- stage the inputs (coalesced)
    for (int i = tid; i < N; i += T) {
      sXyz[i] = xyz[i];
      sF[i] = force[i];
    }
    for (int i = tid; i < nJ; i += T) sSup[i] = sup[i];
    for (int i = tid; i < 2 * M; i += T) sConn[i] = conn[i];
    if (tid == 0) {
      sMeta[0] = 0;
      sMeta[1] = oversize ? TB_INFO_BAD_INDEX : 0;
    }
    __syncthreads();

    // ---- DOF map: free DOFs numbered in ascending DOF order (warp 0, ballot scan)
    if (warp == 0) {
      int run = 0;
      for (int base = 0; base < N; base += 32) {
        const int dof = base + lane;
        bool fr = false;
        if (dof < N) {
          const int j = dof / DIM, ax = dof - j * DIM;
          const int s = sSup[j];
          if (tb_support_bad(DIM, s)) atomicMin(&sMeta[1], TB_INFO_BAD_SUPPORT);
          fr = tb_dof_free(s, ax);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, fr);
        const int pos = run + __popc(bal & ((1u << lane) - 1u));
        if (dof < N) {
          sD2F[dof] = fr ? pos : -1;
          if (fr) sFree[pos] = dof;
        }
        run += __popc(bal);
      }
      if (lane == 0) {
        sMeta[0] = run;
        const int nres = N - run;  // every restrained DOF is one resistance (type.py:37-46)
        const bool stable = (DIM == 2) ? (M + nres >= N) : (nres >= 6 && M + nres >= N);
        if (!stable) atomicMin(&sMeta[1], TB_INFO_NOT_STABLE);
      }
    }

    // ---- member geometry (no FMA contraction: keep the reference's roundings)
    for (int m = tid; m < M; m += T) {
      const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
      double ar = 0.0, e = 0.0, rho = 0.0;
      bool ok = ((unsigned)j0 < (unsigned)nJ) && ((unsigned)j1 < (unsigned)nJ);
      if (gene) {
        const int g = gene[m];
        if ((unsigned)g < (unsigned)a.n_type) {
          ar = a.type_table[3 * g];
          e = a.type_table[3 * g + 1];
          rho = a.type_table[3 * g + 2];
        } else {
          ok = false;
        }
      } else {
        ar = aed[3 * m];
        e = aed[3 * m + 1];
        rho = aed[3 * m + 2];
      }
      double k = 0.0, len = 0.0, c[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) c[i] = 0.0;
      if (!ok) {
        atomicMin(&sMeta[1], TB_INFO_BAD_INDEX);
      } else {
        double dx[DIM];
#pragma unroll
        for (int i = 0; i < DIM; ++i) dx[i] = __dsub_rn(sXyz[j1 * DIM + i], sXyz[j0 * DIM + i]);
        double l2 = __dmul_rn(dx[0], dx[0]);
#pragma unroll
        for (int i = 1; i < DIM; ++i) l2 = __dadd_rn(l2, __dmul_rn(dx[i], dx[i]));
        len = __dsqrt_rn(l2);
        if (!(len > 0.0)) {
          atomicMin(&sMeta[1], TB_INFO_ZERO_LENGTH);
        } else {
          const TbDivisor dv(len);                  // (one reciprocal for the four quotients of the member)
          k = dv.div(__dmul_rn(e, ar));
#pragma unroll
          for (int i = 0; i < DIM; ++i) c[i] = dv.div(dx[i]);
        }
      }
      sMk[m] = k;
#pragma unroll
      for (int i = 0; i < DIM; ++i) sMc[m * DIM + i] = c[i];
      sArea[m] = ar;
      sMw[m] = __dmul_rn(__dmul_rn(ar, len), rho);
      sAx[m] = 0.0;
    }
    __syncthreads();

    const int n = sMeta[0];
    int status = sMeta[1];
    const int ld = (n + 1) | 1;

    if (status == 0 && n > 0) {
      // ---- zero K, then row-owner assembly + the load row
      for (int i = tid; i < ld * n; i += T) sK[i] = 0.0;
      __syncthreads();
      if (tid < n) {
        const int r = tid;
        const int dof = sFree[r];
        const int jr = dof / DIM, ar = dof - jr * DIM;
        double* Krow = sK + r;
        for (int m = 0; m < M; ++m) {
          const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
          if (j0 != jr && j1 != jr) continue;
          const double k = sMk[m];
          const double ca = sMc[m * DIM + ar];
#pragma unroll
          for (int A = 0; A < 2; ++A) {
            if ((A ? j1 : j0) != jr) continue;
#pragma unroll
            for (int B = 0; B < 2; ++B) {
              const int jb = B ? j1 : j0;
#pragma unroll
              for (int j = 0; j < DIM; ++j) {
                const int fc = sD2F[jb * DIM + j];
                if (fc >= 0 && fc <= r) {
                  double p = __dmul_rn(ca, sMc[m * DIM + j]);
                  if (A != B) p = -p;
                  Krow[fc * ld] = __dadd_rn(Krow[fc * ld], __dmul_rn(k, p));
                }
              }
            }
          }
        }
      }
      for (int c = tid; c < n; c += T) sK[n + c * ld] = sF[sFree[c]];
      __syncthreads();

      // ---- left-looking Cholesky, one thread per row (row n = right-hand side).  Every thread
      // also accumulates the pivot itself, so one barrier per column is enough.
      int fail = 0;
      for (int k = 0; k < n; ++k) {
        const bool act = (tid >= k) && (tid <= n);
        const double* rowk = sK + k;
        const double* rowi = sK + (act ? tid : k);
        double d0 = rowk[k * ld], d1 = 0.0;
        double s0 = rowi[k * ld], s1 = 0.0;
        int p = 0;
        for (; p + 1 < k; p += 2) {
          const double b0 = rowk[p * ld], b1 = rowk[(p + 1) * ld];
          const double a0 = rowi[p * ld], a1 = rowi[(p + 1) * ld];
          d0 = fma(-b0, b0, d0);
          d1 = fma(-b1, b1, d1);
          s0 = fma(-a0, b0, s0);
          s1 = fma(-a1, b1, s1);
        }
        if (p < k) {
          const double b0 = rowk[p * ld];
          d0 = fma(-b0, b0, d0);
          s0 = fma(-rowi[p * ld], b0, s0);
        }
        const double d = d0 + d1, s = s0 + s1;
        if (!(d > 0.0)) {  // also catches NaN; identical in every thread, so the exit is uniform
          fail = k + 1;
          break;
        }
        const double lkk = sqrt(d);
        const double rinv = 1.0 / lkk;
        // K[k][k] itself is left untouched: slower warps may still be reading it as their pivot seed
        if (act && tid != k) sK[tid + k * ld] = s * rinv;
        if (tid == k) sDinv[k] = rinv;
        __syncthreads();
      }
      status = fail;

      if (status == 0) {
        // ---- back substitution L^T u = y, column oriented: thread p keeps y_p in a register
        double yp = (tid < n) ? sK[n + tid * ld] : 0.0;
        for (int k = n - 1; k >= 0; --k) {
          if (tid == k) sUf[k] = yp * sDinv[k];
          __syncthreads();
          if (tid < k) yp = fma(-sK[k + tid * ld], sUf[k], yp);
        }
        __syncthreads();
      }
    }

    // output locations
    double* u_out = a.u ? a.u + jo * DIM : nullptr;
    double* ext_out = a.ext ? a.ext + jo * DIM : nullptr;
    double* ax_out = a.axial ? a.axial + mo : nullptr;

    if (status != 0) {  // uniform: zero-filled outputs, never NaN
      for (int i = tid; i < N; i += T) {
        if (u_out) u_out[i] = 0.0;
        if (ext_out) ext_out[i] = 0.0;
      }
      for (int m = tid; m < M; m += T)
        if (ax_out) ax_out[m] = 0.0;
      if (tid == 0) {
        if (a.weight) a.weight[b] = 0.0;
        if (a.info) a.info[b] = status;
        if (a.fitness_mode) {
          if (a.fitness) a.fitness[b] = INFINITY;
          if (a.flags) { a.flags[2 * b] = 0; a.flags[2 * b + 1] = 0; }
        }
      }
      __syncthreads();
      continue;
    }

    // ---- expand to all DOFs (0 at supports), axial forces, reactions
    for (int i = tid; i < N; i += T) {
      const int fr = sD2F[i];
      const double v = fr >= 0 ? sUf[fr] : 0.0;
      sU[i] = v;
      if (u_out) u_out[i] = v;
    }
    __syncthreads();
    for (int m = tid; m < M; m += T) {
      const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < DIM; ++i) t = fma(sMc[m * DIM + i], sU[j1 * DIM + i] - sU[j0 * DIM + i], t);
      const double nm = sMk[m] * t;
      sAx[m] = nm;
      if (ax_out) ax_out[m] = nm;
    }
    __syncthreads();
    if (ext_out) {
      for (int dof = tid; dof < N; dof += T) {
        double e;
        if (sD2F[dof] >= 0) {
          e = sF[dof];
        } else {  // row of K times u, summed member by member in ascending id
          const int J = dof / DIM, ax = dof - J * DIM;
          e = 0.0;
          for (int m = 0; m < M; ++m) {
            const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
            if (j0 == J) e = fma(-sMc[m * DIM + ax], sAx[m], e);
            if (j1 == J) e = fma(sMc[m * DIM + ax], sAx[m], e);
          }
        }
        ext_out[dof] = e;
      }
    }

    // ---- weight (+ GA fitness)
    double w = 0.0;
    for (int m = tid; m < M; m += T) w += sMw[m];
    w = block_sum(w, sRed, tid, T);
    if (tid == 0) {
      if (a.weight) a.weight[b] = w;
      if (a.info) a.info[b] = 0;
    }
    if (a.fitness_mode) {
      double vs = 0.0, vd = 0.0;
      for (int m = tid; m < M; m += T) {  // truss.py:429-433
        const double f = fabs(sAx[m]);
        if (!(f < TB_ZERO_EPS)) {
          const double sg = f / sArea[m];
          if (sg > a.allow_stress) vs += sg - a.allow_stress;
        }
      }
      for (int j = tid; j < nJ; j += T) {  // truss.py:447-451
        bool any = false;
        double l2 = 0.0;
#pragma unroll
        for (int i = 0; i < DIM; ++i) {
          const double v = sU[j * DIM + i];
          any |= !(fabs(v) < TB_ZERO_EPS);
          l2 += v * v;
        }
        if (any) {
          const double l = sqrt(l2);
          if (l > a.allow_displace) vd += l - a.allow_displace;
        }
      }
      vs = block_sum(vs, sRed, tid, T);
      vd = block_sum(vd, sRed, tid, T);
      if (tid == 0) {
        const bool ok_s = fabs(vs) < TB_ZERO_EPS, ok_d = fabs(vd) < TB_ZERO_EPS;
        double fit = w;  // ga.py:146-148
        if (!ok_s) fit += vs / a.allow_stress * 1e5;
        if (!ok_d) fit += vd / a.allow_displace * 1e5;
        if (a.fitness) a.fitness[b] = fit;
        if (a.flags) { a.flags[2 * b] = ok_s; a.flags[2 * b + 1] = ok_d; }
      }
    }
    __syncthreads();  // shared arrays are reused by the next system
  }
}

}  // namespace

int tb_small_smem_bytes(int dim, int nJ, int M, int max_n, int* threads) {
  const int N = nJ * dim;
  const int ldmax = (max_n + 1) | 1;
  size_t dbl = (size_t)ldmax * max_n + 3 * (size_t)N + 2 * (size_t)max_n + (size_t)M * (5 + dim) + 8;
  size_t bytes = dbl * 8 + (2 * (size_t)M + 2 * (size_t)N + 4) * 4 + (size_t)nJ + 16;
  if (threads) {
    int t = ((max_n + 1) + 31) / 32 * 32;
    if (t < 32) t = 32;
    *threads = t;
  }
  return (int)bytes;
}

bool tb_small_fits(int dim, int nJ, int M, int max_n) {
  if (nJ * dim > TB_SMALL_MAX_DOF || M > TB_SMALL_MAX_MEMBER || nJ > TB_SMALL_MAX_JOINT) return false;
  const int nbm = max_n > 0 ? (max_n + 15) / 16 : 1;
  if (nbm <= 10 && tb_dense16_smem_bytes(dim, nJ, M, max_n) <= 110 * 1024) return true;      // k_dense16: one warp per truss
  int threads = 0;
  const int smem = tb_small_smem_bytes(dim, nJ, M, max_n, &threads);                         // k_small: one CTA per truss
  return threads <= SMALL_MAX_THREADS && smem <= 227 * 1024;
}

int tb_launch_small(const SmallArgs& a, int dim, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  // warp-per-system kernel (tb_dense16.cu) first; this CTA-per-truss kernel takes what does not fit its budget
  static const bool legacy = [] { const char* s = getenv("TB_SMALL_LEGACY"); return s && s[0] == '1'; }();
  if (!legacy) {
    const int rc = tb_launch_dense16(a, dim, st);
    if (rc != -1) return rc;
  }
  int threads = 0;
  const int smem = tb_small_smem_bytes(dim, a.nJ, a.M, a.max_n, &threads);
  if (threads > SMALL_MAX_THREADS || smem > 227 * 1024) return TB_ERR_TOO_LARGE;
  auto kern = (dim == 3) ? k_small<3> : k_small<2>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  int per_sm = 0, dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem);
  if (e != cudaSuccess) return (int)e;
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)sms * per_sm;   // persistent: a multiple of the SM count
  if (grid > a.batch) grid = a.batch;
  tb_prof_begin(TB_PROF_SMALL, st);
  kern<<<(unsigned)grid, threads, smem, st>>>(a);
  tb_prof_end(TB_PROF_SMALL, st);
  tb_count_launch();
  return (int)cudaGetLastError();
}
