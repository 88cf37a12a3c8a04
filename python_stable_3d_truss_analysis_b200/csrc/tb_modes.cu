// Batched modal analysis (tb_modes, DESIGN.md section 11): the n_modes lowest eigenpairs of K_ff phi = lambda M_ff phi for
// every system of a uniform batch, n <= TB_SMALL_MAX_DOF free DOFs.
//
// k_modes<DIM> runs one CTA per system in a persistent grid-stride loop, with the whole reduced matrix in dynamic shared
// memory (n x P doubles, P = n | 1: an odd row pitch keeps row-strided and column-strided accesses free of bank
// conflicts).  Per system:
//   1. status guards of the static solve (counting rule, gene index, zero length), then K_ff assembled densely through the
//      plan's scatter map (the same products and ascending-member sums as every other path: bit-identical to
//      GetKMatrix()[mask][:, mask]) and the mass: lumped per free DOF in shared memory, consistent into the CTA's slot of
//      the plan's modal scratch (global memory, L2-resident).
//   2. standard problem: K~ = M^-1/2 K M^-1/2 (lumped) or K~ = L^-1 K L^-T with M = L L^T (consistent, both triangular
//      solves column-parallel in shared memory).
//   3. Householder tridiagonalisation, tred2 style, with Q accumulated in place.
//   4. implicit QL with shifts, tql2 style: thread 0 runs a sweep's scalar recurrence and records its rotations, then every
//      thread applies them to its own row of Z (three barriers per sweep).  tql2 keeps the vectors of a cluster of equal
//      eigenvalues orthogonal with no extra work (bar-72 and bar-120 have exactly repeated frequencies).
//   5. ascending ranks, back-transform of the requested vectors (M^-1/2 z or L^-T z), sign convention, outputs.
// Every sum runs serially in one thread in a fixed order and no value depends on which thread computes it, so a system's
// bits do not depend on its position in the batch, the batch size, the CTA size or the number of resident CTAs.
//
// Steps 2-5 are __device__ functions (modes_eigen, modes_order) shared with k_modes_ragged<DIM> (tb_modes_ragged), which
// differs in step 1 and in where it writes, and with k_buckling<DIM> (tb_buckling, linear buckling: K_ff phi =
// lambda (-K_G) phi), which differs in step 1 and in its output step; see there.
//
// k_modes_sens<DIM> is the reverse mode (tb_modes_adjoint): eigenvalue gradients from the forward's modes, below, and
// k_modes_sens_ragged<DIM> its ragged form (tb_modes_adjoint_ragged); k_buckling_sens<DIM> is the reverse mode of
// tb_buckling (tb_buckling_adjoint): load-factor gradients from the forward's modes, in the same shape.
#include <cfloat>
#include <math_constants.h>

#include "tb_common.cuh"

namespace {

constexpr int TQL_MAX_ITER = 30;   // QL sweeps per eigenvalue (EISPACK tql2's cap)

struct ModesCtl {
  double h;
  int any, lo, status;
  int piv;   // position (free-DOF row) of the pivot where the Cholesky of the slot stopped
};

// (a, e, density) of member m from the explicit rows or the gene / type table; ok = false for a gene out of range
__device__ __forceinline__ void member_props(const ModesArgs& a, const double* aed, const int32_t* gene, int m, double& ar,
                                             double& e, double& rho, bool& ok) {
  const double* t;
  if (gene) {
    const int g = gene[m];
    ok = (unsigned)g < (unsigned)a.n_type;
    t = a.type_table + 3 * (ok ? g : 0);
  } else {
    ok = true;
    t = aed + 3 * m;
  }
  ar = t[0];
  e = t[1];
  rho = t[2];
}

// EA/L, direction cosines and weight term (a L) density of member m, the reference's roundings (tb_member_geom)
template <int DIM>
__device__ __forceinline__ double member_kcw(const ModesArgs& a, const double* xyz, const double* aed, const int32_t* gene,
                                             int m, double& k, double c[DIM], double& w) {
  double ar, e, rho, dx[DIM];
  bool ok;
  member_props(a, aed, gene, m, ar, e, rho, ok);
  return tb_member_geom<DIM>(xyz, a.conn[2 * m], a.conn[2 * m + 1], ar, e, rho, dx, c, k, w);
}

__host__ __device__ inline size_t modes_smem_bytes(int n) {
  const int P = n | 1;
  return ((size_t)n * P + 8 * (size_t)n) * sizeof(double) + 2 * (size_t)n * sizeof(int);
}

// The per-system arrays of steps 2-5 in dynamic shared memory, for n free DOFs
struct ModesSmem {
  double* Z;     // [n][P] K_ff -> K~ -> Householder data -> Q -> eigenvectors of K~ (columns)
  double* dv;    // diagonal, then eigenvalues
  double* ev;    // sub-diagonal
  double* pv;    // tred2 scratch p = A u / H
  double* qv;    // tred2 scratch q = p - K u
  double* sc;    // lumped: M^-1/2 per free DOF
  double* rc;    // rotations of one QL sweep
  double* rs;
  double* sg;    // sign of each requested mode
  int* perm;     // ascending rank -> column of Z
};

__device__ __forceinline__ ModesSmem modes_smem(double* base, int n, int* perm) {
  ModesSmem s;
  s.Z = base;
  s.dv = s.Z + (size_t)n * (n | 1);
  s.ev = s.dv + n;
  s.pv = s.ev + n;
  s.qv = s.pv + n;
  s.sc = s.qv + n;
  s.rc = s.sc + n;
  s.rs = s.rc + n;
  s.sg = s.rs + n;
  s.perm = perm;
  return s;
}

// Steps 2-4 of one system (n >= 1): standard problem, tred2, tql2.  Entered with K_ff in Z (both triangles) and the mass
// (lumped: s.sc; consistent: M_ff in L, row pitch n); returns the status (TB_INFO_MASS, TB_INFO_NO_CONVERGENCE or 0)
// with the eigenvalues in s.dv and the eigenvectors of K~ in the columns of Z.  Shared by k_modes, k_modes_ragged and
// k_buckling (which enters with K_G in Z and K_ff in L).  TB_INFO_MASS means the Cholesky of L met a pivot that is not
// > 0, at row ctl.piv.
__device__ __forceinline__ int modes_eigen(const ModesSmem& s, int n, int consistent, double* L, ModesCtl& ctl,
                                           int status) {
  const int P = n | 1;
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nth >> 5;
  double* Z = s.Z;
  double* dv = s.dv;
  double* ev = s.ev;
  double* pv = s.pv;
  double* qv = s.qv;
  double* sc = s.sc;
  double* rc = s.rc;
  double* rs = s.rs;
  // ---- standard problem
  if (status == 0 && !consistent) {
    for (int r = wid; r < n; r += nw)
      for (int c = lane; c <= r; c += 32) Z[r * P + c] = (Z[r * P + c] * sc[r]) * sc[c];
  } else if (status == 0) {
    // Cholesky M = L L^T in the slot, left-looking: pivot by thread 0, then the column below it in parallel
    for (int j = 0; j < n; ++j) {
      double* Lj = L + (size_t)j * n;
      if (tid == 0) {
        double x = Lj[j];
        for (int k = 0; k < j; ++k) x -= Lj[k] * Lj[k];
        ctl.status = x > 0.0 ? 0 : TB_INFO_MASS;
        if (!(x > 0.0)) ctl.piv = j;
        Lj[j] = x > 0.0 ? sqrt(x) : 0.0;
      }
      __syncthreads();
      if (ctl.status) break;
      const double djj = Lj[j];
      for (int i = j + 1 + tid; i < n; i += nth) {
        double* Li = L + (size_t)i * n;
        double x = Li[j];
        for (int k = 0; k < j; ++k) x -= Li[k] * Lj[k];
        Li[j] = x / djj;
      }
      __syncthreads();
    }
    status = ctl.status;
    __syncthreads();
    if (status == 0) {
      // K~ = L^-1 (L^-1 K)^T: two column-parallel forward substitutions around an in-place transpose
      for (int pass = 0; pass < 2; ++pass) {
        for (int j = tid; j < n; j += nth)
          for (int i = 0; i < n; ++i) {
            const double* Li = L + (size_t)i * n;
            double x = Z[i * P + j];
            for (int k = 0; k < i; ++k) x -= Li[k] * Z[k * P + j];
            Z[i * P + j] = x / Li[i];
          }
        __syncthreads();
        if (pass == 0) {
          for (int r = wid; r < n; r += nw)
            for (int c = lane; c < r; c += 32) {
              const double t = Z[r * P + c];
              Z[r * P + c] = Z[c * P + r];
              Z[c * P + r] = t;
            }
          __syncthreads();
        }
      }
    }
  }

  if (status == 0) {
    // ---- Householder tridiagonalisation (tred2), lower triangle of Z
    for (int i = n - 1; i > 0; --i) {
      const int l = i - 1;
      double* zi = Z + (size_t)i * P;
      __syncthreads();
      if (tid == 0) {
        double h = 0.0, scale = 0.0;
        int any = 0;
        if (l > 0) {
          for (int k = 0; k < i; ++k) scale += fabs(zi[k]);
          if (scale == 0.0) {
            ev[i] = zi[l];
          } else {
            for (int k = 0; k < i; ++k) {
              zi[k] /= scale;
              h += zi[k] * zi[k];
            }
            const double f = zi[l];
            const double g = f >= 0.0 ? -sqrt(h) : sqrt(h);
            ev[i] = scale * g;
            h -= f * g;
            zi[l] = f - g;
            any = 1;
          }
        } else {
          ev[i] = zi[l];
        }
        dv[i] = h;
        ctl.h = h;
        ctl.any = any;
      }
      __syncthreads();
      if (!ctl.any) continue;
      const double h = ctl.h;
      for (int j = tid; j < i; j += nth) {   // p = A u / H, u / H stored in column i
        const double* zj = Z + (size_t)j * P;
        Z[j * P + i] = zi[j] / h;
        double g = 0.0;
        for (int k = 0; k <= j; ++k) g += zj[k] * zi[k];
        for (int k = j + 1; k < i; ++k) g += Z[k * P + j] * zi[k];
        pv[j] = g / h;
      }
      __syncthreads();
      double f = 0.0;                        // (every thread, same order)
      for (int j = 0; j < i; ++j) f += pv[j] * zi[j];
      const double hh = f / (h + h);
      for (int j = tid; j < i; j += nth) qv[j] = pv[j] - hh * zi[j];
      __syncthreads();
      for (int j = wid; j < i; j += nw) {    // rank-2 update A -= u q^T + q u^T, a warp per row
        const double fj = zi[j], gj = qv[j];
        double* zj = Z + (size_t)j * P;
        for (int k = lane; k <= j; k += 32) zj[k] -= (fj * qv[k] + gj * zi[k]);
      }
    }
    __syncthreads();
    if (tid == 0) {
      dv[0] = 0.0;
      ev[0] = 0.0;
    }
    for (int i = 0; i < n; ++i) {           // accumulate Q in place, a thread per column
      __syncthreads();
      const bool acc = dv[i] != 0.0;
      if (acc)
        for (int j = tid; j < i; j += nth) {
          double g = 0.0;
          for (int k = 0; k < i; ++k) g += Z[i * P + k] * Z[k * P + j];
          for (int k = 0; k < i; ++k) Z[k * P + j] -= g * Z[k * P + i];
        }
      __syncthreads();
      if (tid == 0) {
        dv[i] = Z[i * P + i];
        Z[i * P + i] = 1.0;
      }
      for (int j = tid; j < i; j += nth) Z[j * P + i] = Z[i * P + j] = 0.0;
    }
    __syncthreads();

    // ---- implicit QL with shifts (tql2)
    if (tid == 0) {
      for (int i = 1; i < n; ++i) ev[i - 1] = ev[i];
      ev[n - 1] = 0.0;
    }
    int fail = 0;
    for (int l = 0; l < n && !fail; ++l) {
      int iter = 0;
      for (;;) {
        __syncthreads();
        int m;
        for (m = l; m < n - 1; ++m) {
          const double dd = fabs(dv[m]) + fabs(dv[m + 1]);
          if (fabs(ev[m]) <= DBL_EPSILON * dd) break;
        }
        if (m == l) break;
        if (iter++ == TQL_MAX_ITER) {
          fail = 1;
          break;
        }
        __syncthreads();                     // every thread has read d and e
        if (tid == 0) {
          double g = (dv[l + 1] - dv[l]) / (2.0 * ev[l]);
          double r = hypot(g, 1.0);
          g = dv[m] - dv[l] + ev[l] / (g + copysign(r, g));
          double s = 1.0, c = 1.0, p = 0.0;
          int i;
          bool brk = false;
          for (i = m - 1; i >= l; --i) {
            const double f = s * ev[i], bb = c * ev[i];
            r = hypot(f, g);
            ev[i + 1] = r;
            if (r == 0.0) {
              dv[i + 1] -= p;
              ev[m] = 0.0;
              brk = true;
              break;
            }
            s = f / r;
            c = g / r;
            g = dv[i + 1] - p;
            r = (dv[i] - g) * s + 2.0 * c * bb;
            p = s * r;
            dv[i + 1] = g + p;
            g = c * r - bb;
            rc[i] = c;
            rs[i] = s;
          }
          ctl.lo = brk ? i + 1 : l;
          if (!brk) {
            dv[l] -= p;
            ev[l] = g;
            ev[m] = 0.0;
          }
        }
        __syncthreads();
        if (tid < n) {                       // thread k applies the sweep's rotations to row k of Z
          double* zk = Z + (size_t)tid * P;
          for (int i = m - 1; i >= ctl.lo; --i) {
            const double c = rc[i], s = rs[i], f = zk[i + 1];
            zk[i + 1] = s * zk[i] + c * f;
            zk[i] = c * zk[i] - s * f;
          }
        }
      }
    }
    if (fail) status = TB_INFO_NO_CONVERGENCE;
    __syncthreads();
  }
  return status;
}

// Step 5a of one system: ascending ranks (ties: lower column first), back-transform and sign convention of the nq lowest
// modes, their eigenvalues into erow[0, nq).  Shared by k_modes and k_modes_ragged.
__device__ __forceinline__ void modes_order(const ModesSmem& s, int n, int nq, int consistent, const double* L,
                                            double* erow) {
  const int P = n | 1;
  const int tid = threadIdx.x, nth = blockDim.x;
  double* Z = s.Z;
  const double* dv = s.dv;
  const double* sc = s.sc;
  double* sg = s.sg;
  int* perm = s.perm;
  for (int i = tid; i < n; i += nth) {
    const double di = dv[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += (dv[j] < di || (dv[j] == di && j < i)) ? 1 : 0;
    perm[rank] = i;
  }
  __syncthreads();
  for (int q = tid; q < nq; q += nth) {
    const int col = perm[q];
    if (!consistent) {
      for (int r = 0; r < n; ++r) Z[r * P + col] *= sc[r];
    } else {
      for (int r = n - 1; r >= 0; --r) {  // L^T y = z
        double x = Z[r * P + col];
        for (int k = r + 1; k < n; ++k) x -= L[(size_t)k * n + r] * Z[k * P + col];
        Z[r * P + col] = x / L[(size_t)r * n + r];
      }
    }
    double best = 0.0;
    int bi = 0;
    for (int r = 0; r < n; ++r) {
      const double v = fabs(Z[r * P + col]);
      if (v > best) {
        best = v;
        bi = r;
      }
    }
    sg[q] = Z[bi * P + col] < 0.0 ? -1.0 : 1.0;
    erow[q] = dv[col];
  }
  __syncthreads();
}

template <int DIM>
__global__ void __launch_bounds__(160) k_modes(const ModesArgs a) {
  extern __shared__ __align__(16) double smem[];
  __shared__ ModesCtl ctl;
  const int n = a.n, P = n | 1, N = a.N, nm = a.n_modes;
  const int tid = threadIdx.x, nth = blockDim.x;
  int* i2r = (int*)(smem + (size_t)n * P + 8 * (size_t)n);   // internal row of the plan's scatter map -> free DOF in the reference's order
  const ModesSmem s = modes_smem(smem, n, i2r + n);
  double* Z = s.Z;
  double* sc = s.sc;
  for (int r = tid; r < n; r += nth) i2r[a.dof2free[a.free_ref[r]]] = r;
  double* L = a.slot ? a.slot + (size_t)blockIdx.x * n * n : nullptr;   // consistent mass: M_ff, then its Cholesky factor

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed ? a.aed + b * a.aed_stride : nullptr;
    const int32_t* gene = a.aed ? nullptr : a.gene + b * a.gene_stride;
    const double* jm = a.jmass ? a.jmass + b * a.jmass_stride : nullptr;
    __syncthreads();                           // the previous system's shared data is consumed (and i2r is complete)

    // ---- status guards of the static solve, in its order of precedence
    int bad = 0;
    for (int m = tid; m < a.M; m += nth) {
      double ar, e, rho;
      bool ok;
      member_props(a, aed, gene, m, ar, e, rho, ok);
      if (!ok) {
        bad |= 1;
      } else {
        double k, c[DIM], w;
        if (!(member_kcw<DIM>(a, xyz, aed, gene, m, k, c, w) > 0.0)) bad |= 2;
      }
    }
    const int anyidx = __syncthreads_or(bad & 1), anylen = __syncthreads_or(bad & 2);
    int status = a.plan_stable ? 0 : TB_INFO_NOT_STABLE;
    if (anyidx) status = min(status, TB_INFO_BAD_INDEX);
    else if (anylen) status = min(status, TB_INFO_ZERO_LENGTH);

    if (status == 0) {
      // ---- K_ff (and consistent M_ff) densely, both triangles
      for (int i = tid; i < n * P; i += nth) Z[i] = 0.0;
      if (a.consistent)
        for (int i = tid; i < n * n; i += nth) L[i] = 0.0;
      __syncthreads();
      for (int64_t e = tid; e < a.nnz; e += nth) {
        const int r = i2r[a.ent_row[e]], c = i2r[a.ent_col[e]];
        double kv = 0.0, mv = 0.0;
        for (int64_t q = a.ent_ptr[e]; q < a.ent_ptr[e + 1]; ++q) {
          const int m = a.ctr_member[q], loc = a.ctr_local[q];
          const int la = loc / (2 * DIM), lb = loc - la * (2 * DIM);
          const int A = la / DIM, i = la - A * DIM, B = lb / DIM, j = lb - B * DIM;
          double k, cs[DIM], w;
          member_kcw<DIM>(a, xyz, aed, gene, m, k, cs, w);
          double pr = __dmul_rn(cs[i], cs[j]);   // truss.py:69,80
          if (A != B) pr = -pr;
          kv = __dadd_rn(kv, __dmul_rn(k, pr));  // truss.py:70,314
          if (a.consistent && i == j) {          // (m_e / 6) [[2, 1], [1, 2]] per axis
            const double me6 = __ddiv_rn(w, 6.0);
            mv = __dadd_rn(mv, A == B ? __dmul_rn(2.0, me6) : me6);
          }
        }
        Z[r * P + c] = kv;
        Z[c * P + r] = kv;
        if (a.consistent) {
          L[r * n + c] = mv;
          L[c * n + r] = mv;
        }
      }
      int badm = 0;
      if (!a.consistent) {                     // lumped: m_e / 2 per end joint and axis, ascending member, + joint mass
        for (int r = tid; r < n; r += nth) {
          const int J = a.free_ref[r] / DIM;
          double ms = 0.0;
          for (int q = a.inc_ptr[J]; q < a.inc_ptr[J + 1]; ++q) {
            double k, cs[DIM], w;
            member_kcw<DIM>(a, xyz, aed, gene, a.inc_mem[q] >> 1, k, cs, w);
            ms = __dadd_rn(ms, __dmul_rn(w, 0.5));
          }
          if (jm) ms = __dadd_rn(ms, jm[J]);
          if (!(ms > 0.0)) badm = 1;
          sc[r] = ms > 0.0 ? 1.0 / sqrt(ms) : 0.0;
        }
      }
      __syncthreads();
      if (a.consistent && jm)
        for (int r = tid; r < n; r += nth) L[r * n + r] = __dadd_rn(L[r * n + r], jm[a.free_ref[r] / DIM]);
      if (__syncthreads_or(badm)) status = TB_INFO_MASS;
    }

    status = modes_eigen(s, n, a.consistent, L, ctl, status);

    if (status == 0) {
      modes_order(s, n, nm, a.consistent, L, a.eigval + (int64_t)b * nm);
      if (a.modes) {
        double* mo = a.modes + (int64_t)b * nm * N;
        for (int64_t i = tid; i < (int64_t)nm * N; i += nth) mo[i] = 0.0;
        __syncthreads();
        for (int idx = tid; idx < nm * n; idx += nth) {
          const int q = idx / n, r = idx - q * n;
          mo[(int64_t)q * N + a.free_ref[r]] = s.sg[q] * Z[r * P + s.perm[q]];
        }
      }
    } else {                                   // failed system: zero outputs, never NaN
      for (int q = tid; q < nm; q += nth) a.eigval[(int64_t)b * nm + q] = 0.0;
      if (a.modes) {
        double* mo = a.modes + (int64_t)b * nm * N;
        for (int64_t i = tid; i < (int64_t)nm * N; i += nth) mo[i] = 0.0;
      }
    }
    if (tid == 0) a.info[b] = status;
  }
}

// ---- linear buckling (tb_buckling): K_ff phi = lambda (-K_G) phi for a given member-force state N
// k_buckling<DIM> is k_modes with its own step 1 and output step.  Step 1: the static solve's guards, then one pass over
// the plan's scatter map assembles K_ff into the CTA's slot and the geometric stiffness K_G into Z, both triangles, both
// in ascending member order.  Member m contributes to K_G, per block (A, B) and local (i, j),
//   +-g (delta_ij - c_i c_j),  g = N_m / L_m (correctly rounded), + on the diagonal blocks, c_i c_j rounded as K's product
// (the transverse "I - c c^T" form of the truss geometric stiffness).  Steps 2-5 are modes_eigen / modes_order with K_ff
// as the "mass": nu = eig(L^-1 K_G L^-T), K_ff = L L^T, ascending, modes back-transformed by L^T y = z (so K-normalised).
// Output step: mode q is critical when nu_q < -BUCKLING_TAU max_k |nu_k|; its load factor is -1 / nu_q (ascending with
// q), any other mode gets +inf and a zero row.  A pivot of K_ff that is not > 0 at free-DOF row j gives info j + 1.
// Registers: (160, 4) lets ptxas allocate 85 registers with no spills; with (160) alone it holds the kernel at 72-96
// registers and spills 80-120 bytes.  85 registers and k_modes' shared memory give at least k_modes' residency at every n.
constexpr double BUCKLING_TAU = 1e-12;   // relative threshold below which -nu counts as a critical eigenvalue

template <int DIM>
__global__ void __launch_bounds__(160, 4) k_buckling(const BucklingArgs ba) {
  extern __shared__ __align__(16) double smem[];
  __shared__ ModesCtl ctl;
  const ModesArgs& a = ba.base;
  const int n = a.n, P = n | 1, N = a.N, nm = a.n_modes;
  const int tid = threadIdx.x, nth = blockDim.x;
  int* i2r = (int*)(smem + (size_t)n * P + 8 * (size_t)n);   // internal row of the plan's scatter map -> free DOF in the reference's order
  const ModesSmem s = modes_smem(smem, n, i2r + n);
  double* Z = s.Z;
  for (int r = tid; r < n; r += nth) i2r[a.dof2free[a.free_ref[r]]] = r;
  double* L = a.slot + (size_t)blockIdx.x * n * n;           // K_ff, then its Cholesky factor

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed ? a.aed + b * a.aed_stride : nullptr;
    const int32_t* gene = a.aed ? nullptr : a.gene + b * a.gene_stride;
    __syncthreads();                           // the previous system's shared data is consumed (and i2r is complete)

    // ---- status guards of the static solve, in its order of precedence
    int bad = 0;
    for (int m = tid; m < a.M; m += nth) {
      double ar, e, rho;
      bool ok;
      member_props(a, aed, gene, m, ar, e, rho, ok);
      if (!ok) {
        bad |= 1;
      } else {
        double k, c[DIM], w;
        if (!(member_kcw<DIM>(a, xyz, aed, gene, m, k, c, w) > 0.0)) bad |= 2;
      }
    }
    const int anyidx = __syncthreads_or(bad & 1), anylen = __syncthreads_or(bad & 2);
    int status = a.plan_stable ? 0 : TB_INFO_NOT_STABLE;
    if (anyidx) status = min(status, TB_INFO_BAD_INDEX);
    else if (anylen) status = min(status, TB_INFO_ZERO_LENGTH);

    if (status == 0) {
      // ---- K_ff into the slot, K_G into Z, densely, both triangles, one pass over the scatter map
      const double* ax = ba.axial + b * ba.axial_stride;
      for (int i = tid; i < n * P; i += nth) Z[i] = 0.0;
      for (int i = tid; i < n * n; i += nth) L[i] = 0.0;
      __syncthreads();
      for (int64_t e = tid; e < a.nnz; e += nth) {
        const int r = i2r[a.ent_row[e]], c = i2r[a.ent_col[e]];
        double kv = 0.0, gv = 0.0;
        for (int64_t q = a.ent_ptr[e]; q < a.ent_ptr[e + 1]; ++q) {
          const int m = a.ctr_member[q], loc = a.ctr_local[q];
          const int la = loc / (2 * DIM), lb = loc - la * (2 * DIM);
          const int A = la / DIM, i = la - A * DIM, B = lb / DIM, j = lb - B * DIM;
          double k, cs[DIM], w;
          const double len = member_kcw<DIM>(a, xyz, aed, gene, m, k, cs, w);
          const double g = __ddiv_rn(ax[m], len);
          double pr = __dmul_rn(cs[i], cs[j]);   // truss.py:69,80
          double t = i == j ? __dsub_rn(1.0, pr) : -pr;
          if (A != B) {
            pr = -pr;
            t = -t;
          }
          kv = __dadd_rn(kv, __dmul_rn(k, pr));  // truss.py:70,314
          gv = __dadd_rn(gv, __dmul_rn(g, t));
        }
        Z[r * P + c] = gv;
        Z[c * P + r] = gv;
        L[r * n + c] = kv;
        L[c * n + r] = kv;
      }
      __syncthreads();
    }

    status = modes_eigen(s, n, 1, L, ctl, status);
    if (status == TB_INFO_MASS) status = ctl.piv + 1;   // K_ff is not positive definite: the static solve's info

    double* frow = a.eigval + (int64_t)b * nm;
    double* mo = a.modes ? a.modes + (int64_t)b * nm * N : nullptr;
    if (status == 0) {
      modes_order(s, n, nm, 1, L, frow);
      double vmax = 0.0;                       // (every thread, same value)
      for (int j = 0; j < n; ++j) vmax = fmax(vmax, fabs(s.dv[j]));
      const double thr = -BUCKLING_TAU * vmax;
      for (int q = tid; q < nm; q += nth) {
        const double nu = s.dv[s.perm[q]];
        frow[q] = nu < thr ? -1.0 / nu : CUDART_INF;
      }
      if (mo) {
        for (int64_t i = tid; i < (int64_t)nm * N; i += nth) mo[i] = 0.0;
        __syncthreads();
        for (int idx = tid; idx < nm * n; idx += nth) {
          const int q = idx / n, r = idx - q * n;
          const int col = s.perm[q];
          if (s.dv[col] < thr) mo[(int64_t)q * N + a.free_ref[r]] = s.sg[q] * Z[r * P + col];
        }
      }
    } else {                                   // failed system: zero outputs, never NaN
      for (int q = tid; q < nm; q += nth) frow[q] = 0.0;
      if (mo)
        for (int64_t i = tid; i < (int64_t)nm * N; i += nth) mo[i] = 0.0;
    }
    if (tid == 0) a.info[b] = status;
  }
}


// ---- ragged batches (tb_modes_ragged): one CTA per truss, every truss with its own topology
// Only step 1 differs from k_modes: the static solve's guards on the truss, its free-DOF list (ascending DOF, the
// reference's mask order) in shared memory in place of i2r, and a row-owner assembly: the thread of free row r scans
// the truss's members in ascending order and adds every member incident to r's joint to the whole row (both triangles,
// no atomics).  Per entry that is the plan scatter map's ascending-member order, so K_ff, the lumped mass (ascending
// member * 2 + end) and the consistent M_ff get the bits of k_modes for a plan of the same topology.  Shared memory is
// laid out for the launch's free-DOF bound: [bound] free-DOF list, [bound] ranks, then the arrays of steps 2-5 for the
// truss's own n (modes_smem_bytes(bound) in all).

// free indices of joint J's DIM DOFs (-1 at a supported one): fr is ascending, so a joint's free DOFs are consecutive
template <int DIM>
__device__ __forceinline__ void rag_free_of(const int* fr, int n, int J, int f[DIM]) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (fr[mid] < J * DIM) lo = mid + 1;
    else hi = mid;
  }
#pragma unroll
  for (int i = 0; i < DIM; ++i) {
    const bool hit = lo < n && fr[lo] == J * DIM + i;
    f[i] = hit ? lo : -1;
    lo += hit ? 1 : 0;
  }
}

// (min. 1 CTA: without it ptxas holds the kernel at 96 registers and spills; at 112-116 registers shared memory still
// bounds the residency, e.g. 5 CTAs per SM for a bound of 69 free DOFs)
template <int DIM>
__global__ void __launch_bounds__(160, 1) k_modes_ragged(const ModesRagArgs a) {
  extern __shared__ __align__(16) double smem[];
  __shared__ ModesCtl ctl;
  __shared__ int wcnt[160 / 32];
  const int bound = a.max_free, nm = a.n_modes;
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nth >> 5;
  int* fr = (int*)smem;                        // [bound] DOF index of free DOF r of the current truss
  int* perm = fr + bound;                      // [bound]
  double* base = smem + bound;                 // (2 bound ints)
  double* L = a.slot ? a.slot + (size_t)blockIdx.x * bound * bound : nullptr;   // consistent mass: M_ff, then its factor

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const int64_t jo = a.joint_off[b], mo = a.member_off[b];
    const int64_t nj64 = a.joint_off[b + 1] - jo, nm64 = a.member_off[b + 1] - mo;
    const bool rows = nj64 >= 0 && nm64 >= 0 && jo >= 0 && mo >= 0 && jo + nj64 <= a.joint_off[a.batch] &&
                      mo + nm64 <= a.member_off[a.batch];
    const bool fits = rows && nj64 <= a.max_joint && nm64 <= a.max_member;   // (else TB_INFO_BAD_INDEX, as the solve)
    const int nJ = fits ? (int)nj64 : 0, M = fits ? (int)nm64 : 0, N = nJ * DIM;
    const double* xyz = a.xyz + jo * DIM;
    const uint8_t* sup = a.support + jo;
    const int32_t* conn = a.conn + mo * 2;
    const double* aed = a.aed + mo * 3;
    const double* jm = a.jmass ? a.jmass + jo : nullptr;
    __syncthreads();                           // the previous truss's shared data is consumed

    // ---- free-DOF list (a block-wide ballot scan) and the static solve's guards, its precedence: index / size, support,
    // zero length, counting rule
    int n = 0, bad = 0;
    for (int d0 = 0; d0 < N; d0 += nth) {
      const int dof = d0 + tid;
      bool f = false;
      if (dof < N) {
        const int j = dof / DIM, ax = dof - j * DIM, sj = sup[j];
        if (ax == 0 && tb_support_bad(DIM, sj)) bad |= 4;
        f = tb_dof_free(sj, ax);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, f);
      if (lane == 0) wcnt[wid] = __popc(bal);
      __syncthreads();
      int pre = 0, tot = 0;
      for (int w = 0; w < nw; ++w) {
        pre += w < wid ? wcnt[w] : 0;
        tot += wcnt[w];
      }
      const int pos = n + pre + __popc(bal & ((1u << lane) - 1u));
      if (f && pos < bound) fr[pos] = dof;
      n += tot;
      __syncthreads();
    }
    for (int m = tid; m < M; m += nth) {
      const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
      if ((unsigned)j0 >= (unsigned)nJ || (unsigned)j1 >= (unsigned)nJ) {
        bad |= 1;
      } else {
        double dx[DIM], c[DIM], k, w;
        if (!(tb_member_geom<DIM>(xyz, j0, j1, aed[3 * m], aed[3 * m + 1], aed[3 * m + 2], dx, c, k, w) > 0.0)) bad |= 2;
      }
    }
    const int anyidx = __syncthreads_or(bad & 1), anylen = __syncthreads_or(bad & 2), anysup = __syncthreads_or(bad & 4);
    const int nres = N - n;                    // every restrained DOF is one resistance (type.py:37-46)
    const bool stable = (DIM == 2) ? (M + nres >= N) : (nres >= 6 && M + nres >= N);
    int status = 0;
    if (!fits || anyidx || n > bound) status = TB_INFO_BAD_INDEX;
    else if (anysup) status = TB_INFO_BAD_SUPPORT;
    else if (anylen) status = TB_INFO_ZERO_LENGTH;
    else if (!stable) status = TB_INFO_NOT_STABLE;
    if (status != 0 || n == 0) n = 0;          // (no eigenproblem: only zeros to write)
    const int P = n | 1;
    const ModesSmem s = modes_smem(base, n, perm);

    if (n > 0) {
      // ---- K_ff and the mass, row-owner, both triangles
      int badm = 0;
      for (int r = tid; r < n; r += nth) {
        double* zr = s.Z + (size_t)r * P;
        double* lr = a.consistent ? L + (size_t)r * n : nullptr;
        for (int c = 0; c < P; ++c) zr[c] = 0.0;
        if (lr)
          for (int c = 0; c < n; ++c) lr[c] = 0.0;
        const int jr = fr[r] / DIM, ar = fr[r] - jr * DIM;
        int fs[DIM], fo[DIM];
        rag_free_of<DIM>(fr, n, jr, fs);
        double ms = 0.0;
        for (int m = 0; m < M; ++m) {
          const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
          if (j0 != jr && j1 != jr) continue;
          rag_free_of<DIM>(fr, n, j0 == jr ? j1 : j0, fo);
          double dx[DIM], cs[DIM], k, w;
          tb_member_geom<DIM>(xyz, j0, j1, aed[3 * m], aed[3 * m + 1], aed[3 * m + 2], dx, cs, k, w);
#pragma unroll
          for (int j = 0; j < DIM; ++j) {
            const double pr = __dmul_rn(cs[ar], cs[j]);                   // truss.py:69,80
            if (fs[j] >= 0) zr[fs[j]] = __dadd_rn(zr[fs[j]], __dmul_rn(k, pr));   // same joint: + block
            if (fo[j] >= 0) zr[fo[j]] = __dadd_rn(zr[fo[j]], __dmul_rn(k, -pr));  // other joint: - block
          }
          if (lr) {                            // (m_e / 6) [[2, 1], [1, 2]] per axis
            const double me6 = __ddiv_rn(w, 6.0);
            lr[r] = __dadd_rn(lr[r], __dmul_rn(2.0, me6));
            if (fo[ar] >= 0) lr[fo[ar]] = __dadd_rn(lr[fo[ar]], me6);
          } else {                             // lumped: m_e / 2 per end joint and axis
            ms = __dadd_rn(ms, __dmul_rn(w, 0.5));
          }
        }
        if (lr) {
          if (jm) lr[r] = __dadd_rn(lr[r], jm[jr]);
        } else {
          if (jm) ms = __dadd_rn(ms, jm[jr]);
          if (!(ms > 0.0)) badm = 1;
          s.sc[r] = ms > 0.0 ? 1.0 / sqrt(ms) : 0.0;
        }
      }
      if (__syncthreads_or(badm)) status = TB_INFO_MASS;
      status = modes_eigen(s, n, a.consistent, L, ctl, status);
    }

    // ---- outputs: the n lowest of the n_modes requested are real, the rest (and a failed truss) zeros
    const int nq = status == 0 ? min(nm, n) : 0;
    double* erow = a.eigval + (int64_t)b * nm;
    if (nq > 0) modes_order(s, n, nq, a.consistent, L, erow);
    for (int q = nq + tid; q < nm; q += nth) erow[q] = 0.0;
    if (a.modes && rows) {
      const int64_t Nb = nj64 * DIM;
      double* mo_b = a.modes + (int64_t)nm * DIM * jo;
      for (int64_t i = tid; i < (int64_t)nm * Nb; i += nth) mo_b[i] = 0.0;
      __syncthreads();
      for (int idx = tid; idx < nq * n; idx += nth) {
        const int q = idx / n, r = idx - q * n;
        mo_b[(int64_t)q * Nb + fr[r]] = s.sg[q] * s.Z[r * P + s.perm[q]];
      }
    }
    if (tid == 0) {
      a.info[b] = status;
      if (a.n_free) a.n_free[b] = status == 0 ? n : 0;
    }
  }
}

// CTA size and residency depend on the free-DOF bound n only: cached per device and n (the occupancy query costs more
// than the launch).  KERN: which kernel (MODES_PLAN k_modes, MODES_RAGGED k_modes_ragged, MODES_BUCKLING k_buckling).
enum { MODES_PLAN, MODES_RAGGED, MODES_BUCKLING };

template <int DIM, int KERN>
int modes_config(int n, int* threads, int* smem, int* per_sm) {
  static int cache[64][TB_SMALL_MAX_DOF + 1];
  static int attr[64];   // the kernel's dynamic shared-memory limit set so far (only ever raised)
  static std::mutex mu;
  const void* kern = KERN == MODES_RAGGED ? (const void*)k_modes_ragged<DIM>
                     : KERN == MODES_BUCKLING ? (const void*)k_buckling<DIM> : (const void*)k_modes<DIM>;
  int dev = 0;
  TB_CUDA(cudaGetDevice(&dev));
  *threads = ((n < 32 ? 32 : n) + 31) / 32 * 32;
  *smem = (int)modes_smem_bytes(n);
  std::lock_guard<std::mutex> lock(mu);
  int& c = cache[dev & 63][n];
  if (c == 0) {
    if (*smem > attr[dev & 63]) {   // (the exact size: the opt-in limit also counts the kernel's static shared memory)
      TB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, *smem));
      attr[dev & 63] = *smem;
    }
    int q = 0;
    TB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, *threads, (size_t)*smem));
    if (q < 1) return (int)cudaErrorInvalidConfiguration;
    c = q;
  }
  *per_sm = c;
  return 0;
}

// ---- reverse mode (tb_modes_adjoint): dlambda/dp = phi^T (dK/dp - lambda dM/dp) phi, summed with the cotangent
// k_modes_sens<DIM> runs one warp per system (8 per CTA, persistent grid-stride loop).  Lanes first take members and
// write the (a, e, density) row; then lanes take joints and gather the geometry vector of every incident member,
// recomputed by the same member body (one more member evaluation per end instead of per-member scratch).  Per member
// the modes are summed in ascending k, per joint the incidence list in ascending member*2+end order (gather_joint's
// order), so a system's bits depend on nothing but its own inputs.  No atomics, no shared memory, any M.
// k_modes_sens_ragged<DIM> is the same for a ragged batch: the member body is shared, only the free flags of a joint
// (the support codes instead of the plan's DOF map) and the incidence (a scan of the truss's members) are read otherwise.

constexpr int SENS_WARPS = 8;   // (launch bounds: 3 CTAs per SM, the residency of 74-80 registers; 64-78, no spills)

// free flags of a joint's DOFs: through the plan's DOF map, or from a ragged truss's support codes
template <int DIM>
struct PlanFree {
  const int32_t* dof2free;
  __device__ __forceinline__ bool operator()(int J, int i) const { return dof2free[J * DIM + i] >= 0; }
};
struct RagFree {
  const uint8_t* support;
  __device__ __forceinline__ bool operator()(int J, int i) const { return tb_dof_free(support[J], i); }
};

// phi of joint J in one mode row, read at free DOFs only (supported entries count as 0)
template <int DIM, class Free>
__device__ __forceinline__ void mode_at(const Free& fr, const double* phi, int J, double p[DIM]) {
#pragma unroll
  for (int i = 0; i < DIM; ++i) p[i] = fr(J, i) ? phi[J * DIM + i] : 0.0;
}

// Member m of one system over its first nq modes (rows of N): ga = dL/d(a, e, density) and v = dL/d(x_j1) =
// -dL/d(x_j0), with t = c.dphi and w the mass quadratic form per unit member mass (lumped (|phi0|^2 + |phi1|^2) / 2,
// consistent (|phi0|^2 + |phi1|^2 + phi0.phi1) / 3):
//   dlambda/da = (e/L) t^2 - lambda L rho w,  dlambda/de = (a/L) t^2,  dlambda/drho = -lambda a L w,
//   dlambda/dd = (k/L) (2 t dphi - 3 t^2 c) - lambda rho a w c
template <int DIM, class Free>
__device__ __forceinline__ void modes_sens_member(const Free& fr, const int32_t* conn, int N, int nq, int consistent,
                                                  const double* xyz, const double* aed_m, const double* lam,
                                                  const double* gl, const double* phi, int m, double ga[3], double v[DIM]) {
  const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
  const double ar = aed_m[0], e = aed_m[1], rho = aed_m[2];
  double dx[DIM], c[DIM], k, w;
  const double len = tb_member_geom<DIM>(xyz, j0, j1, ar, e, rho, dx, c, k, w);
  const double il = 1.0 / len, el = e * il, al = ar * il, kl = k * il, lr = len * rho, la = len * ar, ra = rho * ar;
  ga[0] = ga[1] = ga[2] = 0.0;
#pragma unroll
  for (int i = 0; i < DIM; ++i) v[i] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double g = gl[q];
    if (g == 0.0) continue;                    // (skipped, not multiplied by zero: a padded cotangent gives the same bits)
    const double* ph = phi + (int64_t)q * N;
    double p0[DIM], p1[DIM], dp[DIM], t = 0.0, s = 0.0, x = 0.0;
    mode_at<DIM>(fr, ph, j0, p0);
    mode_at<DIM>(fr, ph, j1, p1);
#pragma unroll
    for (int i = 0; i < DIM; ++i) {
      dp[i] = p1[i] - p0[i];
      t = fma(c[i], dp[i], t);
      s = fma(p0[i], p0[i], fma(p1[i], p1[i], s));
      x = fma(p0[i], p1[i], x);
    }
    const double wq = consistent ? (s + x) * (1.0 / 3.0) : 0.5 * s;
    const double lq = lam[q], t2 = t * t, lw = lq * wq;
    ga[0] += g * (el * t2 - lr * lw);
    ga[1] += g * (al * t2);
    ga[2] -= g * (la * lw);
#pragma unroll
    for (int i = 0; i < DIM; ++i) v[i] += g * (kl * (2.0 * t * dp[i] - 3.0 * t2 * c[i]) - ra * lw * c[i]);
  }
}

// dL/dmu_J = -sum_k g_k lambda_k |phi_J|^2 over the first nq modes
template <int DIM, class Free>
__device__ __forceinline__ double modes_sens_jmass(const Free& fr, int N, int nq, const double* lam, const double* gl,
                                                   const double* phi, int J) {
  double s = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double g = gl[q];
    if (g == 0.0) continue;
    double p[DIM], pp = 0.0;
    mode_at<DIM>(fr, phi + (int64_t)q * N, J, p);
#pragma unroll
    for (int i = 0; i < DIM; ++i) pp = fma(p[i], p[i], pp);
    s += g * (lam[q] * pp);
  }
  return -s;
}

template <int DIM>
__global__ void __launch_bounds__(32 * SENS_WARPS, 3) k_modes_sens(const ModesSensArgs a) {
  const int lane = threadIdx.x & 31;
  const int nm = a.n_modes;
  const PlanFree<DIM> fr{a.dof2free};
  for (int b = blockIdx.x * SENS_WARPS + (threadIdx.x >> 5); b < a.batch; b += gridDim.x * SENS_WARPS) {
    double* gx = a.g_xyz ? a.g_xyz + (int64_t)b * a.N : nullptr;
    double* ga = a.g_aed ? a.g_aed + (int64_t)b * a.M * 3 : nullptr;
    double* gj = a.g_jmass ? a.g_jmass + (int64_t)b * a.nJ : nullptr;
    if (a.info[b] != 0) {                      // failed system: zero gradients, never NaN
      for (int i = lane; i < a.N; i += 32)
        if (gx) gx[i] = 0.0;
      for (int i = lane; i < 3 * a.M; i += 32)
        if (ga) ga[i] = 0.0;
      for (int i = lane; i < a.nJ; i += 32)
        if (gj) gj[i] = 0.0;
      continue;
    }
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed + b * a.aed_stride;
    const double* lam = a.eigval + (int64_t)b * nm;
    const double* gl = a.g_eigval + (int64_t)b * nm;
    const double* phi = a.modes + (int64_t)b * nm * a.N;
    if (ga)
      for (int m = lane; m < a.M; m += 32) {
        double r[3], v[DIM];
        modes_sens_member<DIM>(fr, a.conn, a.N, nm, a.consistent, xyz, aed + 3 * m, lam, gl, phi, m, r, v);
        ga[3 * m] = r[0];
        ga[3 * m + 1] = r[1];
        ga[3 * m + 2] = r[2];
      }
    if (!gx && !gj) continue;
    for (int J = lane; J < a.nJ; J += 32) {
      if (gx) {
        double s[DIM];
#pragma unroll
        for (int i = 0; i < DIM; ++i) s[i] = 0.0;
        for (int p = a.inc_ptr[J]; p < a.inc_ptr[J + 1]; ++p) {   // (+) at the member's joint 1, (-) at its joint 0
          const int me = a.inc_mem[p], m = me >> 1;
          double r[3], v[DIM];
          modes_sens_member<DIM>(fr, a.conn, a.N, nm, a.consistent, xyz, aed + 3 * m, lam, gl, phi, m, r, v);
#pragma unroll
          for (int i = 0; i < DIM; ++i) s[i] += (me & 1) ? v[i] : -v[i];
        }
#pragma unroll
        for (int i = 0; i < DIM; ++i) gx[J * DIM + i] = s[i];
      }
      if (gj) gj[J] = modes_sens_jmass<DIM>(fr, a.N, nm, lam, gl, phi, J);   // dlambda/dmu_J = -lambda |phi_J|^2
    }
  }
}

template <int DIM>
__global__ void __launch_bounds__(32 * SENS_WARPS, 3) k_modes_sens_ragged(const ModesSensRagArgs a) {
  const int lane = threadIdx.x & 31;
  const int nm = a.n_modes;
  for (int b = blockIdx.x * SENS_WARPS + (threadIdx.x >> 5); b < a.batch; b += gridDim.x * SENS_WARPS) {
    const int64_t jo = a.joint_off[b], mo = a.member_off[b];
    const int64_t nj64 = a.joint_off[b + 1] - jo, nm64 = a.member_off[b + 1] - mo;
    const bool rows = nj64 >= 0 && nm64 >= 0 && jo >= 0 && mo >= 0 && jo + nj64 <= a.joint_off[a.batch] &&
                      mo + nm64 <= a.member_off[a.batch];
    const bool ok = rows && nj64 <= a.max_joint && nm64 <= a.max_member;
    const int nJ = rows ? (int)nj64 : 0, M = rows ? (int)nm64 : 0, N = nJ * DIM;
    double* gx = a.g_xyz ? a.g_xyz + jo * DIM : nullptr;
    double* ga = a.g_aed ? a.g_aed + mo * 3 : nullptr;
    double* gj = a.g_jmass ? a.g_jmass + jo : nullptr;
    if (!ok || a.info[b] != 0) {               // failed truss: zero gradients (nothing when its rows are not valid)
      for (int i = lane; i < N; i += 32)
        if (gx) gx[i] = 0.0;
      for (int i = lane; i < 3 * M; i += 32)
        if (ga) ga[i] = 0.0;
      for (int i = lane; i < nJ; i += 32)
        if (gj) gj[i] = 0.0;
      continue;
    }
    const RagFree fr{a.support + jo};
    const int32_t* conn = a.conn + mo * 2;
    const double* xyz = a.xyz + jo * DIM;
    const double* aed = a.aed + mo * 3;
    const double* lam = a.eigval + (int64_t)b * nm;
    const double* gl = a.g_eigval + (int64_t)b * nm;
    const double* phi = a.modes + (int64_t)nm * DIM * jo;
    // the truss's free DOFs: modes q >= n are the forward's padding and are skipped, whatever their cotangent
    int nf = 0;
    for (int J = lane; J < nJ; J += 32)
#pragma unroll
      for (int i = 0; i < DIM; ++i) nf += fr(J, i) ? 1 : 0;
    const int nq = min(nm, __reduce_add_sync(0xffffffffu, nf));
    if (ga)
      for (int m = lane; m < M; m += 32) {
        const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
        double r[3] = {0.0, 0.0, 0.0}, v[DIM];
        if ((unsigned)j0 < (unsigned)nJ && (unsigned)j1 < (unsigned)nJ)   // (info == 0 rules this out; never read out of range)
          modes_sens_member<DIM>(fr, conn, N, nq, a.consistent, xyz, aed + 3 * m, lam, gl, phi, m, r, v);
        ga[3 * m] = r[0];
        ga[3 * m + 1] = r[1];
        ga[3 * m + 2] = r[2];
      }
    if (!gx && !gj) continue;
    for (int J = lane; J < nJ; J += 32) {
      if (gx) {
        double s[DIM];
#pragma unroll
        for (int i = 0; i < DIM; ++i) s[i] = 0.0;
        for (int m = 0; m < M; ++m) {          // ascending member, (-) at its joint 0 then (+) at its joint 1: the plan's order
          const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
          if ((j0 != J && j1 != J) || (unsigned)j0 >= (unsigned)nJ || (unsigned)j1 >= (unsigned)nJ) continue;
          double r[3], v[DIM];
          modes_sens_member<DIM>(fr, conn, N, nq, a.consistent, xyz, aed + 3 * m, lam, gl, phi, m, r, v);
          if (j0 == J)
#pragma unroll
            for (int i = 0; i < DIM; ++i) s[i] += -v[i];
          if (j1 == J)
#pragma unroll
            for (int i = 0; i < DIM; ++i) s[i] += v[i];
        }
#pragma unroll
        for (int i = 0; i < DIM; ++i) gx[J * DIM + i] = s[i];
      }
      if (gj) gj[J] = modes_sens_jmass<DIM>(fr, N, nq, lam, gl, phi, J);
    }
  }
}

// ---- reverse mode of linear buckling (tb_buckling_adjoint): for a simple critical mode with phi^T K_ff phi = 1,
//   dlambda/dp = lambda phi^T (dK/dp) phi + lambda^2 phi^T (dK_G/dp) phi,
// the member forces N held fixed (their own gradient is an output: the caller closes the chain through the static
// solve's adjoint).  k_buckling_sens<DIM> has k_modes_sens' shape: one warp per system, lanes over members write the
// (a, e, density) row and the dL/dN row, then lanes over joints gather the geometry vector over the plan's incidence
// lists, recomputing the member body.  Modes are summed in ascending q; a mode with a zero cotangent or a factor that is
// not finite (+inf: not critical, its row is zero) is skipped whatever its cotangent, so lambda 0 inf never turns into
// NaN.  No atomics, no shared memory, no scratch.

// Member m of one system over its first nq modes: ga = dL/d(a, e), gn = dL/dN_m and v = dL/d(x_j1) = -dL/d(x_j0), with
// t = c.dphi, s = |dphi|^2 and g = N / L (phi^T K_m phi = k t^2, phi^T K_G,m phi = g (s - t^2)):
//   dlambda/da = lambda (e/L) t^2,  dlambda/de = lambda (a/L) t^2,  dlambda/dN = lambda^2 (s - t^2) / L,
//   dlambda/dd = lambda (k/L) (2 t dphi - 3 t^2 c) + lambda^2 (g/L) (3 t^2 c - 2 t dphi - s c)
template <int DIM>
__device__ __forceinline__ void buckling_sens_member(const PlanFree<DIM>& fr, const int32_t* conn, int N, int nq,
                                                     const double* xyz, const double* aed_m, double axial_m,
                                                     const double* lam, const double* gl, const double* phi, int m,
                                                     double ga[2], double& gn, double v[DIM]) {
  const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
  const double ar = aed_m[0], e = aed_m[1];
  double dx[DIM], c[DIM], k, w;
  const double len = tb_member_geom<DIM>(xyz, j0, j1, ar, e, aed_m[2], dx, c, k, w);
  const double il = 1.0 / len, el = e * il, al = ar * il, kl = k * il, gll = axial_m * il * il;
  ga[0] = ga[1] = gn = 0.0;
#pragma unroll
  for (int i = 0; i < DIM; ++i) v[i] = 0.0;
  for (int q = 0; q < nq; ++q) {
    const double g = gl[q], lq = lam[q];
    if (g == 0.0 || !isfinite(lq)) continue;
    const double* ph = phi + (int64_t)q * N;
    double p0[DIM], p1[DIM], dp[DIM], t = 0.0, s = 0.0;
    mode_at<DIM>(fr, ph, j0, p0);
    mode_at<DIM>(fr, ph, j1, p1);
#pragma unroll
    for (int i = 0; i < DIM; ++i) {
      dp[i] = p1[i] - p0[i];
      t = fma(c[i], dp[i], t);
      s = fma(dp[i], dp[i], s);
    }
    const double gq = g * lq, gq2 = gq * lq, t2 = t * t;
    ga[0] += gq * (el * t2);
    ga[1] += gq * (al * t2);
    gn += gq2 * ((s - t2) * il);
#pragma unroll
    for (int i = 0; i < DIM; ++i) {
      const double a2 = 2.0 * t * dp[i] - 3.0 * t2 * c[i];
      v[i] += gq * (kl * a2) - gq2 * (gll * (a2 + s * c[i]));
    }
  }
}

template <int DIM>
__global__ void __launch_bounds__(32 * SENS_WARPS, 3) k_buckling_sens(const BucklingSensArgs a) {
  const int lane = threadIdx.x & 31;
  const int nm = a.n_modes;
  const PlanFree<DIM> fr{a.dof2free};
  for (int b = blockIdx.x * SENS_WARPS + (threadIdx.x >> 5); b < a.batch; b += gridDim.x * SENS_WARPS) {
    double* gx = a.g_xyz ? a.g_xyz + (int64_t)b * a.N : nullptr;
    double* ga = a.g_aed ? a.g_aed + (int64_t)b * a.M * 3 : nullptr;
    double* gn = a.g_axial ? a.g_axial + (int64_t)b * a.M : nullptr;
    if (a.info[b] != 0) {                      // failed system: zero gradients, never NaN
      for (int i = lane; i < a.N; i += 32)
        if (gx) gx[i] = 0.0;
      for (int i = lane; i < 3 * a.M; i += 32)
        if (ga) ga[i] = 0.0;
      for (int i = lane; i < a.M; i += 32)
        if (gn) gn[i] = 0.0;
      continue;
    }
    const double* xyz = a.xyz + b * a.xyz_stride;
    const double* aed = a.aed + b * a.aed_stride;
    const double* ax = a.axial + b * a.axial_stride;
    const double* lam = a.factor + (int64_t)b * nm;
    const double* gl = a.g_factor + (int64_t)b * nm;
    const double* phi = a.modes + (int64_t)b * nm * a.N;
    if (ga || gn)
      for (int m = lane; m < a.M; m += 32) {
        double r[2], rn, v[DIM];
        buckling_sens_member<DIM>(fr, a.conn, a.N, nm, xyz, aed + 3 * m, ax[m], lam, gl, phi, m, r, rn, v);
        if (ga) {
          ga[3 * m] = r[0];
          ga[3 * m + 1] = r[1];
          ga[3 * m + 2] = 0.0;                 // the density enters neither K nor K_G
        }
        if (gn) gn[m] = rn;
      }
    if (!gx) continue;
    for (int J = lane; J < a.nJ; J += 32) {
      double s[DIM];
#pragma unroll
      for (int i = 0; i < DIM; ++i) s[i] = 0.0;
      for (int p = a.inc_ptr[J]; p < a.inc_ptr[J + 1]; ++p) {   // (+) at the member's joint 1, (-) at its joint 0
        const int me = a.inc_mem[p], m = me >> 1;
        double r[2], rn, v[DIM];
        buckling_sens_member<DIM>(fr, a.conn, a.N, nm, xyz, aed + 3 * m, ax[m], lam, gl, phi, m, r, rn, v);
#pragma unroll
        for (int i = 0; i < DIM; ++i) s[i] += (me & 1) ? v[i] : -v[i];
      }
#pragma unroll
      for (int i = 0; i < DIM; ++i) gx[J * DIM + i] = s[i];
    }
  }
}

// persistent grid of a warp-per-system kernel: the resident CTAs of the device (the occupancy query costs more than the
// launch: cached per device and kernel)
template <int WHICH>
int sens_grid(const void* kern, int batch, int* grid) {
  static int cache[64];
  static std::mutex mu;
  int dev = 0, per_sm = 0, sms = 0;
  TB_CUDA(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lock(mu);
    int& c = cache[dev & 63];
    if (c == 0) {
      int q = 0;
      TB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, 32 * SENS_WARPS, 0));
      if (q < 1) return (int)cudaErrorInvalidConfiguration;
      c = q;
    }
    per_sm = c;
  }
  TB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  *grid = (int)std::min<int64_t>(((int64_t)batch + SENS_WARPS - 1) / SENS_WARPS, (int64_t)sms * per_sm);
  return 0;
}

}  // namespace

int tb_modes_config(int dim, int n, int* threads, int* smem, int* per_sm) {
  if (n < 1 || n > TB_SMALL_MAX_DOF) return (int)cudaErrorInvalidValue;
  return dim == 3 ? modes_config<3, MODES_PLAN>(n, threads, smem, per_sm) : modes_config<2, MODES_PLAN>(n, threads, smem, per_sm);
}

int tb_modes_ragged_config(int dim, int bound, int* threads, int* smem, int* per_sm) {
  if (bound < 1 || bound > TB_SMALL_MAX_DOF) return (int)cudaErrorInvalidValue;
  return dim == 3 ? modes_config<3, MODES_RAGGED>(bound, threads, smem, per_sm)
                  : modes_config<2, MODES_RAGGED>(bound, threads, smem, per_sm);
}

int tb_buckling_config(int dim, int n, int* threads, int* smem, int* per_sm) {
  if (n < 1 || n > TB_SMALL_MAX_DOF) return (int)cudaErrorInvalidValue;
  return dim == 3 ? modes_config<3, MODES_BUCKLING>(n, threads, smem, per_sm)
                  : modes_config<2, MODES_BUCKLING>(n, threads, smem, per_sm);
}

int tb_launch_modes(const ModesArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  if (dim == 3) k_modes<3><<<grid, threads, smem, st>>>(a);
  else k_modes<2><<<grid, threads, smem, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int tb_launch_buckling(const BucklingArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st) {
  if (a.base.batch <= 0) return 0;
  if (dim == 3) k_buckling<3><<<grid, threads, smem, st>>>(a);
  else k_buckling<2><<<grid, threads, smem, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int tb_launch_modes_ragged(const ModesRagArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  if (dim == 3) k_modes_ragged<3><<<grid, threads, smem, st>>>(a);
  else k_modes_ragged<2><<<grid, threads, smem, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int tb_launch_modes_sens(const ModesSensArgs& a, int dim, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  int grid = 0;
  int rc = dim == 3 ? sens_grid<3>((const void*)k_modes_sens<3>, a.batch, &grid)
                    : sens_grid<2>((const void*)k_modes_sens<2>, a.batch, &grid);
  if (rc) return rc;
  if (dim == 3) k_modes_sens<3><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  else k_modes_sens<2><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int tb_launch_modes_sens_ragged(const ModesSensRagArgs& a, int dim, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  int grid = 0;
  int rc = dim == 3 ? sens_grid<13>((const void*)k_modes_sens_ragged<3>, a.batch, &grid)
                    : sens_grid<12>((const void*)k_modes_sens_ragged<2>, a.batch, &grid);
  if (rc) return rc;
  if (dim == 3) k_modes_sens_ragged<3><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  else k_modes_sens_ragged<2><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}

int tb_launch_buckling_sens(const BucklingSensArgs& a, int dim, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  int grid = 0;
  int rc = dim == 3 ? sens_grid<23>((const void*)k_buckling_sens<3>, a.batch, &grid)
                    : sens_grid<22>((const void*)k_buckling_sens<2>, a.batch, &grid);
  if (rc) return rc;
  if (dim == 3) k_buckling_sens<3><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  else k_buckling_sens<2><<<grid, 32 * SENS_WARPS, 0, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}
