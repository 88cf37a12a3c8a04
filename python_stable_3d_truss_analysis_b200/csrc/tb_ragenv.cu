// Envelope path of ragged batches: the trusses too large for the fused shared-memory kernels (k_dense16 / k_small).
// One CTA per truss in a persistent grid-stride loop; each CTA owns one slot of a scratch arena in global memory.
//
//   stage                          replaces (slientruss3d / this library)
//   status guards                  the fused kernels' oversize / index / support / length / counting-rule checks
//   reverse Cuthill-McKee order    tb_plan_create's internal elimination order (tb_plan.cu), per truss on the device
//   row-owner assembly of K_ff     Member.matK + Truss.GetKMatrix     truss.py:65-86,307-316  (+ mask slicing :343)
//     into row-envelope storage
//   envelope Cholesky + solves     np.linalg.solve (LAPACK dgesv)     truss.py:343
//   axial forces, reactions, ext   truss.py:347-361 (the formulas of k_recover, tb_large.cu)
//
// The envelope of row i is the columns first[i]..i of K_ff (= of L) in the elimination order; it is addressed through one
// pointer that points into dynamic shared memory when the truss's envelope fits the launch's budget and into the CTA's
// slot otherwise.  The factorisation is right-looking, one column at a time: every entry of the trailing envelope is
// updated by one thread in ascending column order, so the result does not depend on the launch shape.  Assembly sums
// every entry's member contributions in ascending member order (row owner over the joint's incidence list), so K has the
// reference's bits.  No atomics touch floating-point data.
#include <math.h>

#include <mutex>

#include "tb_blocks.cuh"
#include "tb_common.cuh"

namespace {

constexpr int RE_THREADS = 256;
constexpr int RE_WARPS = RE_THREADS / 32;
// dynamic shared memory per CTA: two CTAs per SM (2 x 113 KB of the SM's 228 KB)
constexpr int RE_SMEM_BUDGET = 112 * 1024;

// per-CTA slot in global memory (byte offsets, 256-byte aligned)
struct RagEnvSlot {
  int64_t oEnv, oMem, oIncPtr, oInc, oAdj, oJoint, total;
};
// per-member doubles: EA/L, a L rho, axial force, cosines
enum : int { RM_K = 0, RM_W = 1, RM_AX = 2, RM_C = 3 };
// per-joint ints: degree, RCM order, BFS level / mark, seen, first free row (reference / RCM order), smallest row the
// joint couples to (reference / RCM order), free axes
enum : int { RJ_DEG = 0, RJ_ORDER, RJ_LEVEL, RJ_MARK, RJ_SEEN, RJ_NATF, RJ_RCMF, RJ_MINNAT, RJ_MINRCM, RJ_NF, RJ_COUNT };

__host__ __device__ inline int64_t re_al(int64_t x) { return (x + 255) & ~(int64_t)255; }

__host__ __device__ inline RagEnvSlot re_slot(int dim, int max_joint, int max_member) {
  RagEnvSlot s;
  const int64_t N = (int64_t)dim * max_joint, M = max_member, J = max_joint;
  int64_t o = 0;
  s.oEnv = o;    o += re_al(N * (N + 1) / 2 * 8);      // dense lower-triangle bound of the envelope
  s.oMem = o;    o += re_al(M * (3 + dim) * 8);        // member geometry and axial forces
  s.oIncPtr = o; o += re_al((J + 1) * 4);              // joint -> incidences (member * 2 + end), ascending
  s.oInc = o;    o += re_al(2 * M * 4);
  s.oAdj = o;    o += re_al(2 * M * 4);                // joint adjacency (sorted, de-duplicated), same ranges as inc
  s.oJoint = o;  o += re_al(RJ_COUNT * J * 4);         // per-joint integer arrays of the ordering
  s.total = o;
  return s;
}

// dynamic shared memory: y, x, 1/L_kk [N] doubles, the envelope budget, then first, ptr [N+1], last, d2f, free [N] ints
inline size_t re_fixed_smem(int dim, int max_joint) {
  const size_t N = (size_t)dim * max_joint;
  return 3 * N * 8 + ((5 * N + 1 + 1) & ~(size_t)1) * 4;
}

__device__ __forceinline__ double re_block_sum(double v, double* sRed, int tid) {
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(full, v, o);
  __syncthreads();
  if ((tid & 31) == 0) sRed[tid >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < RE_WARPS; ++w) t += sRed[w];
  return t;
}

// Member geometry (tb_member_geom) into the member's record {EA/L, a L rho, axial, cosines}; false for a zero length
// (k and the cosines are then stored as 0).
template <int DIM>
__device__ __forceinline__ bool re_member(const double* xyz, const double* aed, int j0, int j1, int m, double* rec) {
  double dx[DIM], c[DIM], k = 0.0, w = 0.0;
  const double len = tb_member_geom<DIM>(xyz, j0, j1, aed[3 * m], aed[3 * m + 1], aed[3 * m + 2], dx, c, k, w);
  const bool ok = len > 0.0;
  rec[RM_K] = ok ? k : 0.0;
  rec[RM_W] = w;
#pragma unroll
  for (int i = 0; i < DIM; ++i) rec[RM_C + i] = ok ? c[i] : 0.0;
  return ok;
}

template <int DIM>
__global__ void __launch_bounds__(RE_THREADS, 2) k_rag_env(const RagEnvArgs a) {
  extern __shared__ __align__(16) double smem[];
  __shared__ int sMeta[4];                   // [0] status  [1] n  [2] RCM order used
  __shared__ unsigned long long sSum[2];     // sum (i - first_i + 1)^2: natural order, RCM order
  __shared__ double sRed[RE_WARPS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Jmax = a.max_joint, Mmax = a.max_member, Nmax = Jmax * DIM;

  double* sY = smem;                         // rhs -> forward solution
  double* sX = sY + Nmax;                    // free displacements
  double* sDinv = sX + Nmax;                 // 1 / L_kk
  double* sEnv = sDinv + Nmax;               // envelope, when it fits a.env_smem
  int* sFirst = (int*)(sEnv + a.env_smem);   // [N]   first column of row i's envelope
  int* sPtr = sFirst + Nmax;                 // [N+1] offset of row i's envelope
  int* sLast = sPtr + Nmax + 1;              // [N]   last row whose envelope reaches column k
  int* sD2F = sLast + Nmax;                  // [N]   DOF -> elimination row, -1 at supports
  int* sFree = sD2F + Nmax;                  // [n]   elimination row -> DOF

  const RagEnvSlot SL = re_slot(DIM, Jmax, Mmax);
  char* slot = (char*)a.scratch + (size_t)blockIdx.x * a.slot_bytes;
  double* gEnv = (double*)(slot + SL.oEnv);
  double* mem = (double*)(slot + SL.oMem);
  int* incPtr = (int*)(slot + SL.oIncPtr);
  int* inc = (int*)(slot + SL.oInc);
  int* adj = (int*)(slot + SL.oAdj);
  int* jnt = (int*)(slot + SL.oJoint);
#define MK(m) mem[(m) * (3 + DIM) + RM_K]
#define MW(m) mem[(m) * (3 + DIM) + RM_W]
#define AXW(m) mem[(m) * (3 + DIM) + RM_AX]
#define MC(m, i) mem[(m) * (3 + DIM) + RM_C + (i)]
#define JA(f, j) jnt[(j) * RJ_COUNT + (f)]

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const int64_t jo = a.joint_off[b], mo = a.member_off[b];
    int nJ = (int)(a.joint_off[b + 1] - jo), M = (int)(a.member_off[b + 1] - mo);
    // routed launch: the fused kernels solved the trusses up to (route_joint, route_member)
    if (a.route_joint > 0 && nJ >= 0 && M >= 0 && nJ <= a.route_joint && M <= a.route_member) continue;
    // ---- 1. guards.  A truss over the slot's sizes touches nothing of the slot.
    const bool oversize = nJ > Jmax || M > Mmax || nJ < 0 || M < 0;
    if (oversize) { nJ = 0; M = 0; }
    const int N = nJ * DIM;
    const double* xyz = a.xyz + jo * DIM;
    const uint8_t* sup = a.support + jo;
    const int32_t* conn = a.conn + mo * 2;
    const double* aed = a.aed + mo * 3;
    if (tid == 0) {
      sMeta[0] = oversize ? TB_INFO_BAD_INDEX : 0;
      sMeta[1] = 0;
      sMeta[2] = 0;
      sSum[0] = 0;
      sSum[1] = 0;
    }
    for (int j = tid; j < nJ; j += RE_THREADS) {
      incPtr[j + 1] = 0;
      JA(RJ_MARK, j) = -1;
      JA(RJ_SEEN, j) = 0;
    }
    if (tid == 0) incPtr[0] = 0;
    __syncthreads();
    for (int j = tid; j < nJ; j += RE_THREADS)
      if (tb_support_bad(DIM, sup[j])) atomicMin(&sMeta[0], TB_INFO_BAD_SUPPORT);
    for (int m = tid; m < M; m += RE_THREADS) {
      const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
      if ((unsigned)j0 < (unsigned)nJ && (unsigned)j1 < (unsigned)nJ) {
        if (!re_member<DIM>(xyz, aed, j0, j1, m, &MK(m))) atomicMin(&sMeta[0], TB_INFO_ZERO_LENGTH);
        atomicAdd(&incPtr[j0 + 1], 1);         // incidence counts (integers: order-free)
        atomicAdd(&incPtr[j1 + 1], 1);
      } else {
        atomicMin(&sMeta[0], TB_INFO_BAD_INDEX);
        MK(m) = 0.0;
        MW(m) = 0.0;
#pragma unroll
        for (int i = 0; i < DIM; ++i) MC(m, i) = 0.0;
      }
    }
    __syncthreads();
    const bool indices_ok = sMeta[0] > TB_INFO_BAD_INDEX;

    if (indices_ok) {
      // ---- 2a. DOF counts, incidence offsets, counting rule (one thread: O(nJ))
      if (tid == 0) {
        int n = 0, run = 0;
        for (int j = 0; j < nJ; ++j) {
          int f = 0;
          for (int ax = 0; ax < DIM; ++ax) f += tb_dof_free(sup[j], ax) ? 1 : 0;
          JA(RJ_NF, j) = f;
          JA(RJ_NATF, j) = n;
          n += f;
          run += incPtr[j + 1];
          incPtr[j + 1] = run;
        }
        const int nres = N - n;                // every restrained DOF is one resistance (type.py:37-46)
        const bool stable = (DIM == 2) ? (M + nres >= N) : (nres >= 6 && M + nres >= N);
        if (!stable) atomicMin(&sMeta[0], TB_INFO_NOT_STABLE);
        sMeta[1] = n;
      }
      __syncthreads();
      // ---- 2b. incidence lists in ascending (member, end) and the joint adjacency (sorted, de-duplicated, no self-loops)
      for (int j = tid; j < nJ; j += RE_THREADS) {
        int p = incPtr[j];
        for (int m = 0; m < M; ++m) {
          if (conn[2 * m] == j) inc[p++] = 2 * m;
          if (conn[2 * m + 1] == j) inc[p++] = 2 * m + 1;
        }
        int* nb = adj + incPtr[j];
        int cnt = 0;
        for (int q = incPtr[j]; q < incPtr[j + 1]; ++q) {
          const int me = inc[q], v = conn[2 * (me >> 1) + 1 - (me & 1)];
          if (v == j) continue;
          int lo = 0, hi = cnt;                  // insert v into the sorted list unless present
          while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (nb[mid] < v) lo = mid + 1; else hi = mid;
          }
          if (lo < cnt && nb[lo] == v) continue;
          for (int t = cnt; t > lo; --t) nb[t] = nb[t - 1];
          nb[lo] = v;
          ++cnt;
        }
        JA(RJ_DEG, j) = cnt;
      }
      __syncthreads();
      // ---- 2c. reverse Cuthill-McKee (one thread), exactly tb_plan_create's rule: each component from its lowest
      // unseen joint, three passes of bfs_far to a pseudo-peripheral start, newly seen neighbours stable-sorted by degree,
      // the whole order reversed
      if (tid == 0) {
        int stamp = 0, nord = 0;
        for (int s0 = 0; s0 < nJ; ++s0) {
          if (JA(RJ_SEEN, s0)) continue;
          int start = s0;
          for (int it = 0; it < 3; ++it) {       // bfs_far: a farthest joint of minimum degree (the queue lives in order[])
            ++stamp;
            int qt = 0;
            JA(RJ_ORDER, nord + qt++) = start;
            JA(RJ_MARK, start) = stamp;
            JA(RJ_LEVEL, start) = 0;
            for (int h = 0; h < qt; ++h) {
              const int v = JA(RJ_ORDER, nord + h);
              for (int e = incPtr[v]; e < incPtr[v] + JA(RJ_DEG, v); ++e) {
                const int w = adj[e];
                if (JA(RJ_MARK, w) != stamp) { JA(RJ_MARK, w) = stamp; JA(RJ_LEVEL, w) = JA(RJ_LEVEL, v) + 1; JA(RJ_ORDER, nord + qt++) = w; }
              }
            }
            int best = JA(RJ_ORDER, nord + qt - 1);
            const int lv = JA(RJ_LEVEL, best);
            for (int h = 0; h < qt; ++h) {
              const int v = JA(RJ_ORDER, nord + h);
              if (JA(RJ_LEVEL, v) == lv && JA(RJ_DEG, v) < JA(RJ_DEG, best)) best = v;
            }
            start = best;
          }
          int h = nord;
          JA(RJ_ORDER, nord++) = start;
          JA(RJ_SEEN, start) = 1;
          for (; h < nord; ++h) {                // Cuthill-McKee
            const int v = JA(RJ_ORDER, h), s = nord;
            for (int e = incPtr[v]; e < incPtr[v] + JA(RJ_DEG, v); ++e) {
              const int w = adj[e];
              if (!JA(RJ_SEEN, w)) { JA(RJ_SEEN, w) = 1; JA(RJ_ORDER, nord++) = w; }
            }
            for (int i = s + 1; i < nord; ++i) {   // stable insertion sort by degree
              const int x = JA(RJ_ORDER, i), dx = JA(RJ_DEG, x);
              int k = i - 1;
              while (k >= s && JA(RJ_DEG, JA(RJ_ORDER, k)) > dx) { JA(RJ_ORDER, k + 1) = JA(RJ_ORDER, k); --k; }
              JA(RJ_ORDER, k + 1) = x;
            }
          }
        }
        for (int i = 0; i < nJ / 2; ++i) {
          const int t = JA(RJ_ORDER, i);
          JA(RJ_ORDER, i) = JA(RJ_ORDER, nJ - 1 - i);
          JA(RJ_ORDER, nJ - 1 - i) = t;
        }
        int r = 0;                               // free DOFs by (RCM rank of the joint, reference free index)
        for (int i = 0; i < nJ; ++i) {
          JA(RJ_RCMF, JA(RJ_ORDER, i)) = r;
          r += JA(RJ_NF, JA(RJ_ORDER, i));
        }
      }
      __syncthreads();
      // ---- 2d. row envelopes of both orders: row i of joint j starts at min(i, smallest row of a joint j couples to);
      // a joint couples to its adjacent joints, and to itself when a member touches it
      for (int j = tid; j < nJ; j += RE_THREADS) {
        int mn = 0x7fffffff, mr = 0x7fffffff;
        if (incPtr[j + 1] > incPtr[j] && JA(RJ_NF, j) > 0) { mn = JA(RJ_NATF, j); mr = JA(RJ_RCMF, j); }
        for (int e = incPtr[j]; e < incPtr[j] + JA(RJ_DEG, j); ++e) {
          const int v = adj[e];
          if (JA(RJ_NF, v) > 0) { mn = min(mn, JA(RJ_NATF, v)); mr = min(mr, JA(RJ_RCMF, v)); }
        }
        JA(RJ_MINNAT, j) = mn;
        JA(RJ_MINRCM, j) = mr;
        unsigned long long s0 = 0, s1 = 0;
        for (int t = 0; t < JA(RJ_NF, j); ++t) {
          const long long i0 = JA(RJ_NATF, j) + t, i1 = JA(RJ_RCMF, j) + t;
          const long long w0 = i0 - min(i0, (long long)mn) + 1, w1 = i1 - min(i1, (long long)mr) + 1;
          s0 += (unsigned long long)(w0 * w0);
          s1 += (unsigned long long)(w1 * w1);
        }
        if (s0) atomicAdd(&sSum[0], s0);
        if (s1) atomicAdd(&sSum[1], s1);
      }
      __syncthreads();
      const int n = sMeta[1];
      const bool use = n > 0 && (double)sSum[1] < 0.85 * (double)sSum[0];
      // ---- 2e. the chosen order: DOF maps and envelope rows
      for (int i = tid; i < N; i += RE_THREADS) sD2F[i] = -1;
      __syncthreads();
      for (int j = tid; j < nJ; j += RE_THREADS) {
        const int f0 = use ? JA(RJ_RCMF, j) : JA(RJ_NATF, j), mn = use ? JA(RJ_MINRCM, j) : JA(RJ_MINNAT, j);
        int t = 0;
        for (int ax = 0; ax < DIM; ++ax) {
          if (!tb_dof_free(sup[j], ax)) continue;
          const int r = f0 + t++;
          sD2F[j * DIM + ax] = r;
          sFree[r] = j * DIM + ax;
          sFirst[r] = min(r, mn);
        }
      }
      __syncthreads();
      if (tid == 0) {                            // envelope offsets and column extents (O(n))
        int p = 0;
        for (int i = 0; i < n; ++i) {
          sPtr[i] = p;
          p += i - sFirst[i] + 1;
          sLast[i] = i;
        }
        sPtr[n] = p;
        for (int i = 0; i < n; ++i) sLast[sFirst[i]] = max(sLast[sFirst[i]], i);
        for (int i = 1; i < n; ++i) sLast[i] = max(sLast[i], sLast[i - 1]);
        sMeta[2] = use ? 1 : 0;
      }
      __syncthreads();

      if (a.order) {                             // ordering mode: the elimination order of the joints and the envelope size
        for (int i = tid; i < nJ; i += RE_THREADS) a.order[jo + i] = sMeta[2] ? JA(RJ_ORDER, i) : i;
        if (tid == 0 && a.envelope) a.envelope[b] = sPtr[n];
      }
    } else if (a.order) {
      for (int i = tid; i < nJ; i += RE_THREADS) a.order[jo + i] = -1;
      if (tid == 0 && a.envelope) a.envelope[b] = -1;
    }
    if (a.order) {
      __syncthreads();
      continue;
    }

    int status = sMeta[0];
    const int n = sMeta[1];
    double* u_out = a.u ? a.u + jo * DIM : nullptr;
    double* ext_out = a.ext ? a.ext + jo * DIM : nullptr;
    double* ax_out = a.axial ? a.axial + mo : nullptr;

    if (status == 0 && n > 0) {
      const int esz = sPtr[n];
      double* env = esz <= a.env_smem ? sEnv : gEnv;
      // ---- 3. assembly: row owner over its joint's incidence list (ascending member, then end) + the load
      for (int e = tid; e < esz; e += RE_THREADS) env[e] = 0.0;
      const double* force = a.force + jo * DIM;
      for (int r = tid; r < n; r += RE_THREADS) sY[r] = force[sFree[r]];
      __syncthreads();
      for (int r = tid; r < n; r += RE_THREADS) {
        const int dof = sFree[r], jr = dof / DIM, ar = dof - jr * DIM;
        double* row = env + sPtr[r] - sFirst[r];
        for (int q = incPtr[jr]; q < incPtr[jr + 1]; ++q) {
          const int me = inc[q], m = me >> 1, A = me & 1;
          const double k = MK(m), ca = MC(m, ar);
#pragma unroll
          for (int B = 0; B < 2; ++B) {
            const int jb = conn[2 * m + B];
#pragma unroll
            for (int j = 0; j < DIM; ++j) {
              const int fc = sD2F[jb * DIM + j];
              if (fc >= 0 && fc <= r) {
                double p = __dmul_rn(ca, MC(m, j));
                if (A != B) p = -p;
                row[fc] = __dadd_rn(row[fc], __dmul_rn(k, p));
              }
            }
          }
        }
      }
      __syncthreads();
      // ---- 4. right-looking envelope Cholesky, the load riding along (L y = f); then L^T x = y
      int fail = 0;
      for (int k = 0; k < n; ++k) {
        const double d = env[sPtr[k] + k - sFirst[k]];
        if (!(d >= 2.2250738585072014e-308)) {   // non-positive, NaN or subnormal (its rsqrt would not be finite); uniform
          fail = k + 1;
          break;
        }
        const double rinv = tbblk::rsqrt_pos(d);   // (hardware seed + one third-order step, as k_dense16)
        const int lk = sLast[k];
        for (int i = k + 1 + tid; i <= lk; i += RE_THREADS) {
          const int fi = sFirst[i];
          if (fi <= k) env[sPtr[i] + k - fi] *= rinv;
        }
        if (tid == 0) {
          sDinv[k] = rinv;
          sY[k] *= rinv;
        }
        __syncthreads();
        const double yk = sY[k];
        for (int i = k + 1 + warp; i <= lk; i += RE_WARPS) {   // warp per row, lanes over its columns (k, i]
          const int fi = sFirst[i];
          if (fi > k) continue;
          double* rowi = env + sPtr[i] - fi;
          const double lik = rowi[k];
          if (lane == 0) sY[i] = fma(-lik, yk, sY[i]);
          for (int j = k + 1 + lane; j <= i; j += 32) {
            const int fj = sFirst[j];
            if (fj <= k) rowi[j] = fma(-lik, env[sPtr[j] + k - fj], rowi[j]);
          }
        }
        __syncthreads();
      }
      status = fail;
      if (status == 0) {
        for (int k = n - 1; k >= 0; --k) {
          const double xk = sY[k] * sDinv[k];
          if (tid == 0) sX[k] = xk;
          const int fk = sFirst[k];
          const double* rowk = env + sPtr[k] - fk;
          for (int j = fk + tid; j < k; j += RE_THREADS) sY[j] = fma(-rowk[j], xk, sY[j]);
          __syncthreads();
        }
      }
    }

    if (status != 0) {                           // zero-filled outputs, never NaN
      for (int i = tid; i < N; i += RE_THREADS) {
        if (u_out) u_out[i] = 0.0;
        if (ext_out) ext_out[i] = 0.0;
      }
      if (ax_out)
        for (int m = tid; m < M; m += RE_THREADS) ax_out[m] = 0.0;
      if (tid == 0) {
        if (a.weight) a.weight[b] = 0.0;
        if (a.info) a.info[b] = status;
      }
      __syncthreads();
      continue;
    }

    // ---- 5. recovery (k_recover's formulas): u, axial forces, weight, then ext (reactions over the incidence lists)
    if (u_out)
      for (int i = tid; i < N; i += RE_THREADS) {
        const int fr = sD2F[i];
        u_out[i] = fr >= 0 ? sX[fr] : 0.0;
      }
    double w = 0.0;
    for (int m = tid; m < M; m += RE_THREADS) {
      const int j0 = conn[2 * m], j1 = conn[2 * m + 1];
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        const int f1 = sD2F[j1 * DIM + i], f0 = sD2F[j0 * DIM + i];
        const double u1 = f1 >= 0 ? sX[f1] : 0.0, u0 = f0 >= 0 ? sX[f0] : 0.0;
        t = fma(MC(m, i), u1 - u0, t);
      }
      const double nm = MK(m) * t;
      w += MW(m);
      AXW(m) = nm;
      if (ax_out) ax_out[m] = nm;
    }
    w = re_block_sum(w, sRed, tid);              // (its barriers also publish axw)
    if (ext_out) {
      const double* f = a.force + jo * DIM;
      for (int dof = tid; dof < N; dof += RE_THREADS) {
        double e;
        if (sD2F[dof] >= 0) {
          e = f[dof];
        } else {                                 // row of K times u, member by member (ascending)
          const int J = dof / DIM, ax = dof - J * DIM;
          e = 0.0;
          for (int q = incPtr[J]; q < incPtr[J + 1]; ++q) {
            const int me = inc[q], m = me >> 1;
            const double g = (me & 1) ? MC(m, ax) : -MC(m, ax);
            e = fma(g, AXW(m), e);
          }
        }
        ext_out[dof] = e;
      }
    }
    if (tid == 0) {
      if (a.weight) a.weight[b] = w;
      if (a.info) a.info[b] = 0;
    }
    __syncthreads();                             // shared arrays and the slot are reused by the next truss
  }
#undef MK
#undef MW
#undef AXW
#undef MC
#undef JA
}

}  // namespace

size_t tb_rag_env_slot_bytes(int dim, int max_joint, int max_member) {
  return (size_t)re_slot(dim, max_joint, max_member).total;
}

int tb_rag_env_config(int dim, int max_joint, int max_member, int batch, int* grid, int* smem_bytes, int* env_smem) {
  const size_t fixed = re_fixed_smem(dim, max_joint);
  const size_t N = (size_t)dim * max_joint, dense = N * (N + 1) / 2;
  size_t env = fixed < (size_t)RE_SMEM_BUDGET ? ((size_t)RE_SMEM_BUDGET - fixed) / 8 : 0;
  if (env > dense) env = dense;
  const size_t smem = fixed + env * 8;
  if (smem > (size_t)227 * 1024) return TB_ERR_TOO_LARGE;
  auto kern = (dim == 3) ? k_rag_env<3> : k_rag_env<2>;
  struct Choice { int smem = -1, per_sm = 0, sms = 0; };
  static Choice cache[64][2];
  static std::mutex cache_mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return (int)cudaGetLastError();
  Choice ch;
  {
    std::lock_guard<std::mutex> lock(cache_mu);
    Choice& c = cache[dev & 63][dim - 2];
    if (c.smem != (int)smem) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      int q = 0;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, RE_THREADS, smem);
      if (e != cudaSuccess) return (int)e;
      cudaDeviceGetAttribute(&c.sms, cudaDevAttrMultiProcessorCount, dev);
      c.per_sm = q < 1 ? 1 : q;
      c.smem = (int)smem;
    }
    ch = c;
  }
  long long g = (long long)ch.sms * ch.per_sm;   // persistent: one slot per resident CTA
  if (g > batch) g = batch;
  if (g < 1) g = 1;
  *grid = (int)g;
  *smem_bytes = (int)smem;
  *env_smem = (int)env;
  return 0;
}

int tb_launch_rag_env(const RagEnvArgs& a, int grid, int smem_bytes, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  auto kern = (a.dim == 3) ? k_rag_env<3> : k_rag_env<2>;
  kern<<<(unsigned)grid, RE_THREADS, smem_bytes, st>>>(a);
  tb_count_launch();
  return (int)cudaGetLastError();
}
