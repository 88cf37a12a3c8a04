// Fused small-system path, second generation: ONE WARP per truss, everything between the inputs and the results
// stays on chip (HBM sees only the per-truss inputs and outputs), no block-level barrier anywhere.
//
//   stage                              replaces (slientruss3d)
//   DOF map (ballot scan)              Truss.GetDisplacementUnknownMask   truss.py:319-326, type.py:48-74
//   stability counting rule            Truss.isStable                     truss.py:154-164
//   member geometry                    Member.length/k/cosines            truss.py:19,56-63
//   joint incidence lists              (the "+=" loop of GetKMatrix visits members in ascending id; the lists keep
//                                       that order per joint, built with match_any ranks: deterministic, no atomics)
//   row-owner assembly of K_ff         Member.matK + Truss.GetKMatrix     truss.py:65-86,307-316  (+ mask slicing :343)
//   dense block Cholesky (16x16, DMMA) np.linalg.solve (LAPACK dgesv)     truss.py:343
//   + fused forward / back solve
//   axial forces, reactions            truss.py:347-361
//   weight, GA fitness                 truss.py:166-168,429-462; ga.py:139-149
//
// K_ff lives in shared memory as the lower triangle of 16x16 blocks in the DMMA fragment layout (tb_blocks.cuh), so the
// factorisation is the band kernel's block column loop with a full "band": products on the FP64 tensor cores, the
// 16x16 diagonal blocks and their inverses in registers (lanes = rows), triangular solves as products with the
// inverses.  Every entry of K_ff is summed in ascending member order (the reference's order), by the lane that owns
// its row.  Systems too large for this kernel's shared-memory budget fall back to tb_small.cu's CTA-per-truss kernel.
#include <math.h>

#include <mutex>

#include "tb_common.cuh"
#include "tb_blocks.cuh"

namespace {

using namespace tbblk;

struct D16Layout {   // per-warp shared-memory carve, in doubles from the warp's base
  int nblk, oK, oY, oXyz, oF, oU, oMk, oMc, oAx, oArea, oT, oCol, oConn, oInc, oIncPtr, oD2F, oFree, oSup, total;
};

__host__ __device__ inline D16Layout d16_layout(int dim, int nJ, int M, int nbm) {
  D16Layout L;
  const int N = nJ * dim;
  L.nblk = nbm * (nbm + 1) / 2;
  int o = 0;
  L.oK = o;      o += L.nblk * BE;
  L.oY = o;      o += nbm * BT;
  L.oT = o;      o += BT;                  // sT / sCol are read as double2: keep them at even offsets
  L.oCol = o;    o += 32;
  L.oXyz = o;    o += N;
  L.oF = o;      o += N;
  L.oU = o;      o += N;
  L.oMk = o;     o += M;
  L.oMc = o;     o += M * dim;
  L.oAx = o;     o += M;
  L.oArea = o;   o += M;
  L.oConn = o;   o += M;                   // [M][2] int32
  L.oInc = o;    o += M;                   // [2M]   int32: member * 2 + end, grouped by joint
  L.oIncPtr = o; o += (nJ + 2 + 1) / 2;    // [nJ+1] int32
  L.oD2F = o;    o += (N + 1) / 2;         // [N]    int32
  L.oFree = o;   o += (nbm * BT + 1) / 2;  // [n]    int32
  L.oSup = o;    o += (nJ + 7) / 8;        // [nJ]   uint8
  L.total = (o + 1) & ~1;                  // keep every warp's base 16-byte aligned
  return L;
}

__device__ __forceinline__ double warp_sum(double v) {   // fixed-shape tree: same bits every run
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int DIM>
__global__ void __launch_bounds__(128) k_dense16(const SmallArgs a, const int nbm, const int nwarp) {
  extern __shared__ __align__(16) double sm_all[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, lsw = lane_swz(lane);
  const int NJmax = a.nJ, Mmax = a.M;
  const D16Layout L = d16_layout(DIM, NJmax, Mmax, nbm);
  double* sm = sm_all + (size_t)wid * L.total;
  double* sK = sm + L.oK;
  double* sY = sm + L.oY;
  double* sXyz = sm + L.oXyz;
  double* sF = sm + L.oF;
  double* sU = sm + L.oU;
  double* sMk = sm + L.oMk;
  double* sMc = sm + L.oMc;
  double* sAx = sm + L.oAx;
  double* sArea = sm + L.oArea;
  double* sT = sm + L.oT;
  double* sCol = sm + L.oCol;
  int* sConn = (int*)(sm + L.oConn);
  int* sInc = (int*)(sm + L.oInc);
  int* sIncPtr = (int*)(sm + L.oIncPtr);
  int* sD2F = (int*)(sm + L.oD2F);
  int* sFree = (int*)(sm + L.oFree);
  uint8_t* sSup = (uint8_t*)(sm + L.oSup);
  const int qr = lane >> 2, qc = lane & 3;
  const unsigned FULL = 0xffffffffu;

  for (int b = blockIdx.x * nwarp + wid; b < a.batch; b += gridDim.x * nwarp) {
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
    int status = oversize ? TB_INFO_BAD_INDEX : 0;

    // ---- stage the inputs (coalesced)
    for (int i = lane; i < N; i += 32) {
      sXyz[i] = xyz[i];
      sF[i] = force[i];
    }
    for (int i = lane; i < nJ; i += 32) sSup[i] = sup[i];
    for (int i = lane; i < 2 * M; i += 32) sConn[i] = conn[i];
    __syncwarp();

    // ---- DOF map: free DOFs numbered in ascending DOF order (ballot scan), counting rule
    int n = 0;
    {
      bool badsup = false;
      for (int base = 0; base < N; base += 32) {
        const int dof = base + lane;
        bool fr = false;
        if (dof < N) {
          const int j = dof / DIM, ax = dof - j * DIM;
          const int s = sSup[j];
          badsup |= tb_support_bad(DIM, s);
          fr = tb_dof_free(s, ax);
        }
        const unsigned bal = __ballot_sync(FULL, fr);
        const int pos = n + __popc(bal & ((1u << lane) - 1u));
        if (dof < N) {
          sD2F[dof] = fr ? pos : -1;
          if (fr && pos < nbm * BT) sFree[pos] = dof;
        }
        n += __popc(bal);
      }
      const int nres = N - n;   // every restrained DOF is one resistance (type.py:37-46)
      const bool stable = (DIM == 2) ? (M + nres >= N) : (nres >= 6 && M + nres >= N);
      if (__any_sync(FULL, badsup)) status = min(status, TB_INFO_BAD_SUPPORT);
      else if (!stable) status = min(status, TB_INFO_NOT_STABLE);
      if (n > nbm * BT) status = min(status, TB_INFO_BAD_INDEX);   // cannot happen when the launcher sized nbm from max_n
    }

    // ---- member geometry (no FMA contraction: keep the reference's roundings), weight
    double wsum = 0.0;
    {
      int bad = 0;   // bit 0: index out of range, bit 1: zero length
      for (int m = lane; m < M; m += 32) {
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
          bad |= 1;
          sConn[2 * m] = 0;          // keep later gathers in range; the system is flagged and its outputs zeroed
          sConn[2 * m + 1] = 0;
        } else {
          double dx[DIM];
#pragma unroll
          for (int i = 0; i < DIM; ++i) dx[i] = __dsub_rn(sXyz[j1 * DIM + i], sXyz[j0 * DIM + i]);
          double l2 = __dmul_rn(dx[0], dx[0]);
#pragma unroll
          for (int i = 1; i < DIM; ++i) l2 = __dadd_rn(l2, __dmul_rn(dx[i], dx[i]));
          len = __dsqrt_rn(l2);
          if (!(len > 0.0)) {
            bad |= 2;
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
        sAx[m] = 0.0;
        wsum += __dmul_rn(__dmul_rn(ar, len), rho);
      }
      const unsigned anyidx = __ballot_sync(FULL, bad & 1), anylen = __ballot_sync(FULL, bad & 2);
      if (anyidx) status = min(status, TB_INFO_BAD_INDEX);
      else if (anylen) status = min(status, TB_INFO_ZERO_LENGTH);
    }
    __syncwarp();

    // ---- joint incidence lists: entries (member * 2 + end) grouped by joint, ascending inside a joint.
    // Lane l of a 16-member chunk handles member l/2, end l&1, so lane order == (member, end) order and the
    // match_any rank of a lane among the lanes with the same joint is its position in that joint's list.
    for (int j = lane; j <= nJ; j += 32) sIncPtr[j] = 0;
    __syncwarp();
    for (int m0 = 0; m0 < M; m0 += 16) {          // pass 1: degrees (into sIncPtr[j + 1])
      const int m = m0 + (lane >> 1);
      const int key = m < M ? sConn[2 * m + (lane & 1)] : -1 - lane;   // inactive lanes: unique negative keys
      const unsigned grp = __match_any_sync(FULL, key);
      if (key >= 0 && (grp & ((1u << lane) - 1u)) == 0) sIncPtr[key + 1] += __popc(grp);   // group leader
      __syncwarp();
    }
    {                                             // exclusive scan over the joints
      int carry = 0;
      for (int base = 0; base < nJ; base += 32) {
        const int j = base + lane;
        int v = j < nJ ? sIncPtr[j + 1] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(FULL, v, o);
          if (lane >= o) v += t;
        }
        if (j < nJ) sIncPtr[j + 1] = carry + v;
        carry += __shfl_sync(FULL, v, 31);
      }
    }
    __syncwarp();
    // pass 2: fill.  sU is free until the recovery stage: its first nJ words serve as per-joint write cursors.
    int* sCur = (int*)sU;
    for (int j = lane; j < nJ; j += 32) sCur[j] = sIncPtr[j];
    __syncwarp();
    for (int m0 = 0; m0 < M; m0 += 16) {
      const int m = m0 + (lane >> 1);
      const int key = m < M ? sConn[2 * m + (lane & 1)] : -1 - lane;
      const unsigned grp = __match_any_sync(FULL, key);
      const int rank = __popc(grp & ((1u << lane) - 1u));
      int basepos = 0;
      if (key >= 0) basepos = sCur[key];
      __syncwarp();
      if (key >= 0) {
        sInc[basepos + rank] = 2 * m + (lane & 1);
        if (rank == 0) sCur[key] = basepos + __popc(grp);
      }
      __syncwarp();
    }

    const int nb = (n + BT - 1) / BT;             // block columns of this system
    int fail = 0;
    if (status == 0 && n > 0) {
      // ---- zero K, then row-owner assembly (ascending member order per entry) + identity on the padded diagonal
      {
        const double2 z = make_double2(0.0, 0.0);
        const int nd2 = nb * (nb + 1) / 2 * (BE / 2);
        for (int i = lane; i < nd2; i += 32) reinterpret_cast<double2*>(sK)[i] = z;
      }
      __syncwarp();
      for (int r = lane; r < nb * BT; r += 32) {
        const int br = r >> 4;
        double* rowbase = sK + (br * (br + 1) / 2) * BE;      // block row br starts at slot br(br+1)/2
        if (r >= n) {
          rowbase[br * BE + b16_off(r & 15, r & 15)] = 1.0;
          sY[r] = 0.0;
          continue;
        }
        const int dof = sFree[r];
        const int jr = dof / DIM, ar = dof - jr * DIM;
        sY[r] = sF[dof];
        for (int p = sIncPtr[jr]; p < sIncPtr[jr + 1]; ++p) {
          const int e = sInc[p], m = e >> 1, end = e & 1;
          const int jb = sConn[2 * m + (end ^ 1)];
          const double k = sMk[m];
          const double ca = sMc[m * DIM + ar];
#pragma unroll
          for (int j = 0; j < DIM; ++j) {
            const double kp = __dmul_rn(k, __dmul_rn(ca, sMc[m * DIM + j]));   // truss.py:69-70: product first, then k
            const int fs = sD2F[jr * DIM + j];                                  // same joint: + block
            if (fs >= 0 && fs <= r) {
              double* q = rowbase + (fs >> 4) * BE + b16_off(r & 15, fs & 15);
              *q = __dadd_rn(*q, kp);
            }
            const int fo = sD2F[jb * DIM + j];                                  // other joint: - block
            if (fo >= 0 && fo <= r) {
              double* q = rowbase + (fo >> 4) * BE + b16_off(r & 15, fo & 15);
              *q = __dadd_rn(*q, -kp);
            }
          }
        }
      }
      __syncwarp();

      // ---- dense block Cholesky, left-looking by block columns; block (i, j) at slot i(i+1)/2 + j
      for (int c = 0; c < nb && !fail; ++c) {
        double* Dc = sK + (c * (c + 1) / 2 + c) * BE;
        {   // diagonal block: P = K(c,c) - sum_d L(c,d) L(c,d)^T, rhs t = f_c - sum_d L(c,d) y_d
          double acc[3][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
          double tp[2] = {0.0, 0.0};
          for (int d = 0; d < c; ++d) {
            const double* Bm = sK + (c * (c + 1) / 2 + d) * BE;
            double bf[2][4];
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) bf[h][ks] = Bm[fo(h * 4 + ks, lsw)];
            const double* yv = sY + d * BT;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const double y4 = yv[ks * 4 + qc];
              tp[0] = fma(bf[0][ks], y4, tp[0]);
              tp[1] = fma(bf[1][ks], y4, tp[1]);
            }
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              dmma(acc[0][0], acc[0][1], bf[0][ks], bf[0][ks]);
              dmma(acc[1][0], acc[1][1], bf[1][ks], bf[0][ks]);
              dmma(acc[2][0], acc[2][1], bf[1][ks], bf[1][ks]);
            }
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            tp[h] += __shfl_xor_sync(FULL, tp[h], 1);
            tp[h] += __shfl_xor_sync(FULL, tp[h], 2);
          }
          double2* p0 = reinterpret_cast<double2*>(Dc + cpair_off(0, 0, lane));
          double2* p1 = reinterpret_cast<double2*>(Dc + cpair_off(1, 0, lane));
          double2* p2 = reinterpret_cast<double2*>(Dc + cpair_off(1, 1, lane));
          double2 v0 = *p0, v1 = *p1, v2 = *p2;
          v0.x -= acc[0][0]; v0.y -= acc[0][1];
          v1.x -= acc[1][0]; v1.y -= acc[1][1];
          v2.x -= acc[2][0]; v2.y -= acc[2][1];
          *p0 = v0; *p1 = v1; *p2 = v2;
          if (qc == 0) {
            sT[qr] = sY[c * BT + qr] - tp[0];
            sT[8 + qr] = sY[c * BT + 8 + qr] - tp[1];
          }
        }
        __syncwarp();
        fail = factor_diag16(Dc, sCol, lane, c * BT);       // Dc now holds W_c = L(c,c)^{-1} (B-operand layout)
        __syncwarp();
        if (fail) break;   // uniform
        double wf[2][4];
#pragma unroll
        for (int nbp = 0; nbp < 2; ++nbp)
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) wf[nbp][ks] = Dc[fo(nbp * 4 + ks, lsw)];
        {   // y_c = W t
          double yp[2] = {0.0, 0.0};
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const double t4 = sT[ks * 4 + qc];
            yp[0] = fma(wf[0][ks], t4, yp[0]);
            yp[1] = fma(wf[1][ks], t4, yp[1]);
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            yp[h] += __shfl_xor_sync(FULL, yp[h], 1);
            yp[h] += __shfl_xor_sync(FULL, yp[h], 2);
          }
          __syncwarp();
          if (qc == 0) {
            sY[c * BT + qr] = yp[0];
            sY[c * BT + 8 + qr] = yp[1];
          }
        }
        // blocks below the diagonal: P = K(i,c) - sum_d L(i,d) L(c,d)^T, then L(i,c) = P W^T, in place
        for (int i = c + 1; i < nb; ++i) {
          double* blk = sK + (i * (i + 1) / 2 + c) * BE;
          double acc[2][2][2] = {};
          for (int d = 0; d < c; ++d) {
            const double* A = sK + (i * (i + 1) / 2 + d) * BE;
            const double* Bm = sK + (c * (c + 1) / 2 + d) * BE;
            double af[2][4], bf[2][4];
#pragma unroll
            for (int h = 0; h < 2; ++h)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                af[h][ks] = A[fo(h * 4 + ks, lsw)];
                bf[h][ks] = Bm[fo(h * 4 + ks, lsw)];
              }
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
#pragma unroll
              for (int mb = 0; mb < 2; ++mb)
#pragma unroll
                for (int nbp = 0; nbp < 2; ++nbp) dmma(acc[mb][nbp][0], acc[mb][nbp][1], af[mb][ks], bf[nbp][ks]);
          }
#pragma unroll
          for (int mb = 0; mb < 2; ++mb)
#pragma unroll
            for (int nbp = 0; nbp < 2; ++nbp) {
              double2* p = reinterpret_cast<double2*>(blk + cpair_off(mb, nbp, lane));
              double2 v = *p;
              v.x -= acc[mb][nbp][0];
              v.y -= acc[mb][nbp][1];
              *p = v;
            }
          __syncwarp();
          double a4[2][4];
#pragma unroll
          for (int mb = 0; mb < 2; ++mb)
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) a4[mb][ks] = blk[fo(mb * 4 + ks, lsw)];
          __syncwarp();
          double x[2][2][2] = {};
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
#pragma unroll
            for (int mb = 0; mb < 2; ++mb)
#pragma unroll
              for (int nbp = 0; nbp < 2; ++nbp)
                if (ks < 2 * nbp + 2) dmma(x[mb][nbp][0], x[mb][nbp][1], a4[mb][ks], wf[nbp][ks]);   // W is lower triangular
#pragma unroll
          for (int mb = 0; mb < 2; ++mb)
#pragma unroll
            for (int nbp = 0; nbp < 2; ++nbp)
              *reinterpret_cast<double2*>(blk + cpair_off(mb, nbp, lane)) = make_double2(x[mb][nbp][0], x[mb][nbp][1]);
        }
        __syncwarp();
      }

      if (!fail) {
        // ---- back substitution: u_c = W_c^T (y_c - sum_{i>c} L(i,c)^T u_i), in place in sY
        for (int c = nb - 1; c >= 0; --c) {
          double tp[4] = {0.0, 0.0, 0.0, 0.0};
          for (int i = c + 1; i < nb; ++i) {
            const double* blk = sK + (i * (i + 1) / 2 + c) * BE;
            const double* uv = sY + i * BT;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const double ur = uv[h * 8 + qr];
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) tp[ks] = fma(blk[fo(h * 4 + ks, lsw)], ur, tp[ks]);
            }
          }
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            tp[ks] += __shfl_xor_sync(FULL, tp[ks], 4);
            tp[ks] += __shfl_xor_sync(FULL, tp[ks], 8);
            tp[ks] += __shfl_xor_sync(FULL, tp[ks], 16);
          }
          if (qr == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) sT[ks * 4 + qc] = sY[c * BT + ks * 4 + qc] - tp[ks];
          }
          __syncwarp();
          const double* W = sK + (c * (c + 1) / 2 + c) * BE;
          double up[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const double rr = sT[h * 8 + qr];
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) up[ks] = fma(W[fo(h * 4 + ks, lsw)], rr, up[ks]);
          }
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            up[ks] += __shfl_xor_sync(FULL, up[ks], 4);
            up[ks] += __shfl_xor_sync(FULL, up[ks], 8);
            up[ks] += __shfl_xor_sync(FULL, up[ks], 16);
          }
          if (qr == 0) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) sY[c * BT + ks * 4 + qc] = up[ks];
          }
          __syncwarp();
        }
      }
      if (fail) status = fail;
    }

    // output locations
    double* u_out = a.u ? a.u + jo * DIM : nullptr;
    double* ext_out = a.ext ? a.ext + jo * DIM : nullptr;
    double* ax_out = a.axial ? a.axial + mo : nullptr;

    if (status != 0) {  // uniform: zero-filled outputs, never NaN
      for (int i = lane; i < N; i += 32) {
        if (u_out) u_out[i] = 0.0;
        if (ext_out) ext_out[i] = 0.0;
      }
      for (int m = lane; m < M; m += 32)
        if (ax_out) ax_out[m] = 0.0;
      if (lane == 0) {
        if (a.weight) a.weight[b] = 0.0;
        if (a.info) a.info[b] = status;
        if (a.fitness_mode) {
          if (a.fitness) a.fitness[b] = INFINITY;
          if (a.flags) { a.flags[2 * b] = 0; a.flags[2 * b + 1] = 0; }
        }
      }
      __syncwarp();
      continue;
    }

    // ---- expand to all DOFs (0 at supports), axial forces, reactions
    __syncwarp();
    for (int i = lane; i < N; i += 32) {
      const int fr = sD2F[i];
      const double v = fr >= 0 ? sY[fr] : 0.0;
      sU[i] = v;
      if (u_out) u_out[i] = v;
    }
    __syncwarp();
    double vs = 0.0, vd = 0.0;
    for (int m = lane; m < M; m += 32) {
      const int j0 = sConn[2 * m], j1 = sConn[2 * m + 1];
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < DIM; ++i) t = fma(sMc[m * DIM + i], sU[j1 * DIM + i] - sU[j0 * DIM + i], t);
      const double nm = sMk[m] * t;
      sAx[m] = nm;
      if (ax_out) ax_out[m] = nm;
      if (a.fitness_mode) {   // truss.py:429-433
        const double f = fabs(nm);
        if (!(f < TB_ZERO_EPS)) {
          const double sg = f / sArea[m];
          if (sg > a.allow_stress) vs += sg - a.allow_stress;
        }
      }
    }
    __syncwarp();
    if (ext_out) {
      for (int dof = lane; dof < N; dof += 32) {
        double e;
        if (sD2F[dof] >= 0) {
          e = sF[dof];
        } else {  // row of K times u, summed member by member in ascending id over the joint's incidence list
          const int J = dof / DIM, ax = dof - J * DIM;
          e = 0.0;
          for (int p = sIncPtr[J]; p < sIncPtr[J + 1]; ++p) {
            const int en = sInc[p], m = en >> 1;
            const double g = (en & 1) ? sMc[m * DIM + ax] : -sMc[m * DIM + ax];
            e = fma(g, sAx[m], e);
          }
        }
        ext_out[dof] = e;
      }
    }

    // ---- weight (+ GA fitness)
    const double w = warp_sum(wsum);
    if (lane == 0) {
      if (a.weight) a.weight[b] = w;
      if (a.info) a.info[b] = 0;
    }
    if (a.fitness_mode) {
      for (int j = lane; j < nJ; j += 32) {  // truss.py:447-451
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
      vs = warp_sum(vs);
      vd = warp_sum(vd);
      if (lane == 0) {
        const bool ok_s = fabs(vs) < TB_ZERO_EPS, ok_d = fabs(vd) < TB_ZERO_EPS;
        double fit = w;  // ga.py:146-148
        if (!ok_s) fit += vs / a.allow_stress * 1e5;
        if (!ok_d) fit += vd / a.allow_displace * 1e5;
        if (a.fitness) a.fitness[b] = fit;
        if (a.flags) { a.flags[2 * b] = ok_s; a.flags[2 * b + 1] = ok_d; }
      }
    }
    __syncwarp();  // shared arrays are reused by the next system
  }
}

}  // namespace

// Shared memory per system (bytes) of the warp-per-system kernel.
int tb_dense16_smem_bytes(int dim, int nJ, int M, int max_n) {
  const int nbm = max_n > 0 ? (max_n + 15) / 16 : 1;
  return d16_layout(dim, nJ, M, nbm).total * 8;
}

// Returns -1 when the batch does not fit this kernel (caller falls back to the CTA-per-truss kernel).
int tb_launch_dense16(const SmallArgs& a, int dim, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  const int nbm = a.max_n > 0 ? (a.max_n + 15) / 16 : 1;
  if (nbm > 10) return -1;
  const int per = d16_layout(dim, a.nJ, a.M, nbm).total * 8;
  if (per > 110 * 1024) return -1;             // fewer than two systems per SM: the CTA-per-truss kernel takes it (tb_small_fits)
  auto kern = (dim == 3) ? k_dense16<3> : k_dense16<2>;
  // Warps per CTA: whatever puts the most warps (= systems in flight) on an SM.  The kernel is latency-bound per warp, so
  // throughput follows the resident warps; shared memory per system decides (bar-72: 19.6 KB per warp -> 11 one-warp CTAs
  // per SM against 8 warps with four-warp CTAs).  Attribute / occupancy queries are cached per device, instantiation and
  // per-system size: they cost more than the launch.
  struct Choice { int per = -1, nwarp = 0, per_sm = 0, sms = 0; };
  static Choice cache[64][2];
  static std::mutex cache_mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return (int)cudaGetLastError();
  Choice ch;
  {
    std::lock_guard<std::mutex> lock(cache_mu);
    Choice& c = cache[dev & 63][dim - 2];
    if (c.per != per) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
      if (e != cudaSuccess) return (int)e;
      e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
      if (e != cudaSuccess) return (int)e;
      Choice best;
      for (int nw = 4; nw >= 1; --nw) {
        if ((size_t)per * nw > (size_t)227 * 1024) continue;
        int q = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, 32 * nw, (size_t)per * nw);
        if (e != cudaSuccess) return (int)e;
        if (q * nw > best.per_sm * best.nwarp) { best.nwarp = nw; best.per_sm = q; }
      }
      if (best.nwarp == 0) return -1;
      cudaDeviceGetAttribute(&best.sms, cudaDevAttrMultiProcessorCount, dev);
      best.per = per;
      c = best;
    }
    ch = c;
  }
  const int nwarp = ch.nwarp, smem = per * nwarp;
  const int per_sm = ch.per_sm, sms = ch.sms;
  long long grid = (long long)sms * per_sm;    // persistent: a multiple of the SM count
  const long long need = (a.batch + nwarp - 1) / nwarp;
  if (grid > need) grid = need;
  tb_prof_begin(TB_PROF_SMALL, st);
  kern<<<(unsigned)grid, 32 * nwarp, smem, st>>>(a, nbm, nwarp);
  tb_prof_end(TB_PROF_SMALL, st);
  tb_count_launch();
  return (int)cudaGetLastError();
}
