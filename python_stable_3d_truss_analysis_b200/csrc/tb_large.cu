// Blocked global-memory path for systems that do not fit the fused shared-memory kernel
// (bar-942: n = 696; cube 12^3: n = 6084).  Four kernels per batch:
//
//   k_geom      member length / EA/L / cosines / weight terms      Member.length,k,cosines  truss.py:19,56-63
//   k_assemble  K_ff tiles through the plan's scatter map          Truss.GetKMatrix + mask  truss.py:307-316,343
//   k_chol      tiled left-looking Cholesky, DMMA updates,         np.linalg.solve          truss.py:343
//               fused forward substitution, back substitution
//   k_recover   displacements, axial forces, reactions, weight,    truss.py:344-361,166-168; ga.py:139-149
//               optional GA fitness
//
// Storage: only the lower triangle, as 64x64 tiles, tile (i,j) at index i(i+1)/2+j.  Inside a tile
// elements are kept "fragment-major" (tb_tile_off): the 8x4 operand fragment of one FP64
// mma.m8n8k4 is 32 consecutive doubles, so a warp's operand load is one conflict-free 256 B
// shared-memory read, and a 64-row x 32-k half tile is one contiguous 16 KB chunk in HBM.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "tb_common.cuh"
#include "tb_ts.cuh"

#ifdef TB_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[16];
#define PH_DECL long long _ph_t = clock64(); unsigned long long _ph_acc[16] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0};
#define PH(i) { long long _n = clock64(); _ph_acc[i] += (unsigned long long)(_n - _ph_t); _ph_t = _n; }
#define PH_FLUSH if (threadIdx.x == 0) { for (int _i = 0; _i < 16; ++_i) atomicAdd(&g_phase_cycles[_i], _ph_acc[_i]); }
extern "C" int tb_phase_read(unsigned long long* out) {
  cudaMemcpyFromSymbol(out, g_phase_cycles, sizeof(unsigned long long) * 16);
  unsigned long long z[16] = {0};
  cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z));
  return 0;
}
#else
#define PH_DECL
#define PH(i) {}
#define PH_FLUSH
#endif

namespace {

constexpr int T = TB_TILE;          // 64
constexpr int HALF = T * 32;        // doubles in a 64 x 32 half tile (16 KB)
constexpr int CH_THREADS = 256;

// ------------------------------------------------------------------------------------------
// k_geom
// ------------------------------------------------------------------------------------------
template <int DIM>
__global__ void k_geom(const LargeArgs a) {
  const int64_t total = (int64_t)a.batch * a.M;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(idx / a.M), m = (int)(idx - (int64_t)b * a.M);
    const double* xyz = a.xyz + b * a.xyz_stride;
    double ar, e, rho;
    bool ok = true;
    if (a.gene) {
      const int g = a.gene[b * a.gene_stride + m];
      if ((unsigned)g < (unsigned)a.n_type) {
        ar = a.type_table[3 * g];
        e = a.type_table[3 * g + 1];
        rho = a.type_table[3 * g + 2];
      } else {
        ok = false;
        ar = e = rho = 0.0;
      }
    } else {
      const double* t = a.aed + b * a.aed_stride + 3 * (int64_t)m;
      ar = t[0];
      e = t[1];
      rho = t[2];
    }
    const int j0 = a.conn[2 * m], j1 = a.conn[2 * m + 1];
    double dx[DIM], c[DIM];
#pragma unroll
    for (int i = 0; i < DIM; ++i) dx[i] = __dsub_rn(xyz[j1 * DIM + i], xyz[j0 * DIM + i]);
    double l2 = __dmul_rn(dx[0], dx[0]);
#pragma unroll
    for (int i = 1; i < DIM; ++i) l2 = __dadd_rn(l2, __dmul_rn(dx[i], dx[i]));
    const double len = __dsqrt_rn(l2);
    double k = 0.0;
#pragma unroll
    for (int i = 0; i < DIM; ++i) c[i] = 0.0;
    if (!ok) {
      atomicMin(&a.status[b], TB_INFO_BAD_INDEX);
    } else if (!(len > 0.0)) {
      atomicMin(&a.status[b], TB_INFO_ZERO_LENGTH);
    } else {
      const TbDivisor dv(len);                  // (one reciprocal for the four quotients of the member)
      k = dv.div(__dmul_rn(e, ar));
#pragma unroll
      for (int i = 0; i < DIM; ++i) c[i] = dv.div(dx[i]);
    }
    a.mk[idx] = k;
#pragma unroll
    for (int i = 0; i < DIM; ++i) a.mc[idx * DIM + i] = c[i];
    a.mw[idx] = __dmul_rn(__dmul_rn(ar, len), rho);
    {   // k * (c_i c_j) for i <= j: product first, then the scale, exactly as truss.py:69-70 / 80-81
      constexpr int NV = DIM * (DIM + 1) / 2;
      double* o = a.mkc + idx * NV;
      int t = 0;
#pragma unroll
      for (int i = 0; i < DIM; ++i)
#pragma unroll
        for (int j = i; j < DIM; ++j) o[t++] = __dmul_rn(k, __dmul_rn(c[i], c[j]));
    }
  }
}

// K_ff non-zeros of one system per CTA (the member products it gathers stay in L1), one thread per
// structural non-zero, summed in ascending member order (truss.py:310) and written in the plan's
// tile-grouped order so the factorisation scatters a tile's entries with coalesced reads.
__global__ void __launch_bounds__(256) k_kval(const LargeArgs a) {
  const int nv = a.dim * (a.dim + 1) / 2;
  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const double* mkc = a.mkc + (int64_t)b * a.M * nv;
    double* kv = a.kv + (int64_t)b * a.nnz;
    for (int q = threadIdx.x; q < a.nnz; q += 256) {
      const int f = a.q_first[q];
      if (f < 0) continue;                                          // several members contribute: second loop
      const double t0 = mkc[(f >> 4) * nv + (f & 7)];
      kv[q] = __dadd_rn(0.0, (f & 8) ? -t0 : t0);
    }
    for (int i = threadIdx.x; i < a.n_multi; i += 256) {             // same-joint entries: ascending member order
      const int q = a.q_multi[i];
      double v = 0.0;
      for (int p = a.q_ptr[q]; p < a.q_ptr[q + 1]; ++p) {
        const int pk = a.q_pack[p];
        const double t = mkc[(pk >> 4) * nv + (pk & 7)];
        v = __dadd_rn(v, (pk & 8) ? -t : t);                       // truss.py:71-76 signs, :314 accumulation
      }
      kv[q] = v;
    }
  }
}

// Fused k_geom + k_kval for systems whose member products fit in shared memory (M * d(d+1)/2 doubles): one CTA per
// system computes the products k (c_i c_j) of every member into shared memory and gathers the K_ff non-zeros from there;
// nothing but the K values goes to HBM (k_recover recomputes the member geometry it needs).
template <int DIM>
__global__ void __launch_bounds__(256) k_prep(const LargeArgs a) {
  extern __shared__ __align__(16) double sMkc[];
  constexpr int NV = DIM * (DIM + 1) / 2;
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    const double* xyz = a.xyz + b * a.xyz_stride;
    int flag = 0;
    if (tid == 0) a.status[b] = 0;             // no separate initialisation kernel on this path
    __syncthreads();
    // two members per thread and pass: the connectivity / property loads of both, then the joint positions of both
    // (which wait on the connectivity), then the arithmetic -- half as many exposed load latencies
    for (int mbase = tid; mbase < a.M; mbase += 2 * 256) {
      double ar[2], e[2], x0[2][DIM], x1[2][DIM];
      int j0[2], j1[2];
      bool ok[2], live[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int m = mbase + 256 * u;
        live[u] = m < a.M;
        ok[u] = true;
        ar[u] = e[u] = 0.0;
        j0[u] = j1[u] = 0;
        if (!live[u]) continue;
        if (a.gene) {
          const int g = a.gene[b * a.gene_stride + m];
          if ((unsigned)g < (unsigned)a.n_type) {
            ar[u] = a.type_table[3 * g];
            e[u] = a.type_table[3 * g + 1];
          } else {
            ok[u] = false;
          }
        } else {
          const double* t = a.aed + b * a.aed_stride + 3 * (int64_t)m;
          ar[u] = t[0];
          e[u] = t[1];
        }
        j0[u] = a.conn[2 * m];
        j1[u] = a.conn[2 * m + 1];
      }
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int i = 0; i < DIM; ++i) {
          x0[u][i] = live[u] ? xyz[j0[u] * DIM + i] : 0.0;
          x1[u][i] = live[u] ? xyz[j1[u] * DIM + i] : 0.0;
        }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        if (!live[u]) continue;
        const int m = mbase + 256 * u;
        double dx[DIM], c[DIM];
#pragma unroll
        for (int i = 0; i < DIM; ++i) dx[i] = __dsub_rn(x1[u][i], x0[u][i]);
        double l2 = __dmul_rn(dx[0], dx[0]);
#pragma unroll
        for (int i = 1; i < DIM; ++i) l2 = __dadd_rn(l2, __dmul_rn(dx[i], dx[i]));
        const double len = __dsqrt_rn(l2);
        double k = 0.0;
#pragma unroll
        for (int i = 0; i < DIM; ++i) c[i] = 0.0;
        if (!ok[u]) {
          flag = min(flag, TB_INFO_BAD_INDEX);
        } else if (!(len > 0.0)) {
          flag = min(flag, TB_INFO_ZERO_LENGTH);
        } else {
          const TbDivisor dv(len);                  // (one reciprocal for the four quotients of the member)
          k = dv.div(__dmul_rn(e[u], ar[u]));
#pragma unroll
          for (int i = 0; i < DIM; ++i) c[i] = dv.div(dx[i]);
        }
        double* o = sMkc + m * NV;
        int t = 0;
#pragma unroll
        for (int i = 0; i < DIM; ++i)
#pragma unroll
          for (int j = i; j < DIM; ++j) o[t++] = __dmul_rn(k, __dmul_rn(c[i], c[j]));   // truss.py:69-70 / 80-81
      }
    }
    if (flag) atomicMin(&a.status[b], flag);
    __syncthreads();
    double* kv = a.kv + (int64_t)b * a.nnz;
    // the map loads of four entries are issued together: one exposed L2 latency per four entries instead of per entry
    for (int q = tid; q < a.nnz; q += 4 * 256) {
      int f[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) f[u] = q + 256 * u < a.nnz ? a.q_first[q + 256 * u] : -1;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (f[u] < 0) continue;                                     // several members contribute: second loop
        const double t0 = sMkc[(f[u] >> 4) * NV + (f[u] & 7)];
        kv[q + 256 * u] = __dadd_rn(0.0, (f[u] & 8) ? -t0 : t0);
      }
    }
    for (int i = tid; i < a.n_multi; i += 256) {             // same-joint entries: ascending member order
      int q, p0, p1;
      if (a.q_multi4) {
        const int4 mr = __ldg(a.q_multi4 + i);
        q = mr.x; p0 = mr.y; p1 = mr.z;
      } else {
        q = a.q_multi[i];
        p0 = a.q_ptr[q]; p1 = a.q_ptr[q + 1];
      }
      double v = 0.0;
      for (int p = p0; p < p1; p += 8) {                     // eight contributions' map loads in flight, summed in order
        int pk[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) pk[u] = p + u < p1 ? a.q_pack[p + u] : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (pk[u] < 0) continue;
          const double t = sMkc[(pk[u] >> 4) * NV + (pk[u] & 7)];
          v = __dadd_rn(v, (pk[u] & 8) ? -t : t);                  // truss.py:71-76 signs, :314 accumulation
        }
      }
      kv[q] = v;
    }
    __syncthreads();
  }
}

__global__ void k_init_status(int32_t* status, int batch, int value) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < batch; i += gridDim.x * blockDim.x) status[i] = value;
}

// ------------------------------------------------------------------------------------------
// k_assemble: one CTA builds one 64x64 tile of one system in shared memory (zero fill, then one
// thread per structural non-zero sums its member contributions in ascending member order) and
// streams it out as one contiguous 32 KB block.  Also gathers the reduced load vector.
// ------------------------------------------------------------------------------------------
template <int DIM>
__global__ void __launch_bounds__(256) k_assemble(const LargeArgs a) {
  __shared__ __align__(16) double sT[TB_TILE_ELEMS];
  const int tid = threadIdx.x;
  const int64_t ntiles = (int64_t)a.nt * (a.nt + 1) / 2;
  const int64_t work = ntiles * a.batch;
  for (int64_t w = blockIdx.x; w < work; w += gridDim.x) {
    const int b = (int)(w / ntiles);
    const int64_t t = w - (int64_t)b * ntiles;
    // decode t -> (ti, tj)
    int ti = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
    while ((int64_t)(ti + 1) * (ti + 2) / 2 <= t) ++ti;
    while ((int64_t)ti * (ti + 1) / 2 > t) --ti;
    const int tj = (int)(t - (int64_t)ti * (ti + 1) / 2);

    for (int i = tid; i < TB_TILE_ELEMS; i += 256) sT[i] = 0.0;
    __syncthreads();
    const double* mk = a.mk + (int64_t)b * a.M;
    const double* mc = a.mc + (int64_t)b * a.M * DIM;
    const int64_t e0 = a.tile_ent_ptr[t], e1 = a.tile_ent_ptr[t + 1];
    for (int64_t q = e0 + tid; q < e1; q += 256) {
      const int e = a.tile_ent[q];
      const int r = a.ent_row[e], c = a.ent_col[e];
      double v = 0.0;
      for (int64_t p = a.ent_ptr[e]; p < a.ent_ptr[e + 1]; ++p) {
        const int m = a.ctr_member[p], loc = a.ctr_local[p];
        const int la = loc / (2 * DIM), lb = loc - la * (2 * DIM);
        const int A = la / DIM, i = la - A * DIM, B = lb / DIM, j = lb - B * DIM;
        double pr = __dmul_rn(mc[m * DIM + i], mc[m * DIM + j]);   // truss.py:69,80
        if (A != B) pr = -pr;
        v = __dadd_rn(v, __dmul_rn(mk[m], pr));                    // truss.py:70,314
      }
      sT[tb_tile_off(r - ti * T, c - tj * T)] = v;
    }
    if (ti == tj) {  // identity on the padded part of the diagonal
      for (int r = tid; r < T; r += 256)
        if (ti * T + r >= a.n) sT[tb_tile_off(r, r)] = 1.0;
    }
    __syncthreads();
    double2* dst = reinterpret_cast<double2*>(a.L + ((int64_t)b * ntiles + t) * TB_TILE_ELEMS);
    const double2* src = reinterpret_cast<const double2*>(sT);
    for (int i = tid; i < TB_TILE_ELEMS / 2; i += 256) dst[i] = src[i];
    // reduced load vector (rows of this tile row, written once by the diagonal tile's CTA)
    if (ti == tj) {
      const double* f = a.force + b * a.force_stride;
      for (int r = tid; r < T; r += 256) {
        const int fr = ti * T + r;
        a.y[(int64_t)b * a.n_pad + fr] = fr < a.n ? f[a.free_idx[fr]] : 0.0;
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// k_chol
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// shared-memory carve of k_chol (doubles)
constexpr int KCH = 16;                                // k-depth of one pipeline stage
constexpr int CHUNK = T * KCH;                         // doubles in a 64-row x 16-k chunk (8 KB)
constexpr int STAGE_DOUBLES = 2 * CHUNK + KCH;         // A chunk, B chunk, 16 y values
constexpr int SM_STAGE = 2 * STAGE_DOUBLES;            // two stages (aliased: C staging tile, scratch)
constexpr int SCR_LD = 67;                             // back-substitution scratch: column-major 64 x 64
constexpr int SM_LJJ = TB_TILE_ELEMS;                  // L(j,j), fragment-major
constexpr int SM_WD = 4 * 256;                         // the four 16x16 inverse diagonal blocks of L(j,j)
constexpr int SM_MISC = 4 * T + 64;                    // rhs acc, u block, y block, rhs vector, diag16, flag
constexpr int CHOL_SMEM_BYTES = (SM_STAGE + SM_LJJ + SM_WD + SM_MISC) * 8;
static_assert(SCR_LD * T <= SM_STAGE + SM_LJJ, "back-substitution scratch must fit in stage buffers + L(j,j)");
static_assert(TB_TILE_ELEMS <= SM_STAGE, "C staging tile must fit in the stage buffers");

// offset of the 32-double operand fragment (8-row block `blk`, k-slab kS in 0..15) inside a tile
__device__ __forceinline__ int frag_off(int blk, int kS) { return ((((kS >> 3) << 3) + blk) << 8) + ((kS & 7) << 5); }
// offset of this lane's accumulator pair (row 8*mb + lane/4, cols 8*nb + 2*(lane%4) + {0,1})
__device__ __forceinline__ int cfrag_off(int mb, int nb, int lane) {
  return frag_off(mb, 2 * nb + ((lane & 3) >> 1)) + ((lane >> 2) << 2) + ((lane & 1) << 1);
}

struct Frag {
  double c[2][4][2];  // [m-block][n-block][2]
};

// TMA side of the tile pipeline: one elected thread moves a stage with bulk copies (cp.async.bulk: the copy engine writes
// shared memory and signals an mbarrier with the byte count; no thread touches the data on its way in)
__device__ __forceinline__ unsigned ch_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ch_mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ch_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void ch_mbar_expect_tx(uint64_t* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ch_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ch_mbar_wait(uint64_t* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "CH_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra CH_DONE;\n"
      "bra CH_WAIT;\n"
      "CH_DONE:\n"
      "}\n" ::"r"(ch_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void ch_bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ch_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(ch_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void ch_fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// acc += sum over the nk block columns k in klist of L(ti,k) * L(tj,k)^T, streamed as 64-row x 16-k chunks through a two-stage
// TMA pipeline: a chunk of a fragment-major tile is eight contiguous 1 KB pieces (one per 8-row block), so one elected
// thread issues 8 (+8 for the second operand, +1 for y) bulk copies per stage onto the stage's mbarrier and everybody waits
// on its phase.  `phase` (bit s: parity the next wait on stage s expects) lives across calls.  When with_y, also accumulates
// rows of A times the forward solution y.
__device__ __forceinline__ void gemm_stream(const double* __restrict__ Lsys, const double* __restrict__ ysys, int ti,
                                            int tj, const int32_t* __restrict__ klist, int nk, bool with_y,
                                            double* sStage, uint64_t* sBar, unsigned& phase, Frag& acc, double (&accy)[2], int tid) {
  const int lane = tid & 31, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
  const bool same = (ti == tj);
  const int S = 4 * nk;
  if (S == 0) return;
  // The stage buffers alias tiles written with ordinary stores, and the tiles of L in global memory were written with
  // ordinary stores as well: order them before the copy engine's accesses (async proxy)
  ch_fence_proxy_async();
  __syncthreads();
  int kt = 0;
  auto issue = [&](int s) {                      // (thread 0 only)
    const int qd = s & 3;
    if (qd == 0) kt = __ldg(klist + (s >> 2));   // stages are issued in order: one list read per block column
    double* buf = sStage + (s & 1) * STAGE_DOUBLES;
    uint64_t* bar = sBar + (s & 1);
    const int64_t tbase = ((qd >> 1) << 11) + ((qd & 1) << 7);   // k-half offset + slab offset inside the tile
    const double* ga = Lsys + tb_tile_index(ti, kt) * TB_TILE_ELEMS + tbase;
    const double* gb = Lsys + tb_tile_index(tj, kt) * TB_TILE_ELEMS + tbase;
    ch_mbar_expect_tx(bar, (unsigned)((same ? CHUNK : 2 * CHUNK) + (with_y ? KCH : 0)) * 8u);
#pragma unroll
    for (int rb = 0; rb < 8; ++rb) {             // row block stride is 8 slabs (256 doubles) in the tile, 4 slabs in the chunk
      ch_bulk_g2s(buf + rb * 128, ga + rb * 256, 1024u, bar);
      if (!same) ch_bulk_g2s(buf + CHUNK + rb * 128, gb + rb * 256, 1024u, bar);
    }
    if (with_y) ch_bulk_g2s(buf + 2 * CHUNK, ysys + kt * T + qd * KCH, (unsigned)KCH * 8u, bar);
  };
  if (tid == 0) issue(0);
  for (int s = 0; s < S; ++s) {
    if (s + 1 < S && tid == 0) issue(s + 1);     // (its buffer was released by the barrier that ended stage s - 1)
    ch_mbar_wait(sBar + (s & 1), (phase >> (s & 1)) & 1u);
    phase ^= 1u << (s & 1);
    const double* bufA = sStage + (s & 1) * STAGE_DOUBLES;
    const double* bufB = same ? bufA : bufA + CHUNK;
    const double* bufY = bufA + 2 * CHUNK;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      double af[2], bf[4];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) af[mb] = bufA[(((2 * wm + mb) << 2) + ks) * 32 + lane];
#pragma unroll
      for (int q = 0; q < 4; ++q) bf[q] = bufB[(((4 * wn + q) << 2) + ks) * 32 + lane];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (!same || 4 * wn + q <= 2 * wm + mb)   // diagonal tile: only blocks on/below the diagonal (warp-uniform)
            dmma(acc.c[mb][q][0], acc.c[mb][q][1], af[mb], bf[q]);
      if (with_y && wn == 0) {
        const double yv = bufY[ks * 4 + (lane & 3)];
        accy[0] = fma(af[0], yv, accy[0]);
        accy[1] = fma(af[1], yv, accy[1]);
      }
    }
    __syncthreads();
  }
}

// FUSED: K_ff tiles are assembled straight into shared memory from the scatter map when the
// factorisation first touches them (K never exists in HBM); otherwise they are read from the
// tile storage k_assemble filled.
//
// Per block column j:  (1) diagonal tile: C = A(j,j) - sum_k L(j,k) L(j,k)^T by DMMA, then factor it
// in shared memory, left-looking over four 16-column sub-panels (DMMA updates; the 16x16 diagonal
// blocks and their inverses by one warp); (2) every tile below: C = A(i,j) - sum_k L(i,k) L(j,k)^T,
// then X L(j,j)^T = C solved per 8-row block entirely inside one warp using the 16x16 inverses.
template <bool FUSED>
__global__ void __launch_bounds__(CH_THREADS, 3) k_chol(const LargeArgs a) {
  extern __shared__ __align__(16) double sm[];
  double* sStage = sm;                 // stage buffers | C staging tile | small scratches
  double* sScr = sm;                   // alias (back substitution)
  double* sC = sm;                     // alias (panel tiles)
  double* sLjj = sm + SM_STAGE;
  double* sWd = sLjj + SM_LJJ;
  double* sRhs = sWd + SM_WD;          // [64] L(j,:) y accumulations
  double* sUb = sRhs + T;              // [64] one block of u during back substitution
  double* sY = sUb + T;                // [64] y_j
  double* sRv = sY + T;                // [64] rhs of the block
  double* sDiag16 = sRv + T;           // [16]
  double* sT16 = sDiag16 + 16;         // [32]
  int* sFlag = (int*)(sT16 + 32);
  uint64_t* sBar = reinterpret_cast<uint64_t*>(sT16 + 34);   // two stage mbarriers of the tile pipeline

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, wm = warp >> 1, wn = warp & 1;
  const int nt = a.nt;
  const int64_t ntiles = (int64_t)nt * (nt + 1) / 2;
  if (tid == 0) {
    ch_mbar_init(&sBar[0], 1);
    ch_mbar_init(&sBar[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  unsigned phase = 0;                  // bit s: parity the next wait on stage s expects
  __syncthreads();

  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    double* Lsys = a.L + (int64_t)b * ntiles * TB_TILE_ELEMS;
    double* ysys = a.y + (int64_t)b * a.n_pad;
    const double* kvs = a.kv + (int64_t)b * a.nnz;
    double* wds = a.wd + (int64_t)b * nt * 1024;
    int64_t resident = -1;   // tile of L currently held in sC (fragment-major), if any
    const double* fsys = a.force + b * a.force_stride;
    if (a.status[b] != 0) continue;  // input problem flagged by k_geom (uniform per CTA)
    int fail = 0;
    if (tid == 0) *sFlag = 0;
    PH_DECL

    for (int j = 0; j < nt && !fail; ++j) {
      // ================= diagonal tile: C = A(j,j) - sum_k L(j,k) L(j,k)^T =================
      Frag acc;
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc.c[mb][q][0] = acc.c[mb][q][1] = 0.0;
      double accy[2] = {0.0, 0.0};
      {
        const int64_t t = tb_tile_index(j, j);
        const int np = a.prod_ptr[t + 1] - a.prod_ptr[t];
        const int32_t* kl = a.prod_k + a.prod_ptr[t];
        if (np == 1 && resident == tb_tile_index(j, __ldg(kl))) {
          // block-tridiagonal case: the only tile this update needs is the one the previous block
          // column just left in shared memory -- no trip through HBM/L2
#pragma unroll 4
          for (int kS = 0; kS < 16; ++kS) {
            double af[2], bf[4];
#pragma unroll
            for (int mb = 0; mb < 2; ++mb) af[mb] = sC[frag_off(2 * wm + mb, kS) + lane];
#pragma unroll
            for (int q = 0; q < 4; ++q) bf[q] = sC[frag_off(4 * wn + q, kS) + lane];
#pragma unroll
            for (int mb = 0; mb < 2; ++mb)
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (4 * wn + q <= 2 * wm + mb) dmma(acc.c[mb][q][0], acc.c[mb][q][1], af[mb], bf[q]);
            if (wn == 0) {
              const double yv = sY[kS * 4 + (lane & 3)];   // y of the previous block column
              accy[0] = fma(af[0], yv, accy[0]);
              accy[1] = fma(af[1], yv, accy[1]);
            }
          }
        } else {
          gemm_stream(Lsys, ysys, j, j, kl, np, true, sStage, sBar, phase, acc, accy, tid);
          resident = -1;
        }
      }
      PH(0)
      if (wn == 0) {  // rows of L(j,0:j) times y(0:j): reduce over the quad
#pragma unroll
        for (int mb = 0; mb < 2; ++mb) {
          double v = accy[mb];
          v += __shfl_xor_sync(0xffffffffu, v, 1);
          v += __shfl_xor_sync(0xffffffffu, v, 2);
          if ((lane & 3) == 0) sRhs[(2 * wm + mb) * 8 + (lane >> 2)] = v;
        }
      }
      {
        const double* At = Lsys + tb_tile_index(j, j) * TB_TILE_ELEMS;
#pragma unroll
        for (int mb = 0; mb < 2; ++mb)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int off = cfrag_off(2 * wm + mb, 4 * wn + q, lane);
            double2 av = make_double2(0.0, 0.0);
            if (!FUSED) av = *reinterpret_cast<const double2*>(At + off);
            *reinterpret_cast<double2*>(sLjj + off) = make_double2(av.x - acc.c[mb][q][0], av.y - acc.c[mb][q][1]);
          }
      }
      __syncthreads();
      if (tid < T) {
        const int r = tid, row = j * T + r;
        if (FUSED) {
          sRv[r] = (row < a.n ? fsys[a.free_idx[row]] : 0.0) - sRhs[r];
          if (row >= a.n) sLjj[tb_tile_off(r, r)] += 1.0;  // identity on the padded diagonal
        } else {
          sRv[r] = ysys[row] - sRhs[r];
        }
      }
      if (FUSED) {  // scatter-map entries of tile (j,j): one thread per structural non-zero
        const int64_t t = tb_tile_index(j, j);
        for (int64_t q = a.tile_ent_ptr[t] + tid; q < a.tile_ent_ptr[t + 1]; q += CH_THREADS)
          sLjj[a.tile_pos[q]] += kvs[q];
      }

      // ---- factor the tile in place: four 16-column sub-panels, left-looking
      for (int sb = 0; sb < 4; ++sb) {
        __syncthreads();
        PH(1)
        if (sb > 0 && warp >= 2 * sb) {  // P(mb, sub-panel) -= L(mb, 0:16sb) L(sub-panel rows, 0:16sb)^T
          double c2[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
          for (int kS = 0; kS < 4 * sb; ++kS) {
            const double av = sLjj[frag_off(warp, kS) + lane];
#pragma unroll
            for (int nbp = 0; nbp < 2; ++nbp) dmma(c2[nbp][0], c2[nbp][1], av, sLjj[frag_off(2 * sb + nbp, kS) + lane]);
          }
#pragma unroll
          for (int nbp = 0; nbp < 2; ++nbp) {
            double2* pv = reinterpret_cast<double2*>(sLjj + cfrag_off(warp, 2 * sb + nbp, lane));
            double2 v = *pv;
            v.x -= c2[nbp][0];
            v.y -= c2[nbp][1];
            *pv = v;
          }
        }
        __syncthreads();
        PH(2)
        if (warp == 0) {
          // 16x16 diagonal block, right-looking, in registers: lanes 0-15 hold the rows of the block,
          // lanes 16-31 the rows of Z = L^{-T} (identity to start with).  The pivot chain is kept
          // short: the lane that owns row k+1 forms its next pivot from its own registers
          // (d' = a - l*l), one shuffle broadcasts it and the rsqrt for column k+1 is issued before
          // the trailing update of column k.  The eliminated column reaches the other lanes through
          // a double-buffered 16-entry shared array (broadcast reads), not shuffles.
          // (A rolled variant with shifting registers and a shared-memory variant were measured
          // 2-3x slower: tools/scratch/base.cu.)
          const int base = 16 * sb, r = lane & 15;
          const int rowpart = (((base + r) >> 3) << 8) + (((base + r) & 7) << 2);
          const int colpart = ((sb >> 1) << 11) + (((4 * sb) & 7) << 5);
          double row[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const double v = sLjj[rowpart + colpart + ((c >> 2) << 5) + (c & 3)];
            row[c] = lane < 16 ? (c <= r ? v : 0.0) : (c == r ? 1.0 : 0.0);
          }
          PH(11)
          int bad = 0;
          double d = __shfl_sync(0xffffffffu, row[0], 0);
          if (!(d > 0.0)) bad = j * T + base + 1;
          double rinv = rsqrt(bad ? 1.0 : d);
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            const double lk = row[k] * rinv;                       // lane k: d * rsqrt(d) = sqrt(d)
            row[k] = lk;
            double rinv_next = 0.0;
            if (k < 15) {
              const double dn = __shfl_sync(0xffffffffu, fma(-lk, lk, row[k + 1]), k + 1);
              if (!(dn > 0.0) && !bad) bad = j * T + base + k + 2;  // same value in every lane
              rinv_next = rsqrt(bad ? 1.0 : dn);
            }
            double* col = sT16 + ((k & 1) << 4);
            if (lane < 16) col[lane] = lk;
            __syncwarp();
#pragma unroll
            for (int c = k + 1; c < 16; ++c) row[c] = fma(-lk, col[c], row[c]);
            rinv = rinv_next;
          }
          PH(12)
          if (bad) {
            if (lane == 0) *sFlag = bad;
          } else if (lane < 16) {  // L back into the tile (upper part of the block zeroed)
#pragma unroll
            for (int c = 0; c < 16; ++c) sLjj[rowpart + colpart + ((c >> 2) << 5) + (c & 3)] = (c <= r) ? row[c] : 0.0;
          } else {  // W = L^{-1} as a DMMA B operand: W[c'][kk] = Z[kk][c'] for kk <= c' (this lane: kk = r)
#pragma unroll
            for (int cp = 0; cp < 16; ++cp)
              sWd[sb * 256 + ((((cp >> 3) << 2) + (r >> 2)) << 5) + ((cp & 7) << 2) + (r & 3)] = (cp >= r) ? row[cp] : 0.0;
          }
        }
        __syncthreads();
        PH(3)
        fail = *sFlag;
        if (fail) break;  // uniform
        if (warp >= 2 * sb + 2) {  // rows below the block: X = P W^T, in place
          double a4[4];
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) a4[ks] = sLjj[frag_off(warp, 4 * sb + ks) + lane];
          __syncwarp();
#pragma unroll
          for (int nbp = 0; nbp < 2; ++nbp) {
            double x0 = 0.0, x1 = 0.0;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) dmma(x0, x1, a4[ks], sWd[sb * 256 + (nbp * 4 + ks) * 32 + lane]);
            *reinterpret_cast<double2*>(sLjj + cfrag_off(warp, 2 * sb + nbp, lane)) = make_double2(x0, x1);
          }
        }
      }
      if (fail) break;  // uniform
      __syncthreads();
      PH(4)

      // ---- publish L(j,j) (strictly-upper part zeroed) and solve L(j,j) y_j = rhs with the 16x16 inverses
      {
        double* Lt = Lsys + tb_tile_index(j, j) * TB_TILE_ELEMS;
#pragma unroll 4
        for (int q = 0; q < 16; ++q) {
          const int idx = tid + q * 256;
          const int l = idx & 31, slot = idx >> 5;
          const int ks = slot & 7, rb = (slot >> 3) & 7, h = slot >> 6;
          const int r = rb * 8 + (l >> 2), c = h * 32 + ks * 4 + (l & 3);
          Lt[idx] = (c <= r) ? sLjj[idx] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) wds[j * 1024 + tid + q * 256] = sWd[tid + q * 256];
      }
      if (warp == 0) {
        const int c = lane & 15, hh = lane >> 4;
        for (int sb = 0; sb < 4; ++sb) {
          double t = 0.0;
          for (int kk = hh; kk < 16 * sb; kk += 2) t = fma(sLjj[tb_tile_off(16 * sb + c, kk)], sY[kk], t);
          t += __shfl_xor_sync(0xffffffffu, t, 16);
          if (lane < 16) sT16[c] = sRv[16 * sb + c] - t;
          __syncwarp();
          double yv = 0.0;
          for (int cc = hh; cc <= c; cc += 2)
            yv = fma(sWd[sb * 256 + (((c >> 3) * 4 + (cc >> 2)) << 5) + ((c & 7) << 2) + (cc & 3)], sT16[cc], yv);
          yv += __shfl_xor_sync(0xffffffffu, yv, 16);
          if (lane < 16) {
            sY[16 * sb + c] = yv;
            ysys[j * T + 16 * sb + c] = yv;
          }
          __syncwarp();
        }
      }
      __syncthreads();
      PH(5)

      // ================= panel tiles below the diagonal =================
      for (int i = nt - 1; i > j; --i) {   // descending: the tile the next diagonal update needs first is left in sC
        const int64_t tij = tb_tile_index(i, j);
        if (!a.tile_nz[tij]) continue;  // structurally zero tile of L: never touched (uniform)
#pragma unroll
        for (int mb = 0; mb < 2; ++mb)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc.c[mb][q][0] = acc.c[mb][q][1] = 0.0;
        gemm_stream(Lsys, ysys, i, j, a.prod_k + a.prod_ptr[tij], a.prod_ptr[tij + 1] - a.prod_ptr[tij], false, sStage,
                    sBar, phase, acc, accy, tid);
        PH(6)
        double* Xt = Lsys + tb_tile_index(i, j) * TB_TILE_ELEMS;
        // C = A(i,j) - acc  -> shared (fragment-major)
#pragma unroll
        for (int mb = 0; mb < 2; ++mb)
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int off = cfrag_off(2 * wm + mb, 4 * wn + q, lane);
            double2 av = make_double2(0.0, 0.0);
            if (!FUSED) av = *reinterpret_cast<const double2*>(Xt + off);
            *reinterpret_cast<double2*>(sC + off) = make_double2(av.x - acc.c[mb][q][0], av.y - acc.c[mb][q][1]);
          }
        if (FUSED) {
          const int64_t t = tb_tile_index(i, j);
          const int64_t e0 = a.tile_ent_ptr[t], e1 = a.tile_ent_ptr[t + 1];
          if (e1 > e0) {  // uniform
            __syncthreads();
            for (int64_t q = e0 + tid; q < e1; q += CH_THREADS) sC[a.tile_pos[q]] += kvs[q];
          }
        }
        __syncthreads();
        PH(7)
        // X L(j,j)^T = C, row block `warp` (8 rows) handled entirely by this warp:
        //   X[:,sb] = (C[:,sb] - X[:,0:sb] L(sb rows, 0:16sb)^T) W_sb^T      for sb = 0..3
#pragma unroll 1
        for (int sb = 0; sb < 4; ++sb) {
          double c2[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
          for (int kS = 0; kS < 4 * sb; ++kS) {
            const double av = sC[frag_off(warp, kS) + lane];
#pragma unroll
            for (int nbp = 0; nbp < 2; ++nbp) dmma(c2[nbp][0], c2[nbp][1], av, sLjj[frag_off(2 * sb + nbp, kS) + lane]);
          }
#pragma unroll
          for (int nbp = 0; nbp < 2; ++nbp) {
            double2* pv = reinterpret_cast<double2*>(sC + cfrag_off(warp, 2 * sb + nbp, lane));
            double2 v = *pv;
            v.x -= c2[nbp][0];
            v.y -= c2[nbp][1];
            *pv = v;
          }
          __syncwarp();
          double a4[4];
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) a4[ks] = sC[frag_off(warp, 4 * sb + ks) + lane];
          __syncwarp();
#pragma unroll
          for (int nbp = 0; nbp < 2; ++nbp) {
            double x0 = 0.0, x1 = 0.0;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) dmma(x0, x1, a4[ks], sWd[sb * 256 + (nbp * 4 + ks) * 32 + lane]);
            *reinterpret_cast<double2*>(sC + cfrag_off(warp, 2 * sb + nbp, lane)) = make_double2(x0, x1);
          }
          __syncwarp();
        }
        // this warp's 8 rows of X -> HBM: two contiguous 2 KB runs of the fragment-major tile
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int o = ((h * 8 + warp) << 8);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<double2*>(Xt + o + (lane + 32 * q) * 2) = *reinterpret_cast<const double2*>(sC + o + (lane + 32 * q) * 2);
        }
        __syncthreads();  // sC is about to be overwritten by the next stream; X visible to the CTA
        resident = tij;
        PH(8)
      }
    }

    if (fail) {
      if (tid == 0) a.status[b] = fail;
      __syncthreads();
      continue;
    }

    // ================= back substitution  L^T u = y  (u overwrites y) =================
    for (int j = nt - 1; j >= 0; --j) {
      // acc_c = sum_{i>j} sum_r L(i,j)[r][c] u_i[r]; thread (warp w, lane l) owns columns
      // c = h*32 + w*4 + (l&3) and rows r = rb*8 + (l>>2) of every tile (coalesced tile reads)
      double a0 = 0.0, a1 = 0.0;
#pragma unroll 2
      for (int i = j + 1; i < nt; ++i) {
        if (!a.tile_nz[tb_tile_index(i, j)]) continue;
        const double* Lt = Lsys + tb_tile_index(i, j) * TB_TILE_ELEMS;
        const double* ui = ysys + i * T + (lane >> 2);
#pragma unroll
        for (int rb = 0; rb < 8; ++rb) {
          const double uv = __ldcg(ui + rb * 8);
          a0 = fma(__ldcg(Lt + tid + rb * 256), uv, a0);
          a1 = fma(__ldcg(Lt + tid + (rb + 8) * 256), uv, a1);
        }
      }
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
      }
      if (lane < 4) {
        sRhs[warp * 4 + lane] = a0;
        sRhs[32 + warp * 4 + lane] = a1;
      }
      PH(9)
      // L(j,j) and the inverses of its 16x16 diagonal blocks back into shared memory
      {
        const double* Lt = Lsys + tb_tile_index(j, j) * TB_TILE_ELEMS;
#pragma unroll 4
        for (int q = 0; q < 16; ++q) sLjj[tid + q * 256] = __ldcg(Lt + tid + q * 256);
#pragma unroll
        for (int q = 0; q < 4; ++q) sWd[tid + q * 256] = __ldcg(wds + j * 1024 + tid + q * 256);
      }
      __syncthreads();
      if (warp == 0) {  // L^T u = r block by block, last 16 first:  u_sb = W_sb^T (r_sb - L(below, sb)^T u_below)
        sRv[lane] = __ldcg(ysys + j * T + lane) - sRhs[lane];
        sRv[lane + 32] = __ldcg(ysys + j * T + lane + 32) - sRhs[lane + 32];
        __syncwarp();
        const int c = lane & 15, hh = lane >> 4;
        for (int sb = 3; sb >= 0; --sb) {
          double t = 0.0;
          for (int rr = 16 * (sb + 1) + hh; rr < T; rr += 2) t = fma(sLjj[tb_tile_off(rr, 16 * sb + c)], sUb[rr], t);
          t += __shfl_xor_sync(0xffffffffu, t, 16);
          if (lane < 16) sT16[c] = sRv[16 * sb + c] - t;
          __syncwarp();
          double uv = 0.0;
          for (int cc = c + hh; cc < 16; cc += 2)   // W^T: u[c] = sum_{cc >= c} W[cc][c] t[cc]
            uv = fma(sWd[sb * 256 + ((((cc >> 3) << 2) + (c >> 2)) << 5) + ((cc & 7) << 2) + (c & 3)], sT16[cc], uv);
          uv += __shfl_xor_sync(0xffffffffu, uv, 16);
          if (lane < 16) {
            sUb[16 * sb + c] = uv;
            ysys[j * T + 16 * sb + c] = uv;
          }
          __syncwarp();
        }
      }
      __syncthreads();
      PH(10)
    }
    PH_FLUSH
    if (tid == 0) a.status[b] = 0;
  }
}

// ------------------------------------------------------------------------------------------
// k_recover: one CTA per system
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum256(double v, double* sRed, int tid) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((tid & 31) == 0) sRed[tid >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) t += sRed[w];
  return t;
}

// RECOMP: the member geometry (EA/L, cosines, weight term) is recomputed from the inputs instead of being read from the
// k_geom arrays, and cosines / axial forces of the system live in shared memory (used with k_prep).
template <int DIM, bool RECOMP>
__global__ void __launch_bounds__(256) k_recover(const LargeArgs a) {
  __shared__ double sRed[8];
  extern __shared__ __align__(16) double sRec[];   // RECOMP: [M] axial | [M][DIM] cosines
  const int tid = threadIdx.x;
  for (int b = blockIdx.x; b < a.batch; b += gridDim.x) {
    int status = a.status[b];
    if (status == 0 && !a.plan_stable) status = TB_INFO_NOT_STABLE;
    double* u_out = a.u ? a.u + (int64_t)b * a.N : nullptr;
    double* ext_out = a.ext ? a.ext + (int64_t)b * a.N : nullptr;
    double* ax_out = a.axial ? a.axial + (int64_t)b * a.M : nullptr;
    double* uf_out = a.u_free ? a.u_free + (int64_t)b * a.n : nullptr;
    double* re_out = a.react ? a.react + (int64_t)b * a.s : nullptr;
    if (status != 0) {
      for (int i = tid; i < a.N; i += 256) {
        if (u_out) u_out[i] = 0.0;
        if (ext_out) ext_out[i] = 0.0;
      }
      for (int r = tid; r < a.n; r += 256)
        if (uf_out) uf_out[r] = 0.0;
      for (int r = tid; r < a.s; r += 256)
        if (re_out) re_out[r] = 0.0;
      for (int m = tid; m < a.M; m += 256)
        if (ax_out) ax_out[m] = 0.0;
      if (tid == 0) {
        if (a.weight) a.weight[b] = 0.0;
        if (a.info) a.info[b] = status;
        if (a.fitness_mode) {
          if (a.fitness) a.fitness[b] = INFINITY;
          if (a.flags) { a.flags[2 * b] = 0; a.flags[2 * b + 1] = 0; }
        }
      }
      continue;
    }
    const double* uf = a.y + (int64_t)b * a.n_pad;
    const double* mk = RECOMP ? nullptr : a.mk + (int64_t)b * a.M;
    const double* mc = RECOMP ? sRec + a.M : a.mc + (int64_t)b * a.M * DIM;
    const double* mw = RECOMP ? nullptr : a.mw + (int64_t)b * a.M;
    double* axw = RECOMP ? sRec : a.mw + (int64_t)b * a.M;  // non-RECOMP: reuse the weight terms' slot for axial after reading them
    const double* xyz = a.xyz + b * a.xyz_stride;
    double w = 0.0, vs = 0.0, vd = 0.0;
    if (u_out)
      for (int i = tid; i < a.N; i += 256) {
        const int fr = a.dof2free[i];
        u_out[i] = fr >= 0 ? uf[fr] : 0.0;
      }
    if (uf_out)                                  // compact: free DOF r of the reference's order
      for (int r = tid; r < a.n; r += 256) uf_out[r] = uf[a.dof2free[a.free_ref[r]]];
    for (int m = tid; m < a.M; m += 256) {
      const int j0 = a.conn[2 * m], j1 = a.conn[2 * m + 1];
      double km, wm, cm[DIM];
      if (RECOMP) {   // same roundings as k_geom / k_prep (truss.py:19,56-63)
        double ar, e, rho;
        if (a.gene) {
          const int g = a.gene[b * a.gene_stride + m];
          ar = a.type_table[3 * g]; e = a.type_table[3 * g + 1]; rho = a.type_table[3 * g + 2];
        } else {
          const double* tt = a.aed + b * a.aed_stride + 3 * (int64_t)m;
          ar = tt[0]; e = tt[1]; rho = tt[2];
        }
        double dx[DIM];
        tb_member_geom<DIM>(xyz, j0, j1, ar, e, rho, dx, cm, km, wm);
#pragma unroll
        for (int i = 0; i < DIM; ++i) sRec[a.M + m * DIM + i] = cm[i];
      } else {
        km = mk[m];
        wm = mw[m];
#pragma unroll
        for (int i = 0; i < DIM; ++i) cm[i] = mc[m * DIM + i];
      }
      double t = 0.0;
#pragma unroll
      for (int i = 0; i < DIM; ++i) {
        const int f1 = a.dof2free[j1 * DIM + i], f0 = a.dof2free[j0 * DIM + i];
        const double u1 = f1 >= 0 ? uf[f1] : 0.0, u0 = f0 >= 0 ? uf[f0] : 0.0;
        t = fma(cm[i], u1 - u0, t);
      }
      const double nm = km * t;
      w += wm;
      axw[m] = nm;
      if (ax_out) ax_out[m] = nm;
      if (a.fitness_mode) {
        const double f = fabs(nm);
        if (!(f < TB_ZERO_EPS)) {
          double ar;
          if (a.gene) ar = a.type_table[3 * a.gene[b * a.gene_stride + m]];
          else ar = a.aed[b * a.aed_stride + 3 * (int64_t)m];
          const double sg = f / ar;
          if (sg > a.allow_stress) vs += sg - a.allow_stress;
        }
      }
    }
    __syncthreads();  // axial forces of this system are visible to the CTA
    auto reaction = [&](int dof) {               // row of K times u at a supported DOF, member by member (ascending)
      const int J = dof / DIM, ax = dof - J * DIM;
      double e = 0.0;
      for (int p = a.inc_ptr[J]; p < a.inc_ptr[J + 1]; ++p) {
        const int me = a.inc_mem[p], m = me >> 1;
        const double g = (me & 1) ? mc[m * DIM + ax] : -mc[m * DIM + ax];
        e = fma(g, axw[m], e);
      }
      return e;
    };
    if (ext_out) {
      const double* f = a.force + b * a.force_stride;
      for (int dof = tid; dof < a.N; dof += 256) ext_out[dof] = a.dof2free[dof] >= 0 ? f[dof] : reaction(dof);
    }
    if (re_out)                                  // compact: supported DOF r of the reference's order
      for (int r = tid; r < a.s; r += 256) re_out[r] = reaction(a.sup_idx[r]);
    if (a.fitness_mode) {
      for (int j = tid; j < a.nJ; j += 256) {
        bool any = false;
        double l2 = 0.0;
#pragma unroll
        for (int i = 0; i < DIM; ++i) {
          const int fr = a.dof2free[j * DIM + i];
          const double v = fr >= 0 ? uf[fr] : 0.0;
          any |= !(fabs(v) < TB_ZERO_EPS);
          l2 += v * v;
        }
        if (any) {
          const double l = sqrt(l2);
          if (l > a.allow_displace) vd += l - a.allow_displace;
        }
      }
    }
    w = block_sum256(w, sRed, tid);
    if (a.fitness_mode) {
      vs = block_sum256(vs, sRed, tid);
      vd = block_sum256(vd, sRed, tid);
    }
    if (tid == 0) {
      if (a.weight) a.weight[b] = w;
      if (a.info) a.info[b] = 0;
      if (a.fitness_mode) {
        const bool ok_s = fabs(vs) < TB_ZERO_EPS, ok_d = fabs(vd) < TB_ZERO_EPS;
        double fit = w;
        if (!ok_s) fit += vs / a.allow_stress * 1e5;
        if (!ok_d) fit += vd / a.allow_displace * 1e5;
        if (a.fitness) a.fitness[b] = fit;
        if (a.flags) { a.flags[2 * b] = ok_s; a.flags[2 * b + 1] = ok_d; }
      }
    }
    __syncthreads();
  }
}

}  // namespace

size_t tb_large_workspace_bytes(int batch, int dim, int M, int n_pad, int64_t nnz, int path, int nb16, int NB) {
  const int nt = n_pad / TB_TILE;
  const size_t ntiles = (size_t)nt * (nt + 1) / 2;
  size_t per = (size_t)M * (2 + dim + dim * (dim + 1) / 2) + (size_t)nnz;
  if (path == 2) per += (size_t)nb16 * (NB + 1) * 256 + (size_t)nb16 * 256 + (size_t)nb16 * 16;
  else per += ntiles * TB_TILE_ELEMS + (size_t)nt * 1024 + (size_t)n_pad;
  return (size_t)batch * per * 8 + (size_t)batch * 4 + 1024;
}

void tb_large_carve(LargeArgs& a, void* ws, int path) {
  double* p = (double*)ws;
  if (path == 2) {
    a.L = p;  p += (size_t)a.batch * a.nb16 * (a.NB + 1) * 256;   // off-diagonal 16x16 blocks of L
    a.wd = p; p += (size_t)a.batch * a.nb16 * 256;                // inverses of the diagonal blocks
    a.y = p;  p += (size_t)a.batch * a.nb16 * 16;
  } else {
    const size_t ntiles = (size_t)a.nt * (a.nt + 1) / 2;
    a.L = p;  p += (size_t)a.batch * ntiles * TB_TILE_ELEMS;      // first: 32 KB-aligned tiles
    a.wd = p; p += (size_t)a.batch * a.nt * 1024;
    a.y = p;  p += (size_t)a.batch * a.n_pad;
  }
  a.mk = p; p += (size_t)a.batch * a.M;
  a.mc = p; p += (size_t)a.batch * a.M * a.dim;
  a.mw = p; p += (size_t)a.batch * a.M;
  a.mkc = p; p += (size_t)a.batch * a.M * (a.dim * (a.dim + 1) / 2);
  a.kv = p; p += (size_t)a.batch * a.nnz;
  a.status = (int32_t*)p;
}

namespace {

// largest dynamic shared-memory size already granted to a kernel instantiation, per device (cudaFuncSetAttribute is a
// per-device setting: a process that solves on cuda:0 and then on cuda:1 has to opt in on both)
constexpr int TB_MAX_DEV = 64;
struct SmemGrant {
  std::mutex mu;
  size_t granted[TB_MAX_DEV] = {};
  template <typename K>
  int ensure(K kern, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    std::lock_guard<std::mutex> lock(mu);
    size_t& g = granted[dev & (TB_MAX_DEV - 1)];
    if (g >= bytes) return 0;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return (int)e;
    g = bytes;
    return 0;
  }
};
SmemGrant g_prep_grant[2], g_rec_grant[2], g_chol_grant[2];

// recovery of one batch (truss.py:344-361): member geometry recomputed in shared memory when it fits, else from the k_geom arrays
int launch_recover(const LargeArgs& a, int num_sm, cudaStream_t st, bool recomp) {
  const size_t rec_smem = (size_t)a.M * (1 + a.dim) * 8;
  int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
  tb_prof_begin(TB_PROF_RECOVER, st);
  if (recomp) {
    auto kern = a.dim == 3 ? k_recover<3, true> : k_recover<2, true>;
    const int rc = g_rec_grant[a.dim - 2].ensure(kern, rec_smem);
    if (rc) return rc;
    kern<<<grid, 256, rec_smem, st>>>(a);
  } else if (a.dim == 3) {
    k_recover<3, false><<<grid, 256, 0, st>>>(a);
  } else {
    k_recover<2, false><<<grid, 256, 0, st>>>(a);
  }
  tb_prof_end(TB_PROF_RECOVER, st);
  return 0;
}

// Two-sided band kernel (tb_bandts.cu): assembly pass in the kernel's program order, the band kernel, recovery
int launch_ts_path(const LargeArgs& a, int num_sm, cudaStream_t st) {
  const TsPlan* ts = a.ts;
  TsArgs t;
  memset(&t, 0, sizeof(t));
  t.batch = a.batch; t.dim = a.dim; t.nJ = a.nJ; t.M = a.M; t.N = a.N; t.n = a.n;
  t.force = a.force; t.force_stride = a.force_stride;
  tb_ts_fill_sides(t, ts);
  double* kv = nullptr;
  tb_ts_carve(t, ts, a.ts_ws, a.ts_total, a.ts_b0, &kv);
  // assembly (k_prep / k_geom + k_kval) driven by the program-order scatter lists; recovery reads u in the internal order
  LargeArgs r = a;
  r.q_first = ts->d_tq_first; r.q_multi = ts->d_tq_multi; r.q_ptr = ts->d_tq_ptr; r.q_pack = ts->d_tq_pack;
  r.n_multi = (int)ts->tq_multi.size();
  r.q_multi4 = ts->d_tq_multi4;
  r.nnz = (int64_t)ts->epos.size();
  r.kv = kv;
  r.y = t.uf;
  r.n_pad = t.n_pad;
  r.status = t.status;
  const size_t prep_smem = (size_t)a.M * (a.dim * (a.dim + 1) / 2) * 8, rec_smem = (size_t)a.M * (1 + a.dim) * 8;
  const bool prep = prep_smem <= 96 * 1024 && rec_smem <= 96 * 1024;
  int launches = 2;
  if (prep) {
    auto kern = a.dim == 3 ? k_prep<3> : k_prep<2>;
    const int rcg = g_prep_grant[a.dim - 2].ensure(kern, prep_smem);
    if (rcg) return rcg;
    int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
    tb_prof_begin(TB_PROF_ASSEMBLE, st);
    kern<<<grid, 256, prep_smem, st>>>(r);
    tb_prof_end(TB_PROF_ASSEMBLE, st);
  } else {                                       // very many members: products through HBM
    k_init_status<<<(a.batch + 255) / 256, 256, 0, st>>>(r.status, a.batch, 0);
    const int64_t total = (int64_t)a.batch * a.M;
    int grid = (int)((total + 255) / 256 < (int64_t)num_sm * 8 ? (total + 255) / 256 : (int64_t)num_sm * 8);
    if (grid < 1) grid = 1;
    tb_prof_begin(TB_PROF_GEOM, st);
    if (a.dim == 3) k_geom<3><<<grid, 256, 0, st>>>(r);
    else k_geom<2><<<grid, 256, 0, st>>>(r);
    tb_prof_end(TB_PROF_GEOM, st);
    grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
    tb_prof_begin(TB_PROF_ASSEMBLE, st);
    k_kval<<<grid, 256, 0, st>>>(r);
    tb_prof_end(TB_PROF_ASSEMBLE, st);
    launches += 2;
  }
  int rc = tb_launch_band_ts(t, tb_ts_smem_bytes(ts), num_sm, st);
  if (rc) return rc;
  rc = launch_recover(r, num_sm, st, prep);
  if (rc) return rc;
  tb_count_launch(launches);                     // (the band kernel counted itself)
  return (int)cudaGetLastError();
}

}  // namespace

// The assembly pass alone (debug export of the device-assembled K_ff values): k_prep, or k_geom + k_kval when the member
// products do not fit shared memory, driven by whatever scatter lists a.q_* point at; writes a.kv[B][a.nnz].
int tb_launch_assemble_only(const LargeArgs& a, int num_sm, cudaStream_t st) {
  if (a.batch <= 0) return 0;
  if (num_sm <= 0) num_sm = 148;
  const size_t prep_smem = (size_t)a.M * (a.dim * (a.dim + 1) / 2) * 8;
  const int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
  if (prep_smem <= 96 * 1024) {
    auto kern = a.dim == 3 ? k_prep<3> : k_prep<2>;
    const int rcg = g_prep_grant[a.dim - 2].ensure(kern, prep_smem);
    if (rcg) return rcg;
    kern<<<grid, 256, prep_smem, st>>>(a);
  } else {
    k_init_status<<<(a.batch + 255) / 256, 256, 0, st>>>(a.status, a.batch, 0);
    const int64_t total = (int64_t)a.batch * a.M;
    int g2 = (int)((total + 255) / 256 < (int64_t)num_sm * 8 ? (total + 255) / 256 : (int64_t)num_sm * 8);
    if (g2 < 1) g2 = 1;
    if (a.dim == 3) k_geom<3><<<g2, 256, 0, st>>>(a);
    else k_geom<2><<<g2, 256, 0, st>>>(a);
    k_kval<<<grid, 256, 0, st>>>(a);
  }
  tb_count_launch(1);
  return (int)cudaGetLastError();
}

int tb_launch_large(const LargeArgs& a, int num_sm, cudaStream_t st, int path) {
  if (a.batch <= 0) return 0;
  if (num_sm <= 0) num_sm = 148;
  static const bool ts_legacy = [] { const char* s = getenv("TB_BAND_LEGACY"); return s && s[0] == '1'; }();
  const bool use_ts = path == 2 && a.ts && a.ts_ws && !a.shared_k && !ts_legacy;
  // TB_UNFUSED_ASSEMBLY=1 keeps the separate HBM-bound assembly kernel (A/B measurements, tiled path only)
  static const bool fused_env = [] { const char* s = getenv("TB_UNFUSED_ASSEMBLY"); return !(s && s[0] == '1'); }();
  const bool fused = fused_env || path == 2;
  // member products in shared memory (k_prep + recomputing k_recover) when they fit, else the k_geom arrays in HBM
  const size_t prep_smem = (size_t)a.M * (a.dim * (a.dim + 1) / 2) * 8, rec_smem = (size_t)a.M * (1 + a.dim) * 8;
  static const bool no_prep = [] { const char* s = getenv("TB_NO_PREP"); return s && s[0] == '1'; }();
  const bool prep = fused && !no_prep && prep_smem <= 96 * 1024 && rec_smem <= 96 * 1024;
  // Two half-batches on two streams (band path, a batch of a few systems per SM): assembly is two waves of CTAs, so
  // the first half's factorisation starts while the second half is still being assembled, and the first half's
  // recovery runs under the second half's factorisation.  Both halves use the two-warp band kernel (eight systems per
  // SM), so together they occupy the SMs like the unsplit batch.  Not under per-kernel profiling (one stream there).
  static const bool split_env = [] { const char* s = getenv("TB_LARGE_SPLIT"); return !(s && s[0] == '0'); }();
  // (not for the two-sided kernel: its halves start together once both assemblies are done, nothing overlaps -- measured)
  if (split_env && !a.no_split && !tb_prof_on() && path == 2 && prep && !a.shared_k && !use_ts && a.NB <= 5 &&
      a.batch > num_sm * 6 && a.batch <= num_sm * 8) {
    static std::mutex split_mu;                // the second stream and its events are shared by every plan of the process:
    std::lock_guard<std::mutex> split_lock(split_mu);   // fork .. join is enqueued as one unit
    static cudaStream_t aux = nullptr;
    static cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    if (!aux) {
      cudaError_t e = cudaStreamCreateWithFlags(&aux, cudaStreamNonBlocking);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming);
      if (e != cudaSuccess) return (int)e;
    }
    static const int n0_env = [] { const char* s = getenv("TB_LARGE_SPLIT_N0"); return s ? atoi(s) : 0; }();
    const int n0 = n0_env > 0 && n0_env < a.batch ? n0_env : num_sm * 4;   // default: one wave of the assembly kernel
    auto slice = [&](int b0, int nb) {
      LargeArgs h = a;
      h.batch = nb;
      h.no_split = 1;
      h.band_warps = 2;
      h.ts_b0 = a.ts_b0 + b0;
      h.xyz = a.xyz + (int64_t)b0 * a.xyz_stride;
      if (a.aed) h.aed = a.aed + (int64_t)b0 * a.aed_stride;
      if (a.gene) h.gene = a.gene + (int64_t)b0 * a.gene_stride;
      h.force = a.force + (int64_t)b0 * a.force_stride;
      const int nv = a.dim * (a.dim + 1) / 2;
      h.mk = a.mk + (int64_t)b0 * a.M;
      h.mc = a.mc + (int64_t)b0 * a.M * a.dim;
      h.mw = a.mw + (int64_t)b0 * a.M;
      h.mkc = a.mkc + (int64_t)b0 * a.M * nv;
      h.kv = a.kv + (int64_t)b0 * a.nnz;
      h.wd = a.wd + (int64_t)b0 * a.nb16 * 256;
      h.L = a.L + (int64_t)b0 * a.nb16 * (a.NB + 1) * 256;
      h.y = a.y + (int64_t)b0 * a.n_pad;
      h.status = a.status + b0;
      if (a.u) h.u = a.u + (int64_t)b0 * a.N;
      if (a.u_free) h.u_free = a.u_free + (int64_t)b0 * a.n;
      if (a.react) h.react = a.react + (int64_t)b0 * a.s;
      if (a.ext) h.ext = a.ext + (int64_t)b0 * a.N;
      if (a.axial) h.axial = a.axial + (int64_t)b0 * a.M;
      if (a.weight) h.weight = a.weight + b0;
      if (a.info) h.info = a.info + b0;
      if (a.fitness) h.fitness = a.fitness + b0;
      if (a.flags) h.flags = a.flags + 2 * (int64_t)b0;
      return h;
    };
    const LargeArgs hA = slice(0, n0), hB = slice(n0, a.batch - n0);
    TB_CUDA(cudaEventRecord(ev_fork, st));
    TB_CUDA(cudaStreamWaitEvent(aux, ev_fork, 0));
    int rc = tb_launch_large(hA, num_sm, st, path);
    if (rc) return rc;
    rc = tb_launch_large(hB, num_sm, aux, path);
    if (rc) return rc;
    TB_CUDA(cudaEventRecord(ev_join, aux));
    TB_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
    return (int)cudaGetLastError();
  }
  if (use_ts) return launch_ts_path(a, num_sm, st);
  if (!prep) k_init_status<<<(a.batch + 255) / 256, 256, 0, st>>>(a.status, a.batch, 0);   // k_prep clears its own
  // load cases of one truss (shared_k): assembly and factorisation run for system 0 only
  const bool shared = a.shared_k && path == 2 && prep && a.batch > 1;
  LargeArgs a1 = a;
  a1.batch = 1;
  if (prep) {
    auto kern = a.dim == 3 ? k_prep<3> : k_prep<2>;
    {
      const int rcg = g_prep_grant[a.dim - 2].ensure(kern, prep_smem);
      if (rcg) return rcg;
    }
    int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
    tb_prof_begin(TB_PROF_ASSEMBLE, st);
    if (shared) kern<<<1, 256, prep_smem, st>>>(a1);
    else kern<<<grid, 256, prep_smem, st>>>(a);
    tb_prof_end(TB_PROF_ASSEMBLE, st);
  } else {
    {
      const int64_t total = (int64_t)a.batch * a.M;
      int grid = (int)((total + 255) / 256 < (int64_t)num_sm * 8 ? (total + 255) / 256 : (int64_t)num_sm * 8);
      if (grid < 1) grid = 1;
      tb_prof_begin(TB_PROF_GEOM, st);
      if (a.dim == 3) k_geom<3><<<grid, 256, 0, st>>>(a);
      else k_geom<2><<<grid, 256, 0, st>>>(a);
      tb_prof_end(TB_PROF_GEOM, st);
    }
    if (fused) {
      int grid = a.batch < num_sm * 8 ? a.batch : num_sm * 8;
      tb_prof_begin(TB_PROF_ASSEMBLE, st);
      k_kval<<<grid, 256, 0, st>>>(a);
      tb_prof_end(TB_PROF_ASSEMBLE, st);
    } else {
      const int64_t work = (int64_t)a.nt * (a.nt + 1) / 2 * a.batch;
      int grid = (int)(work < (int64_t)num_sm * 16 ? work : (int64_t)num_sm * 16);
      tb_prof_begin(TB_PROF_ASSEMBLE, st);
      if (a.dim == 3) k_assemble<3><<<grid, 256, 0, st>>>(a);
      else k_assemble<2><<<grid, 256, 0, st>>>(a);
      tb_prof_end(TB_PROF_ASSEMBLE, st);
    }
  }
  if (path == 2) {
    int rc = tb_launch_band_chol(shared ? a1 : a, num_sm, st);
    if (rc) return rc;
    if (shared) {                              // every load case against the factor of system 0
      rc = tb_launch_band_subst(a, num_sm, st);
      if (rc) return rc;
    }
  } else {
    auto kern = fused ? k_chol<true> : k_chol<false>;
    {
      const int rcg = g_chol_grant[fused].ensure(kern, CHOL_SMEM_BYTES);
      if (rcg) return rcg;
    }
    static std::atomic<int> chol_per_sm[2];    // blocks per SM: a property of the kernel and the architecture, not of the device ordinal
    if (chol_per_sm[fused].load() == 0) {
      int q = 0;
      cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&q, kern, CH_THREADS, CHOL_SMEM_BYTES);
      if (e != cudaSuccess) return (int)e;
      chol_per_sm[fused].store(q < 1 ? 1 : q);
    }
    const int per_sm = chol_per_sm[fused].load();
    int grid = num_sm * per_sm;
    if (grid > a.batch) grid = a.batch;
    tb_prof_begin(TB_PROF_CHOL, st);
    kern<<<grid, CH_THREADS, CHOL_SMEM_BYTES, st>>>(a);
    tb_prof_end(TB_PROF_CHOL, st);
  }
  {
    const int rcr = launch_recover(a, num_sm, st, prep);
    if (rcr) return rcr;
  }
  tb_count_launch((prep ? 3 : 5) + (shared ? 1 : 0));
  return (int)cudaGetLastError();
}
