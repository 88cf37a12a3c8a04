// Shared declarations for the truss_b200 CUDA library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "truss_b200.h"

struct TsPlan;   // two-sided band program (tb_ts.cuh)

// SupportType codes, slientruss3d/type.py:30-35
enum : int { SUP_NO = 0, SUP_PIN = 1, SUP_ROLLER_X = 2, SUP_ROLLER_Y = 3, SUP_ROLLER_Z = 4 };

// Support code -> DOF rule (type.py:48-74): axis `ax` of a joint is restrained by a pin or by the roller of that axis
__host__ __device__ __forceinline__ bool tb_dof_free(int s, int ax) { return !((s == SUP_PIN) || (s == SUP_ROLLER_X + ax)); }
// a code the dim does not know (TB_INFO_BAD_SUPPORT)
__host__ __device__ __forceinline__ bool tb_support_bad(int dim, int s) { return s > SUP_ROLLER_Z || (dim == 2 && s == SUP_ROLLER_Z); }

// utils.py:79-84 IsZero / IsZeroVector default eps
#define TB_ZERO_EPS 1e-10

// tile geometry of the blocked (global-memory) path
constexpr int TB_TILE = 64;                     // tile order
constexpr int TB_TILE_ELEMS = TB_TILE * TB_TILE;  // doubles per tile

// band path (tb_band.cu): 16x16 blocks, at most TB_BAND_MAX_NB sub-diagonal blocks per block column
constexpr int TB_BAND_MAX_NB = 8;

// limits of the fused shared-memory path
constexpr int TB_SMALL_MAX_DOF = 160;     // max d*nJ (bounds the free-DOF count)
constexpr int TB_SMALL_MAX_MEMBER = 1024;
constexpr int TB_SMALL_MAX_JOINT = 80;

// Ragged batches beyond the fused kernels (tb_ragenv.cu): the envelope kernel k_rag_env takes trusses up to
// TB_RAGGED_MAX_DOF = d*nJ and TB_RAGGED_MAX_MEMBER members (the generator's largest truss on a 6^3 grid is 343 joints
// and 5184 members; bar-942 is 732 DOFs).  A batch that does not fit the fused kernels as a whole is split by truss: the
// trusses up to (TB_RAGGED_ROUTE_J<d>, TB_RAGGED_ROUTE_M<d>) run on the fused kernels in one launch of that size (it stays
// on k_dense16 -- at most 9 blocks of 16 free DOFs and 110 KB of shared memory per warp -- and cube-7's 32 joints / 119
// members are under it), the others on k_rag_env.
constexpr int TB_RAGGED_MAX_DOF = 1536;
constexpr int TB_RAGGED_MAX_MEMBER = 8192;
constexpr int TB_RAGGED_ROUTE_J3 = 48, TB_RAGGED_ROUTE_M3 = 192;
constexpr int TB_RAGGED_ROUTE_J2 = 72, TB_RAGGED_ROUTE_M2 = 224;

extern std::atomic<int64_t> g_tb_launches;
inline void tb_count_launch(int n = 1) { g_tb_launches.fetch_add(n, std::memory_order_relaxed); }

// optional per-kernel CUDA-event timing (bench.py's roofline line); slots:
enum : int { TB_PROF_GEOM = 0, TB_PROF_ASSEMBLE = 1, TB_PROF_CHOL = 2, TB_PROF_RECOVER = 3, TB_PROF_SMALL = 4, TB_PROF_SUBST = 5, TB_PROF_SLOTS = 8 };
bool tb_prof_on();
void tb_prof_begin(int slot, cudaStream_t st);
void tb_prof_end(int slot, cudaStream_t st);

#define TB_CUDA(expr)                         \
  do {                                        \
    cudaError_t _e = (expr);                  \
    if (_e != cudaSuccess) return (int)_e;    \
  } while (0)

// ---------------------------------------------------------------------------------------------
// Plan: host-built integer maps for one topology (truss.py:307-326), mirrored on the device.
// ---------------------------------------------------------------------------------------------
// calls of tb_solve_host_async in flight per plan: one uploading, one computing, one downloading
constexpr int TB_ASYNC_SLOTS = 3;

struct DevBuf { void* ptr = nullptr; size_t bytes = 0; };   // grow-only device buffer (tb_api.cu: reserve_sync / _async)
// Cross-stream order of a scratch buffer (tb_api.cu): acquire makes a call on another stream than the last user's wait
// for its event, release records it after the call's last kernel; neither does anything inside a stream capture.
struct StreamOrder {
  cudaEvent_t ev = nullptr;
  cudaStream_t last = nullptr;   // stream of the last call that used the buffer
  bool used = false;
  int acquire(cudaStream_t st);
  int release(cudaStream_t st);
};

struct tb_plan {
  int dim = 0, nJ = 0, M = 0, N = 0, n = 0, s = 0;
  int n_resist = 0, stable = 0, path = 0, n_pad = 0, nt = 0;
  int64_t half_bw = 0;
  int device = 0;
  int num_sm = 0;

  // host copies
  std::vector<int32_t> conn;       // [M,2]
  std::vector<uint8_t> support;    // [nJ]
  std::vector<int32_t> free_idx;   // [n]
  std::vector<int32_t> dof2free;   // [N]
  std::vector<int32_t> sup_idx;    // [s]
  // internal elimination order (reverse Cuthill-McKee over the joints when it shrinks the envelope)
  int reordered = 0;
  std::vector<int32_t> perm;       // [n] internal index -> reference free index
  std::vector<int32_t> free_int;   // [n] DOF index of internal row i      (device: d_free_idx)
  std::vector<int32_t> d2f_int;    // [N] internal row of a DOF, -1 at supports (device: d_dof2free)
  std::vector<int32_t> int_row, int_col;   // [nnz] entry rows / columns in the internal order (row >= col)
  // scatter map over the lower triangle of K_ff (row-major order of entries)
  std::vector<int32_t> ent_row, ent_col;   // [nnz]
  std::vector<int64_t> ent_ptr;            // [nnz+1]
  std::vector<int32_t> ctr_member;         // [n_contrib]
  std::vector<int32_t> ctr_local;          // [n_contrib] a*2d+b
  std::vector<int64_t> tile_ent_ptr;       // [ntiles+1] entries grouped per 64x64 tile (blocked path)
  std::vector<int32_t> tile_ent;           // [nnz] entry ids sorted by tile
  std::vector<int32_t> tile_pos;           // [nnz] fragment-major offset inside the tile, same order
  std::vector<int32_t> q_ptr;              // [nnz+1] contribution ranges in tile_ent order
  std::vector<int32_t> q_pack;             // [n_contrib] member<<4 | negate<<3 | index of (i<=j) cosine product
  std::vector<int32_t> q_multi, bq_multi;  // entries with more than one contribution (tile / band order positions)
  std::vector<int32_t> q_first, bq_first;  // [nnz] first contribution of an entry (tile / band order) | bit 31: the entry has more
  // block-level symbolic factorisation: which 64x64 tiles of L are structurally non-zero, and for
  // each such tile (i,j) the list of k < j with L(i,k) and L(j,k) both non-zero
  std::vector<uint8_t> tile_nz;            // [ntiles]
  std::vector<int32_t> prod_ptr;           // [ntiles+1]
  std::vector<int32_t> prod_k;             // [n_prod]
  int64_t n_tiles_nz = 0;
  // band view (16x16 blocks): nb16 block columns, NB sub-diagonal blocks; entries grouped per block column
  int nb16 = 0, NB = 0;
  std::vector<int32_t> b16_ptr;            // [2 nb16+1] entry ranges (band order) per block column: diagonal block, blocks below it
  std::vector<int32_t> b16_pos;            // [nnz] (block offset e) << 8 | offset inside the 16x16 block
  std::vector<int32_t> b16_nz;             // [nb16] bit e: block (c+e, c) of L is structurally non-zero (block symbolic factorisation)
  int64_t b16_blocks_nz = 0, b16_products = 0;   // non-zero blocks of L, block products of the factorisation
  std::vector<int32_t> bq_ptr, bq_pack;    // contribution lists in band order (same encoding as q_ptr/q_pack)
  int64_t envelope_size = 0;               // entries inside the row envelope of K_ff (= of L)
  double envelope_flops = 0.0;             // flops of an envelope Cholesky + two triangular solves
  double chol_flops = 0.0;                 // flops of the block-sparse factorisation + two triangular solves
  // joint -> incident (member, end) lists, ascending member (recovery of reactions)
  std::vector<int32_t> inc_ptr;            // [nJ+1]
  std::vector<int32_t> inc_mem;            // [2M]  member*2 + end

  // device mirrors
  int32_t* d_conn = nullptr;
  uint8_t* d_support = nullptr;
  int32_t* d_free_idx = nullptr;
  int32_t* d_dof2free = nullptr;
  int32_t* d_sup_idx = nullptr;
  int32_t* d_free_ref = nullptr;   // [n] DOF index of free DOF r in the reference's order (host: free_idx): compact outputs
  int32_t* d_ent_row = nullptr;
  int32_t* d_ent_col = nullptr;
  int64_t* d_ent_ptr = nullptr;
  int32_t* d_ctr_member = nullptr;
  int32_t* d_ctr_local = nullptr;
  int64_t* d_tile_ent_ptr = nullptr;
  int32_t* d_tile_ent = nullptr;
  int32_t* d_tile_pos = nullptr;
  int32_t* d_q_ptr = nullptr;
  int32_t* d_q_pack = nullptr;
  int32_t* d_q_first = nullptr;
  int32_t* d_bq_first = nullptr;
  int32_t* d_q_multi = nullptr;
  int32_t* d_bq_multi = nullptr;
  int32_t* d_b16_ptr = nullptr;
  int32_t* d_b16_pos = nullptr;
  int32_t* d_b16_nz = nullptr;
  int32_t* d_bq_ptr = nullptr;
  int32_t* d_bq_pack = nullptr;
  uint8_t* d_tile_nz = nullptr;
  int32_t* d_prod_ptr = nullptr;
  int32_t* d_prod_k = nullptr;
  int32_t* d_inc_ptr = nullptr;
  int32_t* d_inc_mem = nullptr;

  // two-sided band program of the fused band kernel (tb_tsplan.cu); ts->ok == 0 when the band is too wide for it
  TsPlan* ts = nullptr;

  // grow-only device workspace of the blocked path.  One workspace per plan: `mu` serialises the calls that enqueue work
  // on it (and the growth of the arenas), `ws_order` orders its use, and that of adj_buf and modes_buf, across streams.
  // See the threading contract in truss_b200.h.
  DevBuf ws;
  std::mutex mu;
  StreamOrder ws_order;
  // grow-only staging for the *_host entry points
  DevBuf stage_dev;
  // dense u / ext of a call that asks for the compact outputs only (grow-only, [capacity][N] each)
  DevBuf compact_u, compact_ext;
  // tb_adjoint scratch (grow-only, grown stream-ordered on the caller's stream): adjoint load and solution [B][N] each,
  // status [B], and the per-member vectors [B][M][d] when they do not fit shared memory
  DevBuf adj_buf;
  // modal scratch of tb_modes' consistent mass and of tb_buckling (grow-only, grown stream-ordered): one n x n slot per CTA
  // of the launch
  DevBuf modes_buf;
  // pipelined host calls (tb_solve_host_async): TB_ASYNC_SLOTS more staging arenas used in turn by consecutive calls,
  // the events that chain a call's copies and kernels, and the ticket counters (submitted / known to be complete)
  DevBuf stage_async[TB_ASYNC_SLOTS];
  cudaEvent_t async_in[TB_ASYNC_SLOTS] = {}, async_k[TB_ASYNC_SLOTS] = {}, async_done[TB_ASYNC_SLOTS] = {};
  uint64_t async_submitted = 0, async_completed = 0;
};

// ---------------------------------------------------------------------------------------------
// Several correctly rounded quotients over ONE divisor (a member's EA/L and direction cosines all divide by its length,
// truss.py:19,56-63): y = RN(1/b) once (__drcp_rn), then per numerator Markstein's sequence q = RN(a y), r = a - b q
// (exact, one FMA), RN(q + r y).  With y the correctly rounded reciprocal this IS RN(a / b) -- the result the reference's
// float division produces -- as long as nothing under- or overflows on the way and b's significand is not all ones;
// those (rare) cases take __ddiv_rn.  22 instead of ~110 instructions for the four quotients of a member.
// tb_div_probe checks it against __ddiv_rn on random and adversarial operands (tests/test_gpu_parity.py).
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
struct TbDivisor {
  double b, y;
  bool safe;
  __device__ __forceinline__ explicit TbDivisor(double b_) : b(b_) {
    y = __drcp_rn(b_);
    const int hi = __double2hiint(b_), ex = (hi >> 20) & 0x7ff;
    const bool ones = ((hi & 0xfffff) == 0xfffff) && (__double2loint(b_) == (int)0xffffffff);
    safe = ex > 0x200 && ex < 0x5ff && !ones && hi > 0;       // positive, normal, far from the ends of the exponent range
  }
  __device__ __forceinline__ double div(double a) const {
    const int ea = (__double2hiint(a) >> 20) & 0x7ff;
    if (!safe || ea > 0x5ff || (ea < 0x200 && a != 0.0)) return __ddiv_rn(a, b);
    const double q = __dmul_rn(a, y);
    const double r = __fma_rn(-b, q, a);
    return a == 0.0 ? q : __fma_rn(r, y, q);                   // (a zero keeps its sign: the correction would turn -0 into +0)
  }
};

// Geometry of member (j0, j1) with the reference's roundings (truss.py:19,56-63): dx = x_j1 - x_j0, the length (squares
// summed in axis order), k = EA/L and the cosines through one shared divisor, and the weight term (a L) density.  Returns
// the length; k and c are not finite for a zero-length member (the caller checks the length).
template <int DIM>
__device__ __forceinline__ double tb_member_geom(const double* xyz, int j0, int j1, double ar, double e, double rho,
                                                 double dx[DIM], double c[DIM], double& k, double& w) {
#pragma unroll
  for (int i = 0; i < DIM; ++i) dx[i] = __dsub_rn(xyz[j1 * DIM + i], xyz[j0 * DIM + i]);
  double l2 = __dmul_rn(dx[0], dx[0]);
#pragma unroll
  for (int i = 1; i < DIM; ++i) l2 = __dadd_rn(l2, __dmul_rn(dx[i], dx[i]));
  const double len = __dsqrt_rn(l2);
  const TbDivisor dv(len);                  // (one reciprocal for the four quotients of the member)
  k = dv.div(__dmul_rn(e, ar));
#pragma unroll
  for (int i = 0; i < DIM; ++i) c[i] = dv.div(dx[i]);
  w = __dmul_rn(__dmul_rn(ar, len), rho);
  return len;
}
#endif

// ---------------------------------------------------------------------------------------------
// Kernel argument blocks
// ---------------------------------------------------------------------------------------------
struct SmallArgs {
  int batch, nJ, M;                     // uniform sizes, or the maxima of a ragged batch
  const int64_t* joint_off;             // ragged when non-null
  const int64_t* member_off;
  const double* xyz;      int64_t xyz_stride;
  const uint8_t* support; int64_t support_stride;
  const int32_t* conn;    int64_t conn_stride;
  const double* aed;      int64_t aed_stride;
  const int32_t* gene;    int64_t gene_stride;
  const double* type_table; int n_type;
  const double* force;    int64_t force_stride;
  double* u; double* ext; double* axial; double* weight; int32_t* info;
  double* fitness; uint8_t* flags;
  double allow_stress, allow_displace;
  int fitness_mode;
  int max_n;                            // bound on the free-DOF count (sizes shared memory)
};

struct LargeArgs {
  int batch, dim, nJ, M, N, n, n_pad, nt, s;
  const double* xyz;      int64_t xyz_stride;
  const double* aed;      int64_t aed_stride;
  const int32_t* gene;    int64_t gene_stride;
  const double* type_table; int n_type;
  const double* force;    int64_t force_stride;
  // plan maps (device)
  const int32_t* conn; const int32_t* free_idx; const int32_t* dof2free; const int32_t* sup_idx;
  const int32_t* ent_row; const int32_t* ent_col; const int64_t* ent_ptr;
  const int32_t* ctr_member; const int32_t* ctr_local;
  const int64_t* tile_ent_ptr; const int32_t* tile_ent; const int32_t* tile_pos;
  int64_t nnz;
  const uint8_t* tile_nz; const int32_t* prod_ptr; const int32_t* prod_k;
  const int32_t* q_ptr; const int32_t* q_pack; const int32_t* q_first; const int32_t* q_multi; int n_multi;
  const int4* q_multi4;   // optional: {entry, first contribution, end, 0} per multi-contribution entry (one load instead of a pointer chase)
  int nb16, NB;
  const int32_t* b16_ptr; const int32_t* b16_pos; const int32_t* b16_nz;
  const int32_t* inc_ptr; const int32_t* inc_mem;
  // workspace
  double* mk;      // [B][M]      EA/L
  double* mc;      // [B][M][d]   direction cosines
  double* mw;      // [B][M]      a*L*density
  double* mkc;     // [B][M][d(d+1)/2]  k * (c_i c_j), i <= j  (the distinct entries of truss.py:65-86)
  double* kv;      // [B][nnz]    K_ff non-zeros, grouped by tile (tile_ent order)
  double* wd;      // [B][nt][1024] inverses of the 16x16 diagonal blocks of every L(j,j) (DMMA B-operand layout)
  double* L;       // [B][ntiles][4096] packed lower tiles, fragment-major
  double* y;       // [B][n_pad]  rhs -> forward solution -> free displacements
  int32_t* status; // [B] 0 ok / k>0 pivot / <0 input problem
  // outputs
  double* u; double* ext; double* axial; double* weight; int32_t* info;
  double* u_free; double* react;      // compact outputs [B][n] / [B][s] (reference order), written by the recovery kernel
  const int32_t* free_ref;            // [n] DOF index of free DOF r in the reference's order
  double* fitness; uint8_t* flags;
  double allow_stress, allow_displace;
  int fitness_mode;
  int plan_stable;
  int band_warps;   // band path: 0 = choose by batch size, 2 = force the two-warp kernel (halves of a split batch share the SMs)
  int no_split;     // internal: this call is one half of a split batch
  int shared_k;     // band path: every system of the batch has the stiffness matrix of system 0 (load cases of one truss)
  // two-sided fused band kernel (tb_bandts.cu): program + its slice of the workspace; null = the 16x16 band kernels
  const TsPlan* ts;
  void* ts_ws;
  int ts_b0, ts_total;   // this call covers systems [ts_b0, ts_b0 + batch) of a workspace carved for ts_total systems
  double* kdebug;   // optional debug export of the assembled K values (tb_debug_assemble)
};

// launchers (return cudaError_t as int)
int tb_launch_small(const SmallArgs& a, int dim, cudaStream_t st);
int tb_small_smem_bytes(int dim, int nJ, int M, int max_n, int* threads);
int tb_launch_dense16(const SmallArgs& a, int dim, cudaStream_t st);   // -1: does not fit, use the CTA-per-truss kernel
int tb_dense16_smem_bytes(int dim, int nJ, int M, int max_n);
// does a system of this size fit one of the two fused shared-memory kernels?  (sizes alone are not enough: many members on
// few joints exhaust the per-warp / per-CTA shared memory long before the DOF limit)
bool tb_small_fits(int dim, int nJ, int M, int max_n);
int tb_launch_large(const LargeArgs& a, int num_sm, cudaStream_t st, int path);
size_t tb_large_workspace_bytes(int batch, int dim, int M, int n_pad, int64_t nnz, int path, int nb16, int NB);
void tb_large_carve(LargeArgs& a, void* ws, int path);
int tb_launch_band_chol(const LargeArgs& a, int num_sm, cudaStream_t st);
int tb_launch_assemble_only(const LargeArgs& a, int num_sm, cudaStream_t st);   // member products + K_ff values (a.kv) through a.q_*
int tb_launch_band_subst(const LargeArgs& a, int num_sm, cudaStream_t st);   // load cases against the factor of system 0
int tb_band_smem_bytes(int NB);

// Reverse mode (tb_adjoint.cu): the adjoint load before the adjoint solve, the sensitivities after it
struct TbAdjArgs {
  int batch, dim, nJ, M, N;
  const double* xyz; int64_t xyz_stride;
  const double* aed; int64_t aed_stride;
  const int32_t* conn; const int32_t* dof2free; const int32_t* inc_ptr; const int32_t* inc_mem;
  const double* g_u; const double* g_ext; const double* g_axial; const double* g_w;   // cotangents, null = 0
  double* r;             // [B][N] adjoint load (k_adj_rhs)
  const double* u;       // [B][N] forward displacements (k_sens)
  const double* lam;     // [B][N] adjoint solution (k_sens)
  const int32_t* info;   // [B]    status of the solve (k_sens)
  double* vec;           // [B][M][dim] per-member vectors in HBM, or null: shared memory (tb_adjoint_vec_in_smem)
  double* g_xyz; double* g_aed; double* g_force;                                      // outputs (g_aed required)
};
bool tb_adjoint_vec_in_smem(int dim, int M);
int tb_launch_adj_rhs(const TbAdjArgs& a, int num_sm, cudaStream_t st);
int tb_launch_sens(const TbAdjArgs& a, int num_sm, cudaStream_t st);

// Reverse mode of a ragged batch (tb_adjoint_ragged): packed layout of tb_ragged_in, local joint ids, one warp per truss
struct TbAdjRaggedArgs {
  int batch, dim, max_joint, max_member;
  const int64_t* joint_off; const int64_t* member_off;
  const double* xyz; const uint8_t* support; const int32_t* conn; const double* aed;
  const double* g_u; const double* g_ext; const double* g_axial; const double* g_w;   // cotangents, null = 0
  double* r;             // [d sum nJ] adjoint load (k_adj_rhs_ragged)
  const double* u;       // [d sum nJ] forward displacements (k_sens_ragged)
  const double* lam;     // [d sum nJ] adjoint solution (k_sens_ragged)
  const int32_t* info;   // [B]        status of the solve (k_sens_ragged)
  double* g_xyz; double* g_aed; double* g_force;                                      // outputs (g_aed required)
};
int tb_launch_adj_rhs_ragged(const TbAdjRaggedArgs& a, cudaStream_t st);
int tb_launch_sens_ragged(const TbAdjRaggedArgs& a, cudaStream_t st);

// Envelope path of ragged batches (tb_ragenv.cu): one CTA per truss, one scratch slot per CTA
struct RagEnvArgs {
  int batch, dim, max_joint, max_member;   // the slots are sized from max_joint / max_member
  int route_joint, route_member;           // > 0: skip the trusses up to these sizes (the fused kernels solved them)
  const int64_t* joint_off; const int64_t* member_off;
  const double* xyz; const uint8_t* support; const int32_t* conn; const double* aed; const double* force;
  double* u; double* ext; double* axial; double* weight; int32_t* info;
  int32_t* order;        // ordering mode when non-null: [sum nJ] joints in elimination order (local ids), nothing solved
  int64_t* envelope;     // ordering mode: [B] row-envelope entries of K_ff in that order
  void* scratch;         // grid * slot_bytes
  size_t slot_bytes;
  int env_smem;          // envelope doubles that fit the launch's dynamic shared memory
};
size_t tb_rag_env_slot_bytes(int dim, int max_joint, int max_member);
// persistent grid (at most one CTA per truss), dynamic shared memory and its envelope budget of a launch
int tb_rag_env_config(int dim, int max_joint, int max_member, int batch, int* grid, int* smem_bytes, int* env_smem);
int tb_launch_rag_env(const RagEnvArgs& a, int grid, int smem_bytes, cudaStream_t st);

// Modal analysis (tb_modes.cu): one CTA per system, the reduced matrix in shared memory
struct ModesArgs {
  int batch, nJ, M, N, n, n_modes, consistent, plan_stable, n_type;
  const double* xyz; int64_t xyz_stride;
  const double* aed; int64_t aed_stride;
  const int32_t* gene; int64_t gene_stride;
  const double* type_table;
  const double* jmass; int64_t jmass_stride;     // [B][nJ] non-structural joint mass, or null
  // plan maps (device): the scatter map's entries are in the internal order, free_ref / dof2free map them back
  const int32_t* conn; const int32_t* free_ref; const int32_t* dof2free;
  const int32_t* ent_row; const int32_t* ent_col; const int64_t* ent_ptr; int64_t nnz;
  const int32_t* ctr_member; const int32_t* ctr_local;
  const int32_t* inc_ptr; const int32_t* inc_mem;
  double* eigval; double* modes; int32_t* info;  // outputs [B][n_modes], [B][n_modes][N] or null, [B]
  double* slot;                                  // consistent mass: grid slots of n x n doubles, else null
};
// CTA size, dynamic shared memory and resident CTAs per SM of k_modes for n free DOFs (1 <= n <= TB_SMALL_MAX_DOF)
int tb_modes_config(int dim, int n, int* threads, int* smem, int* per_sm);
int tb_launch_modes(const ModesArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st);

// Linear buckling (tb_buckling, tb_modes.cu): k_modes' layout and plan maps in `base` (eigval = the load factors
// [B][n_modes], modes = [B][n_modes][N] or null, slot = grid slots of n x n doubles: K_ff and its factor; jmass and
// consistent are not read), plus the member axial forces of the reference state
struct BucklingArgs {
  ModesArgs base;
  const double* axial; int64_t axial_stride;     // [B][M] tension positive, stride 0 = shared
};
// CTA size, dynamic shared memory and resident CTAs per SM of k_buckling for n free DOFs (1 <= n <= TB_SMALL_MAX_DOF)
int tb_buckling_config(int dim, int n, int* threads, int* smem, int* per_sm);
int tb_launch_buckling(const BucklingArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st);

// Reverse mode of the modal analysis (tb_modes_adjoint): one warp per system, no scratch
struct ModesSensArgs {
  int batch, nJ, M, N, n_modes, consistent;
  const double* xyz; int64_t xyz_stride;
  const double* aed; int64_t aed_stride;
  const int32_t* conn; const int32_t* dof2free; const int32_t* inc_ptr; const int32_t* inc_mem;
  const double* eigval; const double* modes; const int32_t* info; const double* g_eigval;   // [B][k], [B][k][N], [B], [B][k]
  double* g_xyz; double* g_aed; double* g_jmass;                                            // outputs, null = skipped
};
int tb_launch_modes_sens(const ModesSensArgs& a, int dim, cudaStream_t st);

// Reverse mode of linear buckling (tb_buckling_adjoint): one warp per system, no scratch
struct BucklingSensArgs {
  int batch, nJ, M, N, n_modes;
  const double* xyz; int64_t xyz_stride;
  const double* aed; int64_t aed_stride;
  const double* axial; int64_t axial_stride;     // [B][M] the forward's member forces, stride 0 = shared
  const int32_t* conn; const int32_t* dof2free; const int32_t* inc_ptr; const int32_t* inc_mem;
  const double* factor; const double* modes; const int32_t* info; const double* g_factor;   // [B][k], [B][k][N], [B], [B][k]
  double* g_xyz; double* g_aed; double* g_axial;                                            // outputs, null = skipped
};
int tb_launch_buckling_sens(const BucklingSensArgs& a, int dim, cudaStream_t st);

// Modal analysis of a ragged batch (tb_modes_ragged): packed layout of tb_ragged_in, one CTA per truss
struct ModesRagArgs {
  int batch, max_joint, max_member, max_free, n_modes, consistent;   // max_free: the launch's free-DOF bound
  const int64_t* joint_off; const int64_t* member_off;
  const double* xyz; const uint8_t* support; const int32_t* conn; const double* aed;
  const double* jmass;                           // [sum nJ] non-structural joint mass, or null
  double* eigval; double* modes; int32_t* n_free; int32_t* info;   // [B][n_modes], [n_modes d sum nJ] or null, [B] or null, [B]
  double* slot;                                  // consistent mass: grid slots of max_free^2 doubles, else null
};
// CTA size, dynamic shared memory and resident CTAs per SM of k_modes_ragged for a free-DOF bound (1 <= bound <= 160)
int tb_modes_ragged_config(int dim, int bound, int* threads, int* smem, int* per_sm);
int tb_launch_modes_ragged(const ModesRagArgs& a, int dim, int grid, int threads, int smem, cudaStream_t st);

// Reverse mode of the ragged modal analysis (tb_modes_adjoint_ragged): one warp per truss, no scratch
struct ModesSensRagArgs {
  int batch, max_joint, max_member, n_modes, consistent;
  const int64_t* joint_off; const int64_t* member_off;
  const double* xyz; const uint8_t* support; const int32_t* conn; const double* aed;
  const double* eigval; const double* modes; const int32_t* info; const double* g_eigval;   // packed as the forward's
  double* g_xyz; double* g_aed; double* g_jmass;                                            // outputs, null = skipped
};
int tb_launch_modes_sens_ragged(const ModesSensRagArgs& a, int dim, cudaStream_t st);

// fragment-major offset of element (r, c) inside one 64x64 tile:
//   [k-half 2][row-block 8][k-slab 8][lane 32], lane = (r%8)*4 + c%4
// so that one DMMA m8n8k4 operand fragment (8 rows x 4 k) is 32 consecutive doubles and a
// 64-row x 32-k half tile is one contiguous 16 KB chunk (a single bulk copy).
__host__ __device__ __forceinline__ int tb_tile_off(int r, int c) {
  return ((((c >> 5) << 3) + (r >> 3)) << 8) + (((c >> 2) & 7) << 5) + ((r & 7) << 2) + (c & 3);
}
__host__ __device__ __forceinline__ int64_t tb_tile_index(int ti, int tj) {  // ti >= tj
  return (int64_t)ti * (ti + 1) / 2 + tj;
}
