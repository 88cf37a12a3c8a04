// Plan construction: the integer maps of the reference's assembly/reduction, built once per
// topology on the host and mirrored on the device.
//   DOF maps      <- Truss.GetDisplacementUnknownMask / SupportType.GetResistanceMask
//                    (slientruss3d/truss.py:319-326, type.py:48-74) + boolean-mask ordering (truss.py:343,348)
//   scatter map   <- the four d x d block "+=" of Truss.GetKMatrix (truss.py:307-316), as a
//                    CSR of per-entry contribution lists in ascending member order (no atomics)
//   stability     <- Truss.isStable / nResistance (truss.py:154-164, type.py:37-46)
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <new>
#include <numeric>
#include <tuple>

#include "tb_common.cuh"
#include "tb_ts.cuh"
#include "tb_blocks.cuh"

std::atomic<int64_t> g_tb_launches{0};

// ---- optional per-kernel event timing ---------------------------------------------------------
namespace {
struct ProfRec { int slot; cudaEvent_t e0, e1; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof_recs;
cudaEvent_t g_prof_open[TB_PROF_SLOTS];
}  // namespace
bool tb_prof_on() { return g_prof_on; }
void tb_prof_begin(int slot, cudaStream_t st) {
  if (!g_prof_on) return;
  cudaEventCreate(&g_prof_open[slot]);
  cudaEventRecord(g_prof_open[slot], st);
}
void tb_prof_end(int slot, cudaStream_t st) {
  if (!g_prof_on) return;
  ProfRec r;
  r.slot = slot;
  r.e0 = g_prof_open[slot];
  cudaEventCreate(&r.e1);
  cudaEventRecord(r.e1, st);
  g_prof_recs.push_back(r);
}
extern "C" int tb_profile_enable(int32_t on) {
  g_prof_on = on != 0;
  return TB_OK;
}
// Adds the elapsed milliseconds / launch counts recorded since the last read to ms[slot] / count[slot]
// (arrays of 8) and clears the records.  Synchronises on the recorded events.
extern "C" int tb_profile_read(float* ms, int64_t* count) {
  for (auto& r : g_prof_recs) {
    float t = 0.f;
    cudaError_t e = cudaEventSynchronize(r.e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, r.e0, r.e1);
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
    if (e != cudaSuccess) { g_prof_recs.clear(); return (int)e; }
    if (ms) ms[r.slot] += t;
    if (count) count[r.slot] += 1;
  }
  g_prof_recs.clear();
  return TB_OK;
}

namespace {

template <typename T>
int upload(T** dptr, const std::vector<T>& h) {
  *dptr = nullptr;
  size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
  cudaError_t e = cudaMalloc((void**)dptr, bytes);
  if (e != cudaSuccess) return (int)e;
  if (!h.empty()) {
    e = cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

struct Contrib {
  int32_t row, col, member, local;
};

}  // namespace

extern "C" int tb_plan_create(const tb_topology* topo, tb_plan** plan_out) {
  if (!topo || !plan_out) return TB_ERR_NULL;
  *plan_out = nullptr;
  const int d = topo->dim;
  if (d != 2 && d != 3) return TB_ERR_DIM;
  if (topo->n_joint < 0 || topo->n_member < 0) return TB_ERR_SIZE;
  if ((topo->n_member > 0 && !topo->conn) || (topo->n_joint > 0 && !topo->support)) return TB_ERR_NULL;
  if ((int64_t)topo->n_joint * d > (int64_t)1 << 24) return TB_ERR_TOO_LARGE;

  // The maps are host work; without a CUDA device the plan is host-only (maps can still be
  // queried) and every solve entry point returns TB_ERR_NO_DEVICE -- there is no CPU fallback.
  int ndev = 0;
  const bool has_dev = (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0);
  if (!has_dev) (void)cudaGetLastError();

  tb_plan* p = new (std::nothrow) tb_plan();
  if (!p) return TB_ERR_ALLOC;
  p->dim = d;
  p->nJ = topo->n_joint;
  p->M = topo->n_member;
  p->N = d * p->nJ;
  p->device = -1;
  if (has_dev) {
    cudaGetDevice(&p->device);
    cudaDeviceGetAttribute(&p->num_sm, cudaDevAttrMultiProcessorCount, p->device);
  }
  p->conn.assign(topo->conn, topo->conn + 2 * (size_t)p->M);
  p->support.assign(topo->support, topo->support + p->nJ);

  for (int m = 0; m < p->M; ++m)
    for (int e = 0; e < 2; ++e) {
      int j = p->conn[2 * m + e];
      if (j < 0 || j >= p->nJ) {
        delete p;
        return TB_ERR_INDEX;
      }
    }

  // ---- DOF maps: free DOFs in ascending DOF order (boolean-mask indexing, truss.py:343)
  p->dof2free.assign(p->N, -1);
  p->n_resist = 0;
  for (int j = 0; j < p->nJ; ++j) {
    int s = p->support[j];
    if (tb_support_bad(d, s)) {  // type.py:62,74
      delete p;
      return TB_ERR_SUPPORT;
    }
    for (int ax = 0; ax < d; ++ax) {
      bool resist = !tb_dof_free(s, ax);
      int dof = j * d + ax;
      if (resist) {
        p->sup_idx.push_back(dof);
        p->n_resist++;
      } else {
        p->dof2free[dof] = (int)p->free_idx.size();
        p->free_idx.push_back(dof);
      }
    }
  }
  p->n = (int)p->free_idx.size();
  p->s = (int)p->sup_idx.size();
  // truss.py:158-164
  if (d == 2)
    p->stable = (p->M + p->n_resist >= p->nJ * d);
  else
    p->stable = (p->n_resist >= 6) && (p->M + p->n_resist >= p->nJ * d);

  // ---- scatter map over the lower triangle of K_ff
  std::vector<Contrib> cs;
  cs.reserve((size_t)p->M * 4 * d * d);
  for (int m = 0; m < p->M; ++m) {
    // block order of truss.py:312-314: (A,B) = (0,0),(0,1),(1,0),(1,1)
    for (int A = 0; A < 2; ++A)
      for (int B = 0; B < 2; ++B)
        for (int i = 0; i < d; ++i)
          for (int j = 0; j < d; ++j) {
            int r = p->dof2free[p->conn[2 * m + A] * d + i];
            int c = p->dof2free[p->conn[2 * m + B] * d + j];
            if (r < 0 || c < 0 || r < c) continue;
            cs.push_back({r, c, m, (A * d + i) * 2 * d + (B * d + j)});
          }
  }
  std::stable_sort(cs.begin(), cs.end(), [](const Contrib& a, const Contrib& b) {
    return a.row != b.row ? a.row < b.row : a.col < b.col;
  });
  p->half_bw = 0;
  for (size_t i = 0; i < cs.size(); ++i) {
    if (i == 0 || cs[i].row != cs[i - 1].row || cs[i].col != cs[i - 1].col) {
      p->ent_row.push_back(cs[i].row);
      p->ent_col.push_back(cs[i].col);
      p->ent_ptr.push_back((int64_t)i);
      p->half_bw = std::max<int64_t>(p->half_bw, cs[i].row - cs[i].col);
    }
    p->ctr_member.push_back(cs[i].member);
    p->ctr_local.push_back(cs[i].local);
  }
  p->ent_ptr.push_back((int64_t)cs.size());

  // ---- internal elimination order.  The maps above are the reference's (ascending DOF index) and are what
  // tb_plan_get_maps / tb_plan_get_scatter report.  The factorisation is free to eliminate the free DOFs in any
  // order (the results agree to rounding), so the joints are renumbered by reverse Cuthill-McKee when that shrinks
  // the row envelope of K_ff (cube 12^3: half-bandwidth 3437 -> ~520, 10x fewer flops); every array the kernels
  // see (free_idx, dof2free, entry rows/columns, tiles, band blocks) is in the internal order.
  {
    const size_t nnz = p->ent_row.size();
    std::vector<int32_t> rank(p->nJ);            // joint -> position in the RCM order
    {
      std::vector<std::vector<int32_t>> adj(p->nJ);
      for (int m = 0; m < p->M; ++m) {
        const int a = p->conn[2 * m], b = p->conn[2 * m + 1];
        if (a != b) { adj[a].push_back(b); adj[b].push_back(a); }
      }
      for (auto& v : adj) { std::sort(v.begin(), v.end()); v.erase(std::unique(v.begin(), v.end()), v.end()); }
      std::vector<int32_t> order; order.reserve(p->nJ);
      std::vector<char> seen(p->nJ, 0);
      std::vector<int32_t> level(p->nJ);
      auto bfs_far = [&](int start, std::vector<int32_t>* visit) {   // BFS inside the component; returns a farthest node of minimum degree
        std::vector<int32_t> q{start};
        std::vector<char> mark(p->nJ, 0);
        mark[start] = 1; level[start] = 0;
        for (size_t h = 0; h < q.size(); ++h)
          for (int v : adj[q[h]]) if (!mark[v]) { mark[v] = 1; level[v] = level[q[h]] + 1; q.push_back(v); }
        int best = q.back();
        for (int v : q) if (level[v] == level[q.back()] && adj[v].size() < adj[best].size()) best = v;
        if (visit) *visit = q;
        return best;
      };
      for (int s0 = 0; s0 < p->nJ; ++s0) {
        if (seen[s0]) continue;
        int start = s0;
        for (int it = 0; it < 3; ++it) start = bfs_far(start, nullptr);   // pseudo-peripheral node
        std::vector<int32_t> q{start};
        seen[start] = 1;
        for (size_t h = 0; h < q.size(); ++h) {
          std::vector<int32_t> nb;
          for (int v : adj[q[h]]) if (!seen[v]) { seen[v] = 1; nb.push_back(v); }
          std::stable_sort(nb.begin(), nb.end(), [&](int x, int y) { return adj[x].size() < adj[y].size(); });
          q.insert(q.end(), nb.begin(), nb.end());
        }
        order.insert(order.end(), q.begin(), q.end());
      }
      std::reverse(order.begin(), order.end());
      for (int i = 0; i < p->nJ; ++i) rank[order[i]] = i;
    }
    // candidate order of the free DOFs: by (RCM rank of the joint, axis)
    std::vector<int32_t> cand(p->n);
    std::iota(cand.begin(), cand.end(), 0);
    std::stable_sort(cand.begin(), cand.end(), [&](int x, int y) {
      const int jx = p->free_idx[x] / d, jy = p->free_idx[y] / d;
      return rank[jx] != rank[jy] ? rank[jx] < rank[jy] : x < y;
    });
    std::vector<int32_t> inv(p->n);
    for (int i = 0; i < p->n; ++i) inv[cand[i]] = i;
    auto envelope = [&](const std::vector<int32_t>* map) {   // sum over rows of (row - first column + 1)^2: flop proxy
      std::vector<int32_t> first(p->n);
      std::iota(first.begin(), first.end(), 0);
      for (size_t e = 0; e < nnz; ++e) {
        int r = p->ent_row[e], c = p->ent_col[e];
        if (map) { r = (*map)[r]; c = (*map)[c]; if (r < c) std::swap(r, c); }
        first[r] = std::min(first[r], c);
      }
      double w = 0.0;
      for (int i = 0; i < p->n; ++i) w += (double)(i - first[i] + 1) * (i - first[i] + 1);
      return w;
    };
    const char* env = getenv("TB_NO_REORDER");
    const bool allow = !(env && env[0] == '1');
    const bool use = allow && p->n > 0 && envelope(&inv) < 0.85 * envelope(nullptr);
    p->reordered = use ? 1 : 0;
    p->perm.resize(p->n);
    for (int i = 0; i < p->n; ++i) p->perm[i] = use ? cand[i] : i;          // internal index -> reference free index
    p->free_int.resize(p->n);
    p->d2f_int.assign(p->N, -1);
    for (int i = 0; i < p->n; ++i) {
      p->free_int[i] = p->free_idx[p->perm[i]];
      p->d2f_int[p->free_int[i]] = i;
    }
    p->int_row.resize(nnz);
    p->int_col.resize(nnz);
    p->half_bw = 0;
    for (size_t e = 0; e < nnz; ++e) {
      int r = p->ent_row[e], c = p->ent_col[e];
      if (use) { r = inv[r]; c = inv[c]; if (r < c) std::swap(r, c); }
      p->int_row[e] = r;
      p->int_col[e] = c;
      p->half_bw = std::max<int64_t>(p->half_bw, r - c);
    }
  }
  // from here on "row/col" are the INTERNAL ones
  const std::vector<int32_t>& irow = p->int_row;
  const std::vector<int32_t>& icol = p->int_col;

  // ---- path + tile grouping of entries for the blocked path
  p->path = tb_small_fits(d, p->nJ, p->M, p->n) ? 0 : 1;     // (the shared-memory budgets of the fused kernels, not just the sizes)
  // (a narrow band promotes path 1 to the band path 2 once the band view is known, below)
  p->n_pad = std::max(TB_TILE, (p->n + TB_TILE - 1) / TB_TILE * TB_TILE);
  p->nt = p->n_pad / TB_TILE;
  {
    const int64_t ntiles = (int64_t)p->nt * (p->nt + 1) / 2;
    const size_t nnz = p->ent_row.size();
    std::vector<int64_t> cnt(ntiles + 1, 0);
    for (size_t e = 0; e < nnz; ++e) cnt[tb_tile_index(irow[e] / TB_TILE, icol[e] / TB_TILE) + 1]++;
    for (int64_t t = 0; t < ntiles; ++t) cnt[t + 1] += cnt[t];
    p->tile_ent_ptr = cnt;
    p->tile_ent.assign(nnz, 0);
    std::vector<int64_t> pos(cnt.begin(), cnt.end() - 1);
    for (size_t e = 0; e < nnz; ++e)
      p->tile_ent[pos[tb_tile_index(irow[e] / TB_TILE, icol[e] / TB_TILE)]++] = (int32_t)e;
    p->tile_pos.assign(nnz, 0);
    p->q_ptr.assign(nnz + 1, 0);
    for (size_t q = 0; q < nnz; ++q) {
      const int e = p->tile_ent[q];
      p->tile_pos[q] = tb_tile_off(irow[e] % TB_TILE, icol[e] % TB_TILE);
      for (int64_t c = p->ent_ptr[e]; c < p->ent_ptr[e + 1]; ++c) {
        const int loc = p->ctr_local[c], la = loc / (2 * d), lb = loc % (2 * d);
        const int A = la / d, i = la % d, B = lb / d, j = lb % d;
        const int lo = std::min(i, j), hi = std::max(i, j);
        const int ij = lo * d - lo * (lo - 1) / 2 + (hi - lo);   // index of (lo,hi), lo <= hi, row-major upper triangle
        p->q_pack.push_back((p->ctr_member[c] << 4) | ((A != B) << 3) | ij);
      }
      p->q_ptr[q + 1] = (int32_t)p->q_pack.size();
    }
  }

  // ---- block-level symbolic Cholesky: a tile of L is structurally non-zero if K_ff has entries in
  // it or an earlier block column couples its block row and block column.  TB_DENSE_TILES=1 treats
  // every tile as non-zero (dense reference mode for roofline measurements).
  {
    const int nt = p->nt;
    const int64_t ntiles = (int64_t)nt * (nt + 1) / 2;
    const char* env = getenv("TB_DENSE_TILES");
    const bool dense = env && env[0] == '1';
    p->tile_nz.assign(ntiles, 0);
    p->prod_ptr.assign(ntiles + 1, 0);
    std::vector<std::vector<int32_t>> lists(ntiles);
    for (int j = 0; j < nt; ++j)
      for (int i = j; i < nt; ++i) {
        const int64_t t = tb_tile_index(i, j);
        bool nz = dense || i == j || p->tile_ent_ptr[t + 1] > p->tile_ent_ptr[t];
        for (int k = 0; k < j; ++k)
          if (p->tile_nz[tb_tile_index(i, k)] && p->tile_nz[tb_tile_index(j, k)]) {
            lists[t].push_back(k);
            nz = true;
          }
        p->tile_nz[t] = nz ? 1 : 0;
      }
    p->n_tiles_nz = 0;
    double fl = 0.0;
    const double T3 = (double)TB_TILE * TB_TILE * TB_TILE;
    for (int64_t t = 0; t < ntiles; ++t) {
      p->prod_ptr[t + 1] = p->prod_ptr[t] + (p->tile_nz[t] ? (int32_t)lists[t].size() : 0);
      if (p->tile_nz[t]) {
        p->n_tiles_nz++;
        p->prod_k.insert(p->prod_k.end(), lists[t].begin(), lists[t].end());
      }
    }
    for (int j = 0; j < nt; ++j)
      for (int i = j; i < nt; ++i) {
        const int64_t t = tb_tile_index(i, j);
        if (!p->tile_nz[t]) continue;
        const double np = (double)lists[t].size();
        if (i == j) fl += np * T3 + T3 / 3.0 + 2.0 * TB_TILE * TB_TILE;          // syrk-like update + potrf + two trsv
        else fl += np * 2.0 * T3 + T3 + 4.0 * TB_TILE * TB_TILE;                 // gemm update + trsm + two gemv
      }
    p->chol_flops = fl;
  }

  // ---- band view: 16x16 blocks, entries grouped per block column (then block offset, row, column);
  // row envelope of K_ff (fill stays inside it) and the flops an envelope Cholesky needs
  {
    const size_t nnz = p->ent_row.size();
    p->nb16 = std::max(1, (p->n + 15) / 16);
    int NB = 1;
    for (size_t e = 0; e < nnz; ++e) NB = std::max(NB, irow[e] / 16 - icol[e] / 16);
    p->NB = NB;
    std::vector<int32_t> order(nnz);
    std::iota(order.begin(), order.end(), 0);
    // order: block column, then diagonal block before the blocks below it (the two-warp kernel gives the diagonal
    // block to its factor warp and the rest to its trailing warp), then block row, row, column
    auto sub = [&](int e) { return irow[e] / 16 == icol[e] / 16 ? 0 : 1; };
    auto key = [&](int e) { return std::make_tuple(icol[e] / 16, irow[e] / 16, irow[e], icol[e]); };
    std::sort(order.begin(), order.end(), [&](int x, int y) { return key(x) < key(y); });
    p->b16_ptr.assign(2 * (size_t)p->nb16 + 1, 0);
    p->b16_pos.assign(nnz, 0);
    p->bq_ptr.assign(nnz + 1, 0);
    for (size_t q = 0; q < nnz; ++q) {
      const int e = order[q], r = irow[e], c = icol[e];
      p->b16_ptr[2 * (c / 16) + sub(e) + 1]++;
      const int rr = r % 16, cc = c % 16;
      p->b16_pos[q] = ((r / 16 - c / 16) << 8) | tbblk::b16_off(rr, cc);   // tb_blocks.cuh: swizzled fragment layout
      for (int64_t k = p->ent_ptr[e]; k < p->ent_ptr[e + 1]; ++k) {
        const int loc = p->ctr_local[k], la = loc / (2 * d), lb = loc % (2 * d);
        const int A = la / d, i = la % d, B = lb / d, j = lb % d;
        const int lo = std::min(i, j), hi = std::max(i, j);
        p->bq_pack.push_back((p->ctr_member[k] << 4) | ((A != B) << 3) | (lo * d - lo * (lo - 1) / 2 + (hi - lo)));
      }
      p->bq_ptr[q + 1] = (int32_t)p->bq_pack.size();
    }
    for (int c = 0; c < 2 * p->nb16; ++c) p->b16_ptr[c + 1] += p->b16_ptr[c];
    // block-level symbolic factorisation of the band: bit e of b16_nz[c] <=> block (c+e, c) of L is non-zero
    p->b16_nz.assign(p->nb16, 1);
    for (size_t e = 0; e < nnz; ++e) {
      const int bc = icol[e] / 16, be = irow[e] / 16 - bc;
      if (be < 31) p->b16_nz[bc] |= (1 << be);
    }
    p->b16_blocks_nz = 0;
    p->b16_products = 0;
    for (int c = 0; c < p->nb16; ++c) {
      const unsigned m = (unsigned)p->b16_nz[c];
      for (int e1 = 1; e1 <= NB && e1 < 31; ++e1) {
        if (!((m >> e1) & 1u)) continue;
        for (int e2 = e1; e2 <= NB && e2 < 31; ++e2)
          if ((m >> e2) & 1u) {
            p->b16_nz[c + e1] |= (1 << (e2 - e1));   // L(c+e2, c) L(c+e1, c)^T lands in block (c+e2, c+e1)
            p->b16_products++;
          }
      }
      for (int e = 0; e <= NB && e < 31; ++e) p->b16_blocks_nz += (m >> e) & 1u;
    }
    std::vector<int32_t> first(p->n);
    std::iota(first.begin(), first.end(), 0);
    for (size_t e = 0; e < nnz; ++e) first[irow[e]] = std::min(first[irow[e]], icol[e]);
    double fl = 0.0;
    int64_t env = 0;
    for (int i = 0; i < p->n; ++i) {
      env += i - first[i] + 1;
      for (int j = first[i]; j <= i; ++j) fl += 2.0 * (j - std::max(first[i], first[j])) + 1.0;   // dot + divide / sqrt
      fl += 4.0 * (i - first[i]) + 2.0;                                                            // two triangular solves
    }
    p->envelope_size = env;
    p->envelope_flops = fl;
  }

  // ---- joint incidence lists (ascending member, then end)
  p->inc_ptr.assign(p->nJ + 1, 0);
  for (int m = 0; m < p->M; ++m)
    for (int e = 0; e < 2; ++e) p->inc_ptr[p->conn[2 * m + e] + 1]++;
  for (int j = 0; j < p->nJ; ++j) p->inc_ptr[j + 1] += p->inc_ptr[j];
  p->inc_mem.assign(2 * (size_t)p->M, 0);
  {
    std::vector<int32_t> pos(p->inc_ptr.begin(), p->inc_ptr.end() - 1);
    for (int m = 0; m < p->M; ++m)
      for (int e = 0; e < 2; ++e) p->inc_mem[pos[p->conn[2 * m + e]]++] = m * 2 + e;
  }

  // first contribution of every entry inline (85 % of the entries of a truss have exactly one: a member joining two
  // different joints), so the K-value kernels need one coalesced load per entry instead of a pointer chase
  // ... and the entries with several contributions (the same-joint entries: one per member at that joint) are listed
  // separately, so that the lanes of a warp either all take the one-load path or all walk lists of similar length
  auto firsts = [](const std::vector<int32_t>& ptr, const std::vector<int32_t>& pack, std::vector<int32_t>& first,
                   std::vector<int32_t>& multi) {
    const size_t nq = ptr.empty() ? 0 : ptr.size() - 1;
    first.assign(nq, 0);
    multi.clear();
    for (size_t q = 0; q < nq; ++q) {
      const int cnt = ptr[q + 1] - ptr[q];
      first[q] = (cnt > 0 ? pack[ptr[q]] : 0) | (cnt > 1 ? (int32_t)0x80000000u : 0);
      if (cnt > 1) multi.push_back((int32_t)q);
    }
  };
  firsts(p->q_ptr, p->q_pack, p->q_first, p->q_multi);
  firsts(p->bq_ptr, p->bq_pack, p->bq_first, p->bq_multi);

  {   // two-sided 8x8 band program of the fused band kernel (host arrays always; device mirrors with a device)
    const int rc_ts = tb_ts_build(p);
    if (rc_ts) {
      tb_plan_destroy(p);
      return rc_ts;
    }
  }
  if (p->path == 1 && p->NB <= TB_BAND_MAX_NB) {
    const char* env = getenv("TB_NO_BAND");
    if (!(env && env[0] == '1')) p->path = 2;
  }
  if (!has_dev) {
    *plan_out = p;
    return TB_OK;
  }
  int rc = 0;
  if (!rc) rc = upload(&p->d_conn, p->conn);
  if (!rc) rc = upload(&p->d_support, p->support);
  if (!rc) rc = upload(&p->d_free_idx, p->free_int);
  if (!rc) rc = upload(&p->d_dof2free, p->d2f_int);
  if (!rc) rc = upload(&p->d_sup_idx, p->sup_idx);
  if (!rc) rc = upload(&p->d_free_ref, p->free_idx);
  if (!rc) rc = upload(&p->d_ent_row, p->int_row);
  if (!rc) rc = upload(&p->d_ent_col, p->int_col);
  if (!rc) rc = upload(&p->d_ent_ptr, p->ent_ptr);
  if (!rc) rc = upload(&p->d_ctr_member, p->ctr_member);
  if (!rc) rc = upload(&p->d_ctr_local, p->ctr_local);
  if (!rc) rc = upload(&p->d_tile_ent_ptr, p->tile_ent_ptr);
  if (!rc) rc = upload(&p->d_tile_ent, p->tile_ent);
  if (!rc) rc = upload(&p->d_tile_pos, p->tile_pos);
  if (!rc) rc = upload(&p->d_q_ptr, p->q_ptr);
  if (!rc) rc = upload(&p->d_q_pack, p->q_pack);
  if (!rc) rc = upload(&p->d_q_first, p->q_first);
  if (!rc) rc = upload(&p->d_bq_first, p->bq_first);
  if (!rc) rc = upload(&p->d_q_multi, p->q_multi);
  if (!rc) rc = upload(&p->d_bq_multi, p->bq_multi);
  if (!rc) rc = upload(&p->d_b16_ptr, p->b16_ptr);
  if (!rc) rc = upload(&p->d_b16_pos, p->b16_pos);
  if (!rc) rc = upload(&p->d_b16_nz, p->b16_nz);
  if (!rc) rc = upload(&p->d_bq_ptr, p->bq_ptr);
  if (!rc) rc = upload(&p->d_bq_pack, p->bq_pack);
  if (!rc) rc = upload(&p->d_tile_nz, p->tile_nz);
  if (!rc) rc = upload(&p->d_prod_ptr, p->prod_ptr);
  if (!rc) rc = upload(&p->d_prod_k, p->prod_k);
  if (!rc) rc = upload(&p->d_inc_ptr, p->inc_ptr);
  if (!rc) rc = upload(&p->d_inc_mem, p->inc_mem);
  if (rc) {
    tb_plan_destroy(p);
    return rc;
  }
  *plan_out = p;
  return TB_OK;
}

extern "C" void tb_plan_destroy(tb_plan* p) {
  if (!p) return;
  tb_ts_destroy(p->ts, p->device >= 0);
  p->ts = nullptr;
  if (p->device < 0) {
    delete p;
    return;
  }
  cudaFree(p->d_conn);
  cudaFree(p->d_support);
  cudaFree(p->d_free_idx);
  cudaFree(p->d_dof2free);
  cudaFree(p->d_sup_idx);
  cudaFree(p->d_free_ref);
  cudaFree(p->compact_u);
  cudaFree(p->compact_ext);
  cudaFree(p->d_ent_row);
  cudaFree(p->d_ent_col);
  cudaFree(p->d_ent_ptr);
  cudaFree(p->d_ctr_member);
  cudaFree(p->d_ctr_local);
  cudaFree(p->d_tile_ent_ptr);
  cudaFree(p->d_tile_ent);
  cudaFree(p->d_tile_pos);
  cudaFree(p->d_q_ptr);
  cudaFree(p->d_q_pack);
  cudaFree(p->d_q_first);
  cudaFree(p->d_bq_first);
  cudaFree(p->d_q_multi);
  cudaFree(p->d_bq_multi);
  cudaFree(p->d_b16_ptr);
  cudaFree(p->d_b16_pos);
  cudaFree(p->d_b16_nz);
  cudaFree(p->d_bq_ptr);
  cudaFree(p->d_bq_pack);
  cudaFree(p->d_tile_nz);
  cudaFree(p->d_prod_ptr);
  cudaFree(p->d_prod_k);
  cudaFree(p->d_inc_ptr);
  cudaFree(p->d_inc_mem);
  if (p->ws_event) {
    cudaEventSynchronize(p->ws_event);          // (the last call's kernels may still read the adjoint scratch)
    cudaEventDestroy(p->ws_event);
  }
  cudaFree(p->adj_buf);
  cudaFree(p->ws);
  cudaFree(p->stage_dev);
  for (int i = 0; i < TB_ASYNC_SLOTS; ++i) {
    if (p->async_done[i]) cudaEventSynchronize(p->async_done[i]);     // (a pipelined call may still be in flight)
    cudaFree(p->stage_async[i]);
    if (p->async_in[i]) cudaEventDestroy(p->async_in[i]);
    if (p->async_k[i]) cudaEventDestroy(p->async_k[i]);
    if (p->async_done[i]) cudaEventDestroy(p->async_done[i]);
  }
  if (p->stage_pinned) cudaFreeHost(p->stage_pinned);
  delete p;
}

extern "C" int tb_plan_query(const tb_plan* p, tb_plan_info* o) {
  if (!p || !o) return TB_ERR_NULL;
  o->dim = p->dim;
  o->n_joint = p->nJ;
  o->n_member = p->M;
  o->n_dof = p->N;
  o->n_free = p->n;
  o->n_support = p->s;
  o->n_resist = p->n_resist;
  o->stable = p->stable;
  o->path = p->path;
  o->n_pad = p->n_pad;
  o->nnz_lower = (int64_t)p->ent_row.size();
  o->n_contrib = (int64_t)p->ctr_member.size();
  o->half_bandwidth = p->half_bw;
  o->n_tiles = (int64_t)p->nt * (p->nt + 1) / 2;
  o->n_tiles_nonzero = p->n_tiles_nz;
  o->n_tile_products = (int64_t)p->prod_k.size();
  o->chol_flops = p->chol_flops;
  o->band_blocks = p->NB;
  o->envelope_size = p->envelope_size;
  o->envelope_flops = p->envelope_flops;
  o->reordered = p->reordered;
  o->band_blocks_nonzero = p->b16_blocks_nz;
  o->band_products = p->b16_products;
  return TB_OK;
}

extern "C" int tb_plan_set_path(tb_plan* p, int32_t path) {
  if (!p) return TB_ERR_NULL;
  if (path < 0 || path > 2) return TB_ERR_SIZE;
  if (path == 2 && p->NB > TB_BAND_MAX_NB) return TB_ERR_TOO_LARGE;
  if (path == 0 && !tb_small_fits(p->dim, p->nJ, p->M, p->n)) return TB_ERR_TOO_LARGE;
  p->path = path;
  return TB_OK;
}

extern "C" int tb_plan_get_maps(const tb_plan* p, int32_t* free_idx, int32_t* dof2free, int32_t* sup_idx) {
  if (!p) return TB_ERR_NULL;
  if (free_idx && p->n) memcpy(free_idx, p->free_idx.data(), sizeof(int32_t) * p->n);
  if (dof2free && p->N) memcpy(dof2free, p->dof2free.data(), sizeof(int32_t) * p->N);
  if (sup_idx && p->s) memcpy(sup_idx, p->sup_idx.data(), sizeof(int32_t) * p->s);
  return TB_OK;
}

extern "C" int tb_plan_get_scatter(const tb_plan* p, int32_t* row, int32_t* col, int64_t* contrib_ptr,
                                   int32_t* contrib_member, int32_t* contrib_local) {
  if (!p) return TB_ERR_NULL;
  size_t nnz = p->ent_row.size(), nc = p->ctr_member.size();
  if (row && nnz) memcpy(row, p->ent_row.data(), sizeof(int32_t) * nnz);
  if (col && nnz) memcpy(col, p->ent_col.data(), sizeof(int32_t) * nnz);
  if (contrib_ptr) memcpy(contrib_ptr, p->ent_ptr.data(), sizeof(int64_t) * (nnz + 1));
  if (contrib_member && nc) memcpy(contrib_member, p->ctr_member.data(), sizeof(int32_t) * nc);
  if (contrib_local && nc) memcpy(contrib_local, p->ctr_local.data(), sizeof(int32_t) * nc);
  return TB_OK;
}

extern "C" int tb_small_path_fits(int32_t dim, int32_t n_joint, int32_t n_member) {
  if (dim != 2 && dim != 3) return 0;
  return tb_small_fits(dim, n_joint, n_member, n_joint * dim) ? 1 : 0;       // (ragged batches size by d * nJ: every DOF free)
}

extern "C" int tb_small_path_limits(int32_t* max_dof, int32_t* max_member) {
  if (max_dof) *max_dof = TB_SMALL_MAX_DOF;
  if (max_member) *max_member = TB_SMALL_MAX_MEMBER;
  return TB_OK;
}

extern "C" int64_t tb_launch_count(void) { return g_tb_launches.load(); }
extern "C" int tb_version(void) { return TB_VERSION; }

extern "C" const char* tb_strerror(int code) {
  switch (code) {
    case TB_OK: return "ok";
    case TB_ERR_NULL: return "required pointer is NULL";
    case TB_ERR_DIM: return "dimension of truss must be 2 or 3";
    case TB_ERR_SIZE: return "negative or inconsistent size";
    case TB_ERR_INDEX: return "member refers to a joint that does not exist";
    case TB_ERR_SUPPORT: return "invalid support type for this dimension";
    case TB_ERR_TOO_LARGE: return "system too large for the selected path";
    case TB_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    case TB_ERR_ALLOC: return "allocation failed";
    case TB_ERR_WRONG_DEVICE: return "the plan belongs to another CUDA device than the current one";
    case TB_ERR_JSON: return "not a truss JSON document of the reference's format";
    default: break;
  }
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
  return "unknown error";
}
