/*
 * truss_b200.h -- C ABI of the B200-native batched direct-stiffness truss solver.
 *
 * The reference (slientruss3d v2.0.3) has no FFI/plugin interface: its boundary for
 * this path is the Python method Truss.Solve() (slientruss3d/truss.py:329-364) and
 * its two batched callers, GA.GetFitness (slientruss3d/ga.py:132-149) and the
 * generator's solve site (slientruss3d/generate.py:354-357).  This header is the
 * C-level boundary a reference-side binding (ctypes, see INTEGRATION.md) attaches to;
 * each entry point names the reference lines it replaces.
 *
 * Conventions
 *   - all floating point is IEEE binary64; all indices are int32 unless noted
 *   - dim d in {2,3}; nJ joints, M members, N = d*nJ DOFs (index j*d + axis, as in
 *     truss.py:303-304), n free DOFs, s = N - n supported DOFs
 *   - support codes are the reference's SupportType ints (type.py:30-35):
 *     NO=0 PIN=1 ROLLER_X=2 ROLLER_Y=3 ROLLER_Z=4
 *   - every function returns 0 on success, <0 for an argument error, >0 for a CUDA
 *     error (cudaError_t value); nothing throws across the ABI; tb_strerror() names codes
 *   - numerical status is PER SYSTEM in info[b]:
 *        0  solved
 *        k>0  leading minor k of the reduced stiffness matrix is not positive definite
 *             (LAPACK potrf convention; the reference would raise numpy LinAlgError or
 *             return garbage for a singular K, truss.py:343).  The two-sided band kernel
 *             (k_band_ts) eliminates its top part top-down and its bottom part bottom-up
 *             at once: k - 1 is the plan-order row of the first non-positive pivot of the
 *             part that failed, and of the bottom part when both fail (DESIGN.md section 3).
 *             The envelope kernel of ragged batches: k - 1 is the position of the first
 *             non-positive (or subnormal) pivot in the truss's elimination order
 *             (tb_ragged_env_order)
 *        -1  fails the counting rule of truss.py:158-164 (reference: TrussNotStableError)
 *        -2  a member has zero length (reference: ZeroDivisionError, truss.py:58)
 *        -3  invalid support code for this dim (device-side check; type.py:48-74)
 *        -4  a member or gene index is out of range (device-side check), or a ragged truss is larger
 *            than the batch's max_joint / max_member
 *     outputs of a system with info != 0 are zero-filled (fitness: +inf), never NaN
 *   - "device" entry points take device pointers, enqueue on the given stream and do not
 *     synchronise; "_host" entry points take host pointers and perform the H2D copies,
 *     the solve, and the D2H copies themselves (they synchronise before returning)
 *   - the caller owns every in/out buffer; a plan owns only its maps and workspace
 *   - devices: a plan belongs to the CUDA device that was current when it was created; every solve checks that this
 *     device is current (TB_ERR_WRONG_DEVICE otherwise).  Kernel attributes, helper streams and staging arenas are kept
 *     per device, so one process may hold plans on several GPUs.
 *   - threads: a plan owns ONE workspace, so calls on the same plan are serialised (a mutex inside the plan) and
 *     ordered across streams (the library records an event after the last kernel of a call and makes a call on a
 *     different stream wait for it) -- two threads / two streams may use one plan, they just do not overlap; use one
 *     plan per thread or stream for concurrency.  The *_host entry points are additionally serialised per process
 *     (they share the helper streams and staging arenas).  A call captured into a CUDA graph must stay on one stream.
 *     On an error return no copy or kernel of the failed call is still in flight against the caller's buffers.
 */
#ifndef TRUSS_B200_H
#define TRUSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TB_VERSION 100

/* error codes (negative = argument errors) */
#define TB_OK 0
#define TB_ERR_NULL (-1)       /* required pointer is NULL */
#define TB_ERR_DIM (-2)        /* dim not in {2,3} (utils.py:70-74 CheckDim) */
#define TB_ERR_SIZE (-3)       /* negative / inconsistent sizes */
#define TB_ERR_INDEX (-4)      /* connectivity refers to a joint that does not exist */
#define TB_ERR_SUPPORT (-5)    /* invalid support code for this dim (type.py:48-74) */
#define TB_ERR_TOO_LARGE (-6)  /* system too large for the selected path / workspace */
#define TB_ERR_NO_DEVICE (-7)  /* no CUDA device: there is NO CPU fallback */
#define TB_ERR_ALLOC (-8)
#define TB_ERR_WRONG_DEVICE (-9) /* the plan was created on another CUDA device than the current one */
#define TB_ERR_JSON (-10)      /* a document is not a truss JSON file of the reference's format (truss.py:401-421) */

/* per-system status codes in info[] */
#define TB_INFO_OK 0
#define TB_INFO_NOT_STABLE (-1)
#define TB_INFO_ZERO_LENGTH (-2)
#define TB_INFO_BAD_SUPPORT (-3)
#define TB_INFO_BAD_INDEX (-4)

typedef struct tb_plan tb_plan; /* opaque */

/* Topology shared by every system of a uniform batch (one Truss, many genes / load cases /
 * geometries).  Host pointers; copied by tb_plan_create. */
typedef struct {
  int32_t dim;            /* Truss(dim), truss.py:110-112 */
  int32_t n_joint;        /* Truss.nJoint */
  int32_t n_member;       /* Truss.nMember */
  const int32_t* conn;    /* [M,2] (jointID0, jointID1), truss.py:184-187 */
  const uint8_t* support; /* [nJ] SupportType codes, truss.py:174-175 */
} tb_topology;

typedef struct {
  int32_t dim, n_joint, n_member;
  int32_t n_dof;       /* N */
  int32_t n_free;      /* n */
  int32_t n_support;   /* s */
  int32_t n_resist;    /* Truss.nResistance, truss.py:154-156 */
  int32_t stable;      /* Truss.isStable, truss.py:158-164 */
  int32_t path;        /* 0 = fused shared-memory kernel, 1 = tiled (64x64) pipeline, 2 = band (16x16 blocks) pipeline */
  int32_t n_pad;       /* padded order used by the blocked pipeline (multiple of the tile) */
  int64_t nnz_lower;   /* structural non-zeros of the lower triangle of K_ff */
  int64_t n_contrib;   /* entries of the scatter map (member contributions to the lower triangle) */
  int64_t half_bandwidth; /* max (row - col) over structural non-zeros of K_ff in the internal elimination order */
  /* blocked pipeline: block-level symbolic factorisation over 64x64 tiles of the lower triangle */
  int64_t n_tiles;          /* nt(nt+1)/2 */
  int64_t n_tiles_nonzero;  /* tiles of L that are structurally non-zero (the only ones touched) */
  int64_t n_tile_products;  /* tile x tile^T updates the factorisation performs */
  double chol_flops;        /* flops of that block-sparse factorisation + the two triangular solves */
  /* band path: 16x16 blocks */
  int32_t band_blocks;      /* sub-diagonal 16x16 blocks per block column (the band path needs <= 8) */
  int64_t envelope_size;    /* entries inside the row envelope of K_ff (fill stays inside it) */
  double envelope_flops;    /* flops of an envelope Cholesky + two triangular solves: the algorithmic work */
  int32_t reordered;        /* 1: the factorisation eliminates the free DOFs in reverse Cuthill-McKee order of the joints
                               (internal only: tb_plan_get_maps / tb_plan_get_scatter stay in the reference's order) */
  int64_t band_blocks_nonzero; /* band path: structurally non-zero 16x16 blocks of L */
  int64_t band_products;       /* band path: 16x16 block products of the factorisation */
} tb_plan_info;

/* Build the integer maps of truss.py:319-326 (free/supported DOF order = ascending DOF index)
 * and the deterministic scatter map replacing the "+=" block loop of truss.py:307-316.
 * The maps are built on the host and mirrored on the device.  Without a CUDA device the
 * plan is host-only: maps can be queried, every solve returns TB_ERR_NO_DEVICE. */
int tb_plan_create(const tb_topology* topo, tb_plan** plan_out);
void tb_plan_destroy(tb_plan* plan);
int tb_plan_query(const tb_plan* plan, tb_plan_info* info_out);
/* Override the automatic path choice (0 fused shared-memory kernel, 1 tiled pipeline, 2 band
 * pipeline); used by the parity tests to push every truss through every pipeline. */
int tb_plan_set_path(tb_plan* plan, int32_t path);

/* Host copies of the DOF maps, for bit-exact checks against
 * np.nonzero(GetDisplacementUnknownMask()) (truss.py:319-326):
 *   free_idx[n]  DOF index of free DOF r;  dof2free[N]  inverse map, -1 at supported DOFs;
 *   sup_idx[s]   DOF index of supported DOF r.  Any pointer may be NULL. */
int tb_plan_get_maps(const tb_plan* plan, int32_t* free_idx, int32_t* dof2free, int32_t* sup_idx);

/* Host copy of the scatter map (CSR over the structural non-zeros of the lower triangle of
 * K_ff, row-major order): entry e covers K_ff[row[e], col[e]] and sums contributions
 * contrib_ptr[e] .. contrib_ptr[e+1]-1 in ascending member order (the order of the
 * reference's loop, truss.py:310); contribution c is member contrib_member[c], local
 * stiffness entry (contrib_local[c] / 2d, contrib_local[c] % 2d) of truss.py:65-86.
 * Any pointer may be NULL; sizes are tb_plan_info.nnz_lower / n_contrib. */
int tb_plan_get_scatter(const tb_plan* plan, int32_t* row, int32_t* col, int64_t* contrib_ptr,
                        int32_t* contrib_member, int32_t* contrib_local);

/* One uniform batch: B systems sharing the plan's topology.  A stride is the distance in
 * ELEMENTS between consecutive systems; stride 0 shares the array across the batch. */
typedef struct {
  int32_t batch;
  const double* joint_xyz;   /* [B][nJ][d]  joint positions, truss.py:174-175 */
  int64_t joint_stride;
  const double* member_aed;  /* [B][M][3]   (a, e, density) per member, type.py:5-9; or NULL with gene */
  int64_t member_stride;
  const int32_t* gene;       /* [B][M]      indices into type_table (ga.py:132-137); or NULL */
  int64_t gene_stride;
  const double* type_table;  /* [T][3]      (a, e, density) per member type */
  int32_t n_type;
  const double* force;       /* [B][N]      dense load vector, truss.py:303-304 */
  int64_t force_stride;
} tb_batch_in;

/* Outputs (dense; the reference's sparse dicts are the |x| >= 1e-10 entries, truss.py:344-361).
 * Any pointer may be NULL to skip that output.  Rows are contiguous per system. */
typedef struct {
  double* u;       /* [B][N]  displacements, 0 at supported DOFs        (truss.py:342-345) */
  double* ext;     /* [B][N]  loads with reactions at supported DOFs    (truss.py:347-351) */
  double* axial;   /* [B][M]  member axial force, tension positive      (truss.py:353-361) */
  double* weight;  /* [B]     sum a*L*density                           (truss.py:166-168) */
  int32_t* info;   /* [B]     per-system status                                           */
  /* Compact layout (uniform batches only; either may be NULL): the same results without their redundant parts -- u is
   * zero at supported DOFs and ext equals the caller's own load vector at free DOFs (truss.py:347-349 only overwrites
   * the supported ones), so (u_free, react, axial) carry all the information of (u, ext, axial) in n + s + M instead of
   * 2N + M doubles per system (bar-942: 1674 instead of 2406: 30 % less to copy back or to gather).  Order: the
   * reference's boolean-mask order, i.e. tb_plan_get_maps' free_idx / sup_idx.  May be requested with or without u / ext. */
  double* u_free;  /* [B][n]  displacement of free DOF r      = u[free_idx[r]]           */
  double* react;   /* [B][s]  reaction at supported DOF r     = ext[sup_idx[r]]          */
} tb_batch_out;

/* Cotangents of tb_solve's outputs for tb_adjoint (device pointers, rows contiguous per system); any may be NULL (= 0). */
typedef struct {
  const double* u;          /* [B][N]  entries at supported DOFs are ignored (u is 0 there) */
  const double* ext;        /* [B][N]  free DOFs flow to the load, supported DOFs through the reactions */
  const double* axial;      /* [B][M] */
  const double* weight;     /* [B]    */
} tb_adj_in;

/* Per-system gradients written by tb_adjoint (device pointers); any but member_aed may be NULL to skip it. */
typedef struct {
  double* joint_xyz;        /* [B][nJ][d] */
  double* member_aed;       /* [B][M][3]  (a, e, density) -- required */
  double* force;            /* [B][N]     0 at supported DOFs (truss.py:349 overwrites those loads) */
  int32_t* info;            /* [B]        per-system status (same K, so the forward's); failed system: gradients 0 */
} tb_adj_out;

/* GA fitness outputs (ga.py:139-149): fitness = weight + penalties; flags[b][0] = stress
 * allowed, flags[b][1] = displacement allowed (truss.py:429-462 with isGetSumViolation). */
typedef struct {
  double* fitness;   /* [B]    */
  uint8_t* flags;    /* [B][2] */
  int32_t* info;     /* [B]    */
} tb_fit_out;

/* Truss.Solve() for B systems (truss.py:329-364). */
int tb_solve(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, void* cuda_stream);
int tb_solve_host(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out);

/* Pipelined form of tb_solve_host for callers that stream batches (a load-case sweep, the dataset generator's solve
 * site generate.py:354-357 called batch after batch): the call enqueues the batch -- host-to-device copies, kernels,
 * device-to-host copies, each on its own stream -- and returns at once with a ticket; tb_host_wait(plan, ticket) blocks
 * until that call's results are in its `out` buffers.  Consecutive calls use three staging areas in turn, so the
 * copies of one batch overlap the kernels of its neighbours (PCIe is full duplex).  At most three calls are in flight per
 * plan (one uploading, one computing, one downloading): a fourth submission first waits for the oldest one.  `in` / `out` buffers must stay valid (and should be
 * page-locked, tb_pinned_alloc) until the ticket has been waited for; tickets complete in submission order.  The
 * blocking *_host calls and tb_plan_destroy first wait for every pipelined call of the plan. */
int tb_solve_host_async(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, uint64_t* ticket);
int tb_host_wait(tb_plan* plan, uint64_t ticket);

/* B load cases of ONE truss: `for f in F: truss.SetForces(f); truss.Solve()` (truss.py:329-364 called B times on
 * the same joints and members).  joint_stride and member_stride (or gene_stride) must be 0; only `force` varies.
 * On the band path the stiffness matrix is assembled and factorised ONCE and every load case runs the two triangular
 * substitutions and the recovery against that factor; plans on the other paths factorise per system as tb_solve does.
 * tb_solve on the same arguments factorises every system independently (the bench's headline mode). */
int tb_solve_loadcases(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out, void* cuda_stream);
int tb_solve_loadcases_host(tb_plan* plan, const tb_batch_in* in, const tb_batch_out* out);

/* Reverse mode of tb_solve (truss.py:329-364) for B systems: the gradients of L = <grad.u, u> + <grad.ext, ext> +
 * <grad.axial, axial> + grad.weight * weight with respect to the joint positions, the member properties and the loads,
 * by one adjoint solve with the same stiffness matrix (K is symmetric) through the plan's own pipeline.  `u` = the
 * forward's dense displacements of the same inputs (device, [B][N]).  Explicit member properties only (member_aed; a
 * gene / type-table batch returns TB_ERR_NULL).  Gradients are written per system even for an input shared with stride 0
 * (reducing them is the caller's job).  shared_factor: the systems are load cases of one truss, as tb_solve_loadcases
 * (joint_stride and member_stride must be 0; on the band path one factorisation and B substitutions).  Enqueues on the
 * stream without synchronising; the adjoint scratch is the plan's (grow-only, grown in stream order). */
int tb_adjoint(tb_plan* plan, const tb_batch_in* in, const double* u, const tb_adj_in* grad, const tb_adj_out* out,
               int32_t shared_factor, void* cuda_stream);

/* GA.GetFitness for B genes (ga.py:139-149); `full` may be NULL or receive the full results. */
int tb_fitness(tb_plan* plan, const tb_batch_in* in, double allow_stress, double allow_displace,
               const tb_fit_out* fit, const tb_batch_out* full, void* cuda_stream);
int tb_fitness_host(tb_plan* plan, const tb_batch_in* in, double allow_stress, double allow_displace,
                    const tb_fit_out* fit, const tb_batch_out* full);

/* ---- GA generation step on the device (slientruss3d/ga.py:151-190; SURVEY.md section 8 f-1) -------------------------
 * One generation = tb_fitness on the gene matrix, then tb_ga_step: rank the population by fitness (stable, like
 * sorted() in GA.Select ga.py:155-160), copy the nElite best genes to the front and fill the rest by the reference's
 * UpdatePop rules (crossover of two distinct elites / mutation of one elite / keep pop[j] / fresh random gene,
 * ga.py:172-190).  Random numbers are counter-based (Philox4x32-10 keyed by `seed`, counter = individual, generation),
 * so a run is reproducible from (seed, generation) but does NOT replay Python's `random` stream -- the host GA class
 * keeps that property.  All pointers are device pointers.  The ranking counts, for every individual, the individuals that
 * precede it (N^2 comparisons over a 2-D grid): no sort, no population limit. */
typedef struct {
  int32_t n_pop, n_elite, n_member, n_type;
  double p_crossover, p_mutate, p_origin;   /* GA(pCrossover, pMutate, pOrigin); the rest re-seeds */
  uint64_t seed;
} tb_ga_params;

typedef struct {
  int32_t best_index;         /* individual with the lowest fitness (rank 0) */
  int32_t feasible_index;     /* first individual in rank order with both flags set, -1 if none (_RecordFeasible, ga.py:101-108) */
  double best_fitness;
  double feasible_fitness;
  uint8_t best_stress_ok, best_displace_ok;
  uint8_t pad_[6];
} tb_ga_report;

/* GA.Initialize (ga.py:151-153): gene[n_pop][n_member] drawn from the member-type distribution; type_cum = normalised
 * cumulative weights [n_type] (device) or NULL for uniform. */
int tb_ga_init(const tb_ga_params* params, const double* type_cum, int32_t* gene, void* cuda_stream);

/* GA.Select + GA.UpdatePop (ga.py:155-190).  order[n_pop] receives the ranking (individual indices, best first);
 * gene_out may be NULL (ranking and report only, e.g. the last Select of a run); report may be NULL. */
int tb_ga_step(const tb_ga_params* params, uint64_t generation, const double* fitness, const uint8_t* flags,
               const int32_t* gene_in, int32_t* gene_out, int32_t* order, tb_ga_report* report, void* cuda_stream);

/* Ragged batch: B independent trusses with their own topology (the generator's solve site,
 * generate.py:354-357).  Arrays are packed back to back; system b owns joints
 * joint_off[b]..joint_off[b+1]-1 and members member_off[b]..member_off[b+1]-1; conn holds
 * LOCAL joint ids.  Outputs are packed the same way (u/ext: d*joint_off, axial: member_off). */
typedef struct {
  int32_t dim;
  int32_t batch;
  const int64_t* joint_off;   /* [B+1] */
  const int64_t* member_off;  /* [B+1] */
  const double* joint_xyz;    /* [sum nJ][d] */
  const uint8_t* support;     /* [sum nJ]    */
  const int32_t* conn;        /* [sum M][2]  */
  const double* member_aed;   /* [sum M][3]  */
  const double* force;        /* [d * sum nJ] */
  int32_t max_joint;          /* max nJ over the batch (sizes the shared-memory kernel) */
  int32_t max_member;         /* max M over the batch */
} tb_ragged_in;

/* Routing: a batch whose (max_joint, max_member) fits the fused shared-memory kernels (tb_small_path_fits) runs on them
 * in one launch.  Any other batch is split by truss: the trusses up to 48 joints and 192 members (3D; 2D: 72 joints, 224
 * members) run in one launch of the fused warp-per-truss kernel sized at those limits, and every larger truss runs on the
 * envelope kernel (one CTA per truss: its own reverse Cuthill-McKee order, row-envelope Cholesky; DESIGN.md section 10),
 * which overwrites that truss's rows and status.  Either kernel gives a truss the same bits wherever it sits in the
 * batch.  Accepted sizes: d * max_joint <= 1536 and max_member <= 8192 (tb_ragged_limits); larger: TB_ERR_TOO_LARGE.
 * The compact outputs (u_free / react) are refused (TB_ERR_SIZE): a ragged batch has no common n and s.
 * Scratch of the envelope kernel: one grow-only device arena per device, one slot per CTA of its persistent grid (a
 * slot holds a dense lower-triangle bound of d * max_joint DOFs, the truss's incidence and adjacency lists and member
 * geometry: about 9.4 MB at 1536 DOFs, under 1 MB for a batch of 40-cube trusses).  It is grown stream-ordered on the
 * caller's stream (cudaFreeAsync / cudaMallocAsync).  Threads and streams: calls on one device that need it do not
 * overlap (a mutex), and a call on another stream than the previous one waits for it (an event).  A captured call must
 * stay on one stream, and a call inside a stream capture never grows the arena: it returns TB_ERR_ALLOC with nothing
 * enqueued; a warm-up call of the same sizes outside the capture grows it (and a later growth invalidates graphs
 * captured before it).  Batches that fit the fused kernels use no scratch. */
int tb_solve_ragged(const tb_ragged_in* in, const tb_batch_out* out, void* cuda_stream);
int tb_solve_ragged_host(const tb_ragged_in* in, const tb_batch_out* out);
/* Largest sizes tb_solve_ragged accepts: max_joint = 1536 / dim, max_member = 8192.  TB_ERR_DIM / TB_ERR_NULL. */
int tb_ragged_limits(int32_t dim, int32_t* max_joint, int32_t* max_member);
/* Every truss of the batch through the envelope kernel, whatever its size (tests and tools: the ragged counterpart of
 * tb_plan_set_path).  Device pointers; arguments, outputs, scratch and errors as tb_solve_ragged. */
int tb_solve_ragged_env(const tb_ragged_in* in, const tb_batch_out* out, void* cuda_stream);
/* Ordering mode of the envelope kernel: nothing is solved.  order [sum nJ] receives each truss's joints in elimination
 * order (local ids; 0..nJ-1 when the reverse Cuthill-McKee order does not shrink sum (i - first_i + 1)^2 below 0.85x
 * that of the natural order -- the rule of tb_plan_create), envelope [B] the row-envelope entries of its K_ff in that
 * order (tb_plan_info.envelope_size of a plan of the same topology).  A truss over max_joint / max_member gets envelope
 * -1 and its order rows are not written; one with a joint id outside [0, nJ) gets -1 in both.  order and envelope are
 * required device pointers (TB_ERR_NULL); other argument errors as tb_solve_ragged. */
int tb_ragged_env_order(const tb_ragged_in* in, int32_t* order, int64_t* envelope, void* cuda_stream);

/* Reverse mode of tb_solve_ragged: the gradients of L (as tb_adjoint) for every truss of a ragged batch, by one adjoint
 * ragged solve (the same kernel as the forward of the batch) between two warp-per-truss kernels.  Device pointers in the
 * packed layout: `u` (the forward's displacements of the same inputs), grad->u / grad->ext, out->joint_xyz / out->force
 * [d * sum nJ]; grad->axial [sum M]; out->member_aed [sum M][3]; grad->weight, out->info [B].  Required (TB_ERR_NULL
 * otherwise, when B > 0): in and its packed arrays as for tb_solve_ragged, u, grad, out, out->member_aed, out->info (the
 * solve's per-truss status, the forward's; a failed truss gets zero gradients) and work.  Optional (NULL = a zero
 * cotangent, or the gradient is skipped): grad->u / ext / axial / weight, out->joint_xyz, out->force.
 * `work` is caller-provided device scratch of at least d * joint_off[B] doubles (the adjoint
 * load, overwritten in place by the adjoint solution): the offsets live on the device, so only the caller knows sum nJ.
 * Argument errors as tb_solve_ragged (TB_ERR_NULL / TB_ERR_DIM / TB_ERR_SIZE / TB_ERR_TOO_LARGE; B = 0 is a no-op),
 * TB_ERR_NO_DEVICE without a GPU.  The offsets and arrays are not validated on the host: a truss larger than max_joint /
 * max_member, with a joint id outside [0, nJ) or an unknown support code gets zero gradients (and its status), and
 * nothing is read out of range; the rows of a truss whose offsets do not lie inside [0, joint_off[B]] / [0,
 * member_off[B]] are not written.  Enqueues on the stream without synchronising (capturable into a CUDA graph). */
int tb_adjoint_ragged(const tb_ragged_in* in, const double* u, const tb_adj_in* grad, const tb_adj_out* out, double* work,
                      void* cuda_stream);

/* ---- Dataset generation on the device (slientruss3d/generate.py:12-148; SURVEY.md section 8 f-2) ------------------
 * Expands a pool of trusses (a tb_ragged_in with DEVICE pointers) into n_out augmented trusses in the same packed layout,
 * ready for tb_solve_ragged: output truss o is pool truss src[o] after MoveToCentroid, RandomTranslation, AddJointNoise,
 * RandomResetPin (each optional, applied in this order).  out_joint_off / out_member_off [n_out+1] are the prefix sums of
 * the chosen pool trusses' sizes (device).  Counter-based random numbers keyed by `seed`. */
typedef struct {
  int32_t move_to_centroid;
  int32_t random_translation;
  double translate_lo, translate_hi;     /* RandomTranslation(translateRange) */
  int32_t joint_noise;
  double noise_mean[3], noise_std[3];    /* AddJointNoise(noiseMeans, noiseStds) */
  int32_t reset_pin;
  int32_t min_pin;                       /* RandomResetPin(minNumPin, maxNumPinRatio); ratio <= 0: up to every joint */
  double max_pin_ratio;
  uint64_t seed;
} tb_augment_params;

int tb_augment_ragged(const tb_ragged_in* pool, int32_t n_out, const int32_t* src, const int64_t* out_joint_off,
                      const int64_t* out_member_off, const tb_augment_params* params, double* out_xyz,
                      uint8_t* out_support, int32_t* out_conn, double* out_aed, double* out_force, void* cuda_stream);

/* ---- Random cube-truss topologies on the device (slientruss3d/generate.py:152-336, :338-372; SURVEY.md section 8 f-2)
 * GenerateRandomCubeTrusses draws, per truss, a random walk of numCube unit cells over a grid (CubeGrid.
 * RandomGenerateCubes), numbers the cubes' corners in first-seen order, links one or both diagonals of every face and the
 * twelve edges (CubeTruss.LinkMember, duplicates dropped unless parallel members are allowed), scales the cells by three
 * random lengths, pins the lowest layer, puts random loads on some of the other joints, picks a random type per member
 * and draws again until the counting rule of Truss.isStable holds.  tb_gencube does this for n trusses at once, one
 * thread per truss, with counter-based random numbers keyed by `seed` (reproducible from (seed, index); it does not
 * replay Python's `random` stream -- the host generator keeps that).  Every truss is written at a fixed stride
 * (tb_gencube_limits: max_joint, max_member, max_cube); n_joint / n_member receive the actual sizes, info 0 or
 * TB_INFO_NOT_STABLE when max_attempts draws all failed the counting rule.  After a prefix sum of the sizes,
 * tb_gencube_pack compacts the batch into the packed layout of tb_ragged_in, ready for tb_augment_ragged /
 * tb_solve_ragged.  cells [n][max_cube] (cell index x + gx (y + gy z) of every cube in creation order, -1 padded),
 * picks [n][max_cube][6] (diagonal choice per face: 0 first, 1 second, 2 both) and length [n][3] are optional exports:
 * fed to the host classes CubeTruss / CubeGrid.CubesToTruss they must reproduce the truss exactly (the tests do this).
 * All pointers are device pointers. */
#define TB_GEN_MAX_CELLS 216   /* grid cells (e.g. 6 x 6 x 6) */
#define TB_GEN_MAX_VERTS 343   /* grid corners */
typedef struct {
  int32_t grid[3];              /* gridRange */
  int32_t ncube_lo, ncube_hi;   /* numCube drawn uniformly from [lo, hi] per truss (lo == hi: fixed) */
  int32_t method;               /* GenerateMethod: 0 DFS, 1 BFS, 2 Random */
  int32_t link_type;            /* LinkType: 0 / 1 one diagonal per face, 2 both, 3 Random */
  int32_t add_pin;              /* isAddPinSupport */
  int32_t allow_parallel;       /* isAllowParallel */
  int32_t nforce_lo, nforce_hi; /* nForceRange; -1 = None (1 / every unsupported joint) */
  int32_t n_type;               /* member types to choose from (type_table [n_type][3]) */
  int32_t max_attempts;         /* draws per truss before giving up on the counting rule */
  double length_lo, length_hi;  /* lengthRange */
  double force_lo[3], force_hi[3]; /* forceRange */
  uint64_t seed;
} tb_gencube_params;

int tb_gencube_limits(const tb_gencube_params* params, int32_t* max_joint, int32_t* max_member, int32_t* max_cube);
int tb_gencube(const tb_gencube_params* params, int32_t n, const double* type_table, double* xyz, uint8_t* support,
               double* force, int32_t* conn, double* aed, int32_t* n_joint, int32_t* n_member, int32_t* info,
               int16_t* cells, uint8_t* picks, double* length, void* cuda_stream);
int tb_gencube_pack(const tb_gencube_params* params, int32_t n, const double* xyz, const uint8_t* support,
                    const double* force, const int32_t* conn, const double* aed, const int64_t* joint_off,
                    const int64_t* member_off, double* out_xyz, uint8_t* out_support, double* out_force,
                    int32_t* out_conn, double* out_aed, void* cuda_stream);

/* ---- Bulk JSON loader (slientruss3d/truss.py:401-421 Truss.LoadFromJSON; SURVEY.md section 8 f-3) ------------------
 * Parses n documents of the reference's JSON format ({"joint": [[[x,y,z],"PIN"],...], "force": [[id,[fx,fy,fz]],...],
 * "member": [[[j0,j1],[a,e,density]],...]} and, for output files, the sparse "displace" / "external" / "internal" lists
 * and "weight") straight into the packed arrays of tb_ragged_in -- no per-truss objects -- on `threads` host threads
 * (<= 0: all cores).  Host code only: works without a GPU.  Two passes: tb_json_scan counts the joints and members of
 * every document (the caller turns the counts into the [n+1] prefix sums joint_off / member_off and allocates), then
 * tb_json_fill writes document i's slices.  texts[i] must be NUL-terminated (lens[i] excludes the terminator).  Semantics
 * follow the reference: numbers become the doubles json.load produces, a zero load vector is ignored and a later entry
 * of the same joint replaces an earlier one (truss.py:177-182), results missing from the sparse lists are zeros
 * (truss.py:344-361 dropped them under the 1e-10 filter).  err[i] (may be NULL) receives the status of document i:
 * TB_ERR_JSON malformed / missing keys, TB_ERR_INDEX joint or member id out of range, TB_ERR_SUPPORT unknown support
 * name; the return value is TB_OK or TB_ERR_JSON when any document failed.  u / ext / axial / weight are only written
 * when is_output != 0 (weight may be NULL; it is NaN for documents without the key). */
int tb_json_scan(int32_t n, const char* const* texts, const int64_t* lens, int64_t* n_joint, int64_t* n_member,
                 int32_t* err, int32_t threads);
int tb_json_fill(int32_t n, const char* const* texts, const int64_t* lens, int32_t dim, int32_t is_output,
                 const int64_t* joint_off, const int64_t* member_off, double* xyz, uint8_t* support, double* force,
                 int32_t* conn, double* aed, double* u, double* ext, double* axial, double* weight, int32_t* err,
                 int32_t threads);

/* Page-locked host buffers for callers of the *_host entry points (full-speed H2D/D2H). */
int tb_pinned_alloc(void** ptr, size_t bytes);
int tb_pinned_free(void* ptr);

/* Largest system (free DOFs are bounded by d*nJ) the fused shared-memory kernel accepts. */
int tb_small_path_limits(int32_t* max_dof, int32_t* max_member);
/* 1 when a truss of n_joint joints and n_member members (every DOF possibly free, as in a ragged batch) fits the shared
 * memory of the fused kernels -- the test tb_solve_ragged applies to (max_joint, max_member) to keep a batch on them
 * alone (otherwise it routes by truss, see tb_solve_ragged), and the limit of tb_adjoint_ragged; the size limits above
 * are necessary, not sufficient (many members on few joints run out of shared memory first). */
int tb_small_path_fits(int32_t dim, int32_t n_joint, int32_t n_member);

/* FP64 pipe microbenchmarks used as roofline denominators (MEASURED_PEAKS.json has no FP64
 * entry): which = 0 DFMA (vector), 1 DMMA m8n8k4 (tensor).  Returns TFLOP/s in *tflops. */
int tb_fp64_peak(int32_t which, int32_t iters, double* tflops, float* ms);

/* Accuracy probe of the reciprocal square root the 16x16 pivot blocks use (hardware seed + one third-order
 * step): largest relative error against 1/sqrt(d) over n values spread log-uniformly over [1e-290, 1e300]. */
int tb_rsqrt_probe(int32_t n, double* max_rel_err);

/* Exactness probe of the shared-divisor division the member geometry uses (one correctly rounded reciprocal of the length,
 * then Markstein's multiply / FMA / FMA per numerator instead of four full divisions): counts the operand pairs out of n
 * (random and adversarial significands and exponents, keyed by seed) whose quotient differs from IEEE division. */
int tb_div_probe(int64_t n, uint64_t seed, uint64_t* mismatches);

/* Optional per-kernel CUDA-event timing on the launching stream (bench.py's roofline line).
 * tb_profile_read adds the milliseconds / launch counts recorded since the last read into
 * ms[8] / count[8]; slots: 0 member geometry, 1 assembly, 2 blocked Cholesky+solve, 3 recovery,
 * 4 fused shared-memory kernel. */
int tb_profile_enable(int32_t on);
int tb_profile_read(float* ms, int64_t* count);

/* ---- Introspection of the fused band kernel's program (tests and tools only) ---------------------------------------
 * The band path runs one fused kernel per batch (csrc/tb_bandts.cu): 8x8 blocks, two-sided elimination (the free DOFs
 * are split into a top part, a separator and a bottom part; two warps eliminate towards the separator).  The integer
 * program it executes is built on the host with the plan; these calls expose it so that the CPU tests can replay it in
 * numpy against the oracle (tests/test_ts_program_cpu.py).
 * tb_plan_ts_info: out[16] = {exists, block columns, padded order, first separator block, separator blocks, bottom
 *   blocks, sub-diagonal blocks top / bottom, largest factor chunk, factor doubles per system, block products, block
 *   solves, K entries, member contributions, entries with several contributions}.
 * tb_plan_ts_array: copies array `which` into out (may be NULL) and returns its length in int32 elements, -1 if there is
 *   no program.  Per side: 0 colmask, 1 srcmask, 2 xmask, 3 colent[.][2], 4 rowdof, 5 rownat, 6 lofs; whole program (side
 *   ignored): 7 epos, 8 ent_src, 9 tq_first, 10 tq_multi, 11 tq_ptr, 12 tq_pack (the assembly pass's scatter lists in the
 *   kernel's entry order); 13 colrec[.][8] (per side: the records the kernel reads per block column).
 * tb_ts_phase_read: cycles per kernel phase accumulated by an instrumented build (-DTB_PHASE_TIMING), zeros otherwise. */
/* tb_debug_assemble_host: runs the assembly pass alone on host inputs (explicit member properties) and returns the K_ff
 *   values the DEVICE computed, kv_out[B][nnz_lower] in the entry order of tb_plan_get_scatter -- the gate
 *   "device-assembled K_ff == GetKMatrix()[mask][:, mask]" (truss.py:307-316, 343) of the GPU tests. */
int tb_debug_assemble_host(tb_plan* plan, const tb_batch_in* in, double* kv_out);
int tb_plan_ts_info(const tb_plan* plan, int32_t* out);
int64_t tb_plan_ts_array(const tb_plan* plan, int32_t side, int32_t which, int32_t* out);
int tb_ts_phase_read(unsigned long long* out);

/* Kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t tb_launch_count(void);
const char* tb_strerror(int code);
int tb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TRUSS_B200_H */
