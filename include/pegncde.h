/*
 * pegncde.h -- C-ABI of the B200-native (sm_100a) hot path of
 * hits-mli/perm-equiv-graph-neural-cdes: the Tsit5 solve loop that evaluates the
 * permutation-equivariant graph vector field f_theta(Z_s, A_s) at every stage,
 * forward and exact-discrete-adjoint backward.
 *
 * The reference is pure Python/JAX and has NO FFI for this path; each entry point
 * below names the reference call it replaces (paths relative to the reference root):
 *
 *   pegncde_pack_adj        src/configs/dataset_configs.py:147-173,1073-1100  (coeff layout -> planar planes)
 *   pegncde_pack_x          src/configs/dataset_configs.py:1073-1100          (node-signal coeffs)
 *   pegncde_build_adj       get_graph_interpolation_coeffs, dataset_configs.py:147-173,1073-1100 (snapshots -> planes)
 *   pegncde_vf_fwd          src/models/vector_fields/perm_equiv_graph_vector_field.py:85-129
 *                           + cde_wrapper_vector_field.py:19-26  (the ODETerm callable vf(t, y, args))
 *   pegncde_vf_vjp          jax.vjp of the same callable
 *   pegncde_step_fwd        one diffrax Tsit5.step (call sites pgt_graph_neural_cde.py:65,
 *                           graph_neural_cde.py:53) -> y1, y_err, k7 (FSAL) for host-side controllers
 *   pegncde_solve_fwd       diffrax.diffeqsolve(ODETerm(vf), Tsit5(), ..., ConstantStepSize())
 *                           src/models/pgt_graph_neural_cde.py:119-129, graph_neural_cde.py:94-104,
 *                           tgb_graph_neural_cde.py:152-162
 *   pegncde_solve_bwd       reverse mode through that call (diffrax default RecursiveCheckpointAdjoint,
 *                           reached via eqx.filter_value_and_grad, src/engine/trainer_pgt.py:346,
 *                           src/engine/trainer.py:315)
 *
 * Conventions
 *   - every pointer except `step_ts` is a DEVICE pointer owned by the caller (XLA / torch);
 *     the library never allocates, frees or retains device memory.  Host-side state is limited to: the process-wide
 *     launch counter, the optional profiling hooks (pegncde_profile_*, off by default), a PER-THREAD cache of TMA
 *     descriptors keyed on buffer address and shape, and per-kernel bitmasks of the devices whose kernel attributes
 *     (opt-in shared memory, cluster size) have been set.  Nothing a call computes depends on an earlier call; every
 *     mode is selected through PegDims.flags, the library reads no environment variables.
 *   - functions only ENQUEUE work on `stream` (no device synchronisation, no host callbacks),
 *     so they are safe inside an XLA custom call and capturable in a CUDA graph.
 *   - all floating-point data is fp32 (the reference never enables x64), row-major.
 *   - return value: 0 = ok, otherwise a PEG_ERR_* code; pegncde_strerror() names it.
 *     Nothing throws or exits across this boundary.
 */
#ifndef PEGNCDE_H_
#define PEGNCDE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* peg_stream_t; /* a cudaStream_t */

enum {
  PEG_OK = 0,
  PEG_ERR_BAD_DIMS = 1,      /* a dimension is out of the supported range */
  PEG_ERR_NULL_POINTER = 2,  /* a required pointer is NULL */
  PEG_ERR_WORKSPACE = 3,     /* workspace smaller than pegncde_workspace_bytes() */
  PEG_ERR_CUDA = 4,          /* a CUDA runtime call or launch failed (see pegncde_last_cuda_error) */
  PEG_ERR_UNSUPPORTED = 5,   /* valid request the library does not implement */
  PEG_ERR_ALIGNMENT = 6      /* a pointer or pitch breaks the 16-byte alignment contract */
};

/* flags in PegDims.flags */
enum {
  PEG_FLAG_RELU = 0,            /* reserved */
  PEG_FLAG_TENSOR_CORES = 1,    /* n x n x d contractions on tcgen05 (split operands, fp32 accumulation: fp32-parity) */
  PEG_FLAG_TF32_FAST = 2,       /* with TENSOR_CORES: single-pass TF32 (rna-rounded), looser tolerance */
  PEG_FLAG_DIRECTED = 4,        /* ConvEquivFusionDirectedLayer (layers.py:180-362): 11 parameter pairs, row AND column sums;
                                   needs PegControl.adj_colsum; fusion block = 22 (+2 pad) scalars (see parameter packing) */
  PEG_FLAG_TF32X3 = 16,         /* with TENSOR_CORES: operands of the n x n x d contraction split as 3xTF32 (x = hi + lo, both tf32,
                                   hi*hi + lo*hi + hi*lo on kind::tf32: rounding ~2^-22 per product).  The DEFAULT is the same three-product
                                   split with fp16 parts and block exponents ("fp16x2", 11 + 11 mantissa bits: the same ~2^-22 per
                                   product, fp32 accumulation) on kind::f16 at twice the tf32 rate and half the shared-memory traffic;
                                   it needs PegControl.adj_absmax and falls back to 3xTF32 when that pointer is NULL */
  PEG_FLAG_BF16X2 = 32,         /* with TENSOR_CORES: x = hi + lo with bf16 parts (no block exponents needed; 8 + 8 mantissa bits:
                                   rounding ~2^-17 per product).  A separately stated looser-tolerance mode: Z_T within 1e-4,
                                   gradients within 2e-3 */
  PEG_FLAG_ADJ_LIGHT = 8,       /* with TENSOR_CORES: the adjoint contraction runs two of its four products single-pass; looser
                                   stated tolerance on the param1 / param2 gradients (2.5e-3 instead of 1e-3).  Off by default. */
  PEG_FLAG_NO_FUSED_SMALL = 64, /* opt out of the small-graph path.  By default, graphs with n < 128 (undirected layer, h <= 128; the
                                   shapes the tcgen05 contraction does not take) run a whole evaluation f(t, y) -- and a whole
                                   VJP -- in ONE fp32 kernel, a thread-block cluster per graph with cluster barriers between
                                   the layer phases instead of ~15 / ~40 dependent launches; same arithmetic as the
                                   per-operator fp32 kernels, so the same parity bound */
  PEG_FLAG_FUSED_SMALL = 128    /* take the small-graph path up to n <= 256 (it loses to the per-operator tcgen05 path when one
                                   graph has a wide last layer, e.g. England n=129, 2he=1024: measured in DESIGN.md) */
};

typedef struct PegDims {
  int32_t B;     /* graphs (trajectories) in the batch; each has its own control path      */
  int32_t n;     /* nodes                                                                  */
  int32_t ldn;   /* padded node count of the tiled coefficient planes: n rounded up to 32   */
  int32_t h;     /* hidden_dim = width of the state y [n,h] and of every hidden layer      */
  int32_t e;     /* data_embed_dim; 0 = plain ODETerm(vector_field) (no CDE wrapper)       */
  int32_t L;     /* num_layers of ConvEquivFusionLayer                                     */
  int32_t T;     /* knots of the control path (T-1 cubic pieces)                           */
  int32_t flags; /* PEG_FLAG_*                                                             */
} PegDims;
/* width of the last layer: h if e == 0 else 2*h*e (vector_field_configs.py:71) */

/* Row-sharded mode (SURVEY 8(e): one graph too large for / spread over several GPUs).  Rank r of `world` holds the rows
 * [row0, row0 + PegDims.n) of the n_glob x n_glob adjacency path -- and, to avoid a reduce-scatter, the same rows of its TRANSPOSE
 * (adj_coef_t) -- plus the matching rows of every state / cotangent array.  RMSNorm -> Linear, the Runge-Kutta updates and the
 * weight gradients are row-local; the only exchange step is per layer: the operand V^T of the n x n x d contraction (every rank
 * needs all rows of V) and two d-vectors of column sums.  The library does that exchange itself over peer memory: the producer
 * kernels write this rank's slice of V^T, k_shard_push copies it with 128-bit stores into every peer's buffer over NVLink and
 * raises an epoch flag there, k_shard_wait spins on the local flags and adds the column-sum slots in rank order.  No NCCL on the
 * data path; parameter gradients come out as per-rank partial sums (the caller all-reduces them like in batch-sharded mode).
 * All pointer tables are HOST arrays of `world` (<= 8) device pointers to peer-visible (symmetric) buffers of identical layout.
 * Restrictions: PEG_FLAG_TENSOR_CORES with fp16x2 or 3xTF32 operands, e == 0, undirected layer, PegDims.n a multiple of 128,
 * fixed-step entry points (vf_fwd / vf_vjp / solve_fwd / solve_bwd).
 * CUDA graphs: with epoch_dev == NULL the epoch of every exchange is a launch argument taken from the host counter, so a
 * captured call cannot be replayed.  With epoch_dev set, the kernels add the device word *epoch_dev to a per-call sequence
 * number (the host counter restarts at 0 on every API call), and every call ends by advancing *epoch_dev by its (even; a flag-only
 * exchange pads an odd count, which also keeps the epoch-parity halves alternating across calls) number of exchanges: replays of
 * a captured call then use fresh epochs.  Every rank must replay the same sequence of calls. */
typedef struct PegShard {
  int32_t rank, world;
  int32_t n_glob;            /* global node count = world * PegDims.n                                                  */
  int32_t row0;              /* first global row of this rank = rank * PegDims.n                                        */
  const float* adj_coef_t;   /* [B, T-1, 4 * ldn * n_glob] tiled planes of rows [row0, row0 + n) of the TRANSPOSED path   */
  void* const* vt_hi;        /* [world] -> [2][B * dmax * n_glob] V^T high parts, two epoch-parity halves (bytes: 4 * that) */
  void* const* vt_lo;        /* [world] -> same, low parts                                                              */
  int32_t* const* vexp;      /* [world] -> [2][B * n_glob / 128] block exponents (fp16x2 operands)                        */
  float* const* colsum;      /* [world] -> [2][world][2][B * 2 * dmax] column-sum slots (two vectors per exchange)        */
  uint32_t* const* flags;    /* [world] -> [world + 1] epoch counters (one per source rank) + an error word              */
  uint32_t* epoch;           /* HOST counter of exchanges enqueued so far on this rank (in / out; same on every rank)     */
  uint32_t* epoch_dev;       /* nullable DEVICE word (this rank's own memory, zero-initialised): epoch base for graph replay  */
} PegShard;

/* Sparse (CSR) adjacency path of one batch, built by pegncde_build_adj_sparse / pegncde_pack_adj_sparse.  The batch shares
 * one entry axis: graph b's row i holds the entries [row_ptr[b, i], row_ptr[b, i + 1]) (ABSOLUTE offsets into col and into the
 * entry axis of coef), so a view of one graph needs no copy.  The transposed pattern is stored the same way with its own copy of
 * the coefficients (row i of the transpose = the entries (k, i) of the path), so that both orientations walk contiguous memory.
 *
 * A sparse control runs the n x n x d contraction as an fp32 FMA gather (k_sparse_contract): the operand-format flags
 * PEG_FLAG_TF32X3, PEG_FLAG_BF16X2, PEG_FLAG_TF32_FAST and PEG_FLAG_ADJ_LIGHT mean nothing for it, and the small-graph cluster
 * kernels are not used.  PEG_FLAG_TENSOR_CORES still selects the tcgen05 RMSNorm -> Linear kernels.  Not combinable with
 * PegControl.shard (PEG_ERR_UNSUPPORTED). */
typedef struct PegSparse {
  int64_t nnz;              /* entries of the whole batch (both orientations hold the same count)                            */
  int64_t nnz_stride;       /* entries per coefficient slab, >= nnz                                                          */
  const int32_t* row_ptr;   /* [B, n+1]  absolute offsets of every row                                                       */
  const int32_t* col;       /* [nnz]     column of each entry, ascending inside a row                                        */
  const float* coef;        /* [T-1, nnz_stride, 4]  (a, b, c, d) of each entry for each cubic piece (one 16-byte load)      */
  const int32_t* row_ptr_t; /* the same three arrays for the transposed pattern                                              */
  const int32_t* col_t;
  const float* coef_t;
} PegSparse;

/* Planar control path, built once per batch by pegncde_pack_adj / pegncde_pack_x.
 * Coefficient order everywhere is (a, b, c, d):  X(t) = a + s(b + s(c + s d)), s = t - ts[i]. */
typedef struct PegControl {
  const float* ts;         /* [B, T]            knot times                                         */
  const float* adj_coef;   /* [B, T-1, 4*ldn*ldn] adjacency channel of the reference's coeffs, four planes
                              (a,b,c,d) zero padded to ldn x ldn and stored as 32x32 tiles of 16 KB
                              (exact element order: peg_tile_off in csrc/peg_common.cuh; written by
                              pegncde_pack_adj)                                                     */
  const float* adj_rowsum; /* [B, T-1, 4, n]    row sums of each plane                              */
  const float* adj_diag;   /* [B, T-1, 4, n]    diagonal of each plane                              */
  const float* adj_total;  /* [B, T-1, 4]       total of each plane                                 */
  const float* tch_coef;   /* [B, T-1, 3, n]    (b,c,d) of the time channel, mean over axis 0       */
  const float* x_coef;     /* [B, T-1, 3, n, 2e] (b,c,d) of the node-signal path, last axis (l,k)
                              interleaved like the reference's [n,e,2]; NULL iff e == 0             */
  const float* adj_colsum; /* [B, T-1, 4, n]    column sums of each plane (pegncde_adj_colsums); only read with
                              PEG_FLAG_DIRECTED, NULL otherwise                                     */
  const float* adj_absmax; /* [B, T-1, 4]       max |entry| of each plane (pegncde_adj_absmax): the range bound the fp16x2 operand
                              format scales the interpolated adjacency with; NULL = not available (3xTF32 operands are used) */
  const PegShard* shard;   /* NULL = the whole graph lives on this GPU; otherwise row-sharded mode (see PegShard): every array
                              above holds this rank's rows only (adj_coef: [B, T-1, 4 * ldn * n_glob]), adj_total / adj_absmax are
                              already reduced over the ranks, adj_diag[i] = entry (row0 + i) of local row i                  */
  const PegSparse* sparse; /* NULL = dense planes (adj_coef).  Otherwise the adjacency path is the CSR path of PegSparse: adj_coef may be
                              NULL, adj_absmax is unused, adj_rowsum / adj_diag / adj_total / adj_colsum / tch_coef keep their meaning
                              (the sparse builders fill all of them, adj_colsum included)                                    */
} PegControl;

/* ---- parameter packing ---------------------------------------------------------------
 * params / g_params are one flat fp32 buffer, layer after layer:
 *   weight [d_out, d_in] | bias [d_out] | norm_weight [d_in] | norm_bias [d_in] |
 *   fusion [8,2] = param1[0],param1[1],param2[0],...,param8[1]
 *   (PEG_FLAG_DIRECTED: fusion [12,2] = param1..param8 as above, then param4_prime, param5_prime, param6_prime and one
 *    unused pair that keeps the next layer 16-byte aligned)
 * (leaf names: gnn_layers[l].conv_layer.linear.{weight,bias}, .conv_layer.norm.{weight,bias},
 *  gnn_layers[l].param1..param8 -- src/models/vector_fields/layers.py:19-20,66-74). */
size_t pegncde_param_count(const PegDims* dims);
/* offsets[5*l + {0,1,2,3,4}] = float offset of weight, bias, norm_weight, norm_bias, fusion of layer l */
int pegncde_param_offsets(const PegDims* dims, int64_t* offsets /* [5*L] */);

/* ---- control-path packing (device) ---------------------------------------------------- */
/* d,c,b,a: the four arrays diffrax.backward_hermite_coefficients returns, each
 * [B, T-1, n, n, 2] with the last axis (time, adjacency).  Writes every PegControl adj_* / tch_* field. */
int pegncde_pack_adj(peg_stream_t stream, const PegDims* dims, const float* d, const float* c, const float* b,
                     const float* a, float* adj_coef, float* adj_rowsum, float* adj_diag, float* adj_total,
                     float* tch_coef);
/* Streaming variant: d,c,b,a hold only the cubic pieces [piece_begin, piece_begin + piece_count) -- each
 * [B, piece_count, n, n, 2] -- and only those pieces of the (full-size) outputs are written.  A fixed-step solve walks the
 * pieces in order, so the host can copy and pack piece i+1 while the steps inside piece i run (solve.py, streamed controls). */
int pegncde_pack_adj_range(peg_stream_t stream, const PegDims* dims, int32_t piece_begin, int32_t piece_count, const float* d,
                           const float* c, const float* b, const float* a, float* adj_coef, float* adj_rowsum, float* adj_diag,
                           float* adj_total, float* tch_coef);
/* same for already-tiled adjacency planes (adj_coef given): fills the statistics only;
 * tch_coef is written as d(time)/dt == 1 (b=1, c=d=0). */
int pegncde_adj_stats(peg_stream_t stream, const PegDims* dims, const float* adj_coef, float* adj_rowsum,
                      float* adj_diag, float* adj_total, float* tch_coef);
/* Control-path builder (SURVEY N2): graph snapshots A_k [B, T, n, n] + knot times ts [B, T] (device) -> the same
 * outputs as pegncde_pack_adj, with diffrax.backward_hermite_coefficients (call sites
 * src/configs/dataset_configs.py:168-170, 1094-1096) fused in: 4 n^2 T bytes cross the bus instead of 32 n^2 (T-1).
 * The time channel is implied (X_time(t) = t): tch_coef is written as (1, 0, 0). */
int pegncde_build_adj(peg_stream_t stream, const PegDims* dims, const float* ts, const float* snapshots, float* adj_coef,
                      float* adj_rowsum, float* adj_diag, float* adj_total, float* tch_coef);
/* Rectangular variant for row-sharded controls: snapshots [B, T, n, n_cols] = this rank's rows of the path (or of its transpose),
 * planes tiled with n_cols/32 tiles per row, diagonal taken at column diag_col0 + i (pass -1 to skip it), adj_total = the partial
 * totals of these rows.  n_cols must be a multiple of 32.  adj_rowsum / adj_diag / adj_total / tch_coef may be NULL (transpose). */
int pegncde_build_adj_rect(peg_stream_t stream, const PegDims* dims, int32_t n_cols, int32_t diag_col0, const float* ts,
                           const float* snapshots, float* adj_coef, float* adj_rowsum, float* adj_diag, float* adj_total, float* tch_coef,
                           float* adj_absmax);
/* bytes of each symmetric buffer of a PegShard for these dims (dmax = widest layer): out[0] = vt_hi (= vt_lo), out[1] = vexp,
 * out[2] = colsum, out[3] = flags */
int pegncde_shard_buffer_bytes(const PegDims* dims, int32_t world, size_t* out /* [4] */);
/* column sums of the tiled planes (fixed summation order) -> adj_colsum [B, T-1, 4, n]; needed by PEG_FLAG_DIRECTED only */
int pegncde_adj_colsums(peg_stream_t stream, const PegDims* dims, const float* adj_coef, float* adj_colsum);
/* max |entry| of the tiled planes of the cubic pieces [piece_begin, piece_begin + piece_count) -> adj_absmax [B, T-1, 4] (order
 * independent, hence reproducible) */
int pegncde_adj_absmax(peg_stream_t stream, const PegDims* dims, int32_t piece_begin, int32_t piece_count, const float* adj_coef,
                       float* adj_absmax);
/* Sparse control-path builders (see PegSparse).  `sp` describes the pattern (row_ptr, col, row_ptr_t, col_t, nnz, nnz_stride);
 * its coef / coef_t are the OUTPUTS (cast away const).  perm_t [nnz] scatters entry e of the pattern to position perm_t[e] of the
 * transposed pattern.  Both write coef, coef_t, adj_rowsum, adj_diag, adj_total, adj_colsum ([B, T-1, 4, n] each, totals [B, T-1, 4])
 * and tch_coef = (1, 0, 0) (the time channel is implied).  Every reduction runs in a fixed order: the control is reproducible.
 *   pegncde_build_adj_sparse: knot times ts [B, T] and the values of the path on the pattern, values [T, nnz] (0 where an edge is
 *     absent at a knot); backward_hermite_coefficients is fused in with the per-element arithmetic of pegncde_build_adj, so the
 *     coefficients are bit-identical to the dense builder's at every pattern position.
 *   pegncde_pack_adj_sparse: coefficients given, d, c, b, a each [T-1, nnz] (adjacency channel only; the sparse form of the
 *     reference's coeffs_adj -- linear interpolation is c = d = 0). */
int pegncde_build_adj_sparse(peg_stream_t stream, const PegDims* dims, const PegSparse* sp, const int32_t* perm_t, const float* ts,
                             const float* values, float* adj_rowsum, float* adj_diag, float* adj_total, float* adj_colsum, float* tch_coef);
int pegncde_pack_adj_sparse(peg_stream_t stream, const PegDims* dims, const PegSparse* sp, const int32_t* perm_t, const float* d,
                            const float* c, const float* b, const float* a, float* adj_rowsum, float* adj_diag, float* adj_total,
                            float* adj_colsum, float* tch_coef);
/* d,c,b,a each [B, T-1, n, e, 2] -> x_coef [B, T-1, 3, n, 2e] */
int pegncde_pack_x(peg_stream_t stream, const PegDims* dims, const float* d, const float* c, const float* b,
                   const float* a, float* x_coef);

/* ---- workspace ------------------------------------------------------------------------- */
enum { PEG_WS_VF_FWD = 0, PEG_WS_VF_VJP = 1, PEG_WS_SOLVE_FWD = 2, PEG_WS_SOLVE_BWD = 3, PEG_WS_STEP = 4 };
/* bytes of caller-provided scratch for one call of kind `which` with `steps` solver steps */
size_t pegncde_workspace_bytes(const PegDims* dims, int32_t which, int32_t steps);

/* ---- vector field ----------------------------------------------------------------------- */
/* dy[b] = vf(t, y[b], args) for every graph of the batch; t is a host scalar (shared stage time). */
int pegncde_vf_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                   const float* y /* [B,n,h] */, float* dy /* [B,n,h] */, void* workspace, size_t workspace_bytes);
/* g_y = (d vf/d y)^T g_dy ; g_params += (d vf/d theta)^T g_dy summed over the batch (caller zeroes it);
 * g_xdot (nullable) [B,n,2e] = cotangent of control_data.derivative(t). */
int pegncde_vf_vjp(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                   const float* y, const float* g_dy, float* g_y, float* g_params, float* g_xdot, void* workspace,
                   size_t workspace_bytes);
/* pegncde_vf_vjp plus the cotangent of a sparse control's coefficients: g_adj_coef [T-1, nnz_stride, 4] (a,b,c,d per entry, in
 * pattern order, like PegSparse.coef) ACCUMULATES d loss / d coef (caller zeroes it).  The control's statistics (row / column sums,
 * diagonal, totals) are functions of the coefficients and are differentiated through; the knot times are not.  Every entry has one
 * owner per layer, so the result is reproducible bit for bit.  Same workspace as pegncde_vf_vjp.  A dense control with a non-NULL
 * g_adj_coef returns PEG_ERR_UNSUPPORTED, a pointer that is not 16-byte aligned PEG_ERR_ALIGNMENT; with g_adj_coef == NULL the
 * call is pegncde_vf_vjp. */
int pegncde_vf_vjp_adj(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                       const float* y, const float* g_dy, float* g_y, float* g_params, float* g_xdot, float* g_adj_coef,
                       void* workspace, size_t workspace_bytes);

/* ---- one Tsit5 step (adaptive controllers stay on the host) ----------------------------- */
/* k1 = f(t, y) when k1_valid == 0 (first step) else taken from k1 (FSAL).  Writes y1, y_err
 * (= dt * sum_i (b_i - bhat_i) k_i) and k7 = f(t + dt, y1).  k_stages (nullable) [5,B,n,h] receives k2..k6
 * (needed for dense output). */
int pegncde_step_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                     float dt, const float* y, float* k1, int32_t k1_valid, float* y1, float* y_err, float* k7,
                     float* k_stages, void* workspace, size_t workspace_bytes);

/* ---- batched adaptive solves: the step-size controller on the device --------------------------------------------------
 * diffrax PIDController(rtol, atol) (pcoeff = 0, icoeff = 1, dcoeff = 0) + _clip_to_end under jax.vmap(model)
 * (src/models/graph_neural_cde.py:53-54,86-104; src/configs/loss_configs.py:44): every trajectory of the batch has its own step
 * sequence.  pegncde_step_fwd_batched attempts one step of EVERY trajectory (per-trajectory start t_dev[b] and size dt_dev[b], both
 * device arrays); pegncde_adaptive_control evaluates the scaled error norms, accepts / rejects per trajectory, emits the dense-output
 * samples of accepted steps (SaveAt(ts)), advances y / k1 (FSAL) / the checkpoints and writes the next (t_dev, dt_dev) -- no host round
 * trip per step; the host polls `done` every few attempts.  Finished trajectories are stepped with dt = 0 and left untouched. */
typedef struct PegAdaptState {
  float tprev, tnext;                        /* the step being / to be attempted (host initialises: t0, first tnext)        */
  int32_t done, nacc, attempts, rejected;    /* host initialises to 0                                                       */
  int32_t mi;                                /* next save time to emit (0)                                                   */
  int32_t mi0, mi1, keep;                    /* scratch of the last decision                                                 */
  float h;
  int32_t overflow;                          /* set when the accepted-step table (cap entries) is full: the host must grow it */
} PegAdaptState;
int pegncde_step_fwd_batched(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, const float* t_dev /* [B] */,
                             const float* dt_dev /* [B] */, const float* y, float* k1, int32_t k1_valid, float* y1, float* y_err, float* k7,
                             float* k_stages, void* workspace, size_t workspace_bytes);
/* y_ckpt [B, cap+1, n, h] (slot 0 = y0, written by the host), step_tab [B, cap+1] (slot 0 = t0), ys_save [n_save, B, n, h],
 * sample_step / sample_theta [n_save, B]: for every save time the accepted step that emitted it and the position inside it
 * (what the adjoint needs), sumsq_scratch [B]. */
int pegncde_adaptive_control(peg_stream_t stream, const PegDims* dims, PegAdaptState* state /* [B] device */, float rtol, float atol, float t1,
                             float safety, float factormin, float factormax, int32_t error_order, const float* save_ts, int32_t n_save,
                             int32_t cap, float* y, const float* y1, const float* y_err, float* k1, const float* k7, const float* k_stages,
                             float* y_ckpt, float* ys_save, float* step_tab, int32_t* sample_step, float* sample_theta, float* t_dev,
                             float* dt_dev, float* sumsq_scratch);

/* ---- Tsit5 dense output: diffrax SaveAt(ts=...) (call site src/models/graph_neural_cde.py:86-104) ---------- */
/* out = y + dt * sum_i b_i(theta) k_i with Tsitouras' 4th-order interpolant, theta in [0,1] inside the step
 * [t, t+dt]; k_stages = k2..k6 as written by pegncde_step_fwd. */
int pegncde_tsit5_dense(peg_stream_t stream, const PegDims* dims, float dt, float theta, const float* y, const float* k1,
                        const float* k_stages, const float* k7, float* out);
/* Scaled error norms of adaptive step-size control -- diffrax PIDController(rtol, atol) (call site
 * src/models/graph_neural_cde.py:53-54) and its initial-step heuristic:
 *   out[b] = sum_i ((x - x2)_i / (atol + rtol * max(|s0_i|, |s1_i|)))^2   over the n*h entries of graph b
 * (x2, s1 nullable: 0 / s0).  The host takes sqrt(out / (n h)) (rms norm) and runs the controller. */
int pegncde_scaled_sumsq(peg_stream_t stream, const PegDims* dims, const float* x, const float* x2, const float* s0,
                         const float* s1, float rtol, float atol, float* out /* [B] */);
/* host helper: the seven weights b_i(theta) */
void pegncde_tsit5_dense_weights(float theta, float* w /* [7] */);

/* ---- fixed-step solve -------------------------------------------------------------------- */
/* step_ts: HOST array [steps+1] of fp32 step boundaries, built by the caller with diffrax's
 * ConstantStepSize + end-clipping rule.  y_ckpt [steps+1, B, n, h] receives y at every boundary
 * (y_ckpt[0] = y0, y_ckpt[steps] = y(T)); it is the SaveAt(steps) output and the checkpoint set
 * pegncde_solve_bwd restarts from.  yT (nullable) [B,n,h] = y_ckpt[steps]. */
int pegncde_solve_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                      const float* step_ts, int32_t steps, const float* y0, float* yT, float* y_ckpt,
                      float* stage_store, void* workspace, size_t workspace_bytes);
/* stage_store (nullable, pegncde_stage_store_bytes() bytes): when given, solve_fwd keeps the input of every layer
 * of every stage there and solve_bwd, handed the same buffer, skips its forward recompute (36 instead of 54 passes
 * over the coefficient planes per step).  NULL = checkpoint-per-step mode: solve_bwd recomputes each step.
 * Layout, per step and stage 0..5 (steps x 6 blocks of equal size):
 *   L slots [B,n,h]: the input of every layer (layer 0 of stage 0 is y_ckpt[step] itself, that slot stays unused);
 *   K slots [B,n,h]: M_l = Linear(RMSNorm(input)) of the layers whose output is h wide, K = L (e == 0) or L - 1 (e > 0: the
 *                    last layer is 2he wide and is recomputed);
 *   K slots [B][2][h]: the column sums of those M_l (plain and weighted by the layer's contraction vector).
 * The tensor-core adjoint reads M_l back instead of recomputing it.  A caller streaming the solve in segments offsets the
 * buffer by pegncde_stage_store_bytes(dims, 1) per step. */
size_t pegncde_stage_store_bytes(const PegDims* dims, int32_t steps);
/* g_ckpt (nullable) [steps+1, B, n, h]: cotangents injected at step boundaries (SaveAt(steps) losses);
 * g_yT [B,n,h] cotangent of y(T) (either of the two may be NULL, not both).
 * g_stage (nullable) [steps, 7, B, n, h]: direct cotangents of the stage slopes k1..k7 of every step -- what a loss
 * on dense-output samples (SaveAt(ts=...)) contributes: dt * b_i(theta) * g_sample, summed over the samples of the step.
 * g_xcoef (nullable, e > 0) [B, T-1, 3, n, 2e]: ACCUMULATES the cotangent of PegControl.x_coef (caller zeroes it) --
 * the TGB models learn the node-signal path (src/models/tgb_graph_neural_cde.py:118-137), so reverse mode continues
 * through backward_hermite_coefficients into their data_encoder.
 * Writes g_y0; accumulates g_params (caller zeroes it).  The step table may be any accepted-step sequence (adaptive
 * controllers): the adjoint is that of the discrete scheme with the step sizes held fixed. */
int pegncde_solve_bwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                      const float* step_ts, int32_t steps, const float* y_ckpt, const float* stage_store,
                      const float* g_yT, const float* g_ckpt, const float* g_stage, float* g_y0, float* g_params,
                      float* g_xcoef, void* workspace, size_t workspace_bytes);
/* pegncde_solve_bwd plus g_adj_coef (nullable, sparse controls only) [T-1, nnz_stride, 4]: ACCUMULATES the cotangent of
 * PegSparse.coef over every stage of every step, as pegncde_vf_vjp_adj does for one evaluation.  Entries are absolute, so the
 * per-graph views of one batch (B = 1 controls whose row_ptr points into the batch's entry axis) all write the one shared buffer.
 * Outputs other than g_adj_coef equal pegncde_solve_bwd's bit for bit. */
int pegncde_solve_bwd_adj(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                          const float* step_ts, int32_t steps, const float* y_ckpt, const float* stage_store,
                          const float* g_yT, const float* g_ckpt, const float* g_stage, float* g_y0, float* g_params,
                          float* g_xcoef, float* g_adj_coef, void* workspace, size_t workspace_bytes);

/* ---- introspection ------------------------------------------------------------------------ */
const char* pegncde_strerror(int code);
int pegncde_last_cuda_error(void); /* cudaError_t of the most recent PEG_ERR_CUDA on this thread */
const char* pegncde_version(void);
/* kernels launched by this library since process start (for bench.py's gpu_launches) */
uint64_t pegncde_launch_count(void);

/* ---- measurement hooks (bench.py's roofline) -------------------------------------------------
 * When enabled, every `stride`-th launch of the dominant kernel (the n x n x d contraction) is
 * bracketed by CUDA events on the launching stream.  pegncde_profile_read synchronises those events
 * and returns, per direction (0 = forward contraction, 1 = backward/adjoint contraction): launches seen,
 * launches timed, summed milliseconds of the timed ones and the algorithmic bytes / flops of one launch.  For a sparse control
 * the bytes are its HBM traffic (both orientations' coefficients and columns, row pointers, V, OUT, M in the adjoint); the
 * gathers of V rows (2 nnz d 4 bytes, mostly served from L2) are not included.
 * stride <= 0 disables and frees the events. */
int pegncde_profile_enable(int32_t stride);
int pegncde_profile_read(int32_t direction, uint64_t* launches, uint64_t* timed, double* ms_total,
                         double* bytes_per_launch, double* flops_per_launch);

#ifdef __cplusplus
}
#endif
#endif /* PEGNCDE_H_ */
