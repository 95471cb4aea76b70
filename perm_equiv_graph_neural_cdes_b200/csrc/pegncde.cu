// C-ABI of the pegncde hot path (see include/pegncde.h).  Host code here only validates,
// carves the caller's workspace and enqueues kernels on the caller's stream.
#include <atomic>
#include <cstdio>
#include <cstring>
#include <vector>

#include "peg_kernels.cuh"
#include "peg_small.cuh"
#include "peg_sparse.cuh"
#include "peg_tc.cuh"

namespace peg {

static std::atomic<uint64_t> g_launches{0};
static thread_local int g_last_cuda = 0;
void set_last_cuda(int err) { g_last_cuda = err; }

#define PEG_LAUNCH_CHECK()                         \
  do {                                             \
    g_launches.fetch_add(1);                       \
    cudaError_t _e = cudaPeekAtLastError();        \
    if (_e != cudaSuccess) {                       \
      g_last_cuda = (int)_e;                       \
      (void)cudaGetLastError();                    \
      return PEG_ERR_CUDA;                         \
    }                                              \
  } while (0)

#define PEG_CUDA(call)                             \
  do {                                             \
    cudaError_t _e = (call);                       \
    if (_e != cudaSuccess) {                       \
      g_last_cuda = (int)_e;                       \
      return PEG_ERR_CUDA;                         \
    }                                              \
  } while (0)

// ---- optional per-launch timing of the contraction kernel (bench.py roofline) ----
struct Prof {
  int stride = 0;
  std::vector<cudaEvent_t> ev[2];   // pairs (start, stop)
  uint64_t seen[2] = {0, 0};
  double bytes[2] = {0, 0}, flops[2] = {0, 0};
};
static Prof g_prof;
static const size_t kMaxProfPairs = 16384;

// events recorded while the stream is being captured into a CUDA graph must be external event-record nodes
static inline void record_event(cudaEvent_t e, cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cs);
  if (cs == cudaStreamCaptureStatusActive)
    cudaEventRecordWithFlags(e, st, cudaEventRecordExternal);
  else
    cudaEventRecord(e, st);
}

static inline bool prof_begin(int dir, cudaStream_t st, double bytes, double flops) {
  Prof& p = g_prof;
  if (p.stride <= 0) return false;
  const uint64_t k = p.seen[dir]++;
  p.bytes[dir] = bytes;
  p.flops[dir] = flops;
  if (k % (uint64_t)p.stride != 0 || p.ev[dir].size() >= 2 * kMaxProfPairs) return false;
  cudaEvent_t e0, e1;
  if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return false;
  p.ev[dir].push_back(e0);
  p.ev[dir].push_back(e1);
  record_event(e0, st);
  return true;
}
static inline void prof_end(int dir, cudaStream_t st) { record_event(g_prof.ev[dir].back(), st); }

static inline int last_width(const PegDims& d) { return d.e > 0 ? 2 * d.h * d.e : d.h; }

static int check_dims(const PegDims* d) {
  if (!d) return PEG_ERR_NULL_POINTER;
  if (d->B < 1 || d->n < 1 || d->L < 1 || d->L > PEG_MAX_LAYERS || d->T < 2 || d->T > PEG_MAX_T || d->e < 0)
    return PEG_ERR_BAD_DIMS;
  if (d->h < 4 || d->h > PEG_MAX_H || (d->h % 4) != 0) return PEG_ERR_BAD_DIMS;
  if (d->ldn != peg_npad(d->n)) return PEG_ERR_BAD_DIMS;  // planes are tiled 32x32: ldn = n rounded up to 32
  if ((long long)d->B > 65535) return PEG_ERR_BAD_DIMS;
  return PEG_OK;
}

static Model make_model(const PegDims& d) {
  Model m;
  memset(&m, 0, sizeof(m));
  m.L = d.L;
  m.directed = (d.flags & PEG_FLAG_DIRECTED) ? 1 : 0;
  long long off = 0;
  int dmax = d.h;
  for (int l = 0; l < d.L; ++l) {
    LayerDesc& ld = m.layer[l];
    ld.din = d.h;
    ld.dout = (l == d.L - 1) ? last_width(d) : d.h;
    dmax = ld.dout > dmax ? ld.dout : dmax;
    ld.w_off = off;  off += (long long)ld.dout * ld.din;
    ld.b_off = off;  off += ld.dout;
    ld.nw_off = off; off += ld.din;
    ld.nb_off = off; off += ld.din;
    ld.fus_off = off; off += m.directed ? 24 : 16;   // 22 scalars + 2 of padding: every block stays 16-byte aligned
  }
  m.P = (int)off;
  m.dmax = dmax;
  return m;
}

// ------------------------------------------------------------------------------------------
// workspace carving
// ------------------------------------------------------------------------------------------
struct FevalWs {
  StageScalars* sc;
  float* svec;
  float* colM;   // [B][2][dmax]
  float* colG;   // [B][2][dmax]
  float* colPart;          // [B][row chunks][2][dmax] partial column sums
  unsigned int* tickets;   // [B][ceil(dmax/32)] self-resetting arrival counters (zeroed at every API entry)
  size_t tickets_count;
  float* M;      // [B,n,dmax]
  float* Za;     // [B,n,h] ping
  float* Zb;     // [B,n,h] pong
  float* OL;     // [B,n,dmax] last-layer output (control models)
  // vjp
  float* Obar;   // [B,n,dmax]
  float* Mbar;   // [B,n,dmax]
  float* N;      // [B,n,h]
  float* gxd;    // [B,n,2e] cotangent of control_data.derivative(t) (solve_bwd with g_xcoef)
  TcWs tc;       // tensor-core operand buffers (peg_tc.cuh)
  TcLinear lin;  // tf32 hi/lo copies of the Linear weights (tensor-core RMSNorm -> Linear)
};

static void carve_feval(Bump& bp, const PegDims& d, const Model& m, bool vjp, FevalWs& w) {
  const size_t B = d.B, n = d.n, h = d.h, dm = m.dmax;
  w.sc = bp.take<StageScalars>(B);
  w.svec = bp.take<float>(B * svec_stride(d.n, d.L, d.e));
  w.colM = bp.take<float>(B * 2 * dm);
  w.colG = bp.take<float>(B * 2 * dm);
  w.colPart = bp.take<float>(B * ((n + 31) / 32) * 2 * dm);   // chunks: 256 rows (k_colsums), 64 (norm_linear), 32 (linear_bwd)
  w.tickets_count = B * ((dm + 31) / 32) + 1;      // + the arrival counter of k_shard_push (row-sharded mode)
  w.tickets = bp.take<unsigned int>(w.tickets_count);
  w.M = bp.take<float>(B * n * dm);
  w.Za = bp.take<float>(B * n * h);
  w.Zb = bp.take<float>(B * n * h);
  w.OL = d.e > 0 ? bp.take<float>(B * n * dm) : nullptr;
  if (vjp) {
    w.Obar = bp.take<float>(B * n * dm);
    w.Mbar = bp.take<float>(B * n * dm);
    w.N = bp.take<float>(B * n * h);
    w.gxd = d.e > 0 ? bp.take<float>(B * n * 2 * d.e) : nullptr;
  } else {
    w.Obar = w.Mbar = w.N = w.gxd = nullptr;
  }
  tc_carve(bp, d, m.dmax, w.tc);
  tc_carve_linear(bp, d, m, w.lin);
}

struct Ctx {
  cudaStream_t st;
  PegDims d;
  PegControl ctl;
  const float* params;
  Model m;
  FevalWs w;
  size_t sv_stride;
  bool use_tc;
  int fmt;   // operand format of the tensor-core contraction for this call (set by make_ctx, copied into w.tc after plan())
  const PegShard* sh;   // row-sharded mode (nullptr otherwise)
  const float* t_dev;   // batched adaptive steps: per-graph step start / size (nullptr otherwise) and the stage's c_i
  const float* dt_dev;
  float tcoef;
  unsigned int* xticket;   // arrival counter of k_shard_push (in the tickets area)
  int small_C;             // > 0: the cluster-per-graph kernels of peg_small.cuh evaluate f and its VJP (CTAs per graph)
  size_t small_smem;
  float* g_adj;            // (nullable) the VJP also accumulates the cotangent of PegSparse.coef (sparse controls) or of the
                           // static adjacency [B, ldn, ldn] (static controls) here
};

// ------------------------------------------------------------------------------------------
// one vector-field evaluation: dy = f(t, yin)
//   save[l] (nullable array of L pointers): where to keep the input of layer l (l = 0: yin itself is
//   the input, nothing is copied; save[l>=1] receives relu(O_l)).
//   msave[l] / csave[l] (nullable arrays, nullable entries): where to keep M_l [B,n,dout] and its column sums [B][2][dout]
//   (written in place of the scratch copies, the contraction reads them from there).  The small-graph kernels keep neither.
// ------------------------------------------------------------------------------------------
static int stage_prep(Ctx& c, float t) {
  PrepArgs a;
  a.t_dev = c.t_dev; a.dt_dev = c.dt_dev; a.tcoef = c.tcoef;
  a.ctl = c.ctl;
  a.params = c.params;
  a.model = c.m;
  a.B = c.d.B; a.n = c.d.n; a.e = c.d.e; a.T = c.d.T;
  a.n_glob = c.sh ? c.sh->n_glob : c.d.n;
  a.t = t;
  a.sc = c.w.sc;
  a.svec = c.w.svec;
  // enough blocks for the widest loop of the kernel (the node-signal derivative, n * 2e elements) to be one or two passes
  const size_t work = (size_t)c.d.n * (c.d.e > 0 ? 2 * c.d.e : 1);
  size_t gx = (work + 255) / 256;
  gx = gx > 64 ? 64 : gx;
  dim3 grid((unsigned)gx, c.d.B);
  k_stage_prep<<<grid, 256, 0, c.st>>>(a);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

// producer-side fused outputs (V^T hi/lo for the tensor-core contraction, deterministic column sums).
// `bfp_capable`: the producer kernel that will run can emit the fp16x2 format (a tcgen05 producer whose CTA holds every column of
// its 128 nodes, so it knows the block maximum); otherwise the contraction converts V itself (k_split_transpose16).
static ProducerOut producer_out(Ctx& c, int dcols, bool want_vt, float* cb, bool with_vec, size_t vec_off, bool bfp_capable) {
  ProducerOut po;
  memset(&po, 0, sizeof(po));
  if (want_vt && c.use_tc && !c.ctl.sparse && tc_supported(c.d, dcols) && (c.w.tc.fmt != PEG_FMT_FP16X2 || bfp_capable)) {
    po.Thi = c.w.tc.Vt_hi;
    po.Tlo = c.w.tc.Vt_lo;
    po.npad = c.w.tc.npad;
    po.t16 = c.w.tc.fmt;
    po.vexp = c.w.tc.vexp;
    po.vexp_stride = c.w.tc.vexp_stride;
    po.npad = c.w.tc.ldk;            // row pitch of V^T (all nodes); this rank's rows start at column col0
    po.col0 = c.w.tc.col0;
    po.blk0 = c.w.tc.blk0;
    po.rows_pad = c.w.tc.npad;
  }
  po.cb = cb;
  po.partial = c.w.colPart;
  po.tickets = c.w.tickets;
  po.vec = with_vec ? c.w.svec + vec_off : nullptr;
  po.vec_stride = c.sv_stride;
  return po;
}
static bool norm_linear_on_tc(const Ctx& c, int l) {
  return c.use_tc && c.w.lin.ready && tc_linear_supported(c.m.layer[l].din, c.m.layer[l].dout);
}

// Nout (nullable): the normalised input, for k_weight_grad; the tensor-core path never needs it (k_tc_linear_bwd forms N itself)
static int norm_linear(Ctx& c, int l, const float* Zin, float* M, float* Nout, const ProducerOut& po) {
  const LayerDesc& ld = c.m.layer[l];
  if (norm_linear_on_tc(c, l)) {
    if (Nout != nullptr) return PEG_ERR_UNSUPPORTED;
    const int rc = tc_norm_linear(c.st, c.d, c.w.lin, l, Zin, ld.din, ld.dout, M, po);
    if (rc == PEG_OK) g_launches.fetch_add(1);
    return rc;
  }
  dim3 grid((c.d.n + NL_BM - 1) / NL_BM, (ld.dout + NL_BN - 1) / NL_BN, c.d.B);
  k_norm_linear<<<grid, 256, 0, c.st>>>(Zin, c.d.n, ld.din, ld.dout, c.params + ld.w_off, c.params + ld.b_off,
                                        c.params + ld.nw_off, c.params + ld.nb_off, M, Nout, po);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

static int colsums(Ctx& c, const float* V, int dcols, size_t vec_off, bool with_vec, float* cb) {
  dim3 grid((dcols + 31) / 32, (c.d.n + CS_ROWS - 1) / CS_ROWS, c.d.B), block(32, 8);
  k_colsums<<<grid, block, 0, c.st>>>(V, c.d.n, dcols, with_vec ? c.w.svec + vec_off : nullptr, c.sv_stride, cb,
                                      c.w.colPart, c.w.tickets);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

// ---- row-sharded mode: one exchange (see PegShard in pegncde.h).  `with_vt`: this rank's slice of V^T (+ block exponents) travels;
// cs0 / cs1 (nullable): [B][2][dcols] column-sum vectors that are partial sums over this rank's rows and come back summed over all ranks.
static int shard_exchange(Ctx& c, bool with_vt, int dcols, float* cs0, float* cs1) {
  const PegShard& sh = *c.sh;
  const uint32_t epoch = ++(*sh.epoch);
  ShardXchg x;
  memset(&x, 0, sizeof(x));
  for (int q = 0; q < sh.world; ++q) {
    x.vt_hi[q] = sh.vt_hi[q]; x.vt_lo[q] = sh.vt_lo[q]; x.vexp[q] = sh.vexp[q]; x.colsum[q] = sh.colsum[q]; x.flags[q] = sh.flags[q];
  }
  x.rank = sh.rank; x.world = sh.world; x.epoch = epoch; x.epoch_base = sh.epoch_dev;
  const size_t esz = c.w.tc.fmt == PEG_FMT_TF32X3 ? 4 : 2;
  const size_t ldk = (size_t)peg_npad(sh.n_glob);
  x.half_bytes = (size_t)c.d.B * c.m.dmax * ldk * 4;          // the halves are sized for fp32 words (3xTF32), 16-bit parts use the front
  x.push_vt = with_vt ? 1 : 0;
  x.rows = c.d.B * dcols;
  x.pitch_bytes = ldk * esz;
  x.col0_bytes = (size_t)sh.row0 * esz;
  x.slice_bytes = (size_t)c.d.ldn * esz;
  x.vexp_stride = c.w.tc.vexp_stride; x.vexp_half = c.d.B * c.w.tc.vexp_stride; x.blk0 = sh.row0 / 128; x.nblk_loc = c.d.ldn / 128; x.B = c.d.B;
  x.push_vexp = (with_vt && c.w.tc.fmt == PEG_FMT_FP16X2) ? 1 : 0;
  x.cs_src[0] = cs0; x.cs_src[1] = cs1; x.cs_dst[0] = cs0; x.cs_dst[1] = cs1;
  x.cs_len = c.d.B * 2 * dcols;
  x.cs_cap = (size_t)c.d.B * 2 * c.m.dmax;
  x.cs_half = (size_t)sh.world * 2 * x.cs_cap;
  x.ticket = c.xticket;
  // the producers / tc_convert_v wrote the half of parity (epoch & 1): point the local operand buffers at the other half for the next one
  const size_t bytes = (size_t)x.rows * x.slice_bytes * 2;
  unsigned gx = (unsigned)((bytes / 16 + 255) / 256);
  gx = gx < 1 ? 1 : (gx > 64 ? 64 : gx);      // a few dozen CTAs saturate the NVLink ports; the copy is small next to the contraction
  k_shard_push<<<dim3(gx, sh.world), 256, 0, c.st>>>(x);
  PEG_LAUNCH_CHECK();
  k_shard_wait<<<1, 256, 0, c.st>>>(x);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}
// graph-replayable mode: every API call leaves the epoch base even and past its own exchanges
static int shard_finish(Ctx& c) {
  if (!c.sh || !c.sh->epoch_dev) return PEG_OK;
  if (*c.sh->epoch & 1u) PEG_TRY(shard_exchange(c, false, 0, nullptr, nullptr));     // flag-only exchange: keeps the parity halves alternating
  k_epoch_advance<<<1, 1, 0, c.st>>>(c.sh->epoch_dev, *c.sh->epoch);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}
// operand buffers of the NEXT exchange: the epoch-parity half the producers must write and the contraction will read
static void shard_select_half(Ctx& c) {
  if (!c.sh) return;
  const PegShard& sh = *c.sh;
  const uint32_t next = *sh.epoch + 1;
  const size_t half_bytes = (size_t)c.d.B * c.m.dmax * peg_npad(sh.n_glob) * 4;
  c.w.tc.Vt_hi = (float*)((char*)sh.vt_hi[sh.rank] + (next & 1u) * half_bytes);
  c.w.tc.Vt_lo = (float*)((char*)sh.vt_lo[sh.rank] + (next & 1u) * half_bytes);
  c.w.tc.vexp = sh.vexp[sh.rank] + (size_t)(next & 1u) * c.d.B * c.w.tc.vexp_stride;
}

static bool contract_on_tc(const Ctx& c, int l) { return c.use_tc && !c.ctl.sparse && tc_supported(c.d, c.m.layer[l].dout); }

// cbM_global: cbM is already summed over all ranks (solve_fwd kept it after its own exchange), so the exchange leaves it alone
static int contract(Ctx& c, int l, bool bwd, const float* V, const float* Mref, const float* colbuf, float* out,
                    bool relu, bool scale_tg, float* g_fus, bool vt_ready, const float* cbM = nullptr, bool cbM_global = false) {
  const LayerDesc& ld = c.m.layer[l];
  ContractArgs a;
  a.stat = c.ctl.adj_static ? 1 : 0;
  a.planes = a.stat ? c.ctl.adj_static : c.ctl.adj_coef;
  a.graph_stride = a.stat ? (size_t)c.d.ldn * c.d.ldn : (size_t)(c.d.T - 1) * 4 * c.d.ldn * c.d.ldn;
  a.sc = c.w.sc;
  a.svec = c.w.svec;
  a.sv_stride = c.sv_stride;
  a.rowc_off = bwd ? svec_c(c.d.n, l) : svec_r(c.d.n, l);
  a.v_off = svec_v(c.d.n, l);
  a.tg_off = svec_tg(c.d.n, c.d.L);
  a.fus = c.params + ld.fus_off;
  a.V = V;
  a.Mref = Mref;
  a.colbuf = colbuf;
  a.cbM = cbM;
  a.L = c.d.L;
  a.out = out;
  a.g_fus = g_fus;
  a.n = c.d.n; a.ldn = c.d.ldn; a.d = ld.dout; a.layer = l;
  a.relu = relu ? 1 : 0;
  a.scale_tg = scale_tg ? 1 : 0;
  a.vt_ready = vt_ready ? 1 : 0;
  a.planes_t = c.sh ? c.sh->adj_coef_t : nullptr;
  a.ldk = c.sh ? peg_npad(c.sh->n_glob) : c.d.ldn;
  a.n_glob = c.sh ? c.sh->n_glob : c.d.n;
  a.row_block0 = c.sh ? c.sh->row0 / 128 : 0;
  if (c.sh) a.graph_stride = (size_t)(c.d.T - 1) * 4 * c.d.ldn * a.ldk;
  // algorithmic work of one launch: the four coefficient planes are traversed once (16 n^2 B per graph; a static control's one
  // plane: 4 n^2 B), V is read and OUT written once; 2 (fwd) or 4 (bwd) n x n x d products.
  const double nn = (double)c.d.n * c.d.n, nd = (double)c.d.n * ld.dout;
  double bytes = c.d.B * ((a.stat ? 4.0 : 16.0) * nn + 4.0 * nd * (bwd ? 3.0 : 2.0));
  double flops = c.d.B * (bwd ? 8.0 : 4.0) * nn * ld.dout;
  if (c.ctl.sparse) {
    // sparse path: both orientations' coefficients (one piece) and columns, both row-pointer arrays, V and OUT once (+ M in the
    // adjoint).  The gathers of V rows (2 nnz d 4 bytes, mostly served from L2) are not HBM traffic and are not counted here.
    const double nnz = (double)c.ctl.sparse->nnz;
    bytes = 2.0 * nnz * (16.0 + 4.0) + 2.0 * c.d.B * (c.d.n + 1.0) * 4.0 + c.d.B * 4.0 * nd * (bwd ? 3.0 : 2.0);
    flops = (bwd ? 8.0 : 4.0) * nnz * ld.dout;
  }
  const int dir = bwd ? 1 : 0;
  const bool timed = prof_begin(dir, c.st, bytes, flops);
  int rc = PEG_OK;
  if (c.ctl.sparse) {
    const int glog = sparse_glog(ld.dout), G = 1 << glog;
    dim3 grid((unsigned)((c.d.n + 8 * (32 / G) - 1) / (8 * (32 / G))), (unsigned)((ld.dout + 4 * G - 1) / (4 * G)), c.d.B);
    if (!bwd)
      k_sparse_contract<1><<<grid, 256, 0, c.st>>>(a, *c.ctl.sparse, glog);
    else
      k_sparse_contract<4><<<grid, 256, 0, c.st>>>(a, *c.ctl.sparse, glog);
    g_launches.fetch_add(1);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) { g_last_cuda = (int)e; (void)cudaGetLastError(); rc = PEG_ERR_CUDA; }
  } else if (c.sh) {
    // row-sharded: every rank needs ALL rows of V^T and the column sums over ALL nodes -> convert V if no producer did, then the
    // exchange over peer memory (push + flags, wait + rank-ordered column sums), then the local row blocks of the contraction
    if (!vt_ready) { rc = tc_convert_v(c.st, c.d, c.w.tc, a); g_launches.fetch_add(c.w.tc.fmt == PEG_FMT_FP16X2 ? 2 : 1); }
    if (rc == PEG_OK) rc = shard_exchange(c, true, ld.dout, const_cast<float*>(colbuf), cbM_global ? nullptr : const_cast<float*>(cbM));
    a.vt_ready = 1;
    if (rc == PEG_OK) rc = tc_contract(c.st, c.d, c.w.tc, a, bwd);
    if (rc == PEG_OK) g_launches.fetch_add(1);
    shard_select_half(c);     // the producers of the next layer write the other epoch-parity half
  } else if (c.use_tc && tc_supported(c.d, ld.dout)) {
    rc = tc_contract(c.st, c.d, c.w.tc, a, bwd);
    if (rc == PEG_OK) g_launches.fetch_add(vt_ready ? 1 : (c.w.tc.fmt == PEG_FMT_FP16X2 ? 3 : 2));
  } else {
    dim3 grid((c.d.n + CT_TI - 1) / CT_TI, (ld.dout + CT_TC - 1) / CT_TC, c.d.B);
    if (a.stat) {
      if (!bwd) k_dual_contract<1, true><<<grid, 256, 0, c.st>>>(a);
      else k_dual_contract<4, true><<<grid, 256, 0, c.st>>>(a);
    } else if (!bwd) {
      k_dual_contract<1><<<grid, 256, 0, c.st>>>(a);
    } else {
      k_dual_contract<4><<<grid, 256, 0, c.st>>>(a);
    }
    g_launches.fetch_add(1);
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) { g_last_cuda = (int)e; (void)cudaGetLastError(); rc = PEG_ERR_CUDA; }
  }
  if (timed) prof_end(dir, c.st);
  return rc;
}

// ------------------------------------------------------------------------------------------
// small graphs: one cluster kernel per evaluation / per VJP (peg_small.cuh)
// ------------------------------------------------------------------------------------------
// decides whether this call runs on the small-graph kernels and with how many CTAs per graph
static void small_plan(Ctx& c) {
  c.small_C = 0;
  c.small_smem = 0;
  const PegDims& d = c.d;
  if (d.flags & PEG_FLAG_NO_FUSED_SMALL) return;
  // default: below the smallest tcgen05 shape; PEG_FLAG_FUSED_SMALL widens it
  const int max_n = (d.flags & PEG_FLAG_FUSED_SMALL) ? 256 : 127;
  if (c.sh || c.ctl.sparse || c.m.directed || d.n > max_n || d.n > SG_MAX_N || d.h > SG_MAX_DIN) return;
  const size_t smem = small_smem_floats(d.n, d.L) * sizeof(float);
  if (smem > 220 * 1024) return;
  int dev = 0, sm_count = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { (void)cudaGetLastError(); return; }
  // a static control is planned exactly like a dense one (same cluster width): only the kernels' plane loads differ
  static std::atomic<unsigned> smem_done[4] = {}, cluster_done[4] = {};
  const bool stat = c.ctl.adj_static != nullptr;
  auto fwd = stat ? k_small_fwd<true> : k_small_fwd<false>;
  auto vjp = stat ? k_small_vjp<true> : k_small_vjp<false>;
  const int k0 = stat ? 2 : 0;
  if (optin_smem(fwd, smem_done[k0]) != PEG_OK || optin_smem(vjp, smem_done[k0 + 1]) != PEG_OK) return;
  const bool nonportable = optin_nonportable_cluster(fwd, cluster_done[k0]) == PEG_OK &&
                           optin_nonportable_cluster(vjp, cluster_done[k0 + 1]) == PEG_OK;
  // CTAs per graph: as many as keep the batch within one wave of SMs, no more than the widest phase has work items
  const int dL = c.m.layer[d.L - 1].dout;
  const int items = ((d.n + SG_RB - 1) / SG_RB) * ((dL + SG_WB - 1) / SG_WB);
  int C = 1;
  for (int cand = nonportable ? 16 : 8; cand >= 1; cand >>= 1)
    if ((long long)d.B * cand <= sm_count && cand <= items) { C = cand; break; }
  c.small_C = C;
  c.small_smem = smem;
}

static void small_args(const Ctx& c, float t, SmallArgs& a) {
  memset(&a, 0, sizeof(a));
  a.ctl = c.ctl; a.params = c.params; a.model = c.m;
  a.B = c.d.B; a.n = c.d.n; a.e = c.d.e; a.T = c.d.T; a.L = c.d.L; a.h = c.d.h; a.npad = c.d.ldn; a.C = c.small_C;
  a.t = t;
  a.sc = c.w.sc;
  a.M = c.w.M; a.Za = c.w.Za; a.Zb = c.w.Zb; a.OL = c.w.OL; a.Obar = c.w.Obar; a.Mbar = c.w.Mbar; a.N = c.w.N;
}

static int small_launch(Ctx& c, const SmallArgs& a, bool vjp) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(c.d.B * c.small_C));
  cfg.blockDim = dim3(SG_THREADS);
  cfg.dynamicSmemBytes = c.small_smem;
  cfg.stream = c.st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)c.small_C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  const bool stat = c.ctl.adj_static != nullptr;
  const cudaError_t e = vjp ? cudaLaunchKernelEx(&cfg, stat ? k_small_vjp<true> : k_small_vjp<false>, a)
                            : cudaLaunchKernelEx(&cfg, stat ? k_small_fwd<true> : k_small_fwd<false>, a);
  g_launches.fetch_add(1);
  if (e != cudaSuccess) { g_last_cuda = (int)e; (void)cudaGetLastError(); return PEG_ERR_CUDA; }
  return PEG_OK;
}

static int feval_fwd(Ctx& c, float t, const float* yin, float* dy, float* const* save, int nlayers = -1, float* const* msave = nullptr,
                     float* const* csave = nullptr) {
  const PegDims& d = c.d;
  if (nlayers < 0) nlayers = d.L;
  if (c.small_C > 0 && !c.t_dev) {
    SmallArgs a;
    small_args(c, t, a);
    a.yin = yin; a.dy = dy; a.nlayers = nlayers;
    for (int l = 0; l < d.L; ++l) a.save[l] = save ? save[l] : nullptr;
    return small_launch(c, a, false);
  }
  PEG_TRY(stage_prep(c, t));
  const float* Zin = yin;
  for (int l = 0; l < nlayers; ++l) {
    const LayerDesc& ld = c.m.layer[l];
    const bool last = (l == d.L - 1);
    float* M = (msave && msave[l]) ? msave[l] : c.w.M;
    float* colM = (csave && csave[l]) ? csave[l] : c.w.colM;
    const ProducerOut po = producer_out(c, ld.dout, true, colM, true, svec_c(d.n, l), norm_linear_on_tc(c, l) && tc_norm_linear_full_columns(ld.dout));
    PEG_TRY(norm_linear(c, l, Zin, M, nullptr, po));
    float* out;
    if (!last) {
      out = (save && save[l + 1]) ? save[l + 1] : ((l & 1) ? c.w.Zb : c.w.Za);
    } else {
      out = d.e > 0 ? c.w.OL : dy;
    }
    PEG_TRY(contract(c, l, false, M, nullptr, colM, out, !last, last, nullptr, po.Thi != nullptr));
    Zin = out;
  }
  if (d.e > 0 && nlayers == d.L) {
    const size_t cnt = (size_t)d.B * d.n * d.h;
    k_wrapper_fwd<<<(unsigned)((cnt + 255) / 256), 256, 0, c.st>>>(c.w.OL, c.w.svec, c.sv_stride,
                                                                   svec_xd(d.n, d.L), d.n, d.h, 2 * d.e, d.B, dy);
    PEG_LAUNCH_CHECK();
  }
  return PEG_OK;
}

// cotangent of the sparse coefficients, or of the static adjacency, through layer l (peg_sparse.cuh, peg_tc.cu).  The node tables
// live in Za / Zb, which the VJP does not use otherwise: [B][4][n] fits in Za and [B][n] + [B][2] in Zb, since h >= 4.
// The static n x n product runs on k_tc_adj_grad with PEG_FLAG_TENSOR_CORES and n >= 128, on the fp32 k_adj_grad otherwise.
static bool adj_grad_on_tc(const Ctx& c) { return c.use_tc && c.d.n >= 128; }

static int adj_grad(Ctx& c, int l, const float* M, const float* colM) {
  const PegDims& d = c.d;
  const LayerDesc& ld = c.m.layer[l];
  AdjGradArgs a;
  a.G = c.w.Obar; a.M = M; a.cbM = colM; a.cbG = c.w.colG;
  a.fus = c.params + ld.fus_off;
  a.sc = c.w.sc;
  a.node = c.w.Za;
  a.q = c.w.Zb;
  a.tot = c.w.Zb + (size_t)d.B * d.n;
  a.g_coef = c.g_adj;
  a.n = d.n; a.d = ld.dout; a.directed = c.m.directed;
  k_sparse_adj_node<<<dim3((d.n + 7) / 8, d.B), 256, 0, c.st>>>(a);
  PEG_LAUNCH_CHECK();
  k_sparse_adj_tot<<<d.B, 1024, 0, c.st>>>(a);
  PEG_LAUNCH_CHECK();
  if (c.ctl.adj_static) {
    if (adj_grad_on_tc(c)) {
      PEG_TRY(tc_adj_grad(c.st, d, a.G, a.M, ld.dout, a.fus, a.node, a.q, a.tot, c.g_adj));
      g_launches.fetch_add(1);
    } else {
      const unsigned tiles = (unsigned)((d.n + AG_TILE - 1) / AG_TILE);
      k_adj_grad<<<dim3(tiles, tiles, d.B), 256, 0, c.st>>>(a, c.g_adj, d.ldn);
      PEG_LAUNCH_CHECK();
    }
    return PEG_OK;
  }
  const int glog = sparse_adj_glog(ld.dout), G = 1 << glog;
  k_sparse_adj_grad<<<dim3((unsigned)((d.n + 8 * (32 / G) - 1) / (8 * (32 / G))), d.B), 256, 0, c.st>>>(a, *c.ctl.sparse, glog);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

// VJP of one evaluation.  zin[l] = input of layer l (l = 0..L-1) as saved by feval_fwd.
// kbar: cotangent of dy.  Writes ybar (cotangent of the stage input), accumulates g_params.
// If g_xd != null (control models) also writes the cotangent of control_data.derivative(t).
// mkept / ckept (nullable arrays, nullable entries): M_l and its column sums as feval_fwd kept them (msave / csave); the
// tensor-core path then skips the RMSNorm -> Linear recompute of that layer.
static int feval_vjp(Ctx& c, float t, float* const* zin, const float* kbar, float* ybar, float* g_params,
                     float* g_xd, float* const* mkept = nullptr, float* const* ckept = nullptr) {
  const PegDims& d = c.d;
  const int dL = last_width(d);
  if (g_xd != nullptr && d.e == 0) return PEG_ERR_BAD_DIMS;
  if (c.small_C > 0 && !c.t_dev) {
    SmallArgs a;
    small_args(c, t, a);
    for (int l = 0; l < d.L; ++l) a.zin[l] = zin[l];
    a.kbar = kbar; a.ybar = ybar; a.g_params = g_params; a.g_xd = g_xd;
    return small_launch(c, a, true);
  }
  PEG_TRY(stage_prep(c, t));
  if (g_xd != nullptr) {
    if (d.e == 0) return PEG_ERR_BAD_DIMS;
    // recompute the (tg-scaled) last-layer output, then contract it with kbar
    const int l = d.L - 1;
    const ProducerOut po = producer_out(c, dL, true, c.w.colM, true, svec_c(d.n, l), norm_linear_on_tc(c, l) && tc_norm_linear_full_columns(dL));
    PEG_TRY(norm_linear(c, l, zin[l], c.w.M, nullptr, po));
    PEG_TRY(contract(c, l, false, c.w.M, nullptr, c.w.colM, c.w.OL, false, true, nullptr, po.Thi != nullptr));
    const size_t cnt = (size_t)d.B * d.n * 2 * d.e;
    k_wrapper_xbar<<<(unsigned)((cnt + 255) / 256), 256, 0, c.st>>>(kbar, c.w.OL, d.n, d.h, 2 * d.e, d.B, g_xd);
    PEG_LAUNCH_CHECK();
  }
  bool obar_ready = false;   // column sums / V^T of Obar already produced by the previous k_linear_bwd
  bool obar_vt = false;
  // without the CDE wrapper the top cotangent is tg (.) kbar: on the tensor-core path one kernel writes it together with its
  // column sums, block exponents and V^T (otherwise: k_wrapper_bwd here, k_colsums / tc_convert_v further down)
  const bool top_fused = d.e == 0 && contract_on_tc(c, d.L - 1) && dL <= 256 && (dL % 4) == 0;
  if (top_fused) {
    static std::atomic<unsigned> smem_done{0u};
    PEG_TRY(optin_smem(k_top_producer, smem_done));
    const ProducerOut po = producer_out(c, dL, true, c.w.colG, true, svec_r(d.n, d.L - 1), true);
    if (po.Thi == nullptr) return PEG_ERR_WORKSPACE;
    dim3 grid((unsigned)((po.rows_pad + 127) / 128), d.B);
    k_top_producer<<<grid, 256, 128 * (dL + 1) * sizeof(float), c.st>>>(kbar, c.w.svec, c.sv_stride, svec_tg(d.n, d.L), d.n, dL, c.w.Obar, po);
    PEG_LAUNCH_CHECK();
    obar_ready = true;
    obar_vt = true;
  } else {
    const size_t cnt = (size_t)d.B * d.n * dL;
    k_wrapper_bwd<<<(unsigned)((cnt + 255) / 256), 256, 0, c.st>>>(kbar, c.w.svec, c.sv_stride, svec_xd(d.n, d.L),
                                                                   svec_tg(d.n, d.L), d.n, d.h, 2 * d.e, d.B,
                                                                   c.w.Obar);
    PEG_LAUNCH_CHECK();
  }
  for (int l = d.L - 1; l >= 0; --l) {
    const LayerDesc& ld = c.m.layer[l];
    float* g_fus = g_params + ld.fus_off;
    const bool lb_tc = c.use_tc && c.w.lin.ready && tc_linear_bwd_supported(ld.din, ld.dout);
    const bool wg_fused = lb_tc && tc_linear_bwd_fuses_weight_grad(d, ld.din, ld.dout);
    // M_l and 1^T M_l: as the forward kept them, or recomputed from the saved layer input.  Without tensor cores the recompute
    // also writes the normalised input N_l for k_weight_grad (k_tc_linear_bwd forms N_l itself).
    const bool kept = lb_tc && mkept && mkept[l] && ckept && ckept[l];
    const float* M = kept ? mkept[l] : c.w.M;
    const float* colM = kept ? ckept[l] : c.w.colM;
    if (!kept) PEG_TRY(norm_linear(c, l, zin[l], c.w.M, lb_tc ? nullptr : c.w.N, producer_out(c, ld.dout, false, c.w.colM, false, 0, false)));
    if (!obar_ready) PEG_TRY(colsums(c, c.w.Obar, ld.dout, svec_r(d.n, l), true, c.w.colG));
    // the tcgen05 adjoint epilogue also emits the param3..8 gradients (undirected layer; the directed one keeps the separate kernel)
    const bool fused_vec_grads = contract_on_tc(c, l) && !c.m.directed;
    PEG_TRY(contract(c, l, true, c.w.Obar, M, c.w.colG, c.w.Mbar, false, false, g_fus, obar_vt, fused_vec_grads ? colM : nullptr, kept));
    if (!fused_vec_grads) {
      FusGradArgs a;
      a.G = c.w.Obar; a.M = M; a.cbM = colM; a.cbG = c.w.colG;
      a.sc = c.w.sc; a.svec = c.w.svec; a.sv_stride = c.sv_stride;
      a.n = d.n; a.d = ld.dout; a.L = d.L; a.g_fus = g_fus; a.directed = c.m.directed;
      dim3 grid((d.n + 7) / 8, d.B);
      k_fusion_vec_grads<<<grid, 256, 0, c.st>>>(a);
      PEG_LAUNCH_CHECK();
    }
    if (c.g_adj) PEG_TRY(adj_grad(c, l, M, colM));   // reads Obar: before the Linear backward overwrites it
    {
      dim3 grid((d.n + 31) / 32, d.B);
      float* zb = (l == 0) ? ybar : c.w.Obar;
      // for l > 0 the output is the cotangent Obar of layer l-1: emit its column sums (vec = r_{l-1}) and V^T here
      ProducerOut po;
      memset(&po, 0, sizeof(po));
      if (l > 0) po = producer_out(c, ld.din, true, c.w.colG, true, svec_r(d.n, l - 1), lb_tc);
      if (lb_tc) {
        PEG_TRY(tc_linear_bwd(c.st, c.d, c.w.lin, l, c.w.Mbar, zin[l], c.params + ld.nw_off, c.params + ld.nb_off, ld.din, ld.dout, l > 0 ? 1 : 0,
                              zb, g_params + ld.nw_off, g_params + ld.nb_off, wg_fused ? g_params + ld.w_off : nullptr,
                              wg_fused ? g_params + ld.b_off : nullptr, wg_fused ? nullptr : c.w.N, po));
        g_launches.fetch_add(1);
      } else {
        k_linear_bwd<<<grid, 256, 0, c.st>>>(c.w.Mbar, c.params + ld.w_off, zin[l], c.params + ld.nw_off, d.n,
                                                ld.din, ld.dout, l > 0 ? 1 : 0, zb, g_params + ld.nw_off,
                                                g_params + ld.nb_off, po);
        PEG_LAUNCH_CHECK();
      }
      obar_ready = l > 0;
      obar_vt = po.Thi != nullptr;
    }
    // Linear weight / bias gradient from Mbar and N (unless k_tc_linear_bwd already added it)
    if (!wg_fused) {
      const size_t rows = (size_t)d.B * d.n;
      if (lb_tc) {
        PEG_TRY(tc_weight_grad(c.st, c.d, c.w.Mbar, c.w.N, rows, ld.din, ld.dout, g_params + ld.w_off, g_params + ld.b_off));
        g_launches.fetch_add(1);
      } else {
        // slices of the node dimension: enough blocks to fill the GPU even for small d_out x d_in
        const int tiles = ((ld.dout + 63) / 64) * ((ld.din + 63) / 64);
        int rps = 512;
        while (rps > 64 && tiles * ((rows + rps - 1) / rps) < 296) rps >>= 1;
        dim3 grid((ld.dout + 63) / 64, (ld.din + 63) / 64, (unsigned)((rows + rps - 1) / rps));
        k_weight_grad<<<grid, 256, 0, c.st>>>(c.w.Mbar, c.w.N, rows, ld.din, ld.dout, rps, g_params + ld.w_off,
                                              g_params + ld.b_off);
        PEG_LAUNCH_CHECK();
      }
    }
  }
  return PEG_OK;
}

// out = sum_j cs[j] xs[j]; with `gscale` ([B], device) the coefficients of xs[1..] are multiplied by the graph's own factor (its step size)
static int combine(Ctx& c, float* out, int cnt, const float* const* xs, const double* cs, const float* gscale = nullptr) {
  CombArgs a;
  memset(&a, 0, sizeof(a));
  int k = 0;
  for (int j = 0; j < cnt; ++j) {
    if (cs[j] == 0.0) continue;
    a.x[k] = xs[j];
    a.c[k] = (float)cs[j];
    ++k;
  }
  a.cnt = k;
  a.out = out;
  a.count4 = (size_t)c.d.B * c.d.n * c.d.h / 4;
  a.gscale = gscale;
  a.per_graph4 = (size_t)c.d.n * c.d.h / 4;
  k_rk_combine<<<(unsigned)((a.count4 + 255) / 256), 256, 0, c.st>>>(a);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

// a PegSparse the kernels can walk: every array present, coefficient slabs 16-byte aligned (one float4 per entry)
static int check_sparse(const PegSparse* sp) {
  if (!sp->row_ptr || !sp->col || !sp->coef || !sp->row_ptr_t || !sp->col_t || !sp->coef_t) return PEG_ERR_NULL_POINTER;
  if (sp->nnz < 0 || sp->nnz > INT32_MAX || sp->nnz_stride < sp->nnz) return PEG_ERR_BAD_DIMS;
  if ((((uintptr_t)sp->coef | (uintptr_t)sp->coef_t) & 15) != 0) return PEG_ERR_ALIGNMENT;
  return PEG_OK;
}

static int make_ctx(Ctx& c, peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params) {
  PEG_TRY(check_dims(dims));
  if (!ctl || !params) return PEG_ERR_NULL_POINTER;
  if (!ctl->ts || (!ctl->adj_coef && !ctl->sparse && !ctl->adj_static) || !ctl->adj_rowsum || !ctl->adj_diag || !ctl->adj_total ||
      !ctl->tch_coef)
    return PEG_ERR_NULL_POINTER;
  if (dims->e > 0 && !ctl->x_coef) return PEG_ERR_NULL_POINTER;
  if ((dims->flags & PEG_FLAG_DIRECTED) && !ctl->adj_colsum) return PEG_ERR_NULL_POINTER;
  if (ctl->adj_static) {
    if (ctl->sparse || ctl->shard) return PEG_ERR_UNSUPPORTED;   // a static control is one dense plane on one GPU
    if (((uintptr_t)ctl->adj_static & 15) != 0) return PEG_ERR_ALIGNMENT;
  } else if (ctl->sparse) {
    if (ctl->shard) return PEG_ERR_UNSUPPORTED;     // row-sharded sparse controls are not implemented
    PEG_TRY(check_sparse(ctl->sparse));
  } else if (((uintptr_t)ctl->adj_coef & 15) != 0) {
    return PEG_ERR_ALIGNMENT;
  }
  c.st = (cudaStream_t)stream;
  c.d = *dims;
  if (ctl->adj_static) c.d.flags &= ~PEG_FLAG_ADJ_LIGHT;   // no A'_s product to lighten: the static adjoint is the exact one
  c.ctl = *ctl;
  c.params = params;
  c.m = make_model(*dims);
  c.sv_stride = svec_stride(dims->n, dims->L, dims->e);
  c.use_tc = (dims->flags & PEG_FLAG_TENSOR_CORES) != 0;
  c.fmt = tc_fmt(c.d, ctl->adj_absmax != nullptr);
  c.t_dev = c.dt_dev = nullptr;
  c.tcoef = 0.f;
  c.g_adj = nullptr;
  c.sh = ctl->shard;
  small_plan(c);
  if (c.sh) {
    const PegShard& sh = *c.sh;
    if (sh.world < 1 || sh.world > PEG_MAX_WORLD || sh.rank < 0 || sh.rank >= sh.world) return PEG_ERR_BAD_DIMS;
    if ((dims->n % 128) != 0 || sh.n_glob != sh.world * dims->n || sh.row0 != sh.rank * dims->n) return PEG_ERR_BAD_DIMS;
    if (!c.use_tc || dims->e != 0 || (dims->flags & (PEG_FLAG_DIRECTED | PEG_FLAG_BF16X2)) || (dims->h % 32) != 0 || c.fmt == PEG_FMT_BF16X2) return PEG_ERR_UNSUPPORTED;
    if (!sh.adj_coef_t || !sh.vt_hi || !sh.vt_lo || !sh.vexp || !sh.colsum || !sh.flags || !sh.epoch) return PEG_ERR_NULL_POINTER;
  }
  return PEG_OK;
}

// start of every compute entry point: arrival counters zeroed, tensor-core weight copies refreshed (params may have
// changed since the previous call; the copies live in the caller's workspace)
static int reset_tickets(Ctx& c) {
  c.w.tc.fmt = c.fmt;   // plan() carved the workspace after make_ctx chose the format
  c.xticket = c.w.tickets + (c.w.tickets_count - 1);
  if (c.sh && c.sh->epoch_dev) *c.sh->epoch = 0;     // per-call sequence numbers on top of the device-side base
  if (c.sh) {           // row-sharded: V^T spans all n_glob nodes and lives in the peer-visible buffers
    c.w.tc.ldk = peg_npad(c.sh->n_glob);
    c.w.tc.col0 = c.sh->row0;
    c.w.tc.blk0 = c.sh->row0 / 128;
    c.w.tc.vexp_stride = c.w.tc.ldk / 128;
    shard_select_half(c);
  }
  PEG_CUDA(cudaMemsetAsync(c.w.tickets, 0, c.w.tickets_count * sizeof(unsigned int), c.st));
  if (c.w.tc.vmax) PEG_CUDA(cudaMemsetAsync(c.w.tc.vmax, 0, 2 * (size_t)c.d.B * ((c.w.tc.npad + 127) / 128) * sizeof(unsigned int), c.st));
  if (c.use_tc && c.small_C == 0) {
    PEG_TRY(tc_prep_weights(c.st, c.m, c.params, c.w.lin));
    g_launches.fetch_add(c.m.L);
  }
  return PEG_OK;
}

// stage_store[step][stage 0..5], one block per stage:
//   Z: the input of every layer, L slots of [B,n,h] (layer 0 of stage 0 is y_ckpt[step] itself and stays unused);
//   M: the output M_l = RMSNorm -> Linear of every layer whose output is h wide (all but the 2he-wide last layer of a control
//      model), one slot of [B,n,h] each;
//   C: the column sums of those M_l, [B][2][h] each (row 0 = 1^T M, row 1 = 1^T diag(c_l) M).
// With it solve_bwd needs no forward recompute, and its tensor-core path no RMSNorm -> Linear recompute for the kept layers.
static int kept_m_layers(const PegDims& d) { return d.e > 0 ? d.L - 1 : d.L; }
static size_t store_stage_elems(const PegDims& d) {
  const size_t st = (size_t)d.B * d.n * d.h;
  return (size_t)(d.L + kept_m_layers(d)) * st + (size_t)kept_m_layers(d) * d.B * 2 * d.h;
}
struct StoreSlots {
  float* z[PEG_MAX_LAYERS];
  float* m[PEG_MAX_LAYERS];
  float* cm[PEG_MAX_LAYERS];
};
static StoreSlots store_slots(const PegDims& d, float* store, int step, int stage) {
  StoreSlots s;
  memset(&s, 0, sizeof(s));
  const size_t st = (size_t)d.B * d.n * d.h;
  float* base = store + ((size_t)step * 6 + stage) * store_stage_elems(d);
  for (int l = 0; l < d.L; ++l) s.z[l] = base + (size_t)l * st;
  for (int l = 0; l < kept_m_layers(d); ++l) {
    s.m[l] = base + (size_t)(d.L + l) * st;
    s.cm[l] = base + (size_t)(d.L + kept_m_layers(d)) * st + (size_t)l * d.B * 2 * d.h;
  }
  return s;
}

struct SolveWs {
  float* k[7];
  float* Z0;         // stage input
  float* ytmp;
  // bwd
  float* save[6][PEG_MAX_LAYERS];  // per stage, per layer input
  float* Ybar[6];
  float* kbar;
  float* gcur;
  float* gnext;
};

static size_t plan(const PegDims& d, int which, int steps, void* base, FevalWs* fw, SolveWs* sw) {
  Model m = make_model(d);
  Bump bp(base);
  FevalWs w;
  SolveWs s;
  memset(&s, 0, sizeof(s));
  const size_t st = (size_t)d.B * d.n * d.h;
  const bool vjp = (which == PEG_WS_VF_VJP || which == PEG_WS_SOLVE_BWD);
  carve_feval(bp, d, m, vjp, w);
  if (which == PEG_WS_VF_VJP) {
    for (int l = 1; l < d.L; ++l) s.save[0][l] = bp.take<float>(st);
  }
  if (which == PEG_WS_SOLVE_FWD || which == PEG_WS_STEP) {
    for (int i = 0; i < 7; ++i) s.k[i] = bp.take<float>(st);
    s.Z0 = bp.take<float>(st);
    s.ytmp = bp.take<float>(st);
  }
  if (which == PEG_WS_SOLVE_BWD) {
    for (int i = 0; i < 6; ++i) s.k[i] = bp.take<float>(st);
    for (int i = 0; i < 6; ++i)
      for (int l = 0; l < d.L; ++l) s.save[i][l] = bp.take<float>(st);
    for (int i = 0; i < 6; ++i) s.Ybar[i] = bp.take<float>(st);
    s.kbar = bp.take<float>(st);
    s.gcur = bp.take<float>(st);
    s.gnext = bp.take<float>(st);
  }
  (void)steps;
  if (fw) *fw = w;
  if (sw) *sw = s;
  return (bp.off + 255) & ~(size_t)255;
}

}  // namespace peg

using namespace peg;

extern "C" {

size_t pegncde_param_count(const PegDims* dims) {
  if (check_dims(dims) != PEG_OK) return 0;
  return (size_t)make_model(*dims).P;
}

int pegncde_param_offsets(const PegDims* dims, int64_t* offsets) {
  PEG_TRY(check_dims(dims));
  if (!offsets) return PEG_ERR_NULL_POINTER;
  Model m = make_model(*dims);
  for (int l = 0; l < m.L; ++l) {
    offsets[5 * l + 0] = m.layer[l].w_off;
    offsets[5 * l + 1] = m.layer[l].b_off;
    offsets[5 * l + 2] = m.layer[l].nw_off;
    offsets[5 * l + 3] = m.layer[l].nb_off;
    offsets[5 * l + 4] = m.layer[l].fus_off;
  }
  return PEG_OK;
}

int pegncde_shard_buffer_bytes(const PegDims* dims, int32_t world, size_t* out) {
  PEG_TRY(check_dims(dims));
  if (!out) return PEG_ERR_NULL_POINTER;
  if (world < 1 || world > PEG_MAX_WORLD || (dims->n % 128) != 0) return PEG_ERR_BAD_DIMS;
  const Model m = make_model(*dims);
  const size_t ldk = (size_t)world * dims->n;
  out[0] = 2 * (size_t)dims->B * m.dmax * ldk * 4;
  out[1] = 2 * (size_t)dims->B * (ldk / 128) * sizeof(int32_t);
  out[2] = 2 * (size_t)world * 2 * ((size_t)dims->B * 2 * m.dmax) * sizeof(float);
  out[3] = ((size_t)world + 1) * sizeof(uint32_t);
  return PEG_OK;
}

size_t pegncde_stage_store_bytes(const PegDims* dims, int32_t steps) {
  if (check_dims(dims) != PEG_OK || steps < 1) return 0;
  return (size_t)steps * 6 * store_stage_elems(*dims) * sizeof(float);
}

size_t pegncde_workspace_bytes(const PegDims* dims, int32_t which, int32_t steps) {
  if (check_dims(dims) != PEG_OK) return 0;
  if (which < PEG_WS_VF_FWD || which > PEG_WS_STEP) return 0;
  return plan(*dims, which, steps, nullptr, nullptr, nullptr);
}

static int pack_common(peg_stream_t stream, const PegDims* dims, const float* d, const float* c, const float* b,
                       const float* a, const float* planar, const float* snap, const float* ts, float* adj_coef,
                       float* adj_rowsum, float* adj_diag, float* adj_total, float* tch_coef, int piece0 = 0, int count = -1,
                       int ncols = -1, int diag_col0 = 0) {
  PEG_TRY(check_dims(dims));
  const bool rect = ncols >= 0;          // row-sharded controls: statistics are optional (the transposed shard needs none)
  if (!rect) ncols = dims->n;
  if (!rect && (!adj_rowsum || !adj_diag || !adj_total || !tch_coef)) return PEG_ERR_NULL_POINTER;
  if (rect && (ncols % 32) != 0) return PEG_ERR_BAD_DIMS;
  const int ncpad = peg_npad(ncols);
  cudaStream_t st = (cudaStream_t)stream;
  const int Tm1 = dims->T - 1;
  if (count < 0) count = Tm1;
  if (piece0 < 0 || count < 1 || piece0 + count > Tm1) return PEG_ERR_BAD_DIMS;
  const int nt = dims->ldn / 32;
  dim3 grid(nt, count, dims->B);   // one block per column of tiles (fixed-order column means of the time channel)
  const bool unit_time = planar || snap;   // no time channel in the source: d(time)/dt == 1
  grid.x = ncpad / 32;                    // one block per column of tiles
  k_pack_adj<<<grid, 256, 0, st>>>(d, c, b, a, planar, snap, ts, dims->n, dims->ldn, Tm1, piece0, count, adj_coef, adj_rowsum,
                                   adj_diag, adj_total, tch_coef, ncols, diag_col0, 4);
  PEG_LAUNCH_CHECK();
  if (adj_rowsum && adj_total) {   // row sums and totals of the tiled planes, reduced in a fixed order (deterministic)
    const float* tiled = planar ? planar : adj_coef;
    k_adj_rowsums<<<dim3(nt, count, dims->B), 256, 0, st>>>(tiled, dims->n, dims->ldn, Tm1, piece0, adj_rowsum, ncpad, 4);
    PEG_LAUNCH_CHECK();
    k_adj_totals<<<dim3(4 * count, dims->B), 256, 0, st>>>(adj_rowsum, dims->n, Tm1, piece0, adj_total);
    PEG_LAUNCH_CHECK();
  }
  if (unit_time && tch_coef) {
    const size_t slabs = (size_t)dims->B * Tm1;
    const size_t cnt = slabs * 3 * dims->n;
    k_fill_tch_unit<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(tch_coef, dims->n, slabs);
    PEG_LAUNCH_CHECK();
  }
  return PEG_OK;
}

int pegncde_pack_adj(peg_stream_t stream, const PegDims* dims, const float* d, const float* c, const float* b,
                     const float* a, float* adj_coef, float* adj_rowsum, float* adj_diag, float* adj_total,
                     float* tch_coef) {
  if (!d || !c || !b || !a || !adj_coef) return PEG_ERR_NULL_POINTER;
  return pack_common(stream, dims, d, c, b, a, nullptr, nullptr, nullptr, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef);
}

int pegncde_pack_adj_range(peg_stream_t stream, const PegDims* dims, int32_t piece_begin, int32_t piece_count, const float* d,
                           const float* c, const float* b, const float* a, float* adj_coef, float* adj_rowsum, float* adj_diag,
                           float* adj_total, float* tch_coef) {
  if (!d || !c || !b || !a || !adj_coef) return PEG_ERR_NULL_POINTER;
  return pack_common(stream, dims, d, c, b, a, nullptr, nullptr, nullptr, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef,
                     piece_begin, piece_count);
}

int pegncde_adj_stats(peg_stream_t stream, const PegDims* dims, const float* adj_coef, float* adj_rowsum,
                      float* adj_diag, float* adj_total, float* tch_coef) {
  if (!adj_coef) return PEG_ERR_NULL_POINTER;
  return pack_common(stream, dims, nullptr, nullptr, nullptr, nullptr, adj_coef, nullptr, nullptr, nullptr, adj_rowsum,
                     adj_diag, adj_total, tch_coef);
}

int pegncde_build_adj(peg_stream_t stream, const PegDims* dims, const float* ts, const float* snapshots, float* adj_coef,
                      float* adj_rowsum, float* adj_diag, float* adj_total, float* tch_coef) {
  if (!ts || !snapshots || !adj_coef) return PEG_ERR_NULL_POINTER;
  return pack_common(stream, dims, nullptr, nullptr, nullptr, nullptr, nullptr, snapshots, ts, adj_coef, adj_rowsum,
                     adj_diag, adj_total, tch_coef);
}

int pegncde_adj_colsums(peg_stream_t stream, const PegDims* dims, const float* adj_coef, float* adj_colsum) {
  PEG_TRY(check_dims(dims));
  if (!adj_coef || !adj_colsum) return PEG_ERR_NULL_POINTER;
  const int nt = dims->ldn / 32;
  k_adj_colsums<<<dim3(nt, dims->T - 1, dims->B), 256, 0, (cudaStream_t)stream>>>(adj_coef, dims->n, dims->ldn, dims->T - 1, adj_colsum, 4);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_adj_absmax(peg_stream_t stream, const PegDims* dims, int32_t piece_begin, int32_t piece_count, const float* adj_coef,
                       float* adj_absmax) {
  PEG_TRY(check_dims(dims));
  if (!adj_coef || !adj_absmax) return PEG_ERR_NULL_POINTER;
  const int Tm1 = dims->T - 1;
  if (piece_begin < 0 || piece_count < 1 || piece_begin + piece_count > Tm1) return PEG_ERR_BAD_DIMS;
  cudaStream_t st = (cudaStream_t)stream;
  PEG_CUDA(cudaMemset2DAsync(adj_absmax + (size_t)piece_begin * 4, (size_t)Tm1 * 4 * sizeof(float), 0, (size_t)piece_count * 4 * sizeof(float),
                             dims->B, st));
  const int nt = dims->ldn / 32, ntiles = nt * nt;
  k_adj_absmax<<<dim3(ntiles < 64 ? ntiles : 64, piece_count, dims->B), 256, 0, st>>>(adj_coef, dims->ldn, Tm1, piece_begin, adj_absmax, dims->ldn, 4);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_build_adj_rect(peg_stream_t stream, const PegDims* dims, int32_t n_cols, int32_t diag_col0, const float* ts,
                           const float* snapshots, float* adj_coef, float* adj_rowsum, float* adj_diag, float* adj_total, float* tch_coef,
                           float* adj_absmax) {
  if (!ts || !snapshots || !adj_coef) return PEG_ERR_NULL_POINTER;
  if (n_cols < 32) return PEG_ERR_BAD_DIMS;
  PEG_TRY(pack_common(stream, dims, nullptr, nullptr, nullptr, nullptr, nullptr, snapshots, ts, adj_coef, adj_rowsum, adj_diag, adj_total,
                      tch_coef, 0, -1, n_cols, diag_col0));
  if (adj_absmax) {
    cudaStream_t st = (cudaStream_t)stream;
    const int Tm1 = dims->T - 1, ncpad = peg_npad(n_cols);
    PEG_CUDA(cudaMemsetAsync(adj_absmax, 0, (size_t)dims->B * Tm1 * 4 * sizeof(float), st));
    const int ntiles = (dims->ldn / 32) * (ncpad / 32);
    k_adj_absmax<<<dim3(ntiles < 64 ? ntiles : 64, Tm1, dims->B), 256, 0, st>>>(adj_coef, dims->ldn, Tm1, 0, adj_absmax, ncpad, 4);
    PEG_LAUNCH_CHECK();
  }
  return PEG_OK;
}

// every piece of a static control's tables = piece 0: t [B][Tm1][per] <- t[b][0] for pieces 1 .. Tm1-1
__global__ void k_repeat_piece0(float* __restrict__ t, size_t per, int Tm1, int B) {
  const size_t total = (size_t)B * (Tm1 - 1) * per;
  for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t j = idx % per, r = idx / per, b = r / (Tm1 - 1), iv = 1 + r % (Tm1 - 1);
    t[(b * Tm1 + iv) * per + j] = t[b * Tm1 * per + j];
  }
}

int pegncde_build_adj_static(peg_stream_t stream, const PegDims* dims, const float* adjacency, float* adj_static, float* adj_rowsum,
                             float* adj_diag, float* adj_total, float* adj_colsum, float* adj_absmax, float* tch_coef) {
  PEG_TRY(check_dims(dims));
  if (!adjacency || !adj_static || !adj_rowsum || !adj_diag || !adj_total || !adj_colsum || !adj_absmax || !tch_coef)
    return PEG_ERR_NULL_POINTER;
  if (((uintptr_t)adj_static & 15) != 0) return PEG_ERR_ALIGNMENT;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = dims->B, n = dims->n, npad = dims->ldn, nt = npad / 32, Tm1 = dims->T - 1;
  const size_t vec = (size_t)B * Tm1 * 4 * n, sc = (size_t)B * Tm1 * 4;
  // slots b, c, d of every table stay zero (A' = 0); slot a of piece 0 is written by the dense kernels run with one plane, in their
  // summation order, then repeated for every piece
  PEG_CUDA(cudaMemsetAsync(adj_rowsum, 0, vec * sizeof(float), st));
  PEG_CUDA(cudaMemsetAsync(adj_diag, 0, vec * sizeof(float), st));
  PEG_CUDA(cudaMemsetAsync(adj_colsum, 0, vec * sizeof(float), st));
  PEG_CUDA(cudaMemsetAsync(adj_absmax, 0, sc * sizeof(float), st));
  k_pack_adj<<<dim3(nt, 1, B), 256, 0, st>>>(nullptr, nullptr, nullptr, nullptr, nullptr, adjacency, nullptr, n, npad, Tm1, 0, 1,
                                             adj_static, nullptr, adj_diag, nullptr, nullptr, n, 0, 1);
  PEG_LAUNCH_CHECK();
  k_adj_rowsums<<<dim3(nt, 1, B), 256, 0, st>>>(adj_static, n, npad, Tm1, 0, adj_rowsum, npad, 1);
  PEG_LAUNCH_CHECK();
  k_adj_totals<<<dim3(4, B), 256, 0, st>>>(adj_rowsum, n, Tm1, 0, adj_total);
  PEG_LAUNCH_CHECK();
  k_adj_colsums<<<dim3(nt, 1, B), 256, 0, st>>>(adj_static, n, npad, Tm1, adj_colsum, 1);
  PEG_LAUNCH_CHECK();
  k_adj_absmax<<<dim3(nt * nt < 64 ? nt * nt : 64, 1, B), 256, 0, st>>>(adj_static, npad, Tm1, 0, adj_absmax, npad, 1);
  PEG_LAUNCH_CHECK();
  if (Tm1 > 1) {
    float* per_n[3] = {adj_rowsum, adj_diag, adj_colsum};
    for (float* t : per_n) {
      k_repeat_piece0<<<(unsigned)std::min<size_t>(4096, ((size_t)B * (Tm1 - 1) * 4 * n + 255) / 256), 256, 0, st>>>(t, (size_t)4 * n, Tm1, B);
      PEG_LAUNCH_CHECK();
    }
    float* per_4[2] = {adj_total, adj_absmax};
    for (float* t : per_4) {
      k_repeat_piece0<<<(unsigned)std::min<size_t>(4096, ((size_t)B * (Tm1 - 1) * 4 + 255) / 256), 256, 0, st>>>(t, 4, Tm1, B);
      PEG_LAUNCH_CHECK();
    }
  }
  const size_t cnt = (size_t)B * Tm1 * 3 * n;
  k_fill_tch_unit<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(tch_coef, n, (size_t)B * Tm1);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

static int sparse_common(peg_stream_t stream, const PegDims* dims, const PegSparse* sp, const int32_t* perm_t, const float* ts,
                         const float* values, const float* d, const float* c, const float* b, const float* a, float* adj_rowsum,
                         float* adj_diag, float* adj_total, float* adj_colsum, float* tch_coef) {
  PEG_TRY(check_dims(dims));
  if (!sp || !perm_t || !adj_rowsum || !adj_diag || !adj_total || !adj_colsum || !tch_coef) return PEG_ERR_NULL_POINTER;
  PEG_TRY(check_sparse(sp));
  cudaStream_t st = (cudaStream_t)stream;
  const int Tm1 = dims->T - 1, n = dims->n;
  const dim3 grid((unsigned)((n + 7) / 8), Tm1, dims->B);
  k_sparse_build<<<grid, 256, 0, st>>>(*sp, perm_t, ts, values, d, c, b, a, n, Tm1, adj_rowsum, adj_diag);
  PEG_LAUNCH_CHECK();
  k_sparse_colsums<<<grid, 256, 0, st>>>(*sp, n, Tm1, adj_colsum);
  PEG_LAUNCH_CHECK();
  k_adj_totals<<<dim3(4 * Tm1, dims->B), 256, 0, st>>>(adj_rowsum, n, Tm1, 0, adj_total);
  PEG_LAUNCH_CHECK();
  const size_t slabs = (size_t)dims->B * Tm1;
  k_fill_tch_unit<<<(unsigned)((slabs * 3 * n + 255) / 256), 256, 0, st>>>(tch_coef, n, slabs);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_build_adj_sparse(peg_stream_t stream, const PegDims* dims, const PegSparse* sp, const int32_t* perm_t, const float* ts,
                             const float* values, float* adj_rowsum, float* adj_diag, float* adj_total, float* adj_colsum, float* tch_coef) {
  if (!ts || !values) return PEG_ERR_NULL_POINTER;
  return sparse_common(stream, dims, sp, perm_t, ts, values, nullptr, nullptr, nullptr, nullptr, adj_rowsum, adj_diag, adj_total,
                       adj_colsum, tch_coef);
}

int pegncde_pack_adj_sparse(peg_stream_t stream, const PegDims* dims, const PegSparse* sp, const int32_t* perm_t, const float* d,
                            const float* c, const float* b, const float* a, float* adj_rowsum, float* adj_diag, float* adj_total,
                            float* adj_colsum, float* tch_coef) {
  if (!d || !c || !b || !a) return PEG_ERR_NULL_POINTER;
  return sparse_common(stream, dims, sp, perm_t, nullptr, nullptr, d, c, b, a, adj_rowsum, adj_diag, adj_total, adj_colsum, tch_coef);
}

int pegncde_pack_x(peg_stream_t stream, const PegDims* dims, const float* d, const float* c, const float* b,
                   const float* a, float* x_coef) {
  PEG_TRY(check_dims(dims));
  if (dims->e <= 0) return PEG_ERR_BAD_DIMS;
  if (!d || !c || !b || !x_coef) return PEG_ERR_NULL_POINTER;
  (void)a;
  const size_t slabs = (size_t)dims->B * (dims->T - 1);
  const size_t cnt = slabs * dims->n * 2 * dims->e;
  k_pack_x<<<(unsigned)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, c, b, dims->n, 2 * dims->e, slabs,
                                                                            x_coef);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_vf_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                   const float* y, float* dy, void* workspace, size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  if (!y || !dy || !workspace) return PEG_ERR_NULL_POINTER;
  if (workspace_bytes < plan(*dims, PEG_WS_VF_FWD, 0, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  plan(*dims, PEG_WS_VF_FWD, 0, workspace, &c.w, nullptr);
  PEG_TRY(reset_tickets(c));
  PEG_TRY(feval_fwd(c, t, y, dy, nullptr));
  return shard_finish(c);
}

// g_adj (nullable): the cotangent of the sparse coefficients, [T-1, nnz_stride, 4], accumulated
static int set_adj_grad(Ctx& c, const PegControl* ctl, float* g_adj) {
  if (!g_adj) return PEG_OK;
  if (!ctl->sparse) return PEG_ERR_UNSUPPORTED;     // dense controls get no coefficient cotangent
  if (((uintptr_t)g_adj & 15) != 0) return PEG_ERR_ALIGNMENT;
  c.g_adj = g_adj;
  return PEG_OK;
}

// g_static (nullable): the cotangent of a static control's adjacency, [B, ldn, ldn] row-major, accumulated.  The small-graph cluster
// kernels compute no adjacency gradient: a call that asks for one runs the per-operator path, as with PEG_FLAG_NO_FUSED_SMALL.
static int set_adj_grad_static(Ctx& c, const PegControl* ctl, float* g_static) {
  if (!g_static) return PEG_OK;
  if (!ctl->adj_static) return PEG_ERR_UNSUPPORTED;
  if (((uintptr_t)g_static & 15) != 0) return PEG_ERR_ALIGNMENT;
  c.g_adj = g_static;
  c.small_C = 0;
  return PEG_OK;
}

static int vf_vjp(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t, const float* y,
                  const float* g_dy, float* g_y, float* g_params, float* g_xdot, float* g_adj, bool adj_static, void* workspace,
                  size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  PEG_TRY(adj_static ? set_adj_grad_static(c, ctl, g_adj) : set_adj_grad(c, ctl, g_adj));
  if (!y || !g_dy || !g_y || !g_params || !workspace) return PEG_ERR_NULL_POINTER;
  if (workspace_bytes < plan(*dims, PEG_WS_VF_VJP, 0, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  SolveWs s;
  plan(*dims, PEG_WS_VF_VJP, 0, workspace, &c.w, &s);
  PEG_TRY(reset_tickets(c));
  float* save[PEG_MAX_LAYERS];
  save[0] = const_cast<float*>(y);
  for (int l = 1; l < dims->L; ++l) save[l] = s.save[0][l];
  // forward over the first L-1 layers only: the VJP needs the layer inputs, not the evaluation's output
  PEG_TRY(feval_fwd(c, t, y, nullptr, save, dims->L - 1));
  PEG_TRY(feval_vjp(c, t, save, g_dy, g_y, g_params, g_xdot));
  return shard_finish(c);
}

int pegncde_vf_vjp(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                   const float* y, const float* g_dy, float* g_y, float* g_params, float* g_xdot, void* workspace,
                   size_t workspace_bytes) {
  return vf_vjp(stream, dims, ctl, params, t, y, g_dy, g_y, g_params, g_xdot, nullptr, false, workspace, workspace_bytes);
}

int pegncde_vf_vjp_adj(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                       const float* y, const float* g_dy, float* g_y, float* g_params, float* g_xdot, float* g_adj_coef,
                       void* workspace, size_t workspace_bytes) {
  return vf_vjp(stream, dims, ctl, params, t, y, g_dy, g_y, g_params, g_xdot, g_adj_coef, false, workspace, workspace_bytes);
}

int pegncde_vf_vjp_adj_static(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                              const float* y, const float* g_dy, float* g_y, float* g_params, float* g_xdot, float* g_adj_static,
                              void* workspace, size_t workspace_bytes) {
  return vf_vjp(stream, dims, ctl, params, t, y, g_dy, g_y, g_params, g_xdot, g_adj_static, true, workspace, workspace_bytes);
}

int pegncde_step_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, float t,
                     float dt, const float* y, float* k1, int32_t k1_valid, float* y1, float* y_err, float* k7,
                     float* k_stages, void* workspace, size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  if (!y || !k1 || !y1 || !k7 || !workspace) return PEG_ERR_NULL_POINTER;
  if (workspace_bytes < plan(*dims, PEG_WS_STEP, 0, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  SolveWs s;
  plan(*dims, PEG_WS_STEP, 0, workspace, &c.w, &s);
  PEG_TRY(reset_tickets(c));
  const Tsit5& tb = tsit5();
  const size_t st = (size_t)dims->B * dims->n * dims->h;
  float* k[7] = {k1, s.k[1], s.k[2], s.k[3], s.k[4], s.k[5], k7};
  if (k_stages)   // the caller keeps k2..k6 (dense output / SaveAt(ts=...))
    for (int i = 1; i < 6; ++i) k[i] = k_stages + (size_t)(i - 1) * st;
  if (!k1_valid) PEG_TRY(feval_fwd(c, t, y, k[0], nullptr));
  for (int i = 1; i < 7; ++i) {
    const float* xs[8];
    double cs[8];
    xs[0] = y; cs[0] = 1.0;
    for (int j = 0; j < i; ++j) { xs[j + 1] = k[j]; cs[j + 1] = (double)dt * tb.a[i][j]; }
    float* zin = (i == 6) ? y1 : s.Z0;
    PEG_TRY(combine(c, zin, i + 1, xs, cs));
    const float ti = (i == 6) ? (t + dt) : (t + (float)tb.c[i] * dt);
    PEG_TRY(feval_fwd(c, ti, zin, k[i], nullptr));
  }
  if (y_err) {
    const float* xs[8];
    double cs[8];
    for (int j = 0; j < 7; ++j) { xs[j] = k[j]; cs[j] = (double)dt * tb.berr[j]; }
    PEG_TRY(combine(c, y_err, 7, xs, cs));
  }
  return PEG_OK;
}

int pegncde_step_fwd_batched(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, const float* t_dev,
                             const float* dt_dev, const float* y, float* k1, int32_t k1_valid, float* y1, float* y_err, float* k7,
                             float* k_stages, void* workspace, size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  c.small_C = 0;    // per-trajectory stage times: the per-operator kernels
  if (!t_dev || !dt_dev || !y || !k1 || !y1 || !k7 || !workspace) return PEG_ERR_NULL_POINTER;
  if (c.sh) return PEG_ERR_UNSUPPORTED;
  if (workspace_bytes < plan(*dims, PEG_WS_STEP, 0, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  SolveWs s;
  plan(*dims, PEG_WS_STEP, 0, workspace, &c.w, &s);
  PEG_TRY(reset_tickets(c));
  const Tsit5& tb = tsit5();
  const size_t st = (size_t)dims->B * dims->n * dims->h;
  float* k[7] = {k1, s.k[1], s.k[2], s.k[3], s.k[4], s.k[5], k7};
  if (k_stages)
    for (int i = 1; i < 6; ++i) k[i] = k_stages + (size_t)(i - 1) * st;
  c.t_dev = t_dev; c.dt_dev = dt_dev;
  if (!k1_valid) { c.tcoef = 0.f; PEG_TRY(feval_fwd(c, 0.f, y, k[0], nullptr)); }
  for (int i = 1; i < 7; ++i) {
    const float* xs[8];
    double cs[8];
    xs[0] = y; cs[0] = 1.0;
    for (int j = 0; j < i; ++j) { xs[j + 1] = k[j]; cs[j + 1] = tb.a[i][j]; }     // times the graph's own dt (gscale)
    float* zin = (i == 6) ? y1 : s.Z0;
    PEG_TRY(combine(c, zin, i + 1, xs, cs, dt_dev));
    c.tcoef = (i == 6) ? 1.f : (float)tb.c[i];
    PEG_TRY(feval_fwd(c, 0.f, zin, k[i], nullptr));
  }
  if (y_err) {
    const float* xs[8];
    double cs[8];
    // y_err = dt sum_j berr_j k_j: entry 0 would stay unscaled, so lead with a zero-weight copy of y
    xs[0] = y; cs[0] = 0.0;
    CombArgs a;
    memset(&a, 0, sizeof(a));
    a.x[0] = y; a.c[0] = 0.f;
    for (int j = 0; j < 7; ++j) { a.x[j + 1] = k[j]; a.c[j + 1] = (float)tb.berr[j]; }
    a.cnt = 8; a.out = y_err; a.count4 = st / 4; a.gscale = dt_dev; a.per_graph4 = (size_t)dims->n * dims->h / 4;
    k_rk_combine<<<(unsigned)((a.count4 + 255) / 256), 256, 0, c.st>>>(a);
    PEG_LAUNCH_CHECK();
    (void)xs; (void)cs;
  }
  return PEG_OK;
}

int pegncde_adaptive_control(peg_stream_t stream, const PegDims* dims, PegAdaptState* state, float rtol, float atol, float t1, float safety,
                             float factormin, float factormax, int32_t error_order, const float* save_ts, int32_t n_save, int32_t cap,
                             float* y, const float* y1, const float* y_err, float* k1, const float* k7, const float* k_stages,
                             float* y_ckpt, float* ys_save, float* step_tab, int32_t* sample_step, float* sample_theta, float* t_dev,
                             float* dt_dev, float* sumsq_scratch) {
  PEG_TRY(check_dims(dims));
  if (!state || !y || !y1 || !y_err || !k1 || !k7 || !y_ckpt || !step_tab || !t_dev || !dt_dev || !sumsq_scratch) return PEG_ERR_NULL_POINTER;
  if (n_save > 0 && (!save_ts || !ys_save || !sample_step || !sample_theta || !k_stages)) return PEG_ERR_NULL_POINTER;
  if (cap < 1 || error_order < 1) return PEG_ERR_BAD_DIMS;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t per_graph = (size_t)dims->n * dims->h;
  k_scaled_sumsq<<<dims->B, 1024, 0, st>>>(y_err, nullptr, y, y1, rtol, atol, per_graph, sumsq_scratch);
  PEG_LAUNCH_CHECK();
  k_adapt_decide<<<(dims->B + 63) / 64, 64, 0, st>>>(reinterpret_cast<AdaptState*>(state), sumsq_scratch, dims->B, (float)per_graph, t1, safety, factormin,
                                                       factormax, 1.0f / (float)error_order, save_ts, n_save, cap, step_tab, sample_step, sample_theta,
                                                       dt_dev, t_dev);
  PEG_LAUNCH_CHECK();
  const size_t tot4 = (size_t)dims->B * per_graph / 4;
  k_adapt_apply<<<(unsigned)((tot4 + 255) / 256), 256, 0, st>>>(reinterpret_cast<const AdaptState*>(state), dims->B, per_graph / 4, cap,
                                                                reinterpret_cast<float4*>(y), reinterpret_cast<const float4*>(y1),
                                                                reinterpret_cast<float4*>(k1), reinterpret_cast<const float4*>(k7),
                                                                reinterpret_cast<const float4*>(k_stages), reinterpret_cast<float4*>(y_ckpt),
                                                                reinterpret_cast<float4*>(ys_save), sample_theta);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

// Tsit5 dense output (Tsitouras 2011, the interpolant behind diffrax's SaveAt(ts=...)):
//   y(t + theta dt) = y + dt sum_i b_i(theta) k_i,  b_1 = theta (r11 + theta (r12 + theta (r13 + theta r14))),
//   b_i = theta^2 (r_i2 + theta (r_i3 + theta r_i4)) for i >= 2;  b_i(1) = b_i, b_7(1) = 0.
void pegncde_tsit5_dense_weights(float theta, float* w /* [7] */) {
  static const double r[7][4] = {
      {1.0, -2.763706197274826, 2.9132554618219126, -1.0530884977290216},
      {0.0, 0.13169999999999998, -0.2234, 0.1017},
      {0.0, 3.9302962368947516, -5.941033872131505, 2.490627285651253},
      {0.0, -12.411077166933676, 30.33818863028232, -16.548102889244902},
      {0.0, 37.50931341651104, -88.1789048947664, 47.37952196281928},
      {0.0, -27.896526289197286, 65.09189467479366, -34.87065786149661},
      {0.0, 1.5, -4.0, 2.5}};
  const double th = (double)theta;
  for (int i = 0; i < 7; ++i) w[i] = (float)(th * (r[i][0] + th * (r[i][1] + th * (r[i][2] + th * r[i][3]))));
}

int pegncde_tsit5_dense(peg_stream_t stream, const PegDims* dims, float dt, float theta, const float* y, const float* k1,
                        const float* k_stages, const float* k7, float* out) {
  PEG_TRY(check_dims(dims));
  if (!y || !k1 || !k_stages || !k7 || !out) return PEG_ERR_NULL_POINTER;
  float w[7];
  pegncde_tsit5_dense_weights(theta, w);
  const size_t st = (size_t)dims->B * dims->n * dims->h;
  CombArgs a;
  memset(&a, 0, sizeof(a));
  a.x[0] = y; a.c[0] = 1.f;
  a.x[1] = k1; a.c[1] = dt * w[0];
  for (int i = 1; i < 6; ++i) { a.x[i + 1] = k_stages + (size_t)(i - 1) * st; a.c[i + 1] = dt * w[i]; }
  a.x[7] = k7; a.c[7] = dt * w[6];
  a.cnt = 8;
  a.out = out;
  a.count4 = st / 4;
  k_rk_combine<<<(unsigned)((a.count4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_scaled_sumsq(peg_stream_t stream, const PegDims* dims, const float* x, const float* x2, const float* s0,
                         const float* s1, float rtol, float atol, float* out) {
  PEG_TRY(check_dims(dims));
  if (!x || !s0 || !out) return PEG_ERR_NULL_POINTER;
  const size_t per_graph = (size_t)dims->n * dims->h;
  k_scaled_sumsq<<<dims->B, 1024, 0, (cudaStream_t)stream>>>(x, x2, s0, s1, rtol, atol, per_graph, out);
  PEG_LAUNCH_CHECK();
  return PEG_OK;
}

int pegncde_solve_fwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                      const float* step_ts, int32_t steps, const float* y0, float* yT, float* y_ckpt,
                      float* stage_store, void* workspace, size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  if (!step_ts || !y0 || !y_ckpt || !workspace) return PEG_ERR_NULL_POINTER;
  if (steps < 1) return PEG_ERR_BAD_DIMS;
  if (workspace_bytes < plan(*dims, PEG_WS_SOLVE_FWD, steps, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  SolveWs s;
  plan(*dims, PEG_WS_SOLVE_FWD, steps, workspace, &c.w, &s);
  PEG_TRY(reset_tickets(c));
  const Tsit5& tb = tsit5();
  const size_t st = (size_t)dims->B * dims->n * dims->h;
  PEG_CUDA(cudaMemcpyAsync(y_ckpt, y0, st * sizeof(float), cudaMemcpyDeviceToDevice, c.st));
  float* k[7];
  for (int i = 0; i < 7; ++i) k[i] = s.k[i];
  // the layout of stage_store: store_slots
  StoreSlots slots;
  auto fwd_stage = [&](float ti, const float* zin, float* dy, int step, int stage) -> int {
    if (!stage_store) return feval_fwd(c, ti, zin, dy, nullptr);
    slots = store_slots(*dims, stage_store, step, stage);
    slots.z[0] = nullptr;   // the stage input itself
    return feval_fwd(c, ti, zin, dy, slots.z, -1, slots.m, slots.cm);
  };
  for (int sidx = 0; sidx < steps; ++sidx) {
    const float t = step_ts[sidx];
    const float dt = step_ts[sidx + 1] - step_ts[sidx];
    const float* y = y_ckpt + (size_t)sidx * st;
    float* ynext = y_ckpt + (size_t)(sidx + 1) * st;
    if (sidx == 0) PEG_TRY(fwd_stage(t, y, k[0], 0, 0));
    for (int i = 1; i < 7; ++i) {
      const float* xs[8];
      double cs[8];
      xs[0] = y; cs[0] = 1.0;
      for (int j = 0; j < i; ++j) { xs[j + 1] = k[j]; cs[j + 1] = (double)dt * tb.a[i][j]; }
      float* zin = (i == 6) ? ynext : (stage_store ? store_slots(*dims, stage_store, sidx, i).z[0] : s.Z0);
      PEG_TRY(combine(c, zin, i + 1, xs, cs));
      if (i == 6 && sidx == steps - 1) break;  // the 7th stage only feeds FSAL: unused after the last step
      const float ti = (i == 6) ? step_ts[sidx + 1] : (t + (float)tb.c[i] * dt);
      // the 7th stage IS stage 0 of the next step (FSAL): its layer data are stored there
      PEG_TRY(i == 6 ? fwd_stage(ti, zin, k[i], sidx + 1, 0) : fwd_stage(ti, zin, k[i], sidx, i));
    }
    float* tmp = k[0]; k[0] = k[6]; k[6] = tmp;  // FSAL
  }
  if (yT) PEG_CUDA(cudaMemcpyAsync(yT, y_ckpt + (size_t)steps * st, st * sizeof(float), cudaMemcpyDeviceToDevice, c.st));
  return shard_finish(c);
}

static int solve_bwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params, const float* step_ts,
                     int32_t steps, const float* y_ckpt, const float* stage_store, const float* g_yT, const float* g_ckpt,
                     const float* g_stage, float* g_y0, float* g_params, float* g_xcoef, float* g_adj, bool adj_static,
                     void* workspace, size_t workspace_bytes) {
  Ctx c;
  PEG_TRY(make_ctx(c, stream, dims, ctl, params));
  // a forward on the small-graph kernels keeps no M_l in the stage store: an adjoint moved off them must recompute M_l
  const bool store_has_m = c.small_C == 0;
  PEG_TRY(adj_static ? set_adj_grad_static(c, ctl, g_adj) : set_adj_grad(c, ctl, g_adj));
  if (!step_ts || !y_ckpt || (!g_yT && !g_ckpt) || !g_y0 || !g_params || !workspace) return PEG_ERR_NULL_POINTER;
  if (steps < 1) return PEG_ERR_BAD_DIMS;
  if (g_xcoef && dims->e == 0) return PEG_ERR_BAD_DIMS;
  if (workspace_bytes < plan(*dims, PEG_WS_SOLVE_BWD, steps, nullptr, nullptr, nullptr)) return PEG_ERR_WORKSPACE;
  SolveWs s;
  plan(*dims, PEG_WS_SOLVE_BWD, steps, workspace, &c.w, &s);
  PEG_TRY(reset_tickets(c));
  const Tsit5& tb = tsit5();
  const size_t st = (size_t)dims->B * dims->n * dims->h;
  const int L = dims->L;
  // one evaluation's VJP; with g_xcoef also the cotangent of the node-signal coefficients of the stage's cubic piece
  auto stage_vjp = [&](float t, float* const* save, const float* kbar, float* ybar, float* const* mkept = nullptr,
                       float* const* ckept = nullptr) -> int {
    PEG_TRY(feval_vjp(c, t, save, kbar, ybar, g_params, g_xcoef ? c.w.gxd : nullptr, mkept, ckept));
    if (g_xcoef) {
      const size_t cnt = (size_t)dims->B * dims->n * 2 * dims->e;
      k_xcoef_accum<<<(unsigned)((cnt + 255) / 256), 256, 0, c.st>>>(c.w.gxd, c.w.sc, dims->n, 2 * dims->e, dims->T - 1, dims->B, g_xcoef);
      PEG_LAUNCH_CHECK();
    }
    return PEG_OK;
  };
  // running cotangent of y_{s+1}
  {
    const float* xs[2] = {g_yT, g_ckpt ? g_ckpt + (size_t)steps * st : nullptr};
    double cs[2] = {g_yT ? 1.0 : 0.0, g_ckpt ? 1.0 : 0.0};
    PEG_TRY(combine(c, s.gcur, 2, xs, cs));
  }
  auto stage_cot = [&](int step, int stage) { return g_stage + ((size_t)step * 7 + stage) * st; };
  if (g_stage) {
    // dense output of the last step uses k7 = f(t_S, y_S), which belongs to no later step: its VJP feeds ybar_S directly
    const float* yS = y_ckpt + (size_t)steps * st;
    float* save[PEG_MAX_LAYERS];
    save[0] = const_cast<float*>(yS);
    for (int l = 1; l < L; ++l) save[l] = s.save[0][l];
    PEG_TRY(feval_fwd(c, step_ts[steps], yS, nullptr, save, L - 1));
    PEG_TRY(stage_vjp(step_ts[steps], save, stage_cot(steps - 1, 6), s.Ybar[0]));
    const float* xs[2] = {s.gcur, s.Ybar[0]};
    double cs[2] = {1.0, 1.0};
    PEG_TRY(combine(c, s.gnext, 2, xs, cs));
    float* tmp = s.gcur; s.gcur = s.gnext; s.gnext = tmp;
  }
  for (int sidx = steps - 1; sidx >= 0; --sidx) {
    const float t = step_ts[sidx];
    const float dt = step_ts[sidx + 1] - step_ts[sidx];
    const float* y = y_ckpt + (size_t)sidx * st;
    float tis[6];
    for (int i = 0; i < 6; ++i) tis[i] = (i == 0) ? t : (t + (float)tb.c[i] * dt);
    // ---- recompute the six stages of this step, keeping every layer input (skipped when solve_fwd stored them) ----
    for (int i = 0; i < 6 && !stage_store; ++i) {
      float* zin;
      if (i == 0) {
        zin = const_cast<float*>(y);
      } else {
        const float* xs[8];
        double cs[8];
        xs[0] = y; cs[0] = 1.0;
        for (int j = 0; j < i; ++j) { xs[j + 1] = s.k[j]; cs[j + 1] = (double)dt * tb.a[i][j]; }
        zin = s.save[i][0];
        PEG_TRY(combine(c, zin, i + 1, xs, cs));
      }
      float* save[PEG_MAX_LAYERS];
      save[0] = zin;
      for (int l = 1; l < L; ++l) save[l] = s.save[i][l];
      PEG_TRY(feval_fwd(c, tis[i], zin, s.k[i], save));
    }
    // ---- reverse sweep over the stages: kbar_i = dt (b_i g + sum_{j>i} a_ji Ybar_j) ; Ybar_i = J_i^T kbar_i ----
    for (int i = 5; i >= 0; --i) {
      const float* xs[8];
      double cs[8];
      int cnt = 0;
      xs[cnt] = s.gcur; cs[cnt] = (double)dt * tb.b[i]; ++cnt;
      for (int j = i + 1; j < 6; ++j) { xs[cnt] = s.Ybar[j]; cs[cnt] = (double)dt * tb.a[j][i]; ++cnt; }
      if (g_stage) {   // direct cotangents of the stage slopes (dense output); k7 of the previous step IS this step's k1
        xs[cnt] = stage_cot(sidx, i); cs[cnt] = 1.0; ++cnt;
        if (i == 0 && sidx > 0) { xs[cnt] = stage_cot(sidx - 1, 6); cs[cnt] = 1.0; ++cnt; }
      }
      PEG_TRY(combine(c, s.kbar, cnt, xs, cs));
      if (stage_store) {
        StoreSlots kept = store_slots(*dims, const_cast<float*>(stage_store), sidx, i);
        if (i == 0) kept.z[0] = const_cast<float*>(y);
        PEG_TRY(stage_vjp(tis[i], kept.z, s.kbar, s.Ybar[i], store_has_m ? kept.m : nullptr, store_has_m ? kept.cm : nullptr));
      } else {
        float* save[PEG_MAX_LAYERS];
        save[0] = (i == 0) ? const_cast<float*>(y) : s.save[i][0];
        for (int l = 1; l < L; ++l) save[l] = s.save[i][l];
        PEG_TRY(stage_vjp(tis[i], save, s.kbar, s.Ybar[i]));
      }
    }
    // ---- ybar_s = g + sum_i Ybar_i (+ injected cotangent at this boundary) ----
    {
      const float* xs[8];
      double cs[8];
      int cnt = 0;
      xs[cnt] = s.gcur; cs[cnt] = 1.0; ++cnt;
      for (int i = 0; i < 6; ++i) { xs[cnt] = s.Ybar[i]; cs[cnt] = 1.0; ++cnt; }
      if (g_ckpt) { xs[cnt] = g_ckpt + (size_t)sidx * st; cs[cnt] = 1.0; ++cnt; }
      float* out = (sidx == 0) ? g_y0 : s.gnext;
      PEG_TRY(combine(c, out, cnt, xs, cs));
      float* tmp = s.gcur; s.gcur = s.gnext; s.gnext = tmp;
    }
  }
  return shard_finish(c);
}

int pegncde_solve_bwd(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                      const float* step_ts, int32_t steps, const float* y_ckpt, const float* stage_store,
                      const float* g_yT, const float* g_ckpt, const float* g_stage, float* g_y0, float* g_params,
                      float* g_xcoef, void* workspace, size_t workspace_bytes) {
  return solve_bwd(stream, dims, ctl, params, step_ts, steps, y_ckpt, stage_store, g_yT, g_ckpt, g_stage, g_y0, g_params, g_xcoef,
                   nullptr, false, workspace, workspace_bytes);
}

int pegncde_solve_bwd_adj(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                          const float* step_ts, int32_t steps, const float* y_ckpt, const float* stage_store,
                          const float* g_yT, const float* g_ckpt, const float* g_stage, float* g_y0, float* g_params,
                          float* g_xcoef, float* g_adj_coef, void* workspace, size_t workspace_bytes) {
  return solve_bwd(stream, dims, ctl, params, step_ts, steps, y_ckpt, stage_store, g_yT, g_ckpt, g_stage, g_y0, g_params, g_xcoef,
                   g_adj_coef, false, workspace, workspace_bytes);
}

int pegncde_solve_bwd_adj_static(peg_stream_t stream, const PegDims* dims, const PegControl* ctl, const float* params,
                                 const float* step_ts, int32_t steps, const float* y_ckpt, const float* stage_store,
                                 const float* g_yT, const float* g_ckpt, const float* g_stage, float* g_y0, float* g_params,
                                 float* g_xcoef, float* g_adj_static, void* workspace, size_t workspace_bytes) {
  return solve_bwd(stream, dims, ctl, params, step_ts, steps, y_ckpt, stage_store, g_yT, g_ckpt, g_stage, g_y0, g_params, g_xcoef,
                   g_adj_static, true, workspace, workspace_bytes);
}

const char* pegncde_strerror(int code) {
  switch (code) {
    case PEG_OK: return "ok";
    case PEG_ERR_BAD_DIMS: return "dimension out of the supported range";
    case PEG_ERR_NULL_POINTER: return "required pointer is NULL";
    case PEG_ERR_WORKSPACE: return "workspace too small (see pegncde_workspace_bytes)";
    case PEG_ERR_CUDA: return "CUDA runtime call or kernel launch failed (see pegncde_last_cuda_error)";
    case PEG_ERR_UNSUPPORTED: return "request not implemented by this build";
    case PEG_ERR_ALIGNMENT: return "pointer or pitch breaks the 16-byte alignment contract";
    default: return "unknown pegncde error code";
  }
}

int pegncde_profile_enable(int32_t stride) {
  Prof& p = peg::g_prof;
  for (int d = 0; d < 2; ++d) {
    for (cudaEvent_t e : p.ev[d]) cudaEventDestroy(e);
    p.ev[d].clear();
    p.seen[d] = 0;
  }
  p.stride = stride > 0 ? stride : 0;
  return PEG_OK;
}

int pegncde_profile_read(int32_t direction, uint64_t* launches, uint64_t* timed, double* ms_total,
                         double* bytes_per_launch, double* flops_per_launch) {
  if (direction < 0 || direction > 1) return PEG_ERR_BAD_DIMS;
  Prof& p = peg::g_prof;
  double ms = 0.0;
  uint64_t cnt = 0;
  std::vector<cudaEvent_t>& ev = p.ev[direction];
  for (size_t i = 0; i + 1 < ev.size(); i += 2) {
    if (cudaEventSynchronize(ev[i + 1]) != cudaSuccess) { peg::g_last_cuda = (int)cudaGetLastError(); return PEG_ERR_CUDA; }
    float t = 0.f;
    if (cudaEventElapsedTime(&t, ev[i], ev[i + 1]) != cudaSuccess) { peg::g_last_cuda = (int)cudaGetLastError(); return PEG_ERR_CUDA; }
    ms += t;
    ++cnt;
  }
  if (launches) *launches = p.seen[direction];
  if (timed) *timed = cnt;
  if (ms_total) *ms_total = ms;
  if (bytes_per_launch) *bytes_per_launch = p.bytes[direction];
  if (flops_per_launch) *flops_per_launch = p.flops[direction];
  return PEG_OK;
}

int pegncde_last_cuda_error(void) { return peg::g_last_cuda; }
const char* pegncde_version(void) { return "pegncde-b200 0.1 (sm_100a)"; }
uint64_t pegncde_launch_count(void) { return peg::g_launches.load(); }

}  // extern "C"
