// tcgen05 / TMEM / TMA implementation of the matrix-free equivariant contraction (sm_100a).
//
//   OUT[I] = sum_kc X[I, kc] V[kc]  +  sum_kc Y[kc, I]^T V[kc]      (+ O(n d) epilogue corrections)
//
// X and Y are linear combinations of the four cubic-coefficient planes (the control-path
// interpolation is fused: A_s, A'_s are never written to memory).  Per CTA: one 128-row output
// block x ND columns, accumulators in TMEM.  Work items come in pairs that share one K chunk kc:
// a "direct" item (rows of block I, 32 columns kc) and a "transposed" item (32 rows kc, columns of
// block I) -- both multiply V[kc], so ONE B-operand tile serves the pair.  The chunk order is the
// round-robin schedule J(S) = (S - I) mod nb over the 128-column blocks: CTA I works on blocks
// (I,J) and (J,I) exactly when CTA J does, so HBM sees every plane byte once per pass and L2
// serves the second reader.
//
// Warp roles (576 threads): warps 0-15 converters (LDG.128 planes -> FFMA combine -> 3xTF32 split
// -> swizzled STS of the K-major A operand tiles) in two groups of 8 that work on alternate items (group 0 the
// direct items, group 1 the transposed ones), so one group's conversion overlaps the other group's loads;
// warps 0-7 also run the epilogue (tcgen05.ld); warp 16 = TMA producer of the B operand (V^T hi/lo,
// SWIZZLE_128B); warp 17 = TMEM allocator + the single thread that issues tcgen05.mma.
//
// fp32 parity: 3xTF32 (hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM); PEG_FLAG_TF32_FAST drops
// the two correction products.
#include <cuda.h>
#include <atomic>
#include <cstdio>
#include <cstring>

#include "peg_tc.cuh"
#include "peg_tc_ptx.cuh"

namespace peg {

// ------------------------------------------------------------------------------------------
// V [B,n,d] -> V^T split into tf32 hi / lo, [B][d][npad] (zero padded): the K-major B operand
// grid (npad/32, ceil(d/32), B), block (32, 8)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_split_transpose(const float* __restrict__ V, int n, int d, int npad, const ProducerOut po) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, i0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* Vb = V + (size_t)b * n * d;
  // fp16x2: the block exponent of this tile's 128-node block (written by k_block_exponent just before)
  const float vscale = po.t16 == PEG_FMT_FP16X2 ? exp2_int(po.vexp[(size_t)b * po.vexp_stride + po.blk0 + (i0 >> 7)]) : 1.f;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = i0 + r, c = c0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < n && c < d) ? Vb[(size_t)i * d + c] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int c = c0 + r, i = i0 + threadIdx.x;
    if (c < d) {
      const size_t o = ((size_t)b * d + c) * po.npad + po.col0 + i;     // npad = this rank's padded rows, po.npad = the row pitch of V^T
      if (po.t16 == PEG_FMT_FP16X2) store_vt_f16(po, o, tile[threadIdx.x][r] * vscale);
      else store_vt(po, o, tile[threadIdx.x][r]);
    }
  }
}

// fp16x2 operand format: block exponent e of every 128-node block of V [B,n,d] (vexp[b][block]); k_split_transpose then writes
// V^T * 2^e.  grid (ceil(npad/128), column slices, B), block 256: the CTAs of a block combine their maxima with an atomicMax on the
// bit pattern (non-negative floats order like unsigned integers: order independent) and the last one to arrive turns it into the
// exponent -- a wide layer (d = 2 h e >= 1024 of the control models) no longer hangs on one CTA reading 128 x d values.
// vmax / vtick: [B][vexp_stride] scratch, zero on entry, left zero on exit.
__global__ void __launch_bounds__(256) k_block_exponent(const float* __restrict__ V, int n, int d, int* __restrict__ vexp, int vexp_stride, int blk0,
                                                        unsigned int* __restrict__ vmax, unsigned int* __restrict__ vtick) {
  // vmax / vtick are indexed with the LOCAL block count (gridDim.x blocks per graph); vexp with its own stride and block offset
  __shared__ float bmax_s[8];
  const int b = blockIdx.z, blk = blockIdx.x, i0 = blk * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rows = min(128, n - i0);
  const int c4 = d / 4, per = (c4 + gridDim.y - 1) / gridDim.y;       // float4 columns of this slice
  const int cb = blockIdx.y * per, ce = min(c4, cb + per);
  float mx = 0.f;
  if (rows > 0 && ce > cb) {
    const float4* src = reinterpret_cast<const float4*>(V + ((size_t)b * n + i0) * d);
    const int w = ce - cb;
    for (int i = tid; i < rows * w; i += 256) {
      const int r = i / w, c = cb + (i - r * w);
      const float4 v = __ldg(src + (size_t)r * c4 + c);
      mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
  }
  mx = warp_max(mx);
  if (lane == 0) bmax_s[warp] = mx;
  __syncthreads();
  if (tid == 0) {
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) mx = fmaxf(mx, bmax_s[w8]);
    const size_t slot = (size_t)b * gridDim.x + blk;
    atomicMax(vmax + slot, __float_as_uint(mx));
    __threadfence();
    if (atomicAdd(vtick + slot, 1u) == gridDim.y - 1) {     // last slice of this block: publish the exponent, reset the scratch
      __threadfence();
      const unsigned int bits = atomicExch(vmax + slot, 0u);
      vexp[(size_t)b * vexp_stride + blk0 + blk] = block_exponent(__uint_as_float(bits));
      vtick[slot] = 0u;
    }
  }
}

// ------------------------------------------------------------------------------------------
// the contraction kernel
// ------------------------------------------------------------------------------------------
constexpr int TC_THREADS = 576;   // 2 converter groups x 8 warps + TMA warp + MMA warp
constexpr int TC_CONV_THREADS = 256;
constexpr int TC_BM = 128;   // output rows per CTA (UMMA M)
constexpr int TC_BK = 32;    // K chunk (32 fp32 = 128 B = one swizzle row)
constexpr int TC_ATILE = TC_BM * TC_BK * 4;  // 16 KB

struct TcParams {
  ContractArgs a;
  int nd;        // columns per CTA (UMMA N)
  int nsplit;    // 3 = 3xTF32, 1 = single pass
  int stages_a;  // ring depth of the A-operand tiles (one slot per item; even: the two converter groups alternate)
  int stages_b;  // ring depth of the B-operand tiles (one slot per PAIR of items)
  int nkc;       // number of 32-wide K chunks = npad / 32
  int tmem_cols; // power of two >= 32
  int mode;      // 0 = whole K range + epilogue; 1 = one K slice of `ksplit`, accumulators added into `partial` (no epilogue);
                 // 2 = epilogue only, accumulators read from `partial`  (split-K for grids far smaller than the GPU)
  int ksplit;    // K slices per row block in mode 1 (blockIdx.x = row block * ksplit + slice)
  int pairs_per_slice;
  const int* vexp; // fp16x2 format: [B][vexp_stride] block exponents of V^T (one per 128 nodes)
  int vexp_stride;
  float* partial; // [B][accumulators][n][d] fp32, zeroed by the host before mode 1
};

// Per item type of the LIGHT adjoint: the operand pair is (combined = cA A_s + cD A'_s, 3xTF32: it carries the state cotangent)
// and (sep = A'_s or A_s, ONE tf32 pass: it only feeds two scalar Frobenius gradients).  <sep V, M> and <combined V, M> give
// both <A V, M> and <A' V, M>; sep is the plane with the smaller weight, so the 1-pass error is never amplified.
struct LightCoef { float cA, cD, oc; int sepA; };
__device__ __forceinline__ LightCoef light_coef(float wa, float wd) {
  LightCoef c;
  if (fmaxf(fabsf(wa), fabsf(wd)) < 1e-18f) { c.cA = 1.f; c.cD = 0.f; c.oc = 0.f; c.sepA = 0; }   // no contribution to the output: gradients only
  else { c.cA = wa; c.cD = wd; c.oc = 1.f; c.sepA = fabsf(wa) < fabsf(wd) ? 1 : 0; }
  return c;
}

// fp16x2 (block floating point): V^T holds V * 2^(e_J) per 128-node block J.  The blocks are aligned to the smallest exponent E
// inside the A operand (its entries are multiplied by 2^(E - e_J) <= 1, exact), so every accumulator ends up scaled by 2^E times the
// A scale.  E is cheap enough (one exponent per 128 nodes) for every thread that needs it to recompute it from global memory.
__device__ __forceinline__ int bfp_min_exponent(const int* __restrict__ ve, int nblk) {
  int e = PEG_VEXP_MAX;
  for (int J = 0; J < nblk; ++J) e = min(e, __ldcg(ve + J));     // L2: in row-sharded mode peers write these entries over NVLink
  return e;
}

// KIND 0 = forward, 1 = adjoint with four 3xTF32 products (default), 2 = LIGHT adjoint (two 3xTF32 products + two single-pass
// ones; PEG_FLAG_ADJ_LIGHT, looser tolerance on the param1 / param2 gradients: 2.5e-3 instead of 1e-3)
// FMT 0 = 3xTF32 operands (fp32 words, SWIZZLE_128B tiles, kind::tf32: error ~2^-22 per product);
// FMT 1 = bf16x2 operands (x = hi + lo, both bf16; hi*hi + lo*hi + hi*lo on kind::f16 at twice the tf32 rate and half the
//         shared-memory traffic; SWIZZLE_64B tiles of 8 KB; error ~2^-17 per product, fp32 accumulate in TMEM)
template <int KIND, int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1)
k_tc_contract(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, const TcParams p) {
  constexpr bool BWD = KIND != 0, LIGHT = KIND == 2;
  constexpr bool F16 = FMT != PEG_FMT_TF32X3;       // 16-bit parts: bf16x2 or fp16x2
  constexpr bool BFP = FMT == PEG_FMT_FP16X2;       // block floating point (see PEG_FMT_FP16X2)
  static_assert(!(F16 && LIGHT), "the LIGHT adjoint exists for the tf32 operand format only");

  constexpr int ATILE = F16 ? TC_BM * TC_BK * 2 : TC_ATILE;   // one A-operand tile (hi or lo part)
  constexpr int ESZ = F16 ? 2 : 4;                            // operand element size
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ float fsum[8][16];    // adjoint epilogue: per-warp partials of the fusion-scalar gradients
  constexpr int NA = BWD ? 2 : 1;  // A-operand variants per item: fwd = combined X or Y; bwd = (A_s, A'_s)
  const ContractArgs& a = p.a;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z, I = p.mode == 1 ? (int)blockIdx.x / p.ksplit : (int)blockIdx.x, ntile = blockIdx.y;
  const int kslice = p.mode == 1 ? (int)blockIdx.x - I * p.ksplit : 0;
  const int n = a.n, d = a.d, nd = p.nd;
  const bool split = F16 || p.nsplit == 3;

  // ---- shared memory carve-up (1024-B aligned operand tiles) ----
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int a_bytes = NA * (split ? 2 : 1) * ATILE;             // [variant][hi,lo]
  const int b_tile = nd * TC_BK * ESZ;
  const int b_bytes = (split ? 2 : 1) * b_tile;                 // [hi,lo]
  const int SA = p.stages_a, SB = p.stages_b;
  const uint32_t b_ring = smem_base + SA * a_bytes;
  const uint32_t bar_base = b_ring + SB * b_bytes;  // full_a[SA], empty_a[SA], full_b[SB], empty_b[SB], accum_full, tmem slot
  auto full_a = [&](int s) { return bar_base + 8u * s; };
  auto empty_a = [&](int s) { return bar_base + 8u * (SA + s); };
  auto full_b = [&](int s) { return bar_base + 8u * (2 * SA + s); };
  auto empty_b = [&](int s) { return bar_base + 8u * (2 * SA + SB + s); };
  const uint32_t accum_bar = bar_base + 8u * (2 * SA + 2 * SB);
  const uint32_t tmem_slot = accum_bar + 8u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));  // generic pointer to the aligned base
  // 16-bit formats: the chunk schedule of this CTA as a table (pair -> K chunk; BFP: + per A-operand variant the factor
  // (A scale) * 2^(E - e_J) as float bits), so the conversion loop spends one LDS.128 per item instead of re-deriving the schedule
  // and the plane weights stay warp-uniform (uniform registers): fewer instructions, a dozen fewer live vector registers
  int* sched_kc_s = reinterpret_cast<int*>(smem_gen + (tmem_slot + 8u - smem_base));     // [nkc] K chunk of every pair
  float2* sched_f_s = reinterpret_cast<float2*>(sched_kc_s + ((p.nkc + 1) & ~1));           // [nkc] BFP item factors (variant 0, 1)
  int* emin_s = reinterpret_cast<int*>(sched_f_s + p.nkc);                                   // smallest block exponent of this graph's V^T

  if (tid == 0) {
    for (int s = 0; s < SA; ++s) {
      mbar_init(full_a(s), TC_CONV_THREADS);
      mbar_init(empty_a(s), 1);
    }
    for (int s = 0; s < SB; ++s) {
      mbar_init(full_b(s), 1);
      mbar_init(empty_b(s), 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 17) {  // TMEM allocation (whole warp), address lands in smem
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const StageScalars* scp = a.sc + b;
  struct { float wA[4], wD[4]; int interval; } sc;
#pragma unroll
  for (int q = 0; q < 4; ++q) { sc.wA[q] = scp->wA[q]; sc.wD[q] = scp->wD[q]; }
  sc.interval = scp->interval;
  const int nkc = p.nkc;
  // this CTA's pairs: all of them, or one contiguous slice of the schedule (mode 1); none in mode 2
  const int pr0 = p.mode == 1 ? kslice * p.pairs_per_slice : 0;
  const int npairs = p.mode == 2 ? 0 : (p.mode == 1 ? max(0, min(nkc, pr0 + p.pairs_per_slice) - pr0) : nkc);
  const int items = 2 * npairs;   // local item j = 2 * local pair + type (0 direct, 1 transposed); pair works on chunk kc_of(pr0 + pair)
  // chunk order: 128-column blocks J(S) = (S - I) mod nb, four 32-chunks each (the last block may hold fewer)
  const int nb = (nkc + 3) >> 2, r_last = nkc - 4 * (nb - 1);
  const int Imod = (I + a.row_block0) % nb, Sstar = (nb - 1 + Imod) % nb;   // keyed on the GLOBAL row block (row-sharded mode)
  auto kc_of = [&](int pr) -> int {
    int S, u;
    if (pr < 4 * Sstar) { S = pr >> 2; u = pr & 3; }
    else if (pr < 4 * Sstar + r_last) { S = Sstar; u = pr - 4 * Sstar; }
    else { const int q = pr - 4 * Sstar - r_last; S = Sstar + 1 + (q >> 2); u = q & 3; }
    int J = S - Imod;
    if (J < 0) J += nb;
    return 4 * J + u;
  };
  const float alpha = 1.f + a.fus[0], beta = 1.f + a.fus[1], gamma = a.fus[2], delta = a.fus[3];
  // adjoint: direct items (A V, A' V) enter the output with (gamma, delta), transposed items (A^T V, A'^T V) with (alpha, beta)
  const LightCoef lc_d = light_coef(gamma, delta), lc_t = light_coef(alpha, beta);
  // BFP: power-of-two scale of every A-operand variant from the bound sum_q |w_q| max|plane_q| >= max |combined tile entry|
  // (forward: ONE accumulator takes the direct X items and the transposed Y items, so both share the larger bound).
  // Evaluated twice -- by the converters for their weights and again by the epilogue for the inverse -- rather than kept in
  // registers across the conversion loop (every live register there is a spill at the 96 registers 18 warps allow, and with the
  // whole L1 carved out as shared memory a spill is an L2 round trip on the converters' critical path).
  auto a_scale_exponent = [&](int v) -> int {
    if constexpr (!BFP) return 0;
    const float* am = scp->amax;
    float bound;
    if (BWD) {
      bound = v == 0 ? fabsf(sc.wA[0]) * am[0] + fabsf(sc.wA[1]) * am[1] + fabsf(sc.wA[2]) * am[2] + fabsf(sc.wA[3]) * am[3]
                     : fabsf(sc.wD[1]) * am[1] + fabsf(sc.wD[2]) * am[2] + fabsf(sc.wD[3]) * am[3];
    } else {
      float bx = 0.f, by = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        bx += fabsf(alpha * sc.wA[q] + beta * sc.wD[q]) * am[q];
        by += fabsf(gamma * sc.wA[q] + delta * sc.wD[q]) * am[q];
      }
      bound = fmaxf(bx, by);
    }
    return block_exponent(bound);
  };

  if constexpr (F16) {
    const float as0 = BFP ? exp2_int(a_scale_exponent(0)) : 1.f, as1 = (BFP && BWD) ? exp2_int(a_scale_exponent(NA - 1)) : 1.f;
    const int* ve = BFP ? p.vexp + (size_t)b * p.vexp_stride : nullptr;
    const int Emin = BFP ? bfp_min_exponent(ve, (a.ldk + 127) >> 7) : 0;
    for (int pr = tid; pr < npairs; pr += TC_THREADS) {
      const int kc = kc_of(pr0 + pr);
      const float f = BFP ? exp2_int(max(Emin - __ldcg(ve + (kc >> 2)), -120)) : 1.f;
      sched_kc_s[pr] = kc;
      if (BFP) sched_f_s[pr] = make_float2(f * as0, f * as1);
    }
    if (BFP && tid == 0) *emin_s = Emin;
    __syncthreads();
  }
  if (warp < 16) {
    // =========================== converters ===========================
    const int grp = warp >> 3, w8 = warp & 7;   // group 0: direct items (even j); group 1: transposed items (odd j)
    // row-sharded mode: the transposed products read this rank's rows of the TRANSPOSED path, i.e. they are converted like direct
    // items (operand row = tile row) from planes_t; `dirlike` selects the direct conversion, `tposed` the transposed one
    const bool sharded = a.planes_t != nullptr;
    const bool dirlike = grp == 0 || sharded, tposed = !dirlike;
    // weights of the four planes for each A-operand variant and item type
    float w[NA][4];   // this group's weights: direct items use X (fwd) / (A_s, A'_s) (bwd); transposed items use Y / the same pair
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (LIGHT) {
        const LightCoef lc = grp == 0 ? lc_d : lc_t;
        w[0][q] = lc.cA * sc.wA[q] + lc.cD * sc.wD[q];
        w[NA - 1][q] = lc.sepA ? sc.wA[q] : sc.wD[q];
      } else if (BWD) {
        w[0][q] = sc.wA[q]; w[NA - 1][q] = sc.wD[q];
      } else {
        w[0][q] = grp == 0 ? alpha * sc.wA[q] + beta * sc.wD[q]     // X = (1+p1_0) A + (1+p1_1) A'
                           : gamma * sc.wA[q] + delta * sc.wD[q];   // Y = p2_0 A + p2_1 A'
      }
    }
    const int ntr = a.ldn >> 5, nt = a.ldk >> 5;      // row tiles of this rank's strip, tiles per row of tiles (= K chunks)
    const float* P = ((grp == 1 && sharded) ? a.planes_t : a.planes) + (size_t)b * a.graph_stride + (size_t)sc.interval * 4 * a.ldn * a.ldk;
    // Tiled plane layout (peg_common.cuh): an item is four 16-KB tiles; warp w loads half (g) of tile u, every
    // warp-level LDG.128 is 512 contiguous bytes and the thread ends up with the 4x4 micro tile (rq, cq) of all
    // four planes: buf[plane*4 + m] = row 4*rq + m, columns 4*cq .. 4*cq+3 of the 32x32 tile.
    const int cv_u = w8 >> 1, cv_g = w8 & 1;
    const int cv_cq = lane & 7, cv_rq = ((lane & 7) + 4 * cv_g + (lane >> 3)) & 7;
    const int cv_off = cv_g * 2048 + lane * 4;   // float offset of (g, plane 0, m 0, lane) inside a tile

    // One register buffer per thread (16 x LDG.128 = the thread's 4x4 micro tile of all four planes): a group issues the
    // loads of its next item right after publishing the current one; the two groups run out of phase, so ~2 items
    // (128 KB per SM) are in flight while the other group converts.
    float4 buf[16];
    // 16-bit operand formats, direct items: the 8-byte operand stores of one instruction must hit rows of both parities to be
    // bank-conflict-free (rows are 64 bytes), so the lanes with sw = 1 keep the rows of their micro tile in swapped order
    // (register row m holds tile row m ^ 1).  It costs nothing: only the load addresses and the store offsets change.
    const int sw = (F16 && dirlike) ? ((lane >> 3) & 1) : 0;
    auto load_tile = [&](int rt, int ct) {
      if constexpr (F16) {
        // row tiles beyond the padded matrix (last 128-row block of a ragged n: 4 I + u >= nt, a per-warp, loop-invariant condition)
        // are read from row tile 0 and their weights are zero: no zero-fill path, the loads stay unconditional
        const float* base = P + ((size_t)rt * nt + ct) * 4096 + cv_off;
        const float* base_even = base + sw * 128;
        const float* base_odd = base - sw * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int m = 0; m < 4; ++m) buf[q * 4 + m] = ldg_stream(((m & 1) ? base_odd : base_even) + (q * 4 + m) * 128);
        return;
      }
      if (rt < (tposed ? nt : ntr) && ct < (tposed ? ntr : nt)) {
        const float* base = P + ((size_t)rt * nt + ct) * 4096 + cv_off;
        const float* base_even = base + sw * 128;   // register row m <- tile row m ^ sw: even m read one row up, odd m one row down
        const float* base_odd = base - sw * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int m = 0; m < 4; ++m) buf[q * 4 + m] = ldg_stream(((m & 1) ? base_odd : base_even) + (q * 4 + m) * 128);
      } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) buf[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // item j -> its plane tile: direct = rows of block I x chunk kc, transposed = chunk kc x columns of block I
    // BFP: (A scale of variant v) * 2^(E - e_J) of the item whose planes are in flight.  Fetched in load_item, ahead of the item's
    // 16 plane loads: a shared-memory load issued at the start of the conversion instead queues behind those loads and the operand
    // stores of the other group, and the whole conversion waits for it (measured: 197 vs 155 us per adjoint launch)
    float fitem[NA];
#pragma unroll
    for (int v = 0; v < NA; ++v) fitem[v] = 1.f;
    const bool tile_ok = 4 * I + cv_u < ntr;           // this warp's 32-row (direct) / 32-column (transposed) strip exists
    const int my_tile = tile_ok ? 4 * I + cv_u : 0;
    auto load_item = [&](int j) {
      const int kc = F16 ? sched_kc_s[j >> 1] : kc_of(pr0 + (j >> 1));
      if constexpr (BFP) {
        const float2 e = sched_f_s[j >> 1];
        fitem[0] = e.x;
        if (NA > 1) fitem[NA - 1] = e.y;
      }
      if (dirlike) load_tile(F16 ? my_tile : 4 * I + cv_u, kc);
      else load_tile(kc, F16 ? my_tile : 4 * I + cv_u);
    };
    // store 4 consecutive k (k = 4 * chunk .. 4 * chunk + 3) of operand row r as hi (+ lo) parts into the swizzled K-major tile:
    // tf32: one 16-byte chunk of a 128-byte row (SWIZZLE_128B); bf16x2: 8 bytes of a 64-byte row (SWIZZLE_64B: 16-byte chunk
    // index ^= (row >> 1) & 3 inside 8-row x 64-byte atoms)
    auto store_chunk = [&](uint32_t hi_base, int r, int chunk, float x0, float x1, float x2, float x3, bool with_lo) {
      if constexpr (F16) {
        const uint32_t off = (uint32_t)(r >> 3) * 512u + (uint32_t)(r & 7) * 64u + (uint32_t)(((chunk >> 1) ^ ((r >> 1) & 3)) << 4) + (uint32_t)(chunk & 1) * 8u;
        uint32_t h01, l01, h23, l23;
        split_bf16x2(x0, x1, h01, l01);
        split_bf16x2(x2, x3, h23, l23);
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(hi_base + off), "r"(h01), "r"(h23) : "memory");
        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(hi_base + ATILE + off), "r"(l01), "r"(l23) : "memory");
      } else {
        const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((chunk ^ (r & 7)) << 4);
        const float h0 = tf32_rna(x0), h1 = tf32_rna(x1), h2 = tf32_rna(x2), h3 = tf32_rna(x3);
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(hi_base + off), "f"(h0), "f"(h1), "f"(h2), "f"(h3) : "memory");
        if (split && with_lo)
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(hi_base + ATILE + off), "f"(x0 - h0), "f"(x1 - h1), "f"(x2 - h2), "f"(x3 - h3) : "memory");
      }
    };
    // Conversion of one item: (1) FFMA-combine the four planes (the fused cubic interpolation + fusion weights) while the
    // slot may still be busy, (2) wait for the A slot, (3) 3xTF32-split and store the operand tile, publish it,
    // (4) issue the loads of the group's next item.
    auto convert = [&](int j, bool transposed) {
      float t[NA][16];   // t[v][4 m + e] = element (row 4 rq + m, column 4 cq + e) of the combined tile
#pragma unroll
      for (int v = 0; v < NA; ++v) {
        const float w0 = w[v][0], w1 = w[v][1], w2 = w[v][2], w3 = w[v][3];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const float4 e0 = buf[0 * 4 + m], e1 = buf[1 * 4 + m], e2 = buf[2 * 4 + m], e3 = buf[3 * 4 + m];
          if (BWD && !LIGHT && v == NA - 1) {   // A'_s = b + 2 s c + 3 s^2 d: the derivative has no `a` term (wD[0] == 0)
            t[v][4 * m + 0] = w1 * e1.x + w2 * e2.x + w3 * e3.x;
            t[v][4 * m + 1] = w1 * e1.y + w2 * e2.y + w3 * e3.y;
            t[v][4 * m + 2] = w1 * e1.z + w2 * e2.z + w3 * e3.z;
            t[v][4 * m + 3] = w1 * e1.w + w2 * e2.w + w3 * e3.w;
          } else {
            t[v][4 * m + 0] = w0 * e0.x + w1 * e1.x + w2 * e2.x + w3 * e3.x;
            t[v][4 * m + 1] = w0 * e0.y + w1 * e1.y + w2 * e2.y + w3 * e3.y;
            t[v][4 * m + 2] = w0 * e0.z + w1 * e1.z + w2 * e2.z + w3 * e3.z;
            t[v][4 * m + 3] = w0 * e0.w + w1 * e1.w + w2 * e2.w + w3 * e3.w;
          }
        }
      }
      const int st = j % SA;
      const uint32_t ph = (uint32_t)(j / SA) & 1u;
      const uint32_t a_base = smem_base + st * a_bytes;
      mbar_wait(empty_a(st), ph ^ 1u);   // the MMAs that read this slot's previous contents have completed
#pragma unroll
      for (int v = 0; v < NA; ++v) {
        const uint32_t hi_base = a_base + v * (split ? 2 : 1) * ATILE;
        const bool with_lo = !(LIGHT && v == NA - 1);   // the single-pass operand needs no correction tile
        if (!transposed) {
#pragma unroll
          for (int m = 0; m < 4; ++m)   // operand row = tile row 4 rq + m, chunk = cq (4 consecutive k)
            store_chunk(hi_base, 32 * cv_u + 4 * cv_rq + m, cv_cq, t[v][4 * m + 0], t[v][4 * m + 1], t[v][4 * m + 2], t[v][4 * m + 3], with_lo);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e)   // operand row = tile column 4 cq + e, chunk = rq: the four k values are the rows m = 0..3
            store_chunk(hi_base, 32 * cv_u + 4 * cv_cq + e, cv_rq, t[v][e], t[v][4 + e], t[v][8 + e], t[v][12 + e], with_lo);
        }
      }
      fence_proxy_async();       // generic-proxy smem writes -> visible to the tensor core (async proxy)
      mbar_arrive(full_a(st));
      // the group's next loads go out only now: issued before the slot wait they were measured slower in the forward (159 vs
      // 137 us at n=2048, d=128, B=9), and the adjoint keeps 32 combined values live that would spill at 96 registers
      if (j + 2 < items) load_item(j + 2);
    };

    // ---- 16-bit operand formats: streaming conversion ----
    // With 8-KB tiles there are four A slots, so the slot wait rarely blocks and the conversion needs no staging array: wait for the
    // slot, then combine -> split -> store row by row while the plane registers die (the 3xTF32 path above combines ahead of its
    // slot wait and keeps 32 combined values live, which spills at the 96 registers 18 warps allow).
    // Operand-tile offsets (SWIZZLE_64B): row r, 16-byte chunk c, half hf -> (r >> 3) * 512 + (r & 7) * 64 + ((c ^ ((r >> 1) & 3)) << 4)
    // + 8 hf.  For the four rows r0 + m' (r0 multiple of 4) of one micro tile only (m' >> 1) enters the XOR: two base offsets.
    const int r0 = 32 * cv_u + 4 * (dirlike ? cv_rq : cv_cq);      // first operand row of this thread (direct: tile rows, transposed: tile columns)
    const int kq = dirlike ? cv_cq : cv_rq;                         // its K quad: k = 4 kq .. 4 kq + 3
    const uint32_t o_row = (uint32_t)(r0 >> 3) * 512u + (uint32_t)(r0 & 7) * 64u + (uint32_t)(kq & 1) * 8u;
    const uint32_t o_lo = o_row + (uint32_t)(((kq >> 1) ^ ((r0 >> 1) & 3)) << 4);          // rows r0, r0 + 1
    const uint32_t o_hi = o_row + (uint32_t)(((kq >> 1) ^ (((r0 >> 1) & 3) + 1)) << 4);    // rows r0 + 2, r0 + 3
    // store of row r0 + (m ^ sw) (held in register row m)
    const uint32_t o_m[4] = {o_lo + (uint32_t)(0 ^ sw) * 64u, o_lo + (uint32_t)(1 ^ sw) * 64u, o_hi + (uint32_t)(2 ^ sw) * 64u, o_hi + (uint32_t)(3 ^ sw) * 64u};
    auto split16 = [&](float x0, float x1, uint32_t& hi, uint32_t& lo) {
      if constexpr (BFP) split_f16x2(x0, x1, hi, lo);
      else split_bf16x2(x0, x1, hi, lo);
    };
    // BFP: the launch-wide A scale rides in the (warp-uniform) weights; the per-item block alignment 2^(E - e_J) is one extra
    // multiply per value (a power of two: exact) -- keeping it out of the weights keeps them in uniform registers

    auto comb = [&](int v, float e0, float e1, float e2, float e3) -> float {
      float r;
      if (BWD && v == NA - 1) r = w[v][1] * e1 + w[v][2] * e2 + w[v][3] * e3;    // A'_s has no `a` term (wD[0] == 0)
      else r = w[v][0] * e0 + w[v][1] * e1 + w[v][2] * e2 + w[v][3] * e3;
      return BFP ? r * fitem[v] : r;
    };
    // slot / phase of this group's current item, advanced incrementally (SA is a run-time value: no division per item)
    int cur_st = grp % SA;
    uint32_t cur_ph = 0u;
    auto sts2 = [&](uint32_t addr, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory"); };
    // A warp whose 32-row / 32-column strip lies beyond the padded matrix (last 128-row block of a ragged n) converts nothing: it
    // zeroes its rows of each A slot the first time its group uses the slot (a slot is only ever written by one group) and then
    // just keeps the barrier protocol going.  This keeps the plane weights of every working warp warp-uniform (uniform registers).
    auto idle16 = [&](int j) {
      mbar_wait(empty_a(cur_st), cur_ph ^ 1u);
      if (j < SA) {
        const uint32_t a_base = smem_base + cur_st * a_bytes;
#pragma unroll
        for (int m = 0; m < 4; ++m)
#pragma unroll
          for (int t = 0; t < 2 * NA; ++t) asm volatile("st.shared.v2.b32 [%0], {%1, %1};" ::"r"(a_base + o_m[m] + t * ATILE), "r"(0u) : "memory");
      }
      fence_proxy_async();
      mbar_arrive(full_a(cur_st));
      cur_st += 2;
      if (cur_st >= SA) { cur_st -= SA; cur_ph ^= 1u; }
    };
    auto convert16 = [&](int j, bool transposed) {

      const uint32_t a_base = smem_base + cur_st * a_bytes;
      mbar_wait(empty_a(cur_st), cur_ph ^ 1u);   // the MMAs that read this slot's previous contents have completed
      if (!transposed) {
#pragma unroll
        for (int m = 0; m < 4; ++m) {   // operand row = tile row, the four k values are the columns 4 cq .. 4 cq + 3
          const float4 e0 = buf[0 * 4 + m], e1 = buf[1 * 4 + m], e2 = buf[2 * 4 + m], e3 = buf[3 * 4 + m];
          const uint32_t addr = a_base + o_m[m];
#pragma unroll
          for (int v = 0; v < NA; ++v) {
            uint32_t h01, l01, h23, l23;
            split16(comb(v, e0.x, e1.x, e2.x, e3.x), comb(v, e0.y, e1.y, e2.y, e3.y), h01, l01);
            split16(comb(v, e0.z, e1.z, e2.z, e3.z), comb(v, e0.w, e1.w, e2.w, e3.w), h23, l23);
            sts2(addr + v * 2 * ATILE, h01, h23);
            sts2(addr + v * 2 * ATILE + ATILE, l01, l23);
          }
        }
      } else {
        // operand row = tile column 4 cq + e, the four k values are the tile rows 4 rq + m: rows (0,1) and (2,3) are packed as they
        // are combined, so only 16 packed registers per variant outlive the plane registers
        uint32_t ph[NA][4][2], pl[NA][4][2];   // [variant][column e][row pair]
#pragma unroll
        for (int mp = 0; mp < 2; ++mp) {
          const float4 a0 = buf[0 * 4 + 2 * mp], a1 = buf[1 * 4 + 2 * mp], a2 = buf[2 * 4 + 2 * mp], a3 = buf[3 * 4 + 2 * mp];
          const float4 c0 = buf[0 * 4 + 2 * mp + 1], c1 = buf[1 * 4 + 2 * mp + 1], c2 = buf[2 * 4 + 2 * mp + 1], c3 = buf[3 * 4 + 2 * mp + 1];
#pragma unroll
          for (int v = 0; v < NA; ++v) {
            split16(comb(v, a0.x, a1.x, a2.x, a3.x), comb(v, c0.x, c1.x, c2.x, c3.x), ph[v][0][mp], pl[v][0][mp]);
            split16(comb(v, a0.y, a1.y, a2.y, a3.y), comb(v, c0.y, c1.y, c2.y, c3.y), ph[v][1][mp], pl[v][1][mp]);
            split16(comb(v, a0.z, a1.z, a2.z, a3.z), comb(v, c0.z, c1.z, c2.z, c3.z), ph[v][2][mp], pl[v][2][mp]);
            split16(comb(v, a0.w, a1.w, a2.w, a3.w), comb(v, c0.w, c1.w, c2.w, c3.w), ph[v][3][mp], pl[v][3][mp]);
          }
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint32_t addr = a_base + o_m[e];
#pragma unroll
          for (int v = 0; v < NA; ++v) {
            sts2(addr + v * 2 * ATILE, ph[v][e][0], ph[v][e][1]);
            sts2(addr + v * 2 * ATILE + ATILE, pl[v][e][0], pl[v][e][1]);
          }
        }
      }
      fence_proxy_async();       // generic-proxy smem writes -> visible to the tensor core (async proxy)
      mbar_arrive(full_a(cur_st));
      cur_st += 2;               // this group's next item is j + 2
      if (cur_st >= SA) { cur_st -= SA; cur_ph ^= 1u; }
      if (j + 2 < items) load_item(j + 2);
    };

    if constexpr (F16) {
      if (!tile_ok) {
        for (int j = grp; j < items; j += 2) idle16(j);
      } else {
        // The two groups must run OUT of phase (one converts while the other's loads are in flight).  Started together they can
        // lock in phase -- both wait for loads, then both convert and share the issue slots -- which costs a conversion time per
        // item pair (measured on the fp16x2 adjoint: 195 vs 156 us per launch).  Group 1 therefore starts half a cycle late
        // (1200 ns in the adjoint; the forward needs no stagger).
        if (BWD && grp == 1) __nanosleep(1200u);
        if (items > 0) load_item(grp);   // group 0: direct items (even j); group 1: transposed items (odd j)
        if (grp == 0) for (int j = 0; j < items; j += 2) convert16(j, false);
        else          for (int j = 1; j < items; j += 2) convert16(j, tposed);
      }
    } else {
      if (items > 0) load_item(grp);
      if (grp == 0) for (int j = 0; j < items; j += 2) convert(j, false);
      else          for (int j = 1; j < items; j += 2) convert(j, tposed);
    }
  } else if (warp == 16) {
    // =========================== TMA producer (B operand) ===========================
    if (lane == 0) {
      const int row0 = b * d + ntile * nd;
      for (int pr = 0; pr < npairs; ++pr) {   // one B tile per pair of items
        const int st = pr % SB;
        const uint32_t ph = (uint32_t)(pr / SB) & 1u;
        const int kc = kc_of(pr0 + pr);
        mbar_wait(empty_b(st), ph ^ 1u);   // the MMAs have finished reading this slot
        const uint32_t b_base = b_ring + st * b_bytes;
        mbar_expect_tx(full_b(st), (uint32_t)b_bytes);
        tma_load_2d(b_base, &map_hi, kc * TC_BK, row0, full_b(st));
        if (split) tma_load_2d(b_base + b_tile, &map_lo, kc * TC_BK, row0, full_b(st));
      }
    }
  } else {
    // =========================== MMA issuer ===========================
    if (lane == 0) {
      // instruction descriptor: fp32 accumulate, K-major A and B, N = nd, M = 128; operand format tf32 (2) or bf16 (1)
      const uint32_t fmt = BFP ? 0u : (F16 ? 1u : 2u);   // F16 = 0, BF16 = 1, TF32 = 2
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(nd >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      uint32_t started = 0u;  // bit acc set once the accumulator has been written (first MMA overwrites)
      for (int j = 0; j < items; ++j) {
        const int st = j % SA, pr = j >> 1, sb = pr % SB;
        const uint32_t ph = (uint32_t)(j / SA) & 1u;
        const int type = j & 1;
        if (type == 0) mbar_wait(full_b(sb), (uint32_t)(pr / SB) & 1u);   // the pair's B tile
        const uint32_t a_base = smem_base + st * a_bytes;
        const uint32_t b_base = b_ring + sb * b_bytes;
        mbar_wait(full_a(st), ph);
        tc_fence_after();
#pragma unroll
        for (int v = 0; v < NA; ++v) {
          // fwd: one accumulator; bwd: acc index = type*2 + v  (0: A V, 1: A'V, 2: A^T V, 3: A'^T V;
          // LIGHT: 0 / 2 = combined operand, 1 / 3 = the single-pass sep operand of the direct / transposed items)
          const int acc = BWD ? (type * 2 + v) : 0;
          const uint32_t tacc = tmem_base + (uint32_t)(acc * nd);
          const uint32_t ahi = a_base + v * (split ? 2 : 1) * ATILE, alo = ahi + ATILE;
          if constexpr (F16) {
            // one MMA consumes K = 16 bf16 = 32 bytes of every operand row: two K steps per 32-wide chunk, three products each
#pragma unroll
            for (int k16 = 0; k16 < TC_BK / 16; ++k16) {
              const uint64_t dah = make_desc_sw64(ahi + k16 * 32), dbh = make_desc_sw64(b_base + k16 * 32);
              const uint64_t dal = make_desc_sw64(alo + k16 * 32), dbl = make_desc_sw64(b_base + b_tile + k16 * 32);
              umma_bf16(tacc, dah, dbh, idesc, (started >> acc) & 1u);
              started |= 1u << acc;
              umma_bf16(tacc, dal, dbh, idesc, 1u);
              umma_bf16(tacc, dah, dbl, idesc, 1u);
            }
          } else {
#pragma unroll
            for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
              const uint64_t dah = make_desc_sw128(ahi + k8 * 32), dbh = make_desc_sw128(b_base + k8 * 32);
              umma_tf32(tacc, dah, dbh, idesc, (started >> acc) & 1u);
              started |= 1u << acc;
              if (split && !(LIGHT && v == NA - 1)) {
                const uint64_t dal = make_desc_sw128(alo + k8 * 32), dbl = make_desc_sw128(b_base + b_tile + k8 * 32);
                umma_tf32(tacc, dal, dbh, idesc, 1u);
                umma_tf32(tacc, dah, dbl, idesc, 1u);
              }
            }
          }
        }
        umma_commit(empty_a(st));                 // frees this A slot once the MMAs above have read it
        if (type == 1) umma_commit(empty_b(sb));  // ... and the pair's B slot
      }
      if (items > 0) umma_commit(accum_bar);     // all accumulators final
    }
  }

  // =========================== epilogue (warps 0-7) ===========================
  if (warp < 8) {
    if (items > 0) {
      mbar_wait(accum_bar, 0u);
      tc_fence_after();
    }
    const int q = warp & 3;               // TMEM lane quarter this warp may read
    const int row = q * 32 + lane;
    const int gi = I * TC_BM + row;
    const int half = warp >> 2;           // column half handled by this warp
    const int cols_per_half = nd / 2;     // nd % 32 == 0 is required by tc_supported
    const float* sv = a.svec + (size_t)b * a.sv_stride;
    const float* cb0 = a.colbuf + ((size_t)b * 2 + 0) * d;
    const float* cb1 = a.colbuf + ((size_t)b * 2 + 1) * d;
    const float kappa = scp->kappa[a.layer];
    const bool rowok = gi < n;
    const float vi = rowok ? 1.f + sv[a.v_off + gi] : 0.f;
    const float rc = rowok ? sv[a.rowc_off + gi] : 0.f;
    const float tg = (rowok && a.scale_tg) ? sv[a.tg_off + gi] : 1.f;
    const float* Vrow = a.V + ((size_t)b * n + (rowok ? gi : 0)) * d;
    const float* Mrow = BWD ? a.Mref + ((size_t)b * n + (rowok ? gi : 0)) * d : nullptr;
    float* Orow = a.out + ((size_t)b * n + (rowok ? gi : 0)) * d;
    float g4[4] = {0.f, 0.f, 0.f, 0.f};
    // adjoint only: the O(n d) fusion-parameter gradients (param3..8) ride along -- per node q = <G_i, M_i>,
    // u = <G_i, 1^T M>, w = <M_i, 1^T G> (k_fusion_vec_grads of the CUDA-core path, fused here)
    float fq = 0.f, fu = 0.f, fw = 0.f;
    const float* cbM = (BWD && a.cbM) ? a.cbM + (size_t)b * 2 * d : nullptr;
    for (int cc = 0; cc < cols_per_half; cc += 16) {
      const int col = half * cols_per_half + cc;      // column inside this CTA's ND tile
      const int gc = ntile * nd + col;                // global feature column
      uint32_t r0[16], r1[16], r2[16], r3[16];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col;
      constexpr int NACC = BWD ? 4 : 1;
      float* prow = p.partial ? p.partial + (((size_t)b * NACC) * n + (rowok ? gi : 0)) * d + gc : nullptr;   // accumulator 0
      const size_t pacc = (size_t)n * d;                                                                      // next accumulator
      if (p.mode == 2) {   // split-K: the summed accumulators come from global memory
        auto ld16 = [&](int acc, uint32_t (&r)[16]) {
#pragma unroll
          for (int v4 = 0; v4 < 4; ++v4) {
            const float4 x = rowok ? __ldcg(reinterpret_cast<const float4*>(prow + acc * pacc + 4 * v4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            r[4 * v4] = __float_as_uint(x.x); r[4 * v4 + 1] = __float_as_uint(x.y); r[4 * v4 + 2] = __float_as_uint(x.z); r[4 * v4 + 3] = __float_as_uint(x.w);
          }
        };
        ld16(0, r0);
        if (BWD) { ld16(1, r1); ld16(2, r2); ld16(3, r3); }
      } else {
        tmem_ld16(taddr, r0);
        if (BWD) {
          tmem_ld16(taddr + nd, r1);
          tmem_ld16(taddr + 2 * nd, r2);
          tmem_ld16(taddr + 3 * nd, r3);
        }
        tmem_wait_ld();
        if constexpr (BFP) {   // undo the block scales (powers of two: exact); accumulator acc = type * 2 + v carries the scale of variant v
          // |exponents| <= 60: both factors are normal numbers
          const int Emin = *emin_s;
          const float d0 = exp2_int(-a_scale_exponent(0)) * exp2_int(-Emin), d1 = BWD ? exp2_int(-a_scale_exponent(NA - 1)) * exp2_int(-Emin) : 1.f;
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            r0[u] = __float_as_uint(__uint_as_float(r0[u]) * d0);
            if (BWD) {
              r1[u] = __float_as_uint(__uint_as_float(r1[u]) * d1);
              r2[u] = __float_as_uint(__uint_as_float(r2[u]) * d0);
              r3[u] = __float_as_uint(__uint_as_float(r3[u]) * d1);
            }
          }
        }
      }
      if (p.mode == 1) {   // split-K: add this slice's accumulators into the partial buffer, epilogue runs in the mode-2 launch
        if (rowok && items > 0) {
          auto add16 = [&](int acc, const uint32_t (&r)[16]) {
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4)
              atomicAdd(reinterpret_cast<float4*>(prow + acc * pacc + 4 * v4),
                        make_float4(__uint_as_float(r[4 * v4]), __uint_as_float(r[4 * v4 + 1]), __uint_as_float(r[4 * v4 + 2]), __uint_as_float(r[4 * v4 + 3])));
          };
          add16(0, r0);
          if (BWD) { add16(1, r1); add16(2, r2); add16(3, r3); }
        }
        continue;
      }
      if (rowok) {
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          const float4 vin = *reinterpret_cast<const float4*>(Vrow + gc + 4 * v4);
          const float4 s4 = __ldg(reinterpret_cast<const float4*>(cb0 + gc + 4 * v4));
          const float4 t4 = __ldg(reinterpret_cast<const float4*>(cb1 + gc + 4 * v4));
          const float vv[4] = {vin.x, vin.y, vin.z, vin.w}, ss[4] = {s4.x, s4.y, s4.z, s4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
          float o[4];
          if (!BWD) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              float val = vv[u] * vi + __uint_as_float(r0[4 * v4 + u]) + rc * ss[u] + tt[u] + kappa * ss[u];
              if (a.relu) val = fmaxf(val, 0.f);
              o[u] = val * tg;
            }
          } else {
            const float4 m4 = *reinterpret_cast<const float4*>(Mrow + gc + 4 * v4);
            const float mm[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float aV = __uint_as_float(r0[4 * v4 + u]), dV = __uint_as_float(r1[4 * v4 + u]);
              const float atV = __uint_as_float(r2[4 * v4 + u]), dtV = __uint_as_float(r3[4 * v4 + u]);
              if (LIGHT) o[u] = vv[u] * vi + lc_t.oc * atV + lc_d.oc * aV + rc * ss[u] + tt[u] + kappa * ss[u];   // combined operands carry the weights
              else o[u] = vv[u] * vi + alpha * atV + beta * dtV + gamma * aV + delta * dV + rc * ss[u] + tt[u] + kappa * ss[u];
              g4[0] = fmaf(atV, mm[u], g4[0]);
              g4[1] = fmaf(dtV, mm[u], g4[1]);
              g4[2] = fmaf(aV, mm[u], g4[2]);
              g4[3] = fmaf(dV, mm[u], g4[3]);
              fq = fmaf(vv[u], mm[u], fq);
              fw = fmaf(mm[u], ss[u], fw);
            }
            if (cbM) {
              const float4 c4 = __ldg(reinterpret_cast<const float4*>(cbM + gc + 4 * v4));
              fu = fmaf(vv[0], c4.x, fmaf(vv[1], c4.y, fmaf(vv[2], c4.z, fmaf(vv[3], c4.w, fu))));
            }
          }
          *reinterpret_cast<float4*>(Orow + gc + 4 * v4) = make_float4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    if (BWD && p.mode != 1) {
      // per-thread partials of the 16 fusion-scalar gradients this CTA contributes to (layout of g_fus: param1..8 x 2)
      float part[14];
#pragma unroll
      for (int k = 0; k < 4; ++k) part[k] = g4[k];
#pragma unroll
      for (int k = 4; k < 14; ++k) part[k] = 0.f;
      if (cbM && rowok) {
        const float rA = sv[svec_rA(n, a.L) + gi], rD = sv[svec_rD(n, a.L) + gi];
        const float dA = sv[svec_dgA(n, a.L) + gi], dD = sv[svec_dgD(n, a.L) + gi];
        part[4] = dA * fq; part[5] = dD * fq;      // param3
        part[6] = rA * fu; part[7] = rD * fu;      // param4 (/n)
        part[8] = rA * fw; part[9] = rD * fw;      // param5 (/n)
        part[10] = rA * fq; part[11] = rD * fq;    // param6 (/n)
        part[12] = fq;                              // param8 (* tot / n^2)
      }
      if (cbM && I + a.row_block0 == 0 && q == 0) {   // param7: tot_A / n^2 * <1^T G, 1^T M>, this CTA's columns once per graph
        float t = 0.f;
        for (int c = half * cols_per_half + lane; c < (half + 1) * cols_per_half; c += 32) t = fmaf(cb0[ntile * nd + c], cbM[ntile * nd + c], t);
        part[13] = t;
      }
      const int nred = cbM ? 14 : 4;
      for (int k = 0; k < nred; ++k) {
        float t = part[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        if (lane == 0) fsum[warp][k] = t;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (BWD && p.mode != 1 && tid < (a.cbM ? 14 : 4)) {   // one atomic per scalar and CTA
    float t = 0.f;
#pragma unroll
    for (int w8i = 0; w8i < 8; ++w8i) t += fsum[w8i][tid];
    const float inv_n = 1.f / (float)a.n_glob, inv_n2 = inv_n * inv_n;
    const float totA = scp->totA, totD = scp->totD;
    if (tid < 4) {
      if (LIGHT) {   // (<combined V, M>, <sep V, M>) -> (<A V, M>, <A' V, M>) of this thread's item type (0,1: transposed; 2,3: direct)
        const int pair = tid >> 1;
        float tc = 0.f, ts = 0.f;
#pragma unroll
        for (int w8i = 0; w8i < 8; ++w8i) { tc += fsum[w8i][2 * pair]; ts += fsum[w8i][2 * pair + 1]; }
        const LightCoef c = pair == 0 ? lc_t : lc_d;
        const float gA = c.sepA ? ts : (tc - c.cD * ts) / c.cA;
        const float gD = c.sepA ? (tc - c.cA * ts) / c.cD : ts;
        t = (tid & 1) ? gD : gA;
      }
      atomicAdd(a.g_fus + tid, t);
    }
    else if (tid < 6) atomicAdd(a.g_fus + tid, t);                     // param3: indices 4, 5
    else if (tid < 12) atomicAdd(a.g_fus + tid, t * inv_n);            // param4..6: indices 6..11
    else if (tid == 12) { atomicAdd(a.g_fus + 14, t * totA * inv_n2); atomicAdd(a.g_fus + 15, t * totD * inv_n2); }
    else { atomicAdd(a.g_fus + 12, t * totA * inv_n2); atomicAdd(a.g_fus + 13, t * totA * inv_n2); }   // reference quirk: both use sum(A)
  }
  __syncwarp();
  if (warp == 17) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols));
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// Tensor maps of a K-major fp32 hi / lo operand pair [rows][cols] (cols contiguous), box = 32 cols x box_rows rows,
// SWIZZLE_128B.  They depend only on (buffers, shape, box): a small per-thread cache keeps the driver call off the
// hot path.  The returned pointers stay valid until 16 further distinct maps have been requested on this thread.
static int get_maps(const float* hi, const float* lo, uint64_t cols, uint64_t rows, int box_rows, const CUtensorMap** mhi,
                    const CUtensorMap** mlo, int fmt16 = 0) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return PEG_ERR_UNSUPPORTED;
  struct MapKey { const void* hi; const void* lo; uint64_t rows, cols; int box; int fmt16; };
  struct MapEntry { MapKey k; CUtensorMap mhi, mlo; bool valid; };
  constexpr int NC = 16;
  static thread_local MapEntry cache[NC];
  static thread_local int cache_next = 0;
  MapEntry* ent = nullptr;
  for (int i = 0; i < NC; ++i)
    if (cache[i].valid && cache[i].k.hi == hi && cache[i].k.lo == lo && cache[i].k.rows == rows && cache[i].k.cols == cols &&
        cache[i].k.box == box_rows && cache[i].k.fmt16 == fmt16) { ent = &cache[i]; break; }
  if (!ent) {
    ent = &cache[cache_next];
    cache_next = (cache_next + 1) % NC;
    ent->valid = false;
    const cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)cols * (fmt16 ? 2 : 4)};   // bf16x2 operands: packed bf16, 64-byte box rows, SWIZZLE_64B
    const cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    for (int which = 0; which < 2; ++which) {
      if (enc(which ? &ent->mlo : &ent->mhi, fmt16 == PEG_FMT_BF16X2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : (fmt16 == PEG_FMT_FP16X2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32), 2, (void*)(which ? lo : hi), gdim, gstr, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, fmt16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
        fprintf(stderr, "pegncde: cuTensorMapEncodeTiled failed: dims %llu x %llu, box 32 x %d\n", (unsigned long long)cols,
                (unsigned long long)rows, box_rows);
        return PEG_ERR_CUDA;
      }
    }
    ent->k = MapKey{hi, lo, rows, cols, box_rows, fmt16};
    ent->valid = true;
  }
  *mhi = &ent->mhi;
  *mlo = &ent->mlo;
  return PEG_OK;
}

static int pick_nd(int d, int maxnd) {
  for (int nd = maxnd; nd >= 32; nd -= 32)
    if (d % nd == 0) return nd;
  return 0;
}

static inline int npad_of(int n) { return peg_npad(n); }

void tc_carve(Bump& bp, const PegDims& d, int dmax, TcWs& w) {
  w.npad = npad_of(d.n);
  w.fmt = PEG_FMT_TF32X3;
  w.vexp = nullptr;
  w.vmax = nullptr;
  w.ldk = w.npad;
  w.col0 = w.blk0 = 0;
  w.vexp_stride = (w.npad + 127) / 128;
  if ((d.flags & PEG_FLAG_TENSOR_CORES) == 0) {
    w.Vt_hi = w.Vt_lo = w.partial = nullptr;
    return;
  }
  w.vexp = bp.take<int>((size_t)d.B * w.vexp_stride);
  w.vmax = bp.take<unsigned int>(2 * (size_t)d.B * ((w.npad + 127) / 128));     // block maxima + arrival counters of k_block_exponent (zeroed per API call)
  const size_t cnt = (size_t)d.B * dmax * w.npad;
  w.Vt_hi = bp.take<float>(cnt);
  w.Vt_lo = bp.take<float>(cnt);
  w.partial = bp.take<float>((size_t)d.B * 4 * d.n * dmax);   // split-K accumulators (small grids only)
}

// operand format of the n x n x d contraction (PEG_FMT_*): fp16x2 with block exponents by default; 3xTF32 on request, for the
// tf32-only accuracy modes, when the control carries no plane maxima, or beyond 65536 nodes (512 block exponents per graph)
int tc_fmt(const PegDims& d, bool have_absmax) {
  if (d.flags & (PEG_FLAG_TF32X3 | PEG_FLAG_TF32_FAST | PEG_FLAG_ADJ_LIGHT)) return PEG_FMT_TF32X3;
  if (d.flags & PEG_FLAG_BF16X2) return PEG_FMT_BF16X2;
  return (have_absmax && d.ldn <= 65536) ? PEG_FMT_FP16X2 : PEG_FMT_TF32X3;
}

bool tc_supported(const PegDims& d, int dcols) {
  if (d.n < 128) return false;
  if (dcols % 32 != 0) return false;
  if (pick_nd(dcols, 256) == 0 || pick_nd(dcols, 128) == 0) return false;
  return get_encode() != nullptr;
}

static int tmem_cols_pow2(int cols) {
  int c = 32;
  while (c < cols) c <<= 1;
  return c;
}

// V [B,n,d] -> the K-major B operand V^T (hi / lo parts in the call's operand format) when no producer kernel wrote it
int tc_convert_v(cudaStream_t st, const PegDims& dm, const TcWs& w, const ContractArgs& a) {
  const int n = a.n, d = a.d, npad = w.npad, ldk = w.ldk, fmt = w.fmt;
  if (!w.Vt_hi || !w.Vt_lo) return PEG_ERR_WORKSPACE;
  ProducerOut po;
  memset(&po, 0, sizeof(po));
  po.Thi = w.Vt_hi; po.Tlo = w.Vt_lo; po.npad = ldk; po.t16 = fmt; po.vexp = w.vexp; po.vexp_stride = w.vexp_stride;
  po.col0 = w.col0; po.blk0 = w.blk0; po.rows_pad = npad;
  if (fmt == PEG_FMT_FP16X2) {
    const int slices = d >= 1024 ? 8 : (d >= 256 ? 2 : 1);
    k_block_exponent<<<dim3((npad + 127) / 128, slices, dm.B), 256, 0, st>>>(a.V, n, d, w.vexp, w.vexp_stride, w.blk0, w.vmax, w.vmax + (size_t)dm.B * ((npad + 127) / 128));
    if (cudaPeekAtLastError() != cudaSuccess) { set_last_cuda((int)cudaGetLastError()); fprintf(stderr, "pegncde: k_block_exponent launch failed\n"); return PEG_ERR_CUDA; }
  }
  dim3 grid(npad / 32, (d + 31) / 32, dm.B), block(32, 8);
  k_split_transpose<<<grid, block, 0, st>>>(a.V, n, d, npad, po);
  if (cudaPeekAtLastError() != cudaSuccess) { set_last_cuda((int)cudaGetLastError()); fprintf(stderr, "pegncde: k_split_transpose launch failed\n"); return PEG_ERR_CUDA; }
  return PEG_OK;
}

int tc_contract(cudaStream_t st, const PegDims& dm, const TcWs& w, const ContractArgs& a, bool bwd) {
  const int n = a.n, d = a.d, npad = w.npad, ldk = w.ldk;
  if (!w.Vt_hi || !w.Vt_lo) return PEG_ERR_WORKSPACE;
  if (!get_encode()) return PEG_ERR_UNSUPPORTED;
  const int fmt = w.fmt, f16 = fmt != PEG_FMT_TF32X3 ? 1 : 0;
  if (!a.vt_ready) PEG_TRY(tc_convert_v(st, dm, w, a));
  TcParams p;
  p.a = a;
  p.nd = pick_nd(d, bwd ? 128 : 256);
  p.nsplit = (dm.flags & PEG_FLAG_TF32_FAST) ? 1 : 3;
  p.nkc = ldk / 32;
  const int na = bwd ? 2 : 1, sp = (f16 || p.nsplit == 3) ? 2 : 1;
  const int a_bytes = na * sp * (f16 ? TC_ATILE / 2 : TC_ATILE), b_bytes = sp * p.nd * TC_BK * (f16 ? 2 : 4);
  // smem rings: two B slots (one per pair in flight), the rest of ~208 KB goes to A slots (even count, at most 4)
  int sb = 2;
  int sa = ((208 * 1024 - sb * b_bytes) / a_bytes) & ~1;
  sa = sa > 4 ? 4 : sa;
  if (sa < 2) { sb = 1; sa = ((208 * 1024 - sb * b_bytes) / a_bytes) & ~1; }
  if (f16) {   // half-size tiles: four A slots always fit, the rest goes to B slots (at most 4)
    sb = (208 * 1024 - sa * a_bytes) / b_bytes;
    sb = sb > 4 ? 4 : sb;
  }
  if (sa < 2) return PEG_ERR_UNSUPPORTED;
  p.stages_a = sa;
  p.stages_b = sb;
  p.tmem_cols = tmem_cols_pow2((bwd ? 4 : 1) * p.nd);
  const int nblk = (n + TC_BM - 1) / TC_BM;
  p.vexp = w.vexp;
  p.vexp_stride = w.vexp_stride;
  const size_t sched_bytes = f16 ? (size_t)12 * p.nkc + 32 : 0;   // chunk-schedule table of the 16-bit formats (at most nkc pairs per CTA)
  const size_t smem = (size_t)sa * a_bytes + (size_t)sb * b_bytes + 1024 + 8 * (2 * sa + 2 * sb + 2) + 64 + sched_bytes;

  const CUtensorMap* mhi_p = nullptr;
  const CUtensorMap* mlo_p = nullptr;
  PEG_TRY(get_maps(w.Vt_hi, w.Vt_lo, (uint64_t)ldk, (uint64_t)dm.B * d, p.nd, &mhi_p, &mlo_p, fmt));
  const CUtensorMap& mhi = *mhi_p;
  const CUtensorMap& mlo = *mlo_p;

  // Split-K for grids far smaller than the GPU (one graph of ~1k nodes: 8 row blocks on 148 SMs): every row block's chunk
  // schedule is cut into `ksplit` slices that run on their own SMs and add their accumulators into `partial` (vector
  // atomics); a second, epilogue-only launch finishes the layer.  Costs a memset and a launch, so only when it pays.
  p.mode = 0; p.ksplit = 1; p.pairs_per_slice = p.nkc; p.partial = nullptr;
  {
    const int total = nblk * (d / p.nd) * dm.B;
    int S = 148 / (total > 0 ? total : 1);
    const int smax = 16, minpairs = 2;   // measured on the Twitter shape: 8/4 -> 288, 16/2 -> 298 solver steps/s
    S = S > smax ? smax : S;
    S = S > p.nkc / minpairs ? p.nkc / minpairs : S;
    if (S >= 2 && p.nkc >= 16 && w.partial != nullptr) {
      p.pairs_per_slice = (p.nkc + S - 1) / S;
      p.ksplit = (p.nkc + p.pairs_per_slice - 1) / p.pairs_per_slice;   // every slice non-empty
      p.partial = w.partial;
      p.mode = 1;
    }
  }
  dim3 grid(nblk * p.ksplit, d / p.nd, dm.B);
  if (p.mode == 1) {
    if (cudaMemsetAsync(w.partial, 0, (size_t)dm.B * (bwd ? 4 : 1) * n * d * sizeof(float), st) != cudaSuccess) {
      set_last_cuda((int)cudaGetLastError());
      return PEG_ERR_CUDA;
    }
  }
  // PEG_FLAG_ADJ_LIGHT (two of the four adjoint products single-pass): measured on B200 at n=2048, d=128, B=9 the adjoint launch
  // goes 213 -> 199 us (+5 % solver steps/s) but the param1/param2 gradients of a whole solve are off by up to 2.5e-3 (the rounding
  // of the slowly varying planes is correlated across launches, it does not average out) -> an accuracy mode the caller asks for
  const int kind = bwd ? ((dm.flags & PEG_FLAG_ADJ_LIGHT) ? 2 : 1) : 0;   // tc_fmt() is 3xTF32 whenever ADJ_LIGHT is set
  // the instantiation for (kind, format): 0..2 = 3xTF32 forward / adjoint / LIGHT adjoint, then bf16x2 and fp16x2 forward / adjoint
  const int inst = fmt == PEG_FMT_TF32X3 ? kind : 3 + 2 * (fmt - 1) + kind;
  {
    static std::atomic<unsigned> done[7] = {{0u}, {0u}, {0u}, {0u}, {0u}, {0u}, {0u}};
    switch (inst) {
      case 0: PEG_TRY(optin_smem(k_tc_contract<0, 0>, done[0])); break;
      case 1: PEG_TRY(optin_smem(k_tc_contract<1, 0>, done[1])); break;
      case 2: PEG_TRY(optin_smem(k_tc_contract<2, 0>, done[2])); break;
      case 3: PEG_TRY(optin_smem(k_tc_contract<0, 1>, done[3])); break;
      case 4: PEG_TRY(optin_smem(k_tc_contract<1, 1>, done[4])); break;
      case 5: PEG_TRY(optin_smem(k_tc_contract<0, 2>, done[5])); break;
      default: PEG_TRY(optin_smem(k_tc_contract<1, 2>, done[6])); break;
    }
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  auto launch = [&]() -> cudaError_t {
    switch (inst) {
      case 0: return cudaLaunchKernelEx(&cfg, k_tc_contract<0, 0>, mhi, mlo, p);
      case 1: return cudaLaunchKernelEx(&cfg, k_tc_contract<1, 0>, mhi, mlo, p);
      case 2: return cudaLaunchKernelEx(&cfg, k_tc_contract<2, 0>, mhi, mlo, p);
      case 3: return cudaLaunchKernelEx(&cfg, k_tc_contract<0, 1>, mhi, mlo, p);
      case 4: return cudaLaunchKernelEx(&cfg, k_tc_contract<1, 1>, mhi, mlo, p);
      case 5: return cudaLaunchKernelEx(&cfg, k_tc_contract<0, 2>, mhi, mlo, p);
      default: return cudaLaunchKernelEx(&cfg, k_tc_contract<1, 2>, mhi, mlo, p);
    }
  };
  const cudaError_t le = launch();
  if (le != cudaSuccess) {
    fprintf(stderr, "pegncde: k_tc_contract<%d> launch failed (%s): grid %u x %u x %u, smem %zu, nd %d, slots A %d B %d, tmem %d\n", kind,
            cudaGetErrorString(le), grid.x, grid.y, grid.z, smem, p.nd, sa, sb, p.tmem_cols);
    set_last_cuda((int)le); (void)cudaGetLastError(); return PEG_ERR_CUDA;
  }
  if (cudaPeekAtLastError() != cudaSuccess) { set_last_cuda((int)cudaGetLastError()); return PEG_ERR_CUDA; }
  if (p.mode == 1) {   // epilogue-only launch over the row blocks
    p.mode = 2;
    cfg.gridDim = dim3((unsigned)nblk, d / p.nd, dm.B);
    const cudaError_t le2 = launch();
    if (le2 != cudaSuccess) { set_last_cuda((int)le2); (void)cudaGetLastError(); return PEG_ERR_CUDA; }
  }
  return PEG_OK;
}


// ==========================================================================================
// RMSNorm -> Linear on tcgen05 (3xTF32):  M = rinv (Z Wn^T) + cvec,  Wn = W diag(norm.weight),
// cvec = W norm.bias + bias (tc_prep_weights), rinv = rsqrt(mean z^2 + eps) per node.
// One CTA per 128 nodes x ND outputs: M = 128 (nodes), N = ND, K = din in chunks of 32.
//   warps 0-7 : load Z rows (coalesced LDG.128, all K chunks of a 128-wide super chunk in flight at once), accumulate
//               sum z^2, 3xTF32-split into the swizzled K-major A tiles; afterwards the epilogue (tcgen05.ld):
//               norm scale + bias, M, V^T hi/lo (coalesced: lane = node), deterministic column sums
//   warp 8    : TMA producer of the weight tiles (hi / lo, SWIZZLE_128B);  warp 9: TMEM allocator + MMA issuer
// grid (ceil(n/128), dout/ND, B), block 320
// ==========================================================================================
// Sums, over the 32 lanes of a warp, 16 per-lane values at once with a transpose-reduce butterfly (16 shuffles instead
// of 80): on return v[0] of lane L holds the full sum of column warp_col16(L) (each column lands in two lanes).
// Fixed order, hence deterministic.
__device__ __forceinline__ int warp_col16(int lane) { return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1); }
__device__ __forceinline__ void warp_colsum16(float (&v)[16], int lane) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool up = (lane & 16) != 0;
    const float send = up ? v[i] : v[i + 8], keep = up ? v[i + 8] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool up = (lane & 8) != 0;
    const float send = up ? v[i] : v[i + 4], keep = up ? v[i + 4] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool up = (lane & 4) != 0;
    const float send = up ? v[i] : v[i + 2], keep = up ? v[i + 2] : v[i];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  {
    const bool up = (lane & 2) != 0;
    const float send = up ? v[0] : v[1], keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

constexpr int NL_THREADS = 320;

struct NlParams {
  const float* Z;      // [B,n,din]
  const float* cvec;   // [dout]
  float* M;            // [B,n,dout]
  ProducerOut po;
  int n, din, dout, nd, stages, tmem_cols, nsplit;
};

__global__ void __launch_bounds__(NL_THREADS, 1)
k_tc_norm_linear(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, const NlParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ float rinv_s[128];
  __shared__ float bmax_s[8];
  __shared__ bool is_last;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z, rb = blockIdx.x, ntile = blockIdx.y;
  const int n = p.n, din = p.din, dout = p.dout, nd = p.nd, S = p.stages;
  const bool split = p.nsplit == 3;
  const int row0 = rb * 128;
  const int nchunks = din >> 5;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int a_bytes = (split ? 2 : 1) * TC_ATILE;
  const int b_tile = nd * TC_BK * 4;
  const int b_bytes = (split ? 2 : 1) * b_tile;
  const int stage_bytes = a_bytes + b_bytes;
  const uint32_t bar_base = smem_base + S * stage_bytes;
  auto full_a = [&](int s) { return bar_base + 8u * s; };
  auto full_b = [&](int s) { return bar_base + 8u * (S + s); };
  auto empty = [&](int s) { return bar_base + 8u * (2 * S + s); };
  const uint32_t accum_bar = bar_base + 8u * (3 * S);
  const uint32_t tmem_slot = accum_bar + 8u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  float* csum = reinterpret_cast<float*>(smem_gen);   // [4 row quarters][2][nd]: reuses stage 0 after the MMAs are done

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full_a(s), 256);
      mbar_init(full_b(s), 1);
      mbar_init(empty(s), 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));
  const float* Zb = p.Z + (size_t)b * n * din;

  if (warp < 8) {
    // ---- loaders / converters: thread -> rows 32 i + (tid >> 3), 16-byte chunk (tid & 7) of every K chunk ----
    const int lr = tid >> 3, lc = tid & 7;
    float rsq[4] = {0.f, 0.f, 0.f, 0.f};
    for (int sc0 = 0; sc0 < nchunks; sc0 += 4) {
      float4 buf[4][4];
#pragma unroll
      for (int kc = 0; kc < 4; ++kc)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = row0 + 32 * i + lr;
          buf[kc][i] = (sc0 + kc < nchunks && row < n) ? __ldg(reinterpret_cast<const float4*>(Zb + (size_t)row * din + (sc0 + kc) * 32 + lc * 4))
                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        const int j = sc0 + kc;
        if (j >= nchunks) break;
        const int st = j % S;
        mbar_wait(empty(st), ((uint32_t)(j / S) & 1u) ^ 1u);
        const uint32_t a_base = smem_base + st * stage_bytes;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = buf[kc][i];
          rsq[i] = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, rsq[i]))));
          const int r = 32 * i + lr;
          const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((lc ^ (r & 7)) << 4);
          const float h0 = tf32_rna(v.x), h1 = tf32_rna(v.y), h2 = tf32_rna(v.z), h3 = tf32_rna(v.w);
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_base + off), "f"(h0), "f"(h1), "f"(h2), "f"(h3) : "memory");
          if (split)
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_base + TC_ATILE + off), "f"(v.x - h0), "f"(v.y - h1),
                         "f"(v.z - h2), "f"(v.w - h3) : "memory");
        }
        fence_proxy_async();
        mbar_arrive(full_a(st));
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {   // the 8 lanes that share a row
      float v = rsq[i];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      if (lc == 0) rinv_s[32 * i + lr] = rsqrtf(v / (float)din + 1e-5f);
    }
  } else if (warp == 8) {
    if (lane == 0) {
      const int wrow0 = ntile * nd;
      for (int j = 0; j < nchunks; ++j) {
        const int st = j % S;
        mbar_wait(empty(st), ((uint32_t)(j / S) & 1u) ^ 1u);
        const uint32_t b_base = smem_base + st * stage_bytes + a_bytes;
        mbar_expect_tx(full_b(st), (uint32_t)b_bytes);
        tma_load_2d(b_base, &map_hi, j * TC_BK, wrow0, full_b(st));
        if (split) tma_load_2d(b_base + b_tile, &map_lo, j * TC_BK, wrow0, full_b(st));
      }
    }
  } else {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(nd >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      for (int j = 0; j < nchunks; ++j) {
        const int st = j % S;
        const uint32_t ph = (uint32_t)(j / S) & 1u;
        mbar_wait(full_b(st), ph);
        mbar_wait(full_a(st), ph);
        tc_fence_after();
        const uint32_t ahi = smem_base + st * stage_bytes, alo = ahi + TC_ATILE;
        const uint32_t bhi = ahi + a_bytes, blo = bhi + b_tile;
#pragma unroll
        for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
          const uint64_t dah = make_desc_sw128(ahi + k8 * 32), dbh = make_desc_sw128(bhi + k8 * 32);
          umma_tf32(tmem_base, dah, dbh, idesc, (j > 0 || k8 > 0) ? 1u : 0u);
          if (split) {
            umma_tf32(tmem_base, make_desc_sw128(alo + k8 * 32), dbh, idesc, 1u);
            umma_tf32(tmem_base, dah, make_desc_sw128(blo + k8 * 32), idesc, 1u);
          }
        }
        umma_commit(empty(st));
      }
      umma_commit(accum_bar);
    }
  }

  // ---- epilogue (warps 0-7): TMEM lane = node, columns = outputs ----
  if (warp < 8) {
    asm volatile("bar.sync 1, 256;" ::: "memory");   // rinv_s complete (loader warps only)
    mbar_wait(accum_bar, 0u);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane, gi = row0 + row;
    const bool rowok = gi < n;
    const float ri = rinv_s[row];
    const float vv = (p.po.vec && rowok) ? p.po.vec[(size_t)b * p.po.vec_stride + gi] : 0.f;
    float* Mrow = p.M + ((size_t)b * n + (rowok ? gi : 0)) * dout;
    const int cols_per_half = nd / 2;
    // fp16x2 operand format: V^T of this 128-node block is stored as M * 2^e with one block exponent e (a first pass over the
    // accumulators finds the block maximum; the host hands out Thi only when this CTA holds every column of the block)
    float vscale = 1.f;
    if (p.po.Thi != nullptr && p.po.t16 == PEG_FMT_FP16X2) {
      float mx = 0.f;
      for (int cc = 0; cc < cols_per_half; cc += 16) {
        const int col = half * cols_per_half + cc, gc = ntile * nd + col;
        uint32_t r[16];
        tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col, r);
        tmem_wait_ld();
        if (rowok) {
#pragma unroll
          for (int u = 0; u < 16; ++u) mx = fmaxf(mx, fabsf(fmaf(ri, __uint_as_float(r[u]), __ldg(p.cvec + gc + u))));
        }
      }
      mx = warp_max(mx);
      if (lane == 0) bmax_s[warp] = mx;
      asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) mx = fmaxf(mx, bmax_s[w8]);
      const int e = block_exponent(mx);
      vscale = exp2_int(e);
      if (tid == 0) p.po.vexp[(size_t)b * p.po.vexp_stride + p.po.blk0 + rb] = e;
    }
    for (int cc = 0; cc < cols_per_half; cc += 16) {
      const int col = half * cols_per_half + cc, gc = ntile * nd + col;
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col, r);
      tmem_wait_ld();
      float m[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) m[u] = rowok ? fmaf(ri, __uint_as_float(r[u]), __ldg(p.cvec + gc + u)) : 0.f;
      if (rowok) {
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4)
          *reinterpret_cast<float4*>(Mrow + gc + 4 * v4) = make_float4(m[4 * v4], m[4 * v4 + 1], m[4 * v4 + 2], m[4 * v4 + 3]);
      }
      if (p.po.Thi != nullptr && gi < p.po.rows_pad) {   // V^T hi/lo: the 32 lanes of a warp are 32 consecutive nodes
        if (p.po.t16 == PEG_FMT_FP16X2) {
#pragma unroll
          for (int u = 0; u < 16; ++u) store_vt_f16(p.po, ((size_t)b * dout + gc + u) * p.po.npad + p.po.col0 + gi, m[u] * vscale);
        } else {
#pragma unroll
          for (int u = 0; u < 16; ++u) store_vt(p.po, ((size_t)b * dout + gc + u) * p.po.npad + p.po.col0 + gi, m[u]);
        }
      }
      if (p.po.cb != nullptr) {   // column sums over this warp's 32 nodes (fixed butterfly order)
        float s1[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) s1[u] = vv * m[u];
        warp_colsum16(m, lane);
        warp_colsum16(s1, lane);
        if ((lane & 1) == 0) {
          csum[(q * 2 + 0) * nd + col + warp_col16(lane)] = m[0];
          csum[(q * 2 + 1) * nd + col + warp_col16(lane)] = s1[0];
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (p.po.cb != nullptr) {
    const int chunks = gridDim.x;
    if (tid < nd) {
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) { t0 += csum[(q * 2 + 0) * nd + tid]; t1 += csum[(q * 2 + 1) * nd + tid]; }
      float* part = p.po.partial + (((size_t)b * chunks + rb) * 2) * dout;
      part[ntile * nd + tid] = t0;
      part[dout + ntile * nd + tid] = t1;
    }
    finalize_colsums(p.po, b, chunks, dout, ntile * nd, nd, p.po.tickets + (size_t)b * gridDim.y + ntile, &is_last);
  }
  if (warp == 9) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols));
  }
}

// weights of one layer -> Wn hi/lo [dout][din] and cvec [dout].  grid (dout), block 128
__global__ void __launch_bounds__(128) k_prep_weights(const float* __restrict__ W, const float* __restrict__ bias,
                                                      const float* __restrict__ nw, const float* __restrict__ nb, int din,
                                                      float* __restrict__ Wn_hi, float* __restrict__ Wn_lo, float* __restrict__ cvec,
                                                      float* __restrict__ Wt_hi, float* __restrict__ Wt_lo) {
  __shared__ float sh[33];
  const int o = blockIdx.x, dout = gridDim.x;
  float c = 0.f;
  for (int k = threadIdx.x; k < din; k += 128) {
    const float w = W[(size_t)o * din + k];
    const float wn = w * nw[k];
    const float hi = tf32_rna(wn);
    Wn_hi[(size_t)o * din + k] = hi;
    Wn_lo[(size_t)o * din + k] = wn - hi;
    const float wh = tf32_rna(w);
    Wt_hi[(size_t)k * dout + o] = wh;
    Wt_lo[(size_t)k * dout + o] = w - wh;
    c = fmaf(nb[k], w, c);
  }
  const float t = block_sum(c, sh);
  if (threadIdx.x == 0) cvec[o] = t + bias[o];
}

void tc_carve_linear(Bump& bp, const PegDims& d, const Model& m, TcLinear& w) {
  memset(&w, 0, sizeof(w));
  if ((d.flags & PEG_FLAG_TENSOR_CORES) == 0) return;
  for (int l = 0; l < m.L; ++l) {
    const size_t cnt = (size_t)m.layer[l].dout * m.layer[l].din;
    w.Wn_hi[l] = bp.take<float>(cnt);
    w.Wn_lo[l] = bp.take<float>(cnt);
    w.cvec[l] = bp.take<float>(m.layer[l].dout);
    w.Wt_hi[l] = bp.take<float>(cnt);
    w.Wt_lo[l] = bp.take<float>(cnt);
  }
  w.ready = true;
}

static int nl_pick_nd(int dout) {
  for (int nd = 256; nd >= 32; nd -= 32)
    if (dout % nd == 0) return nd;
  return 0;
}

bool tc_norm_linear_full_columns(int dout) { return nl_pick_nd(dout) == dout; }

bool tc_linear_supported(int din, int dout) {
  return din % 32 == 0 && din >= 32 && nl_pick_nd(dout) != 0 && get_encode() != nullptr;
}

int tc_prep_weights(cudaStream_t st, const Model& m, const float* params, const TcLinear& w) {
  if (!w.ready) return PEG_OK;
  for (int l = 0; l < m.L; ++l) {
    const LayerDesc& ld = m.layer[l];
    if (!tc_linear_supported(ld.din, ld.dout) && !tc_linear_bwd_supported(ld.din, ld.dout)) continue;
    k_prep_weights<<<ld.dout, 128, 0, st>>>(params + ld.w_off, params + ld.b_off, params + ld.nw_off, params + ld.nb_off, ld.din,
                                            w.Wn_hi[l], w.Wn_lo[l], w.cvec[l], w.Wt_hi[l], w.Wt_lo[l]);
    if (cudaPeekAtLastError() != cudaSuccess) { set_last_cuda((int)cudaGetLastError()); return PEG_ERR_CUDA; }
  }
  return PEG_OK;
}

int tc_norm_linear(cudaStream_t st, const PegDims& dm, const TcLinear& w, int layer, const float* Z, int din, int dout, float* M,
                   const ProducerOut& po) {
  if (!w.ready) return PEG_ERR_WORKSPACE;
  NlParams p;
  memset(&p, 0, sizeof(p));
  p.Z = Z; p.cvec = w.cvec[layer]; p.M = M; p.po = po;
  p.n = dm.n; p.din = din; p.dout = dout;
  p.nd = nl_pick_nd(dout);
  p.nsplit = (dm.flags & PEG_FLAG_TF32_FAST) ? 1 : 3;
  const int sp = p.nsplit == 3 ? 2 : 1;
  const int stage_bytes = sp * TC_ATILE + sp * p.nd * TC_BK * 4;
  int stages = (200 * 1024) / stage_bytes;
  const int nchunks = din / 32;
  stages = stages > nchunks ? nchunks : stages;
  stages = stages > 4 ? 4 : stages;
  if (stages < 1) return PEG_ERR_UNSUPPORTED;
  p.stages = stages;
  p.tmem_cols = tmem_cols_pow2(p.nd);
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 8 * (3 * stages + 2) + 64;
  const CUtensorMap* mhi = nullptr;
  const CUtensorMap* mlo = nullptr;
  PEG_TRY(get_maps(w.Wn_hi[layer], w.Wn_lo[layer], (uint64_t)din, (uint64_t)dout, p.nd, &mhi, &mlo));
  static std::atomic<unsigned> done{0u};
  PEG_TRY(optin_smem(k_tc_norm_linear, done));
  dim3 grid((dm.n + 127) / 128, dout / p.nd, dm.B);
  k_tc_norm_linear<<<grid, NL_THREADS, smem, st>>>(*mhi, *mlo, p);
  if (cudaPeekAtLastError() != cudaSuccess) {
    const cudaError_t e = cudaGetLastError();
    fprintf(stderr, "pegncde: k_tc_norm_linear launch failed (%s): grid %u x %u x %u, smem %zu, nd %d, stages %d\n",
            cudaGetErrorString(e), grid.x, grid.y, grid.z, smem, p.nd, stages);
    set_last_cuda((int)e);
    return PEG_ERR_CUDA;
  }
  return PEG_OK;
}


// ==========================================================================================
// Backward of Linear + RMSNorm wrt the layer input on tcgen05 (3xTF32):
//   Nbar = Mbar W   (M = 128 nodes, N = din, K = dout in chunks of 32; A = Mbar rows converted in flight, B = W^T hi/lo by TMA)
//   Zbar = rinv w Nbar - z rinv^3 <w Nbar, z> / din ; optional ReLU mask (z > 0) ; g_nw += sum Nbar zhat ; g_nb += sum Nbar
// plus the producer outputs of Zbar (V^T hi/lo, deterministic column sums) for the next adjoint contraction.
// A thread of the epilogue owns one node: the per-node reductions are thread-local apart from one exchange between the
// two column halves; per-column reductions use the butterfly above.
// The Linear's own gradient needs the normalised input N = z rinv nw + nb, which this kernel has at hand:
//   dout == 128 (gW set): Wbar += Mbar^T N and bbar += 1^T Mbar of the CTA's 128 nodes on tcgen05 as well.  The epilogue stores
//     both operands transposed (node = K) into the idle operand ring, one 32-node K step per warp quarter, and a second TMEM
//     accumulator takes the 128 x din partial, which is added with vector atomics.
//   otherwise (Nout set): N is written out for k_tc_weight_grad.
// grid (ceil(n/128), 1, B), block 320
// ==========================================================================================
struct LbParams {
  const float* Mbar;   // [B,n,dout]
  const float* Z;      // [B,n,din]
  const float* nw;     // [din]
  const float* nb;     // [din]
  float* Zbar;         // [B,n,din]
  float* g_nw;
  float* g_nb;
  float* gW;           // nullable [dout][din]: fused weight gradient (dout == 128)
  float* gb;           // [dout] (with gW)
  float* Nout;         // nullable [B,n,din]
  ProducerOut po;
  int n, din, dout, stages, tmem_cols, nsplit, relu_mask, wg_col;
};

__global__ void __launch_bounds__(NL_THREADS, 1)
k_tc_linear_bwd(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, const LbParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ float red_s[2][2][128];   // [column half][ss, dot][node]
  __shared__ float bmax_s[8];
  __shared__ bool is_last;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.z, rb = blockIdx.x;
  const int n = p.n, din = p.din, dout = p.dout, nd = din, S = p.stages;
  const bool split = p.nsplit == 3;
  const int row0 = rb * 128;
  const int nchunks = dout >> 5;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int a_bytes = (split ? 2 : 1) * TC_ATILE;
  const int b_tile = nd * TC_BK * 4;
  const int b_bytes = (split ? 2 : 1) * b_tile;
  const int stage_bytes = a_bytes + b_bytes;
  const bool wg = p.gW != nullptr;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  float* csum = reinterpret_cast<float*>(smem_gen + S * stage_bytes);   // [4 row quarters][4 sums][din]
  float* bsum = csum + 16 * din;                                        // [4 row quarters][dout] (wg)
  const uint32_t bar_base = smem_base + S * stage_bytes + (16 * din + (wg ? 4 * dout : 0)) * 4;
  auto full_a = [&](int s) { return bar_base + 8u * s; };
  auto full_b = [&](int s) { return bar_base + 8u * (S + s); };
  auto empty = [&](int s) { return bar_base + 8u * (2 * S + s); };
  auto wg_full = [&](int s) { return bar_base + 8u * (3 * S + s); };
  auto wg_free = [&](int s) { return bar_base + 8u * (4 * S + s); };
  const uint32_t accum_bar = bar_base + 8u * (5 * S);
  const uint32_t wg_bar = accum_bar + 8u;
  const uint32_t tmem_slot = wg_bar + 8u;

  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full_a(s), 256);
      mbar_init(full_b(s), 1);
      mbar_init(empty(s), 1);
      mbar_init(wg_full(s), 64);
      mbar_init(wg_free(s), 1);
    }
    mbar_init(accum_bar, 1);
    mbar_init(wg_bar, 1);
    fence_barrier_init();
  }
  if (warp == 9) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));
  const float* Mb = p.Mbar + (size_t)b * n * dout;
  const float* Zb = p.Z + (size_t)b * n * din;

  if (warp < 8) {
    const int lr = tid >> 3, lc = tid & 7;
    for (int sc0 = 0; sc0 < nchunks; sc0 += 4) {
      float4 buf[4][4];
#pragma unroll
      for (int kc = 0; kc < 4; ++kc)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = row0 + 32 * i + lr;
          buf[kc][i] = (sc0 + kc < nchunks && row < n) ? __ldg(reinterpret_cast<const float4*>(Mb + (size_t)row * dout + (sc0 + kc) * 32 + lc * 4))
                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        const int j = sc0 + kc;
        if (j >= nchunks) break;
        const int st = j % S;
        mbar_wait(empty(st), ((uint32_t)(j / S) & 1u) ^ 1u);
        const uint32_t a_base = smem_base + st * stage_bytes;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 v = buf[kc][i];
          const int r = 32 * i + lr;
          const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((lc ^ (r & 7)) << 4);
          const float h0 = tf32_rna(v.x), h1 = tf32_rna(v.y), h2 = tf32_rna(v.z), h3 = tf32_rna(v.w);
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_base + off), "f"(h0), "f"(h1), "f"(h2), "f"(h3) : "memory");
          if (split)
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_base + TC_ATILE + off), "f"(v.x - h0), "f"(v.y - h1),
                         "f"(v.z - h2), "f"(v.w - h3) : "memory");
        }
        fence_proxy_async();
        mbar_arrive(full_a(st));
      }
    }
  } else if (warp == 8) {
    if (lane == 0) {
      for (int j = 0; j < nchunks; ++j) {
        const int st = j % S;
        mbar_wait(empty(st), ((uint32_t)(j / S) & 1u) ^ 1u);
        const uint32_t b_base = smem_base + st * stage_bytes + a_bytes;
        mbar_expect_tx(full_b(st), (uint32_t)b_bytes);
        tma_load_2d(b_base, &map_hi, j * TC_BK, 0, full_b(st));
        if (split) tma_load_2d(b_base + b_tile, &map_lo, j * TC_BK, 0, full_b(st));
      }
    }
  } else {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(nd >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      for (int j = 0; j < nchunks; ++j) {
        const int st = j % S;
        const uint32_t ph = (uint32_t)(j / S) & 1u;
        mbar_wait(full_b(st), ph);
        mbar_wait(full_a(st), ph);
        tc_fence_after();
        const uint32_t ahi = smem_base + st * stage_bytes, alo = ahi + TC_ATILE;
        const uint32_t bhi = ahi + a_bytes, blo = bhi + b_tile;
#pragma unroll
        for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
          const uint64_t dah = make_desc_sw128(ahi + k8 * 32), dbh = make_desc_sw128(bhi + k8 * 32);
          umma_tf32(tmem_base, dah, dbh, idesc, (j > 0 || k8 > 0) ? 1u : 0u);
          if (split) {
            umma_tf32(tmem_base, make_desc_sw128(alo + k8 * 32), dbh, idesc, 1u);
            umma_tf32(tmem_base, dah, make_desc_sw128(blo + k8 * 32), idesc, 1u);
          }
        }
        umma_commit(empty(st));
      }
      umma_commit(accum_bar);
      if (wg) {   // Wbar partial: K = the 128 nodes, one 32-node step per warp quarter of the epilogue, step c in ring slot c % S
        for (int c = 0; c < 4; ++c) {
          const int st = c % S;
          mbar_wait(wg_full(st), (uint32_t)(c / S) & 1u);
          tc_fence_after();
          const uint32_t ahi = smem_base + st * stage_bytes, alo = ahi + TC_ATILE;
          const uint32_t bhi = ahi + a_bytes, blo = bhi + b_tile;
#pragma unroll
          for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
            const uint64_t dah = make_desc_sw128(ahi + k8 * 32), dbh = make_desc_sw128(bhi + k8 * 32);
            umma_tf32(tmem_base + (uint32_t)p.wg_col, dah, dbh, idesc, (c > 0 || k8 > 0) ? 1u : 0u);
            if (split) {
              umma_tf32(tmem_base + (uint32_t)p.wg_col, make_desc_sw128(alo + k8 * 32), dbh, idesc, 1u);
              umma_tf32(tmem_base + (uint32_t)p.wg_col, dah, make_desc_sw128(blo + k8 * 32), idesc, 1u);
            }
          }
          umma_commit(wg_free(st));
        }
        umma_commit(wg_bar);
      }
    }
  }

  if (warp < 8) {
    mbar_wait(accum_bar, 0u);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane, gi = row0 + row;
    const bool rowok = gi < n;
    const float* Zrow = Zb + (size_t)(rowok ? gi : 0) * din;
    const int cols_per_half = nd / 2;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    // pass 1: this half's share of sum z^2 and <w Nbar, z>
    float ss = 0.f, dot = 0.f;
    for (int cc = 0; cc < cols_per_half; cc += 16) {
      const int col = half * cols_per_half + cc;
      uint32_t r[16];
      tmem_ld16(trow + (uint32_t)col, r);
      tmem_wait_ld();
      if (rowok) {
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          const float4 z4 = *reinterpret_cast<const float4*>(Zrow + col + 4 * v4);
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.nw + col + 4 * v4));
          const float zz[4] = {z4.x, z4.y, z4.z, z4.w}, ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            ss = fmaf(zz[u], zz[u], ss);
            dot = fmaf(ww[u] * __uint_as_float(r[4 * v4 + u]), zz[u], dot);
          }
        }
      }
    }
    red_s[half][0][row] = ss;
    red_s[half][1][row] = dot;
    asm volatile("bar.sync 1, 256;" ::: "memory");
    ss = red_s[0][0][row] + red_s[1][0][row];
    dot = red_s[0][1][row] + red_s[1][1][row];
    const float rinv = rsqrtf(ss / (float)din + 1e-5f);
    const float coef = rinv * rinv * rinv * dot / (float)din;
    if (wg) {
      // K step q of the weight gradient: this quarter's 32 nodes (lane = K index) into ring slot q % S, which the main MMAs have
      // released (accum_bar) or the weight-gradient MMA of step q - S frees.  A' = Mbar^T (row = output), B' = N^T (row = input).
      const int st = q % S;
      if (q >= S) mbar_wait(wg_free(st), 0u);
      const uint32_t a_base = smem_base + st * stage_bytes, b_base = a_base + a_bytes;
      auto put = [&](uint32_t tile, uint32_t lo_off, int r, float x) {
        const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + ((uint32_t)((lane >> 2) ^ (r & 7)) << 4) + (uint32_t)(lane & 3) * 4u;
        const float h = tf32_rna(x);
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(tile + off), "f"(h) : "memory");
        if (split) asm volatile("st.shared.f32 [%0], %1;" ::"r"(tile + lo_off + off), "f"(x - h) : "memory");
      };
      const float* Mrow = Mb + (size_t)(rowok ? gi : 0) * dout;
      for (int oc = half * (dout / 2); oc < (half + 1) * (dout / 2); oc += 16) {
        float m[16];
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          const float4 m4 = rowok ? __ldg(reinterpret_cast<const float4*>(Mrow + oc + 4 * v4)) : make_float4(0.f, 0.f, 0.f, 0.f);
          m[4 * v4] = m4.x; m[4 * v4 + 1] = m4.y; m[4 * v4 + 2] = m4.z; m[4 * v4 + 3] = m4.w;
        }
#pragma unroll
        for (int u = 0; u < 16; ++u) put(a_base, TC_ATILE, oc + u, m[u]);
        warp_colsum16(m, lane);
        if ((lane & 1) == 0) bsum[q * dout + oc + warp_col16(lane)] = m[0];
      }
      for (int kc = half * (din / 2); kc < (half + 1) * (din / 2); kc += 4) {
        float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rowok) z4 = *reinterpret_cast<const float4*>(Zrow + kc);
        const float4 s4 = __ldg(reinterpret_cast<const float4*>(p.nw + kc)), t4 = __ldg(reinterpret_cast<const float4*>(p.nb + kc));
        put(b_base, b_tile, kc + 0, rowok ? z4.x * rinv * s4.x + t4.x : 0.f);
        put(b_base, b_tile, kc + 1, rowok ? z4.y * rinv * s4.y + t4.y : 0.f);
        put(b_base, b_tile, kc + 2, rowok ? z4.z * rinv * s4.z + t4.z : 0.f);
        put(b_base, b_tile, kc + 3, rowok ? z4.w * rinv * s4.w + t4.w : 0.f);
      }
      fence_proxy_async();
      mbar_arrive(wg_full(st));
    }
    const float vv = (p.po.vec && rowok) ? p.po.vec[(size_t)b * p.po.vec_stride + gi] : 0.f;
    float* Zbrow = p.Zbar + ((size_t)b * n + (rowok ? gi : 0)) * din;
    // pass 2: Zbar, its producer outputs, and the per-column sums (g_nw, g_nb, column sums of Zbar)
    float zmax = 0.f;   // max |Zbar| of this thread's entries (block exponent of the fp16x2 operand format)
    for (int cc = 0; cc < cols_per_half; cc += 16) {
      const int col = half * cols_per_half + cc;
      uint32_t r[16];
      tmem_ld16(trow + (uint32_t)col, r);
      tmem_wait_ld();
      float zb[16], gw[16], gb[16], s1[16];
#pragma unroll
      for (int v4 = 0; v4 < 4; ++v4) {
        float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rowok) z4 = *reinterpret_cast<const float4*>(Zrow + col + 4 * v4);
        const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.nw + col + 4 * v4));
        const float zz[4] = {z4.x, z4.y, z4.z, z4.w}, ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = 4 * v4 + u;
          const float nbar = rowok ? __uint_as_float(r[e]) : 0.f;
          float v = rinv * ww[u] * nbar - zz[u] * coef;
          if (!rowok || (p.relu_mask && !(zz[u] > 0.f))) v = 0.f;
          zb[e] = v;
          gw[e] = nbar * zz[u] * rinv;
          gb[e] = nbar;
          s1[e] = vv * v;
        }
      }
      if (rowok) {
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4)
          *reinterpret_cast<float4*>(Zbrow + col + 4 * v4) = make_float4(zb[4 * v4], zb[4 * v4 + 1], zb[4 * v4 + 2], zb[4 * v4 + 3]);
      }
      if (p.Nout != nullptr && rowok) {
        float* Nrow = p.Nout + ((size_t)b * n + gi) * din;
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
          const float4 z4 = *reinterpret_cast<const float4*>(Zrow + col + 4 * v4);
          const float4 s4 = __ldg(reinterpret_cast<const float4*>(p.nw + col + 4 * v4)), t4 = __ldg(reinterpret_cast<const float4*>(p.nb + col + 4 * v4));
          *reinterpret_cast<float4*>(Nrow + col + 4 * v4) =
              make_float4(z4.x * rinv * s4.x + t4.x, z4.y * rinv * s4.y + t4.y, z4.z * rinv * s4.z + t4.z, z4.w * rinv * s4.w + t4.w);
        }
      }
      if (p.po.Thi != nullptr && gi < p.po.rows_pad && p.po.t16 != PEG_FMT_FP16X2) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
          store_vt(p.po, ((size_t)b * din + col + u) * p.po.npad + p.po.col0 + gi, zb[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 16; ++u) zmax = fmaxf(zmax, fabsf(zb[u]));
      warp_colsum16(gw, lane);
      warp_colsum16(gb, lane);
      warp_colsum16(zb, lane);
      warp_colsum16(s1, lane);
      if ((lane & 1) == 0) {
        const int c = col + warp_col16(lane);
        csum[(q * 4 + 0) * nd + c] = gw[0];
        csum[(q * 4 + 1) * nd + c] = gb[0];
        csum[(q * 4 + 2) * nd + c] = zb[0];
        csum[(q * 4 + 3) * nd + c] = s1[0];
      }
    }
    if (p.po.Thi != nullptr && p.po.t16 == PEG_FMT_FP16X2) {
      // pass 3 (fp16x2 operand format): the block maximum is known only now -> V^T = Zbar * 2^e from a third walk over the accumulators
      zmax = warp_max(zmax);
      if (lane == 0) bmax_s[warp] = zmax;
      asm volatile("bar.sync 1, 256;" ::: "memory");
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) zmax = fmaxf(zmax, bmax_s[w8]);
      const int e = block_exponent(zmax);
      const float vscale = exp2_int(e);
      if (tid == 0) p.po.vexp[(size_t)b * p.po.vexp_stride + p.po.blk0 + rb] = e;
      if (gi < p.po.rows_pad) {
        for (int cc = 0; cc < cols_per_half; cc += 16) {
          const int col = half * cols_per_half + cc;
          uint32_t r[16];
          tmem_ld16(trow + (uint32_t)col, r);
          tmem_wait_ld();
#pragma unroll
          for (int v4 = 0; v4 < 4; ++v4) {
            float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rowok) z4 = *reinterpret_cast<const float4*>(Zrow + col + 4 * v4);
            const float4 w4 = __ldg(reinterpret_cast<const float4*>(p.nw + col + 4 * v4));
            const float zz[4] = {z4.x, z4.y, z4.z, z4.w}, ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float nbar = rowok ? __uint_as_float(r[4 * v4 + u]) : 0.f;
              float v = rinv * ww[u] * nbar - zz[u] * coef;   // the same expression as pass 2: bit-identical Zbar
              if (!rowok || (p.relu_mask && !(zz[u] > 0.f))) v = 0.f;
              store_vt_f16(p.po, ((size_t)b * din + col + 4 * v4 + u) * p.po.npad + p.po.col0 + gi, v * vscale);
            }
          }
        }
      }
    }
    if (wg) {   // TMEM lane = output o (dout == 128), columns = inputs: add the CTA's Wbar partial
      mbar_wait(wg_bar, 0u);
      tc_fence_after();
      float* grow = p.gW + (size_t)row * din;
      for (int cc = 0; cc < cols_per_half; cc += 16) {
        const int col = half * cols_per_half + cc;
        uint32_t r[16];
        tmem_ld16(trow + (uint32_t)(p.wg_col + col), r);
        tmem_wait_ld();
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4)
          atomicAdd(reinterpret_cast<float4*>(grow + col + 4 * v4),
                    make_float4(__uint_as_float(r[4 * v4]), __uint_as_float(r[4 * v4 + 1]), __uint_as_float(r[4 * v4 + 2]), __uint_as_float(r[4 * v4 + 3])));
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (wg && tid < dout) atomicAdd(p.gb + tid, bsum[tid] + bsum[dout + tid] + bsum[2 * dout + tid] + bsum[3 * dout + tid]);
  if (tid < nd) {
    float t[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int k = 0; k < 4; ++k) t[k] += csum[(q * 4 + k) * nd + tid];
    atomicAdd(p.g_nw + tid, t[0]);
    atomicAdd(p.g_nb + tid, t[1]);
    if (p.po.cb != nullptr) {
      float* part = p.po.partial + (((size_t)b * gridDim.x + rb) * 2) * din;
      part[tid] = t[2];
      part[din + tid] = t[3];
    }
  }
  if (p.po.cb != nullptr)
    finalize_colsums(p.po, b, gridDim.x, din, 0, nd, p.po.tickets + (size_t)b, &is_last);
  if (warp == 9) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols));
  }
}

bool tc_linear_bwd_supported(int din, int dout) {
  return din % 32 == 0 && din >= 32 && din <= 256 && dout % 32 == 0 && dout >= 32 && get_encode() != nullptr;
}

static int lb_stages(int din, int dout, int nsplit) {
  const int sp = nsplit == 3 ? 2 : 1;
  const int stage_bytes = sp * TC_ATILE + sp * din * TC_BK * 4;
  int stages = (200 * 1024) / stage_bytes;
  const int nchunks = dout / 32;
  stages = stages > nchunks ? nchunks : stages;
  return stages > 4 ? 4 : stages;
}

// the weight-gradient MMA takes all dout outputs as its 128 rows, and its second accumulator (din columns) must fit next to the first
bool tc_linear_bwd_fuses_weight_grad(const PegDims& dm, int din, int dout) {
  return tc_linear_bwd_supported(din, dout) && dout == TC_BM && 2 * tmem_cols_pow2(din) <= 512 &&
         lb_stages(din, dout, (dm.flags & PEG_FLAG_TF32_FAST) ? 1 : 3) >= 2;
}

int tc_linear_bwd(cudaStream_t st, const PegDims& dm, const TcLinear& w, int layer, const float* Mbar, const float* Z,
                  const float* nw, const float* nb, int din, int dout, int relu_mask, float* Zbar, float* g_nw, float* g_nb,
                  float* gW, float* gb, float* Nout, const ProducerOut& po) {
  if (!w.ready) return PEG_ERR_WORKSPACE;
  if (gW != nullptr && !tc_linear_bwd_fuses_weight_grad(dm, din, dout)) return PEG_ERR_UNSUPPORTED;
  LbParams p;
  memset(&p, 0, sizeof(p));
  p.Mbar = Mbar; p.Z = Z; p.nw = nw; p.nb = nb; p.Zbar = Zbar; p.g_nw = g_nw; p.g_nb = g_nb; p.po = po;
  p.gW = gW; p.gb = gb; p.Nout = gW != nullptr ? nullptr : Nout;
  p.n = dm.n; p.din = din; p.dout = dout; p.relu_mask = relu_mask;
  p.nsplit = (dm.flags & PEG_FLAG_TF32_FAST) ? 1 : 3;
  const int sp = p.nsplit == 3 ? 2 : 1;
  const int stage_bytes = sp * TC_ATILE + sp * din * TC_BK * 4;
  const int stages = lb_stages(din, dout, p.nsplit);
  if (stages < 1) return PEG_ERR_UNSUPPORTED;
  p.stages = stages;
  p.wg_col = tmem_cols_pow2(din);
  p.tmem_cols = gW != nullptr ? 2 * p.wg_col : p.wg_col;
  const size_t sums = (size_t)(16 * din + (gW != nullptr ? 4 * dout : 0)) * 4;
  const size_t smem = (size_t)stages * stage_bytes + sums + 1024 + 8 * (5 * stages + 3) + 64;
  const CUtensorMap* mhi = nullptr;
  const CUtensorMap* mlo = nullptr;
  PEG_TRY(get_maps(w.Wt_hi[layer], w.Wt_lo[layer], (uint64_t)dout, (uint64_t)din, din, &mhi, &mlo));
  static std::atomic<unsigned> done{0u};
  PEG_TRY(optin_smem(k_tc_linear_bwd, done));
  dim3 grid((dm.n + 127) / 128, 1, dm.B);
  k_tc_linear_bwd<<<grid, NL_THREADS, smem, st>>>(*mhi, *mlo, p);
  if (cudaPeekAtLastError() != cudaSuccess) {
    const cudaError_t e = cudaGetLastError();
    fprintf(stderr, "pegncde: k_tc_linear_bwd launch failed (%s): grid %u x %u, smem %zu, din %d, stages %d\n", cudaGetErrorString(e),
            grid.x, grid.z, smem, din, stages);
    set_last_cuda((int)e);
    return PEG_ERR_CUDA;
  }
  return PEG_OK;
}


// ==========================================================================================
// Weight / bias gradient of the Linear on tcgen05 (3xTF32):  Wbar[o][k] += sum_r Mbar[r][o] N[r][k],  bbar[o] += sum_r Mbar[r][o]
// over all B*n rows.  The reduction runs along the rows, so BOTH operands are needed row(K)-major: 8 loader warps read
// 4x4 micro tiles (4 rows x 4 columns, 4 LDG.128) and store them transposed (16-byte chunk = 4 consecutive rows of one
// column) into the swizzled K-major tiles -- lanes of a store phase hold 8 different row quads of the same column, which
// makes the transposed stores bank-conflict-free.  M = 128 outputs o, N = din, K = 32 rows per chunk, one accumulator in
// TMEM per CTA; every CTA owns a slice of the rows and adds its 128 x din partial with vector atomics.
// grid (row slices, dout/128), block 288
// ==========================================================================================
constexpr int WG_THREADS = 288;

struct WgParams {
  const float* Mbar;   // [rows, dout]
  const float* N;      // [rows, din]
  float* gW;           // [dout, din]
  float* gb;           // [dout]
  size_t rows;
  int rows_per_slice;  // multiple of 32
  int din, dout, stages, tmem_cols, nsplit;
};

__global__ void __launch_bounds__(WG_THREADS, 1) k_tc_weight_grad(const WgParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int din = p.din, dout = p.dout, S = p.stages;
  const bool split = p.nsplit == 3;
  const int o0 = blockIdx.y * 128;
  const size_t r_begin = (size_t)blockIdx.x * p.rows_per_slice;
  const size_t r_end = min(p.rows, r_begin + (size_t)p.rows_per_slice);
  const int nchunks = (int)((r_end - r_begin + 31) / 32);

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int a_bytes = (split ? 2 : 1) * TC_ATILE;
  const int b_tile = din * TC_BK * 4;
  const int b_bytes = (split ? 2 : 1) * b_tile;
  const int stage_bytes = a_bytes + b_bytes;
  const uint32_t bar_base = smem_base + S * stage_bytes;
  auto full = [&](int s) { return bar_base + 8u * s; };
  auto empty = [&](int s) { return bar_base + 8u * (S + s); };
  const uint32_t accum_bar = bar_base + 8u * (2 * S);
  const uint32_t tmem_slot = accum_bar + 8u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(full(s), 256); mbar_init(empty(s), 1); }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  if (warp < 8) {
    // micro tile of this thread: row quad rq (rows 4 rq .. 4 rq + 3 of the chunk), column quad cq (+ 32 per pass for N)
    const int rq = lane & 7, cq = 4 * warp + (lane >> 3);
    const int npass = (din + 127) / 128;
    float bs[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < nchunks; ++j) {
      const size_t rbase = r_begin + (size_t)j * 32 + 4 * rq;
      float4 a[4], bq[2][4];
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const size_t row = rbase + m;
        const bool ok = row < r_end;
        a[m] = (ok && o0 + 4 * cq < dout) ? __ldg(reinterpret_cast<const float4*>(p.Mbar + row * dout + o0 + 4 * cq)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int ps = 0; ps < 2; ++ps) {
          const int c = 4 * (cq + 32 * ps);
          bq[ps][m] = (ok && ps < npass && c < din) ? __ldg(reinterpret_cast<const float4*>(p.N + row * din + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      const int st = j % S;
      mbar_wait(empty(st), ((uint32_t)(j / S) & 1u) ^ 1u);
      const uint32_t a_base = smem_base + st * stage_bytes, b_base = a_base + a_bytes;
      auto put = [&](uint32_t hi_tile, uint32_t lo_off, int row, float x0, float x1, float x2, float x3) {
        const uint32_t off = (uint32_t)(row >> 3) * 1024u + (uint32_t)(row & 7) * 128u + (uint32_t)((rq ^ (row & 7)) << 4);
        const float h0 = tf32_rna(x0), h1 = tf32_rna(x1), h2 = tf32_rna(x2), h3 = tf32_rna(x3);
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(hi_tile + off), "f"(h0), "f"(h1), "f"(h2), "f"(h3) : "memory");
        if (split)
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(hi_tile + lo_off + off), "f"(x0 - h0), "f"(x1 - h1), "f"(x2 - h2),
                       "f"(x3 - h3) : "memory");
      };
      // A' = Mbar^T: operand row = output o = 4 cq + e, chunk rq = rows 4 rq .. 4 rq + 3
      put(a_base, TC_ATILE, 4 * cq + 0, a[0].x, a[1].x, a[2].x, a[3].x);
      put(a_base, TC_ATILE, 4 * cq + 1, a[0].y, a[1].y, a[2].y, a[3].y);
      put(a_base, TC_ATILE, 4 * cq + 2, a[0].z, a[1].z, a[2].z, a[3].z);
      put(a_base, TC_ATILE, 4 * cq + 3, a[0].w, a[1].w, a[2].w, a[3].w);
#pragma unroll
      for (int m = 0; m < 4; ++m) { bs[0] += a[m].x; bs[1] += a[m].y; bs[2] += a[m].z; bs[3] += a[m].w; }
      // B' = N^T: operand row = input k = 4 (cq + 32 ps) + e
#pragma unroll
      for (int ps = 0; ps < 2; ++ps) {
        const int r4 = 4 * (cq + 32 * ps);
        if (ps < npass && r4 < din) {
          put(b_base, b_tile, r4 + 0, bq[ps][0].x, bq[ps][1].x, bq[ps][2].x, bq[ps][3].x);
          put(b_base, b_tile, r4 + 1, bq[ps][0].y, bq[ps][1].y, bq[ps][2].y, bq[ps][3].y);
          put(b_base, b_tile, r4 + 2, bq[ps][0].z, bq[ps][1].z, bq[ps][2].z, bq[ps][3].z);
          put(b_base, b_tile, r4 + 3, bq[ps][0].w, bq[ps][1].w, bq[ps][2].w, bq[ps][3].w);
        }
      }
      fence_proxy_async();
      mbar_arrive(full(st));
    }
    // bias gradient: the 8 row-quad lanes (lane & 7) of one column quad
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float v = bs[e];
      v += __shfl_xor_sync(0xffffffffu, v, 1);
      v += __shfl_xor_sync(0xffffffffu, v, 2);
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      if (rq == 0 && p.gb != nullptr && o0 + 4 * cq < dout) atomicAdd(p.gb + o0 + 4 * cq + e, v);
    }
  } else {
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(din >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
      for (int j = 0; j < nchunks; ++j) {
        const int st = j % S;
        mbar_wait(full(st), (uint32_t)(j / S) & 1u);
        tc_fence_after();
        const uint32_t ahi = smem_base + st * stage_bytes, alo = ahi + TC_ATILE;
        const uint32_t bhi = ahi + a_bytes, blo = bhi + b_tile;
#pragma unroll
        for (int k8 = 0; k8 < TC_BK / 8; ++k8) {
          const uint64_t dah = make_desc_sw128(ahi + k8 * 32), dbh = make_desc_sw128(bhi + k8 * 32);
          umma_tf32(tmem_base, dah, dbh, idesc, (j > 0 || k8 > 0) ? 1u : 0u);
          if (split) {
            umma_tf32(tmem_base, make_desc_sw128(alo + k8 * 32), dbh, idesc, 1u);
            umma_tf32(tmem_base, dah, make_desc_sw128(blo + k8 * 32), idesc, 1u);
          }
        }
        umma_commit(empty(st));
      }
      umma_commit(accum_bar);
    }
  }

  if (warp < 8 && nchunks > 0) {
    mbar_wait(accum_bar, 0u);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int o = o0 + q * 32 + lane;
    float* grow = p.gW + (size_t)(o < dout ? o : 0) * din;
    const int cols_per_half = din / 2;
    for (int cc = 0; cc < cols_per_half; cc += 16) {
      const int col = half * cols_per_half + cc;
      uint32_t r[16];
      tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col, r);
      tmem_wait_ld();
      if (o >= dout) continue;   // rows of the last 128-row tile beyond dout (zero operand rows)
#pragma unroll
      for (int v4 = 0; v4 < 4; ++v4)
        atomicAdd(reinterpret_cast<float4*>(grow + col + 4 * v4),
                  make_float4(__uint_as_float(r[4 * v4]), __uint_as_float(r[4 * v4 + 1]), __uint_as_float(r[4 * v4 + 2]), __uint_as_float(r[4 * v4 + 3])));
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 8) {
    __syncwarp();
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols));
  }
}

int tc_weight_grad(cudaStream_t st, const PegDims& dm, const float* Mbar, const float* N, size_t rows, int din, int dout,
                   float* gW, float* gb) {
  WgParams p;
  memset(&p, 0, sizeof(p));
  p.Mbar = Mbar; p.N = N; p.gW = gW; p.gb = gb; p.rows = rows; p.din = din; p.dout = dout;
  p.nsplit = (dm.flags & PEG_FLAG_TF32_FAST) ? 1 : 3;
  const int sp = p.nsplit == 3 ? 2 : 1;
  const int stage_bytes = sp * TC_ATILE + sp * din * TC_BK * 4;
  int stages = (200 * 1024) / stage_bytes;
  stages = stages > 4 ? 4 : stages;
  if (stages < 1) return PEG_ERR_UNSUPPORTED;
  p.stages = stages;
  p.tmem_cols = tmem_cols_pow2(din);
  // row slices: about half a wave of CTAs (each adds a 128 x din partial with atomics, so fewer, fatter slices are cheaper)
  const int otiles = (dout + 127) / 128;
  int slices = 74 / otiles;
  slices = slices < 1 ? 1 : slices;
  size_t rps = (rows + slices - 1) / slices;
  rps = (rps + 31) / 32 * 32;
  rps = rps < 64 ? 64 : rps;
  p.rows_per_slice = (int)rps;
  const unsigned nsl = (unsigned)((rows + rps - 1) / rps);
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 8 * (2 * stages + 2) + 64;
  static std::atomic<unsigned> done{0u};
  PEG_TRY(optin_smem(k_tc_weight_grad, done));
  k_tc_weight_grad<<<dim3(nsl, otiles), WG_THREADS, smem, st>>>(p);
  if (cudaPeekAtLastError() != cudaSuccess) {
    const cudaError_t e = cudaGetLastError();
    fprintf(stderr, "pegncde: k_tc_weight_grad launch failed (%s): grid %u x %d, smem %zu\n", cudaGetErrorString(e), nsl, otiles, smem);
    set_last_cuda((int)e);
    return PEG_ERR_CUDA;
  }
  return PEG_OK;
}

}  // namespace peg
