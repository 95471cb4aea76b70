// Small-graph path: ONE kernel per vector-field evaluation and ONE per VJP, a thread-block cluster per graph.
//
// Below a few hundred nodes the per-operator pipeline of pegncde.cu (stage prep -> RMSNorm/Linear -> column sums -> contraction ->
// ... ~15 launches per evaluation, ~40 per VJP) is bound by the dependent-launch latency of kernels that each do microseconds of
// work: England (n=129) and SIR (n=100, B=50) both sat at ~2 ms per Tsit5 step whatever the arithmetic.  Here a cluster of C CTAs
// owns one graph for the whole evaluation: the stage scalars and O(n) vectors live in shared memory, the layer stack runs as
// phases separated by cluster barriers (hardware barrier, ~0.5 us) instead of kernel boundaries, intermediate activations go
// through L2-resident workspace, the operand V of a contraction item sits in shared memory for all its rows (so the column sums
// 1^T V, vec^T V are local and deterministic) and the cubic-coefficient planes stream with register prefetch.
//   phase A  (per layer)  RMSNorm -> Linear tiles 64 x 64                     (layers.py:45-46)
//   phase B  (per layer)  matrix-free equivariant contraction items 64 x 64   (layers.py:114-160), fp32 FFMA -- exact
//   wrapper               dy[n,m] = sum_j out[n, m 2e + j] X'(t)[n, j]        (cde_wrapper_vector_field.py:21-25)
// and the mirrored adjoint phases (A' recompute, B' four products + fusion-scalar gradients, C linear/norm backward + weight
// gradients).  Work items of a phase are dealt to the cluster's CTAs in contiguous ranges.  Undirected fusion layer only.
#pragma once
#include <cooperative_groups.h>
#include "peg_kernels.cuh"

namespace peg {
namespace cg = cooperative_groups;

constexpr int SG_THREADS = 256;
constexpr int SG_RB = 64, SG_WB = 64, SG_KC = 16, SG_LD = SG_RB + 4;
constexpr int SG_SCRATCH = 5632;     // floats: max over phases (linear backward: 32x36 + 32x128 + 2x128)
constexpr int SG_MAX_N = 512, SG_MAX_DIN = 128;
constexpr int SG_RES_N = 128;        // up to this many nodes the interpolated adjacency of the stage stays in shared memory

struct SmallArgs {
  PegControl ctl;
  const float* params;
  Model model;
  int B, n, e, T, L, h, npad, C;
  float t;
  StageScalars* sc;          // [B] (kept for k_xcoef_accum)
  // workspace, per graph [n][dmax] / [n][h]
  float* M; float* Za; float* Zb; float* OL; float* Obar; float* Mbar; float* N;
  // forward
  const float* yin; float* dy; float* save[PEG_MAX_LAYERS]; int nlayers;
  // vjp
  const float* zin[PEG_MAX_LAYERS]; const float* kbar; float* ybar; float* g_params; float* g_xd;
};

struct SmallSm {
  float* vec;    // [(3L+1)][nv]: v_l, r_l, c_l per layer, then tg
  float* rows;   // [4][nv]: rowsum(A_s), rowsum(A'_s), diag(A_s), diag(A'_s)
  float* Vs;     // [n16][64]
  float* S;      // SG_SCRATCH floats
  float* cb0; float* cb1; float* sM;   // [64] each
  float* rinv; float* cvec;            // [64] each
  float* red;    // [160]
  int nv;        // row pitch of vec / rows (n rounded up to 4)
  float* As;     // resident mode (n <= SG_RES_N): A_s and A'_s of the stage, [n16][P] each, P = n16 + 1 (both orientations
  float* Ad;     //   are read from it: the odd pitch keeps row and column walks off the same banks); nullptr otherwise
  int P;
};

__host__ __device__ inline size_t small_smem_floats(int n, int L) {
  const size_t nv = (size_t)(n + 3) / 4 * 4, n16 = (size_t)(n + 15) / 16 * 16;
  const size_t res = n <= SG_RES_N ? 2 * n16 * (n16 + 1) + 4 : 0;
  return (size_t)(3 * L + 1) * nv + 4 * nv + n16 * SG_WB + SG_SCRATCH + 5 * 64 + 160 + res;
}

__device__ __forceinline__ SmallSm small_carve(float* base, int n, int L) {
  SmallSm s;
  s.nv = (n + 3) / 4 * 4;
  const int n16 = (n + 15) / 16 * 16;
  s.vec = base;  base += (size_t)(3 * L + 1) * s.nv;
  s.rows = base; base += 4 * s.nv;
  s.Vs = base;   base += (size_t)n16 * SG_WB;
  s.S = base;    base += SG_SCRATCH;
  s.cb0 = base; s.cb1 = base + 64; s.sM = base + 128; s.rinv = base + 192; s.cvec = base + 256; base += 320;
  s.red = base;  base += 160;
  if (n <= SG_RES_N) {
    s.P = n16 + 1;
    s.As = base;
    s.Ad = base + (size_t)n16 * s.P;
  } else {
    s.P = 0;
    s.As = s.Ad = nullptr;
  }
  return s;
}

// contiguous range of `Q` work items for CTA `rank` of `C`
__device__ __forceinline__ void small_range(int Q, int rank, int C, int& lo, int& hi) {
  lo = (int)(((long long)rank * Q) / C);
  hi = (int)(((long long)(rank + 1) * Q) / C);
}

// per-stage scalars and O(n) vectors of graph b (k_stage_prep, undirected branch), into shared memory
__device__ void small_prep(const SmallArgs& a, int b, int rank, const SmallSm& sm, StageScalars* S) {
  const int tid = threadIdx.x, n = a.n, L = a.L, Tm1 = a.T - 1, nv = sm.nv;
  const float* ts = a.ctl.ts + (size_t)b * a.T;
  const float tq = a.t;
  float cnt = 0.f;
  for (int i = tid; i < a.T; i += SG_THREADS) cnt += (ts[i] < tq) ? 1.f : 0.f;
  cnt = block_sum(cnt, sm.red);
  int iv = (int)(cnt + 0.5f) - 1;
  iv = max(0, min(iv, a.T - 2));
  const float s = tq - ts[iv];
  const float wA[4] = {1.f, s, s * s, s * s * s};
  const float wD[4] = {0.f, 1.f, 2.f * s, 3.f * s * s};
  const size_t slab = (size_t)b * Tm1 + iv;
  const float* tot = a.ctl.adj_total + slab * 4;
  const float totA = wA[0] * tot[0] + wA[1] * tot[1] + wA[2] * tot[2] + wA[3] * tot[3];
  const float totD = wD[1] * tot[1] + wD[2] * tot[2] + wD[3] * tot[3];
  const float inv_n = 1.f / (float)n, inv_n2 = inv_n * inv_n;
  if (tid == 0) {
    S->interval = iv;
    S->s = s;
    for (int p = 0; p < 4; ++p) { S->wA[p] = wA[p]; S->wD[p] = wD[p]; S->amax[p] = 0.f; }
    S->totA = totA;
    S->totD = totD;
    for (int l = 0; l < PEG_MAX_LAYERS; ++l) S->kappa[l] = 0.f;
    for (int l = 0; l < L; ++l) {
      const float* f = a.params + a.model.layer[l].fus_off;
      S->kappa[l] = (f[12] + f[13]) * totA * inv_n2;
    }
    S->pad[0] = S->pad[1] = 0.f;
    if (rank == 0) a.sc[b] = *S;
  }
  const float* rs = a.ctl.adj_rowsum + slab * 4 * n;
  const float* dg = a.ctl.adj_diag + slab * 4 * n;
  const float* tc = a.ctl.tch_coef + slab * 3 * n;
  for (int i = tid; i < n; i += SG_THREADS) {
    const float rA = wA[0] * rs[i] + wA[1] * rs[n + i] + wA[2] * rs[2 * n + i] + wA[3] * rs[3 * n + i];
    const float rD = wD[1] * rs[n + i] + wD[2] * rs[2 * n + i] + wD[3] * rs[3 * n + i];
    const float dA = wA[0] * dg[i] + wA[1] * dg[n + i] + wA[2] * dg[2 * n + i] + wA[3] * dg[3 * n + i];
    const float dD = wD[1] * dg[n + i] + wD[2] * dg[2 * n + i] + wD[3] * dg[3 * n + i];
    sm.rows[i] = rA; sm.rows[nv + i] = rD; sm.rows[2 * nv + i] = dA; sm.rows[3 * nv + i] = dD;
    for (int l = 0; l < L; ++l) {
      const float* f = a.params + a.model.layer[l].fus_off;
      sm.vec[(3 * l + 0) * nv + i] = f[4] * dA + f[5] * dD + (f[10] * rA + f[11] * rD) * inv_n + (f[14] * totA + f[15] * totD) * inv_n2;
      sm.vec[(3 * l + 1) * nv + i] = (f[6] * rA + f[7] * rD) * inv_n;
      sm.vec[(3 * l + 2) * nv + i] = (f[8] * rA + f[9] * rD) * inv_n;
    }
    sm.vec[3 * L * nv + i] = tc[i] + s * (2.f * tc[n + i] + 3.f * s * tc[2 * n + i]);
  }
  __syncthreads();
}

// planes of graph b for the stage's cubic piece; STAT (static control, PegControl.adj_static): the one plane of graph b, which
// serves every piece -- planes b, c, d are exact zeros, so the kernels below compute what the dense control of [A] * T computes
template <bool STAT>
__device__ __forceinline__ const float* small_planes(const SmallArgs& a, int b, int interval) {
  if (STAT) return a.ctl.adj_static + (size_t)b * a.npad * a.npad;
  return a.ctl.adj_coef + ((size_t)b * (a.T - 1) + interval) * 4 * (size_t)a.npad * a.npad;
}

// resident mode: A_s = sum_p wA[p] plane_p and A'_s = sum_p wD[p] plane_p of the stage's cubic piece, once per kernel.  The tiled
// planes are read in storage order (a warp's 128-bit loads are 512 contiguous bytes); thread (g, m, lane) of a 32x32 tile holds
// row 4 rq + m, columns 4 cq .. 4 cq + 3 of all four planes (peg_tile_off).  STAT: the plane is copied (A_s = a, A'_s = 0).
template <bool STAT>
__device__ void small_build_A(const SmallArgs& a, int b, const StageScalars* S, const SmallSm& sm) {
  const int tid = threadIdx.x, n16 = (a.n + 15) / 16 * 16, nt = a.npad >> 5, tiles = (n16 + 31) >> 5, P = sm.P;
  const float* Pl = small_planes<STAT>(a, b, S->interval);
  const int g = tid >> 7, m = (tid >> 5) & 3, lane = tid & 31;
  const int s_ = (g << 2) | (lane >> 3), cq = lane & 7, rq = (s_ + cq) & 7;
  const int r = rq * 4 + m, c = cq * 4;
  const float wA0 = S->wA[0], wA1 = S->wA[1], wA2 = S->wA[2], wA3 = S->wA[3], wD1 = S->wD[1], wD2 = S->wD[2], wD3 = S->wD[3];
#pragma unroll 2
  for (int t = 0; t < tiles * tiles; ++t) {
    const int rt = t / tiles, ct = t - rt * tiles;
    if (STAT) {
      const float4 p0 = __ldg(reinterpret_cast<const float4*>(Pl + ((size_t)rt * nt + ct) * 1024 + (size_t)(g * 4 + m) * 128 + lane * 4));
      const int gi = rt * 32 + r, gk = ct * 32 + c;
      if (gi < n16 && gk < n16) {
        const float e0[4] = {p0.x, p0.y, p0.z, p0.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          sm.As[gi * P + gk + j] = e0[j];
          sm.Ad[gi * P + gk + j] = 0.f;
        }
      }
      continue;
    }
    const float* tb = Pl + ((size_t)rt * nt + ct) * 4096 + (size_t)(g * 16 + m) * 128 + lane * 4;
    const float4 p0 = __ldg(reinterpret_cast<const float4*>(tb));
    const float4 p1 = __ldg(reinterpret_cast<const float4*>(tb + 512));
    const float4 p2 = __ldg(reinterpret_cast<const float4*>(tb + 1024));
    const float4 p3 = __ldg(reinterpret_cast<const float4*>(tb + 1536));
    const int gi = rt * 32 + r, gk = ct * 32 + c;
    if (gi < n16 && gk < n16) {
      const float e0[4] = {p0.x, p0.y, p0.z, p0.w}, e1[4] = {p1.x, p1.y, p1.z, p1.w};
      const float e2[4] = {p2.x, p2.y, p2.z, p2.w}, e3[4] = {p3.x, p3.y, p3.z, p3.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        sm.As[gi * P + gk + j] = wA0 * e0[j] + wA1 * e1[j] + wA2 * e2[j] + wA3 * e3[j];
        sm.Ad[gi * P + gk + j] = wD1 * e1[j] + wD2 * e2[j] + wD3 * e3[j];
      }
    }
  }
  __syncthreads();
}

// X'(t)[i, j] of the node-signal control on the stage's cubic piece
__device__ __forceinline__ float small_xd(const SmallArgs& a, int b, const StageScalars* S, int i, int j) {
  const int e2 = 2 * a.e;
  const size_t per = (size_t)a.n * e2;
  const float* xc = a.ctl.x_coef + ((size_t)b * (a.T - 1) + S->interval) * 3 * per + (size_t)i * e2 + j;
  const float s = S->s;
  return xc[0] + s * (2.f * xc[per] + 3.f * s * xc[2 * per]);
}

// ---- phase A: one 64 x 64 tile of M = RMSNorm(Z) W^T + b (k_norm_linear with BM = 64); optionally the normalised input ----
__device__ void small_linear_tile(const float* Z, int n, int din, int dout, const float* __restrict__ W,
                                  const float* __restrict__ bias, const float* __restrict__ nw, const float* __restrict__ nb,
                                  int row0, int col0, float* M, float* Nout, const SmallSm& sm) {
  float (*zt)[SG_LD] = reinterpret_cast<float (*)[SG_LD]>(sm.S);
  float (*wt)[SG_LD] = reinterpret_cast<float (*)[SG_LD]>(sm.S + 32 * SG_LD);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float sumsq[2] = {0.f, 0.f}, cpart[2] = {0.f, 0.f};
  for (int k0 = 0; k0 < din; k0 += 32) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int idx = tid + SG_THREADS * u, r = idx >> 3, kq = (idx & 7) * 4, k = k0 + kq;
      float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f), w4 = z4;
      if (row0 + r < n && k < din) z4 = __ldcg(reinterpret_cast<const float4*>(Z + (size_t)(row0 + r) * din + k));
      if (col0 + r < dout && k < din) w4 = __ldg(reinterpret_cast<const float4*>(W + (size_t)(col0 + r) * din + k));
      const float zz[4] = {z4.x, z4.y, z4.z, z4.w}, ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        sumsq[u] = fmaf(zz[e], zz[e], sumsq[u]);
        zt[kq + e][r] = zz[e];
        const float sw = (k + e) < din ? nw[k + e] : 0.f, sb = (k + e) < din ? nb[k + e] : 0.f;
        cpart[u] = fmaf(sb, ww[e], cpart[u]);
        wt[kq + e][r] = ww[e] * sw;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 32; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&zt[k][4 * ty]);
      const float4 b4 = *reinterpret_cast<const float4*>(&wt[k][4 * tx]);
      const float aa[4] = {a4.x, a4.y, a4.z, a4.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      sumsq[u] += __shfl_xor_sync(0xffffffffu, sumsq[u], o);
      cpart[u] += __shfl_xor_sync(0xffffffffu, cpart[u], o);
    }
    if ((tid & 7) == 0) {
      const int r = (tid + SG_THREADS * u) >> 3;
      sm.rinv[r] = rsqrtf(sumsq[u] / (float)din + 1e-5f);
      sm.cvec[r] = cpart[u] + ((col0 + r < dout) ? bias[col0 + r] : 0.f);
    }
  }
  __syncthreads();
  if (Nout != nullptr && col0 == 0) {
    const int q4 = din >> 2;
    for (int idx = tid; idx < SG_RB * q4; idx += SG_THREADS) {
      const int r = idx / q4, k = (idx - r * q4) * 4, node = row0 + r;
      if (node >= n) continue;
      const float4 z4 = __ldcg(reinterpret_cast<const float4*>(Z + (size_t)node * din + k));
      const float4 s4 = *reinterpret_cast<const float4*>(nw + k), t4 = *reinterpret_cast<const float4*>(nb + k);
      const float ri = sm.rinv[r];
      *reinterpret_cast<float4*>(Nout + (size_t)node * din + k) =
          make_float4(z4.x * ri * s4.x + t4.x, z4.y * ri * s4.y + t4.y, z4.z * ri * s4.z + t4.z, z4.w * ri * s4.w + t4.w);
    }
  }
  const int oc = col0 + 4 * tx;
  if (oc < dout) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int node = row0 + 4 * ty + i;
      if (node >= n) continue;
      const float ri = sm.rinv[4 * ty + i];
      *reinterpret_cast<float4*>(M + (size_t)node * dout + oc) =
          make_float4(fmaf(ri, acc[i][0], sm.cvec[4 * tx + 0]), fmaf(ri, acc[i][1], sm.cvec[4 * tx + 1]),
                      fmaf(ri, acc[i][2], sm.cvec[4 * tx + 2]), fmaf(ri, acc[i][3], sm.cvec[4 * tx + 3]));
    }
  }
  __syncthreads();
}

// ---- operand V of the contraction items of one column block: all rows into shared memory + its column sums (fixed order) ----
// cb0[c] = sum_k V[k,c], cb1[c] = sum_k vecw[k] V[k,c]; with Mcols also sM[c] = sum_k Mcols[k,c]
__device__ void small_load_V(const float* V, int n, int d, int c0, int wb, const float* vecw, const float* Mcols, const SmallSm& sm) {
  const int tid = threadIdx.x, n16 = (n + 15) / 16 * 16;
  for (int idx = tid; idx < n16 * 16; idx += SG_THREADS) {
    const int k = idx >> 4, c4 = (idx & 15) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (k < n && c4 < wb) v = __ldcg(reinterpret_cast<const float4*>(V + (size_t)k * d + c0 + c4));
    *reinterpret_cast<float4*>(&sm.Vs[k * SG_WB + c4]) = v;
  }
  __syncthreads();
  const int c = tid & 63, part = tid >> 6;
  float s0 = 0.f, s1 = 0.f, m0 = 0.f;
  for (int k = part; k < n; k += 4) {
    const float v = sm.Vs[k * SG_WB + c];
    s0 += v;
    s1 = fmaf(vecw[k], v, s1);
    if (Mcols != nullptr && c < wb) m0 += __ldcg(Mcols + (size_t)k * d + c0 + c);
  }
  sm.S[part * 64 + c] = s0;
  sm.S[256 + part * 64 + c] = s1;
  sm.S[512 + part * 64 + c] = m0;
  __syncthreads();
  if (tid < 64) {
    sm.cb0[tid] = ((sm.S[tid] + sm.S[64 + tid]) + sm.S[128 + tid]) + sm.S[192 + tid];
    sm.cb1[tid] = ((sm.S[256 + tid] + sm.S[320 + tid]) + sm.S[384 + tid]) + sm.S[448 + tid];
    sm.sM[tid] = ((sm.S[512 + tid] + sm.S[576 + tid]) + sm.S[640 + tid]) + sm.S[704 + tid];
  }
  __syncthreads();
}

struct SmallItem {
  const float* P;       // the four planes of the stage's cubic piece of this graph (tiled, npad x npad)
  int npad, n, d;       // d = row pitch of V / Mref / out
  int i0, rows_end;     // row block [i0, rows_end)
  int c0, wb;           // column block
  const float* fus;     // fusion scalars of the layer
  const float* vvec;    // smem: v_l
  const float* rowc;    // smem: r_l (forward) / c_l (adjoint)
  const float* tg;      // smem
  float kappa;
  int relu, scale_tg;
  float* out;           // graph base, pitch d
  // adjoint only
  const float* As;      // resident A_s / A'_s (shared memory, pitch P) or nullptr: stream the planes
  const float* Ad;
  int ldA;
  const float* Mref;    // graph base, pitch d
  const float* rows;    // smem [4][nv]
  int nv;
  float totA, totD;
  int first_row_block;  // this item also adds the once-per-column-block param7 term
  float* g_fus;
};

// ---- phase B / B': one (row block, column block) item of the matrix-free contraction (k_dual_contract, V from shared memory,
// planes prefetched into registers one K chunk ahead).  NACC = 1 forward, 4 adjoint (+ all fusion-scalar gradients of the layer).
template <int NACC, bool STAT>
__device__ void small_contract_item(const SmallItem& it, const StageScalars* S, const SmallSm& sm) {
  constexpr int NS = (NACC == 1) ? 2 : 4;
  float (*Sm_)[SG_KC][SG_LD] = reinterpret_cast<float (*)[SG_KC][SG_LD]>(sm.S);
  const int tid = threadIdx.x, n = it.n, npad = it.npad, nt = npad >> 5, i0 = it.i0;
  const float alpha = 1.f + it.fus[0], beta = 1.f + it.fus[1], gamma = it.fus[2], delta = it.fus[3];
  float wx[4], wy[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    if (NACC == 1) {
      wx[p] = alpha * S->wA[p] + beta * S->wD[p];
      wy[p] = gamma * S->wA[p] + delta * S->wD[p];
    } else {
      wx[p] = S->wA[p];
      wy[p] = S->wD[p];
    }
  }
  float acc[NACC][4][4];
#pragma unroll
  for (int q = 0; q < NACC; ++q)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[q][i][j] = 0.f;
  const int ty = tid >> 4, tx = tid & 15;
  const int drow = tid >> 2, dkq = tid & 3;     // direct tile: element (row i, col k)
  const int tkr = tid >> 4, tiq = tid & 15;     // transposed tile: element (row k, col i)
  float4 pd[4], pt[4];
  auto fetch = [&](int k0) {
    const int gi = i0 + drow, gk = k0 + 4 * dkq;
    const bool okd = gi < npad && gk < npad;
    const int gk2 = k0 + tkr, gi2 = i0 + 4 * tiq;
    const bool okt = gk2 < npad && gi2 < npad;
    constexpr int NPL = STAT ? 1 : 4;   // a static control has plane a only: b, c, d stay exact zeros
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      pd[q] = (okd && q < NPL) ? __ldg(reinterpret_cast<const float4*>(it.P + peg_tile_off(gi, gk, q, nt, NPL))) : make_float4(0.f, 0.f, 0.f, 0.f);
      pt[q] = (okt && q < NPL) ? __ldg(reinterpret_cast<const float4*>(it.P + peg_tile_off(gk2, gi2, q, nt, NPL))) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stage = [&](int k0) {
    {
      const int gk = k0 + 4 * dkq;
      const float* pf = reinterpret_cast<const float*>(pd);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool ok = (gk + j) < n;
        const float e0 = pf[0 * 4 + j], e1 = pf[1 * 4 + j], e2 = pf[2 * 4 + j], e3 = pf[3 * 4 + j];
        Sm_[0][4 * dkq + j][drow] = ok ? (wx[0] * e0 + wx[1] * e1 + wx[2] * e2 + wx[3] * e3) : 0.f;
        if (NACC == 4) Sm_[1][4 * dkq + j][drow] = ok ? (wy[0] * e0 + wy[1] * e1 + wy[2] * e2 + wy[3] * e3) : 0.f;
      }
    }
    {
      const int gi = i0 + 4 * tiq;
      const float* pf = reinterpret_cast<const float*>(pt);
      float y0[4], y1[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool ok = (gi + j) < n;
        const float e0 = pf[0 * 4 + j], e1 = pf[1 * 4 + j], e2 = pf[2 * 4 + j], e3 = pf[3 * 4 + j];
        if (NACC == 1) {
          y0[j] = ok ? (wy[0] * e0 + wy[1] * e1 + wy[2] * e2 + wy[3] * e3) : 0.f;
          y1[j] = 0.f;
        } else {
          y0[j] = ok ? (wx[0] * e0 + wx[1] * e1 + wx[2] * e2 + wx[3] * e3) : 0.f;
          y1[j] = ok ? (wy[0] * e0 + wy[1] * e1 + wy[2] * e2 + wy[3] * e3) : 0.f;
        }
      }
      *reinterpret_cast<float4*>(&Sm_[NS / 2][tkr][4 * tiq]) = make_float4(y0[0], y0[1], y0[2], y0[3]);
      if (NACC == 4) *reinterpret_cast<float4*>(&Sm_[3][tkr][4 * tiq]) = make_float4(y1[0], y1[1], y1[2], y1[3]);
    }
  };
  const bool resident = it.As != nullptr;
  const int n16 = (n + 15) / 16 * 16;
  // resident mode: the operand tiles come straight from A_s / A'_s in shared memory -- no L2 round trip per K chunk
  auto stage_res = [&](int k0) {
    const int P = it.ldA;
    {
      const int gi = i0 + drow, gk = k0 + 4 * dkq;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float a_ = 0.f, d_ = 0.f;
        if (gi < n16) { a_ = it.As[gi * P + gk + j]; d_ = it.Ad[gi * P + gk + j]; }
        if (NACC == 1) {
          Sm_[0][4 * dkq + j][drow] = alpha * a_ + beta * d_;
        } else {
          Sm_[0][4 * dkq + j][drow] = a_;
          Sm_[1][4 * dkq + j][drow] = d_;
        }
      }
    }
    {
      const int gk = k0 + tkr, gi = i0 + 4 * tiq;
      float y0[4], y1[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float a_ = 0.f, d_ = 0.f;
        if (gi + j < n16) { a_ = it.As[gk * P + gi + j]; d_ = it.Ad[gk * P + gi + j]; }
        if (NACC == 1) { y0[j] = gamma * a_ + delta * d_; y1[j] = 0.f; }
        else { y0[j] = a_; y1[j] = d_; }
      }
      *reinterpret_cast<float4*>(&Sm_[NS / 2][tkr][4 * tiq]) = make_float4(y0[0], y0[1], y0[2], y0[3]);
      if (NACC == 4) *reinterpret_cast<float4*>(&Sm_[3][tkr][4 * tiq]) = make_float4(y1[0], y1[1], y1[2], y1[3]);
    }
  };
  if (!resident) fetch(0);
  for (int k0 = 0; k0 < n; k0 += SG_KC) {
    if (resident) stage_res(k0); else stage(k0);
    __syncthreads();
    if (!resident && k0 + SG_KC < n) fetch(k0 + SG_KC);     // in flight while this chunk is multiplied
#pragma unroll
    for (int k = 0; k < SG_KC; ++k) {
      const float4 v4 = *reinterpret_cast<const float4*>(&sm.Vs[(k0 + k) * SG_WB + 4 * tx]);
      const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
      if (NACC == 1) {
        const float4 s0 = *reinterpret_cast<const float4*>(&Sm_[0][k][4 * ty]);
        const float4 s1 = *reinterpret_cast<const float4*>(&Sm_[1][k][4 * ty]);
        const float aa[4] = {s0.x + s1.x, s0.y + s1.y, s0.z + s1.z, s0.w + s1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[0][i][j] = fmaf(aa[i], vv[j], acc[0][i][j]);
      } else {
#pragma unroll
        for (int q = 0; q < NACC; ++q) {
          const float4 s0 = *reinterpret_cast<const float4*>(&Sm_[q][k][4 * ty]);
          const float aa[4] = {s0.x, s0.y, s0.z, s0.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[q][i][j] = fmaf(aa[i], vv[j], acc[q][i][j]);
        }
      }
    }
    __syncthreads();
  }
  // ---- epilogue ----
  const int lc = 4 * tx, gc = it.c0 + lc;
  float g[14];
#pragma unroll
  for (int k = 0; k < 14; ++k) g[k] = 0.f;
  if (lc < it.wb) {
    const float ss[4] = {sm.cb0[lc], sm.cb0[lc + 1], sm.cb0[lc + 2], sm.cb0[lc + 3]};
    const float tt[4] = {sm.cb1[lc], sm.cb1[lc + 1], sm.cb1[lc + 2], sm.cb1[lc + 3]};
    const float sMv[4] = {sm.sM[lc], sm.sM[lc + 1], sm.sM[lc + 2], sm.sM[lc + 3]};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gi = i0 + 4 * ty + i;
      if (gi >= it.rows_end) continue;
      const float vi = 1.f + it.vvec[gi];
      const float rc = it.rowc[gi];
      const float tg = it.scale_tg ? it.tg[gi] : 1.f;
      const float4 vin = *reinterpret_cast<const float4*>(&sm.Vs[gi * SG_WB + lc]);
      const float vv[4] = {vin.x, vin.y, vin.z, vin.w};
      float o[4];
      if (NACC == 1) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float val = vv[j] * vi + acc[0][i][j] + rc * ss[j] + tt[j] + it.kappa * ss[j];
          if (it.relu) val = fmaxf(val, 0.f);
          o[j] = val * tg;
        }
      } else {
        const float4 m4 = __ldcg(reinterpret_cast<const float4*>(it.Mref + (size_t)gi * it.d + gc));
        const float mm[4] = {m4.x, m4.y, m4.z, m4.w};
        float q = 0.f, u = 0.f, w = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // acc[0] = A V, acc[1] = A'V, acc[2] = A^T V, acc[3] = A'^T V   (V = cotangent of the layer output)
          o[j] = vv[j] * vi + alpha * acc[2][i][j] + beta * acc[3][i][j] + gamma * acc[0][i][j] + delta * acc[1][i][j] +
                 rc * ss[j] + tt[j] + it.kappa * ss[j];
          g[0] = fmaf(acc[2][i][j], mm[j], g[0]);   // param1[0]: <A^T g, M>
          g[1] = fmaf(acc[3][i][j], mm[j], g[1]);   // param1[1]: <A'^T g, M>
          g[2] = fmaf(acc[0][i][j], mm[j], g[2]);   // param2[0]: <A g, M>
          g[3] = fmaf(acc[1][i][j], mm[j], g[3]);   // param2[1]: <A' g, M>
          q = fmaf(vv[j], mm[j], q);
          u = fmaf(vv[j], sMv[j], u);
          w = fmaf(mm[j], ss[j], w);
        }
        const float rA = it.rows[gi], rD = it.rows[it.nv + gi], dA = it.rows[2 * it.nv + gi], dD = it.rows[3 * it.nv + gi];
        g[4] = fmaf(dA, q, g[4]); g[5] = fmaf(dD, q, g[5]);       // param3
        g[6] = fmaf(rA, u, g[6]); g[7] = fmaf(rD, u, g[7]);       // param4 (/n)
        g[8] = fmaf(rA, w, g[8]); g[9] = fmaf(rD, w, g[9]);       // param5 (/n)
        g[10] = fmaf(rA, q, g[10]); g[11] = fmaf(rD, q, g[11]);   // param6 (/n)
        g[12] += q;                                               // param8 (* tot / n^2)
      }
      *reinterpret_cast<float4*>(it.out + (size_t)gi * it.d + gc) = make_float4(o[0], o[1], o[2], o[3]);
    }
    if (NACC == 4 && it.first_row_block && ty == 0) {             // param7: tot_A / n^2 (1^T G . 1^T M), once per column block
#pragma unroll
      for (int j = 0; j < 4; ++j) g[13] = fmaf(ss[j], sMv[j], g[13]);
    }
  }
  if (NACC == 4) {
    const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
    for (int k = 0; k < 14; ++k) {
      const float t = warp_sum(g[k]);
      if (lane == 0) sm.red[warp * 16 + k] = t;
    }
    __syncthreads();
    if (tid < 14) {
      float t = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) t += sm.red[w8 * 16 + tid];
      const float inv_n = 1.f / (float)n, inv_n2 = inv_n * inv_n;
      const int k = tid;
      if (k < 4) atomicAdd(it.g_fus + k, t);
      else if (k < 6) atomicAdd(it.g_fus + 4 + (k - 4), t);
      else if (k < 8) atomicAdd(it.g_fus + 6 + (k - 6), t * inv_n);
      else if (k < 10) atomicAdd(it.g_fus + 8 + (k - 8), t * inv_n);
      else if (k < 12) atomicAdd(it.g_fus + 10 + (k - 10), t * inv_n);
      else if (k == 12) {
        atomicAdd(it.g_fus + 14, t * it.totA * inv_n2);
        atomicAdd(it.g_fus + 15, t * it.totD * inv_n2);
      } else {
        atomicAdd(it.g_fus + 12, t * it.totA * inv_n2);
        atomicAdd(it.g_fus + 13, t * it.totA * inv_n2);
      }
    }
  }
  __syncthreads();     // the next item may reload Vs / restage S
}

// ---- phase C (a): backward of Linear + RMSNorm for 32 nodes (k_linear_bwd, din <= 128) ----
__device__ void small_linear_bwd_item(const float* Mbar, const float* __restrict__ W, const float* Z, const float* __restrict__ nw,
                                      int n, int din, int dout, int relu_mask, int node0, float* Zbar, float* g_nw, float* g_nb,
                                      const SmallSm& sm) {
  float (*mt)[36] = reinterpret_cast<float (*)[36]>(sm.S);
  float (*wsm)[SG_MAX_DIN] = reinterpret_cast<float (*)[SG_MAX_DIN]>(sm.S + 32 * 36);
  float* gsw = sm.S + 32 * 36 + 32 * SG_MAX_DIN;
  float* gsb = gsw + SG_MAX_DIN;
  const int tid = threadIdx.x, ty = tid >> 5, tx = tid & 31, c = 4 * tx;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int cc = tid; cc < din; cc += SG_THREADS) { gsw[cc] = 0.f; gsb[cc] = 0.f; }
  for (int o0 = 0; o0 < dout; o0 += 32) {
    {
      const int r = tid >> 3, kq = (tid & 7) * 4, node = node0 + r, o = o0 + kq;
      float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (node < n && o < dout) m4 = __ldcg(reinterpret_cast<const float4*>(Mbar + (size_t)node * dout + o));
      mt[kq + 0][r] = m4.x; mt[kq + 1][r] = m4.y; mt[kq + 2][r] = m4.z; mt[kq + 3][r] = m4.w;
    }
    for (int idx = tid; idx < 32 * (din >> 2); idx += SG_THREADS) {
      const int k = idx / (din >> 2), c4 = idx - k * (din >> 2), o = o0 + k;
      const float4 w4 = (o < dout) ? __ldg(reinterpret_cast<const float4*>(W + (size_t)o * din + 4 * c4)) : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(&wsm[k][4 * c4]) = w4;
    }
    __syncthreads();
    if (c < din) {
#pragma unroll 8
      for (int k = 0; k < 32; ++k) {
        const float4 a4 = *reinterpret_cast<const float4*>(&mt[k][4 * ty]);
        const float4 b4 = *reinterpret_cast<const float4*>(&wsm[k][c]);
        const float aa[4] = {a4.x, a4.y, a4.z, a4.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
  float gw[4] = {0.f, 0.f, 0.f, 0.f}, gb[4] = {0.f, 0.f, 0.f, 0.f};
  float nwv[4] = {0.f, 0.f, 0.f, 0.f};
  if (c < din) { nwv[0] = nw[c]; nwv[1] = nw[c + 1]; nwv[2] = nw[c + 2]; nwv[3] = nw[c + 3]; }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int node = node0 + 4 * ty + i;
    const bool ok = node < n;
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (ok && c < din) {
      const float4 z4 = __ldcg(reinterpret_cast<const float4*>(Z + (size_t)node * din + c));
      z[0] = z4.x; z[1] = z4.y; z[2] = z4.z; z[3] = z4.w;
    }
    float ss = 0.f, dot = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ss = fmaf(z[j], z[j], ss);
      dot = fmaf(nwv[j] * acc[i][j], z[j], dot);
    }
    ss = warp_sum(ss);
    dot = warp_sum(dot);
    const float rinv = rsqrtf(ss / (float)din + 1e-5f);
    const float coef = rinv * rinv * rinv * dot / (float)din;
    if (ok && c < din) {
      float zb[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        zb[j] = rinv * nwv[j] * acc[i][j] - z[j] * coef;
        if (relu_mask && !(z[j] > 0.f)) zb[j] = 0.f;
        gw[j] = fmaf(acc[i][j] * z[j], rinv, gw[j]);
        gb[j] += acc[i][j];
      }
      *reinterpret_cast<float4*>(Zbar + (size_t)node * din + c) = make_float4(zb[0], zb[1], zb[2], zb[3]);
    }
  }
  if (c < din) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { atomicAdd(&gsw[c + j], gw[j]); atomicAdd(&gsb[c + j], gb[j]); }
  }
  __syncthreads();
  for (int cc = tid; cc < din; cc += SG_THREADS) {
    atomicAdd(g_nw + cc, gsw[cc]);
    atomicAdd(g_nb + cc, gsb[cc]);
  }
  __syncthreads();
}

// ---- phase C (b): one 64 x 64 tile of the weight gradient over the graph's n rows (k_weight_grad) ----
__device__ void small_weight_grad_item(const float* Mbar, const float* N, int n, int din, int dout, int o0, int c0, float* gW,
                                       float* gb, const SmallSm& sm) {
  float (*ms)[SG_LD] = reinterpret_cast<float (*)[SG_LD]>(sm.S);
  float (*ns)[SG_LD] = reinterpret_cast<float (*)[SG_LD]>(sm.S + 16 * SG_LD);
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, lk = tid >> 4, lq = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;
  for (int k0 = 0; k0 < n; k0 += 16) {
    const int row = k0 + lk, o = o0 + 4 * lq, c = c0 + 4 * lq;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(&ms[lk][4 * lq]) = (row < n && o < dout) ? __ldcg(reinterpret_cast<const float4*>(Mbar + (size_t)row * dout + o)) : zero4;
    *reinterpret_cast<float4*>(&ns[lk][4 * lq]) = (row < n && c < din) ? __ldcg(reinterpret_cast<const float4*>(N + (size_t)row * din + c)) : zero4;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 m4 = *reinterpret_cast<const float4*>(&ms[k][4 * ty]);
      const float4 n4 = *reinterpret_cast<const float4*>(&ns[k][4 * tx]);
      const float mm[4] = {m4.x, m4.y, m4.z, m4.w}, nn[4] = {n4.x, n4.y, n4.z, n4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(mm[i], nn[j], acc[i][j]);
    }
    if (c0 == 0 && tid < 64) {
#pragma unroll
      for (int k = 0; k < 16; ++k) bsum += ms[k][tid];
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int o = o0 + 4 * ty + i;
    if (o >= dout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + 4 * tx + j;
      if (c < din) atomicAdd(gW + (size_t)o * din + c, acc[i][j]);
    }
  }
  if (c0 == 0 && tid < 64 && o0 + tid < dout) atomicAdd(gb + o0 + tid, bsum);
}

// layer phases shared by the two kernels ---------------------------------------------------------------------------------------
__device__ void small_phase_linear(const SmallArgs& a, int l, const float* Z, float* Mg, float* Ng, int rank, const SmallSm& sm) {
  const LayerDesc& ld = a.model.layer[l];
  const int nrb = (a.n + SG_RB - 1) / SG_RB, ncb = (ld.dout + SG_WB - 1) / SG_WB;
  int lo, hi;
  small_range(nrb * ncb, rank, a.C, lo, hi);
  for (int q = lo; q < hi; ++q) {
    const int cbi = q / nrb, rbi = q - cbi * nrb;
    small_linear_tile(Z, a.n, ld.din, ld.dout, a.params + ld.w_off, a.params + ld.b_off, a.params + ld.nw_off, a.params + ld.nb_off,
                      rbi * SG_RB, cbi * SG_WB, Mg, Ng, sm);
  }
}

// forward contraction of layer l: V = Mg [n][dout] -> out [n][dout]
template <bool STAT>
__device__ void small_phase_contract_fwd(const SmallArgs& a, int b, int l, const float* Mg, float* out, int relu, int scale_tg,
                                         int rank, const StageScalars* S, const SmallSm& sm) {
  const LayerDesc& ld = a.model.layer[l];
  const int n = a.n, nrb = (n + SG_RB - 1) / SG_RB, rbsz = ((n + nrb - 1) / nrb + 3) / 4 * 4, ncb = (ld.dout + SG_WB - 1) / SG_WB;
  int lo, hi;
  small_range(nrb * ncb, rank, a.C, lo, hi);
  SmallItem it;
  it.P = small_planes<STAT>(a, b, S->interval);
  it.npad = a.npad; it.n = n; it.d = ld.dout;
  it.fus = a.params + ld.fus_off;
  it.vvec = sm.vec + (3 * l + 0) * sm.nv;
  it.rowc = sm.vec + (3 * l + 1) * sm.nv;
  it.tg = sm.vec + 3 * a.L * sm.nv;
  it.kappa = S->kappa[l];
  it.relu = relu; it.scale_tg = scale_tg;
  it.out = out;
  it.As = sm.As; it.Ad = sm.Ad; it.ldA = sm.P;
  it.Mref = nullptr; it.rows = nullptr; it.nv = sm.nv; it.totA = it.totD = 0.f; it.first_row_block = 0; it.g_fus = nullptr;
  int cur = -1;
  for (int q = lo; q < hi; ++q) {
    const int cbi = q / nrb, rbi = q - cbi * nrb;
    it.c0 = cbi * SG_WB; it.wb = min(SG_WB, ld.dout - it.c0);
    it.i0 = rbi * rbsz; it.rows_end = min(n, it.i0 + rbsz);
    if (cbi != cur) { small_load_V(Mg, n, ld.dout, it.c0, it.wb, sm.vec + (3 * l + 2) * sm.nv, nullptr, sm); cur = cbi; }
    small_contract_item<1, STAT>(it, S, sm);
  }
}

// =====================================================================================
// dy = f(t, yin) for graph blockIdx.x / C; grid (B * C), cluster (C), block 256
// =====================================================================================
template <bool STAT>
__global__ void __launch_bounds__(SG_THREADS, 1) k_small_fwd(const SmallArgs a) {
  extern __shared__ __align__(16) float sg_smem[];
  __shared__ StageScalars S;
  cg::cluster_group cluster = cg::this_cluster();
  const int b = blockIdx.x / a.C, rank = blockIdx.x - b * a.C;
  const SmallSm sm = small_carve(sg_smem, a.n, a.L);
  const int n = a.n, h = a.h, L = a.L, dmax = a.model.dmax;
  small_prep(a, b, rank, sm, &S);
  if (sm.As) small_build_A<STAT>(a, b, &S, sm);
  float* Mg = a.M + (size_t)b * n * dmax;
  const float* Zin = a.yin + (size_t)b * n * h;
  for (int l = 0; l < a.nlayers; ++l) {
    const bool last = (l == L - 1);
    small_phase_linear(a, l, Zin, Mg, nullptr, rank, sm);
    __threadfence();
    cluster.sync();
    float* out;
    if (!last) out = (a.save[l + 1] ? a.save[l + 1] : ((l & 1) ? a.Zb : a.Za)) + (size_t)b * n * h;
    else out = a.e > 0 ? a.OL + (size_t)b * n * dmax : a.dy + (size_t)b * n * h;
    small_phase_contract_fwd<STAT>(a, b, l, Mg, out, last ? 0 : 1, last ? 1 : 0, rank, &S, sm);
    __threadfence();
    cluster.sync();
    Zin = out;
  }
  if (a.e > 0 && a.nlayers == L) {     // CDE wrapper
    const int e2 = 2 * a.e;
    int r0, r1;
    small_range(n, rank, a.C, r0, r1);
    const float* OLg = a.OL + (size_t)b * n * dmax;
    float* dyg = a.dy + (size_t)b * n * h;
    for (int idx = r0 * h + threadIdx.x; idx < r1 * h; idx += SG_THREADS) {
      const int i = idx / h, m = idx - i * h;
      const float* o = OLg + (size_t)i * h * e2 + (size_t)m * e2;
      float acc = 0.f;
      for (int j = 0; j < e2; ++j) acc = fmaf(__ldcg(o + j), small_xd(a, b, &S, i, j), acc);
      dyg[idx] = acc;
    }
  }
}

// =====================================================================================
// VJP of one evaluation (feval_vjp): ybar = J_y^T kbar, g_params += J_theta^T kbar, optionally g_xd
// =====================================================================================
template <bool STAT>
__global__ void __launch_bounds__(SG_THREADS, 1) k_small_vjp(const SmallArgs a) {
  extern __shared__ __align__(16) float sg_smem[];
  __shared__ StageScalars S;
  cg::cluster_group cluster = cg::this_cluster();
  const int b = blockIdx.x / a.C, rank = blockIdx.x - b * a.C, tid = threadIdx.x;
  const SmallSm sm = small_carve(sg_smem, a.n, a.L);
  const int n = a.n, h = a.h, L = a.L, dmax = a.model.dmax, e2 = 2 * a.e;
  const int dL = a.model.layer[L - 1].dout;
  small_prep(a, b, rank, sm, &S);
  if (sm.As) small_build_A<STAT>(a, b, &S, sm);
  float* Mg = a.M + (size_t)b * n * dmax;
  float* Ng = a.N + (size_t)b * n * h;
  float* Og = a.Obar + (size_t)b * n * dmax;
  float* Bg = a.Mbar + (size_t)b * n * dmax;
  float* OLg = a.OL ? a.OL + (size_t)b * n * dmax : nullptr;
  const float* kb = a.kbar + (size_t)b * n * h;
  int r0, r1;
  small_range(n, rank, a.C, r0, r1);
  if (a.g_xd != nullptr) {
    // recompute the tg-scaled last-layer output, then contract it with kbar
    const int l = L - 1;
    small_phase_linear(a, l, a.zin[l] + (size_t)b * n * h, Mg, nullptr, rank, sm);
    __threadfence();
    cluster.sync();
    small_phase_contract_fwd<STAT>(a, b, l, Mg, OLg, 0, 1, rank, &S, sm);
    __threadfence();
    cluster.sync();
    float* gx = a.g_xd + (size_t)b * n * e2;
    for (int idx = r0 * e2 + tid; idx < r1 * e2; idx += SG_THREADS) {
      const int i = idx / e2, j = idx - i * e2;
      float acc = 0.f;
      for (int m = 0; m < h; ++m) acc = fmaf(kb[(size_t)i * h + m], __ldcg(OLg + (size_t)i * h * e2 + (size_t)m * e2 + j), acc);
      gx[idx] = acc;
    }
  }
  {   // cotangent of the last layer's output
    const float* tg = sm.vec + 3 * L * sm.nv;
    for (int idx = r0 * dL + tid; idx < r1 * dL; idx += SG_THREADS) {
      const int i = idx / dL, col = idx - i * dL;
      float v;
      if (e2 > 0) {
        const int m = col / e2, j = col - m * e2;
        v = tg[i] * kb[(size_t)i * h + m] * small_xd(a, b, &S, i, j);
      } else {
        v = tg[i] * kb[(size_t)i * h + col];
      }
      Og[idx] = v;
    }
  }
  // (the barrier after the first recompute phase below orders Obar before its readers)
  for (int l = L - 1; l >= 0; --l) {
    const LayerDesc& ld = a.model.layer[l];
    const float* Zl = a.zin[l] + (size_t)b * n * h;
    float* g_fus = a.g_params + ld.fus_off;
    small_phase_linear(a, l, Zl, Mg, Ng, rank, sm);        // A': M_l and the normalised input N_l
    __threadfence();
    cluster.sync();
    {   // B': Mbar = adjoint contraction of Obar, fusion-scalar gradients
      const int nrb = (n + SG_RB - 1) / SG_RB, rbsz = ((n + nrb - 1) / nrb + 3) / 4 * 4, ncb = (ld.dout + SG_WB - 1) / SG_WB;
      int lo, hi;
      small_range(nrb * ncb, rank, a.C, lo, hi);
      SmallItem it;
      it.P = small_planes<STAT>(a, b, S.interval);
      it.npad = a.npad; it.n = n; it.d = ld.dout;
      it.fus = a.params + ld.fus_off;
      it.vvec = sm.vec + (3 * l + 0) * sm.nv;
      it.rowc = sm.vec + (3 * l + 2) * sm.nv;      // c_l multiplies 1^T G on the way back
      it.tg = sm.vec + 3 * L * sm.nv;
      it.kappa = S.kappa[l];
      it.relu = 0; it.scale_tg = 0;
      it.out = Bg;
      it.As = sm.As; it.Ad = sm.Ad; it.ldA = sm.P;
      it.Mref = Mg; it.rows = sm.rows; it.nv = sm.nv; it.totA = S.totA; it.totD = S.totD; it.g_fus = g_fus;
      int cur = -1;
      for (int q = lo; q < hi; ++q) {
        const int cbi = q / nrb, rbi = q - cbi * nrb;
        it.c0 = cbi * SG_WB; it.wb = min(SG_WB, ld.dout - it.c0);
        it.i0 = rbi * rbsz; it.rows_end = min(n, it.i0 + rbsz);
        it.first_row_block = rbi == 0;
        if (cbi != cur) { small_load_V(Og, n, ld.dout, it.c0, it.wb, sm.vec + (3 * l + 1) * sm.nv, Mg, sm); cur = cbi; }
        small_contract_item<4, STAT>(it, &S, sm);
      }
    }
    __threadfence();
    cluster.sync();
    {   // C: Linear / RMSNorm backward (32-node items) and weight-gradient tiles
      const int nrb32 = (n + 31) / 32, nwo = (ld.dout + 63) / 64, nwc = (ld.din + 63) / 64;
      int lo, hi;
      small_range(nrb32 + nwo * nwc, rank, a.C, lo, hi);
      float* zb = (l == 0) ? a.ybar + (size_t)b * n * h : Og;
      for (int q = lo; q < hi; ++q) {
        if (q < nrb32) {
          small_linear_bwd_item(Bg, a.params + ld.w_off, Zl, a.params + ld.nw_off, n, ld.din, ld.dout, l > 0 ? 1 : 0, q * 32, zb,
                                a.g_params + ld.nw_off, a.g_params + ld.nb_off, sm);
        } else {
          const int w = q - nrb32, oi = w / nwc, ci = w - oi * nwc;
          small_weight_grad_item(Bg, Ng, n, ld.din, ld.dout, oi * 64, ci * 64, a.g_params + ld.w_off, a.g_params + ld.b_off, sm);
        }
      }
    }
    __threadfence();
    cluster.sync();
  }
}

}  // namespace peg
