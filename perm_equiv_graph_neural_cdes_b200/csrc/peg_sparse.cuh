// Sparse (CSR) adjacency paths: the control-path builders and the gather form of the n x n x d contraction (PegSparse in
// pegncde.h).  Same operator and epilogue as k_dual_contract; the interpolated adjacency is formed per entry instead of per tile.
#pragma once
#include "peg_kernels.cuh"

namespace peg {

// =====================================================================================
// builders: one warp per (row, cubic piece, graph).  grid (ceil(n/8), T-1, B), block 256.
// The warp walks its row's entries in order, computes their (a,b,c,d) -- from the knot values (Hermite, the arithmetic of
// pegncde_build_adj) or taken as given -- writes them to coef and, through perm_t, to coef_t, and reduces the row sums and the
// diagonal with lane-strided partials + a butterfly: a fixed order, so the control is reproducible.
// =====================================================================================
__global__ void __launch_bounds__(256) k_sparse_build(const PegSparse sp, const int32_t* __restrict__ perm_t, const float* __restrict__ ts,
                                                      const float* __restrict__ values, const float* __restrict__ cd,
                                                      const float* __restrict__ cc, const float* __restrict__ cb,
                                                      const float* __restrict__ ca, int n, int Tm1, float* __restrict__ rowsum,
                                                      float* __restrict__ diag) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp, iv = blockIdx.y, b = blockIdx.z;
  if (i >= n) return;
  const int e0 = sp.row_ptr[(size_t)b * (n + 1) + i], e1 = sp.row_ptr[(size_t)b * (n + 1) + i + 1];
  const size_t nnz = (size_t)sp.nnz;
  float dt = 1.f, dtp = 1.f;
  if (values) {
    const float* tb = ts + (size_t)b * (Tm1 + 1);
    dt = tb[iv + 1] - tb[iv];
    dtp = iv > 0 ? tb[iv] - tb[iv - 1] : dt;
  }
  float4* coef = reinterpret_cast<float4*>(const_cast<float*>(sp.coef)) + (size_t)iv * sp.nnz_stride;
  float4* coef_t = reinterpret_cast<float4*>(const_cast<float*>(sp.coef_t)) + (size_t)iv * sp.nnz_stride;
  float rs[4] = {0.f, 0.f, 0.f, 0.f}, dg[4] = {0.f, 0.f, 0.f, 0.f};
  for (int e = e0 + lane; e < e1; e += 32) {
    float hv[4];
    if (values) {
      const float y0 = __ldg(values + (size_t)iv * nnz + e), y1 = __ldg(values + (size_t)(iv + 1) * nnz + e);
      const float yp = iv > 0 ? __ldg(values + (size_t)(iv - 1) * nnz + e) : 0.f;
      hermite_piece(y0, y1, yp, iv == 0, dt, dtp, hv);
    } else {
      const size_t o = (size_t)iv * nnz + e;
      hv[0] = __ldg(ca + o); hv[1] = __ldg(cb + o); hv[2] = __ldg(cc + o); hv[3] = __ldg(cd + o);
    }
    const float4 v = make_float4(hv[0], hv[1], hv[2], hv[3]);
    coef[e] = v;
    coef_t[__ldg(perm_t + e)] = v;
    const bool on_diag = __ldg(sp.col + e) == i;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      rs[p] += hv[p];
      if (on_diag) dg[p] = hv[p];
    }
  }
  const size_t slab = (size_t)b * Tm1 + iv;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const float r = warp_sum(rs[p]), g = warp_sum(dg[p]);   // a coalesced pattern has at most one diagonal entry per row
    if (lane == 0) {
      rowsum[(slab * 4 + p) * n + i] = r;
      diag[(slab * 4 + p) * n + i] = g;
    }
  }
}

// column sums = row sums of the transposed pattern (run after k_sparse_build has written coef_t).  Same grid as k_sparse_build.
__global__ void __launch_bounds__(256) k_sparse_colsums(const PegSparse sp, int n, int Tm1, float* __restrict__ colsum) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp, iv = blockIdx.y, b = blockIdx.z;
  if (i >= n) return;
  const int e0 = sp.row_ptr_t[(size_t)b * (n + 1) + i], e1 = sp.row_ptr_t[(size_t)b * (n + 1) + i + 1];
  const float4* coef_t = reinterpret_cast<const float4*>(sp.coef_t) + (size_t)iv * sp.nnz_stride;
  float cs[4] = {0.f, 0.f, 0.f, 0.f};
  for (int e = e0 + lane; e < e1; e += 32) {
    const float4 v = coef_t[e];
    cs[0] += v.x; cs[1] += v.y; cs[2] += v.z; cs[3] += v.w;
  }
  const size_t slab = (size_t)b * Tm1 + iv;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    const float t = warp_sum(cs[p]);
    if (lane == 0) colsum[(slab * 4 + p) * n + i] = t;
  }
}

// =====================================================================================
// The contraction on a CSR path (k_dual_contract's operator, fp32 FMA):
//   forward  (NACC=1): OUT = V(1+v) + X V + Y^T V + rowc (1^T V) + 1 (vec^T V + kappa 1^T V)
//   backward (NACC=4): A V, A'V, A^T V, A'^T V and the same epilogue (+ the param1 / param2 Frobenius products)
// A group of G lanes (G = 4-column float4 slots of the slab, a power of two <= 32) owns one (row, slab of 4G columns, graph).  It
// walks row i of the pattern (direct terms), then row i of the transposed pattern (transposed terms): G lanes load G entries' col
// and coef (one 16-byte load per entry) and form their interpolated weights, which are broadcast by shuffle, and every lane
// gathers its float4 of V[col] (G * 16 contiguous bytes per entry).  Entry order is fixed: the output is deterministic.
// grid (ceil(n / (8 * 32/G)), ceil(d / 4G), B), block 256.
// =====================================================================================
template <int NACC, bool TRANS>
__device__ __forceinline__ void sparse_walk_row(const int32_t* __restrict__ col, const float4* __restrict__ coef, int e0, int e1, int G,
                                                int lj, unsigned gmask, const float (&w0)[4], const float (&w1)[4],
                                                const float* __restrict__ Vb, int d, int gc, bool col_ok, float (&acc)[NACC][1][4]) {
  constexpr int Q0 = (NACC == 4 && TRANS) ? 2 : 0;   // accumulator of the first weight: A V / A^T V (backward), X V + Y^T V (forward)
  for (int base = e0; base < e1; base += G) {
    const int e = base + lj;
    int k = 0;
    float u0 = 0.f, u1 = 0.f;
    if (e < e1) {
      k = __ldg(col + e);
      const float4 cf = __ldg(coef + e);
      u0 = w0[0] * cf.x + w0[1] * cf.y + w0[2] * cf.z + w0[3] * cf.w;
      if (NACC == 4) u1 = w1[0] * cf.x + w1[1] * cf.y + w1[2] * cf.z + w1[3] * cf.w;
    }
    const int cnt = min(G, e1 - base);
    for (int jj = 0; jj < cnt; ++jj) {
      const int kk = __shfl_sync(gmask, k, jj, G);
      const float x0 = __shfl_sync(gmask, u0, jj, G);
      const float x1 = NACC == 4 ? __shfl_sync(gmask, u1, jj, G) : 0.f;
      if (col_ok) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(Vb + (size_t)kk * d + gc));
        acc[Q0][0][0] = fmaf(x0, v.x, acc[Q0][0][0]); acc[Q0][0][1] = fmaf(x0, v.y, acc[Q0][0][1]);
        acc[Q0][0][2] = fmaf(x0, v.z, acc[Q0][0][2]); acc[Q0][0][3] = fmaf(x0, v.w, acc[Q0][0][3]);
        if (NACC == 4) {
          acc[Q0 + 1][0][0] = fmaf(x1, v.x, acc[Q0 + 1][0][0]); acc[Q0 + 1][0][1] = fmaf(x1, v.y, acc[Q0 + 1][0][1]);
          acc[Q0 + 1][0][2] = fmaf(x1, v.z, acc[Q0 + 1][0][2]); acc[Q0 + 1][0][3] = fmaf(x1, v.w, acc[Q0 + 1][0][3]);
        }
      }
    }
  }
}

template <int NACC>
__global__ void __launch_bounds__(256) k_sparse_contract(const ContractArgs a, const PegSparse sp, int glog) {
  __shared__ float red[40];
  const int G = 1 << glog, rows_per_warp = 32 >> glog;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int sub = lane >> glog, lj = lane & (G - 1);
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (sub * G));
  const int b = blockIdx.z;
  const int gi = (blockIdx.x * 8 + warp) * rows_per_warp + sub;
  const int gc = blockIdx.y * 4 * G + 4 * lj;
  const int n = a.n, d = a.d;
  const StageScalars& sc = a.sc[b];    // read in place: a local copy would put its dynamically indexed kappa[] on the stack
  const float alpha = 1.f + a.fus[0], beta = 1.f + a.fus[1], gamma = a.fus[2], delta = a.fus[3];
  // forward: direct weight X = alpha A + beta A', transposed weight Y = gamma A + delta A'; backward: A and A' in both orientations
  float wx[4], wy[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    if (NACC == 1) {
      wx[p] = alpha * sc.wA[p] + beta * sc.wD[p];
      wy[p] = gamma * sc.wA[p] + delta * sc.wD[p];
    } else {
      wx[p] = sc.wA[p];
      wy[p] = sc.wD[p];
    }
  }
  float acc[NACC][1][4];
#pragma unroll
  for (int q = 0; q < NACC; ++q)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[q][0][j] = 0.f;
  const bool row_ok = gi < n, col_ok = gc < d;
  const float* Vb = a.V + (size_t)b * n * d;
  if (row_ok) {
    const size_t slab = (size_t)sc.interval * sp.nnz_stride;
    const int32_t* rp = sp.row_ptr + (size_t)b * (n + 1);
    const int32_t* rpt = sp.row_ptr_t + (size_t)b * (n + 1);
    const float4* cf = reinterpret_cast<const float4*>(sp.coef) + slab;
    const float4* cft = reinterpret_cast<const float4*>(sp.coef_t) + slab;
    if (NACC == 1) {
      sparse_walk_row<NACC, false>(sp.col, cf, rp[gi], rp[gi + 1], G, lj, gmask, wx, wy, Vb, d, gc, col_ok, acc);
      sparse_walk_row<NACC, true>(sp.col_t, cft, rpt[gi], rpt[gi + 1], G, lj, gmask, wy, wx, Vb, d, gc, col_ok, acc);
    } else {
      sparse_walk_row<NACC, false>(sp.col, cf, rp[gi], rp[gi + 1], G, lj, gmask, wx, wy, Vb, d, gc, col_ok, acc);
      sparse_walk_row<NACC, true>(sp.col_t, cft, rpt[gi], rpt[gi + 1], G, lj, gmask, wx, wy, Vb, d, gc, col_ok, acc);
    }
  }
  float g4[4] = {0.f, 0.f, 0.f, 0.f};
  if (row_ok && col_ok) {
    const float* sv = a.svec + (size_t)b * a.sv_stride;
    const float4 s4 = *reinterpret_cast<const float4*>(a.colbuf + ((size_t)b * 2 + 0) * d + gc);
    const float4 t4 = *reinterpret_cast<const float4*>(a.colbuf + ((size_t)b * 2 + 1) * d + gc);
    const float ss[4] = {s4.x, s4.y, s4.z, s4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
    contract_epilogue4<NACC, 1>(a, b, gi, gc, sv, Vb, acc, 0, ss, tt, sc.kappa[a.layer], alpha, beta, gamma, delta, g4);
  }
  if (NACC == 4) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float t = block_sum(g4[q], red);
      if (tid == 0) atomicAdd(a.g_fus + q, t);
    }
  }
}

// =====================================================================================
// Cotangent of the coefficients (pegncde_vf_vjp_adj / pegncde_solve_bwd_adj).  One layer computes O = M + F M, F = fusion(A, A').
// With Obar = dL/dO, Gbar_ij = <Obar_i, M_j>, q_i = <Obar_i, M_i>, u_i = <Obar_i, 1^T M>, w_i = <M_i, 1^T Obar>, every pattern entry
// (i, j) gets
//   gA = (1 + p1) Gbar_ij + p2 Gbar_ji + [i == j] p3 q_i + rowA_i + colA_j + totA     (gD likewise with the A' coefficients)
// where row* / col* / tot* gather the row-sum, column-sum, diag(sum) and total terms of the fusion (DESIGN.md, "Edge gradients"), and
// adds wA[k] gA + wD[k] gD to coefficient k of the entry on the stage's cubic piece.
// =====================================================================================
struct AdjGradArgs {
  const float* G;          // Obar [B,n,d]
  const float* M;          // [B,n,d]
  const float* cbM;        // [B][2][d]: [0] = 1^T M
  const float* cbG;        // [B][2][d]: [0] = 1^T Obar
  const float* fus;        // the layer's fusion scalars (16, or 22 + 2 for the directed layer)
  const StageScalars* sc;
  float* node;             // [B][4][n]: rowA, rowD, colA, colD
  float* q;                // [B][n]
  float* tot;              // [B][2]: totA, totD
  float* g_coef;           // [T-1, nnz_stride, 4]
  int n, d, directed;
};

// per-node tables: one warp per (node, graph), grid (ceil(n/8), B), block 256
__global__ void __launch_bounds__(256) k_sparse_adj_node(const AdjGradArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp, b = blockIdx.y;
  const int n = a.n, d = a.d;
  if (i >= n) return;
  const float* g = a.G + ((size_t)b * n + i) * d;
  const float* m = a.M + ((size_t)b * n + i) * d;
  const float* sM = a.cbM + (size_t)b * 2 * d;
  const float* sG = a.cbG + (size_t)b * 2 * d;
  float q = 0.f, u = 0.f, w = 0.f;
  for (int c = lane; c < d; c += 32) {
    const float gv = g[c], mv = m[c];
    q = fmaf(gv, mv, q);
    u = fmaf(gv, sM[c], u);
    w = fmaf(mv, sG[c], w);
  }
  q = warp_sum(q); u = warp_sum(u); w = warp_sum(w);
  if (lane != 0) return;
  const float* f = a.fus;
  const float inv_n = 1.f / (float)n;
  float rA, rD, cA = 0.f, cD = 0.f;
  if (!a.directed) {        // term 4: rowsum_i on row i (u_i), term 5: rowsum_j on column j (w_i), term 6: diag(rowsum) (q_i)
    rA = (f[6] * u + f[8] * w + f[10] * q) * inv_n;
    rD = (f[7] * u + f[9] * w + f[11] * q) * inv_n;
  } else {                  // column sums feed terms 4, 5, 6 (and 4' for A'); row sums feed 4' (A), 5', 6'
    rA = ((f[16] + f[18]) * w + f[20] * q) * inv_n;
    rD = (f[19] * w + f[21] * q) * inv_n;
    cA = (f[6] * u + f[8] * w + f[10] * q) * inv_n;
    cD = (f[7] * u + (f[9] + f[17]) * w + f[11] * q) * inv_n;
  }
  float* nv = a.node + (size_t)b * 4 * n;
  nv[i] = rA; nv[n + i] = rD; nv[2 * n + i] = cA; nv[3 * n + i] = cD;
  a.q[(size_t)b * n + i] = q;
}

// per-graph totals, reduced in a fixed order: grid B, block 1024.  Term 7 multiplies sum(A) for both of its coefficients (the
// reference's quirk), so only term 8 puts a total on A'.
__global__ void __launch_bounds__(1024) k_sparse_adj_tot(const AdjGradArgs a) {
  __shared__ float red[40];
  const int b = blockIdx.x, n = a.n, d = a.d;
  const float* q = a.q + (size_t)b * n;
  const float* sM = a.cbM + (size_t)b * 2 * d;
  const float* sG = a.cbG + (size_t)b * 2 * d;
  float sq = 0.f, s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) sq += q[i];
  for (int c = threadIdx.x; c < d; c += blockDim.x) s = fmaf(sG[c], sM[c], s);
  sq = block_sum(sq, red);
  s = block_sum(s, red);
  if (threadIdx.x == 0) {
    const float* f = a.fus;
    const float inv_n2 = 1.f / ((float)n * (float)n);
    a.tot[2 * b] = ((f[12] + f[13]) * s + f[14] * sq) * inv_n2;
    a.tot[2 * b + 1] = f[15] * sq * inv_n2;
  }
}

// the entries: k_sparse_contract's layout with at most 8 lanes per (row i, graph) (sparse_adj_glog), grid (ceil(n / (8 * 32/G)), B),
// block 256.  The group keeps the first ADJ_RESIDENT slabs (4G columns each) of Obar_i and M_i in registers; for each entry (i, j) of
// row i every lane gathers its float4s of M_j and Obar_j, the two dot products are reduced over the group by a butterfly, and the
// lane that loaded the entry read-modify-writes its four coefficients.  Narrow groups keep the butterfly short (3 shuffles per
// product, shared by the 4 rows a warp walks at once).  One owner per entry and stream-ordered launches: no atomics, and the result
// is reproducible bit for bit.
constexpr int ADJ_RESIDENT = 4;

__device__ __forceinline__ void adj_dot4(const float4 o, const float4 m, const float4 mj, const float4 oj, float& sij, float& sji) {
  sij = fmaf(o.x, mj.x, fmaf(o.y, mj.y, fmaf(o.z, mj.z, fmaf(o.w, mj.w, sij))));
  sji = fmaf(oj.x, m.x, fmaf(oj.y, m.y, fmaf(oj.z, m.z, fmaf(oj.w, m.w, sji))));
}

__global__ void __launch_bounds__(256) k_sparse_adj_grad(const AdjGradArgs a, const PegSparse sp, int glog) {
  const int G = 1 << glog, rows_per_warp = 32 >> glog;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane >> glog, lj = lane & (G - 1);
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (sub * G));
  const int b = blockIdx.y, n = a.n, d = a.d;
  const int i = (blockIdx.x * 8 + warp) * rows_per_warp + sub;
  if (i >= n) return;                        // the whole group shares i
  const float* Gb = a.G + (size_t)b * n * d;
  const float* Mb = a.M + (size_t)b * n * d;
  const float* nv = a.node + (size_t)b * 4 * n;
  const StageScalars& sc = a.sc[b];
  const float* f = a.fus;
  const float alpha = 1.f + f[0], beta = 1.f + f[1], gamma = f[2], delta = f[3];
  const float qi = a.q[(size_t)b * n + i];
  const float rA = nv[i] + a.tot[2 * b], rD = nv[n + i] + a.tot[2 * b + 1];
  const int nslab = (d + 4 * G - 1) / (4 * G), c0 = 4 * lj;
  float4 oi[ADJ_RESIDENT], mi[ADJ_RESIDENT];
#pragma unroll
  for (int s = 0; s < ADJ_RESIDENT; ++s) {
    const int c = s * 4 * G + c0;
    oi[s] = make_float4(0.f, 0.f, 0.f, 0.f);
    mi[s] = oi[s];
    if (s < nslab && c < d) {
      oi[s] = __ldg(reinterpret_cast<const float4*>(Gb + (size_t)i * d + c));
      mi[s] = __ldg(reinterpret_cast<const float4*>(Mb + (size_t)i * d + c));
    }
  }
  float4* gc = reinterpret_cast<float4*>(a.g_coef) + (size_t)sc.interval * sp.nnz_stride;
  const int e0 = sp.row_ptr[(size_t)b * (n + 1) + i], e1 = sp.row_ptr[(size_t)b * (n + 1) + i + 1];
  for (int base = e0; base < e1; base += G) {
    const int e = base + lj;
    const int k = e < e1 ? __ldg(sp.col + e) : 0;
    const int cnt = min(G, e1 - base);
    float gij = 0.f, gji = 0.f;
    for (int jj = 0; jj < cnt; ++jj) {
      const int j = __shfl_sync(gmask, k, jj, G);
      const float* Mj = Mb + (size_t)j * d;
      const float* Gj = Gb + (size_t)j * d;
      float sij = 0.f, sji = 0.f;
#pragma unroll
      for (int s = 0; s < ADJ_RESIDENT; ++s) {
        const int c = s * 4 * G + c0;
        if (s < nslab && c < d)
          adj_dot4(oi[s], mi[s], __ldg(reinterpret_cast<const float4*>(Mj + c)), __ldg(reinterpret_cast<const float4*>(Gj + c)), sij, sji);
      }
      for (int s = ADJ_RESIDENT; s < nslab; ++s) {   // rows wider than the resident slabs (the 2he-wide last layer): reload row i
        const int c = s * 4 * G + c0;
        if (c < d)
          adj_dot4(__ldg(reinterpret_cast<const float4*>(Gb + (size_t)i * d + c)), __ldg(reinterpret_cast<const float4*>(Mb + (size_t)i * d + c)),
                   __ldg(reinterpret_cast<const float4*>(Mj + c)), __ldg(reinterpret_cast<const float4*>(Gj + c)), sij, sji);
      }
      for (int o = G >> 1; o > 0; o >>= 1) {
        sij += __shfl_xor_sync(gmask, sij, o, G);
        sji += __shfl_xor_sync(gmask, sji, o, G);
      }
      if (lj == jj) { gij = sij; gji = sji; }
    }
    if (e < e1) {
      const bool on_diag = k == i;
      const float gA = alpha * gij + gamma * gji + rA + nv[2 * n + k] + (on_diag ? f[4] * qi : 0.f);
      const float gD = beta * gij + delta * gji + rD + nv[3 * n + k] + (on_diag ? f[5] * qi : 0.f);
      float4 v = gc[e];
      v.x += sc.wA[0] * gA + sc.wD[0] * gD;
      v.y += sc.wA[1] * gA + sc.wD[1] * gD;
      v.z += sc.wA[2] * gA + sc.wD[2] * gD;
      v.w += sc.wA[3] * gA + sc.wD[3] * gD;
      gc[e] = v;
    }
  }
}

// lanes per row of k_sparse_adj_grad: as k_sparse_contract, at most 8
inline int sparse_adj_glog(int d) {
  int g = 0;
  while (g < 3 && (4 << g) < d) ++g;
  return g;
}

// lanes per row of k_sparse_contract: enough float4 slots for d columns, at most a warp
inline int sparse_glog(int d) {
  int g = 0;
  while (g < 5 && (4 << g) < d) ++g;
  return g;
}

}  // namespace peg
