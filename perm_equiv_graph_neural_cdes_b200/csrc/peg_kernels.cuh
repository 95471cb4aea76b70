// CUDA-core (fp32 FFMA) kernels of the pegncde hot path.  These are the exact-fp32
// building blocks; the n x n x d contraction additionally has a tcgen05 (tensor-core)
// implementation in peg_tc.cu that replaces k_dual_contract when PEG_FLAG_TENSOR_CORES
// is set and the shape is large enough to be a real dense contraction.
#pragma once
#include "peg_common.cuh"

namespace peg {

// warp_sum / block_sum / ProducerOut / finalize_colsums live in peg_common.cuh (shared with peg_tc.cu)

// =====================================================================================
// control-path packing (pre-pass, once per batch)
// reference layout: d,c,b,a each [B, T-1, n, n, 2], last axis (time, adjacency)
// =====================================================================================

// diffrax.backward_hermite_coefficients of one element on one cubic piece (the dense and the sparse builders share it, so both give
// the same bits): a = y0, b = previous secant (first piece: own secant), c = 2 (m - b) / dt, d = -(m - b) / dt^2
__device__ __forceinline__ void hermite_piece(float y0, float y1, float yprev, bool first, float dt, float dtp, float (&hv)[4]) {
  const float m = (y1 - y0) / dt;
  const float bb = first ? m : (y0 - yprev) / dtp;
  hv[0] = y0;
  hv[1] = bb;
  hv[2] = 2.0f * (m - bb) / dt;
  hv[3] = -(m - bb) / (dt * dt);
}

// grid (nt column tiles, T-1, B), block 256: one block per COLUMN of 32x32 tiles, walked top to bottom.  Source is the
// reference layout (d,c,b,a each [B,T-1,n,n,2]), or the already tiled planes (tiled_in, pegncde_adj_stats), or the raw graph
// snapshots A_k [B,T,n,n] + knot times (snap / ts, pegncde_build_adj: backward_hermite_coefficients fused in,
// same operation order as the host formula so both routes give identical planes).
// Reads are coalesced float2 rows of the source, writes are coalesced float4 of the 16-KB tile (staged in smem).
// The column means of the time channel (tch) are summed by the block that owns the column tile, rows in ascending order and
// the 8 warps in a fixed order: no float atomics, so the packed control is reproducible bit for bit.
__global__ void __launch_bounds__(256) k_pack_adj(const float* __restrict__ cd, const float* __restrict__ cc,
                                                  const float* __restrict__ cb, const float* __restrict__ ca,
                                                  const float* __restrict__ tiled_in, const float* __restrict__ snap,
                                                  const float* __restrict__ ts, int n, int npad, int Tm1, int piece0,
                                                  int in_Tm1, float* __restrict__ adj_coef, float* __restrict__ rowsum,
                                                  float* __restrict__ diag, float* __restrict__ total,
                                                  float* __restrict__ tch, int ncols, int diag_col0, int np) {
  // rectangular shards (row-sharded mode): n rows x ncols columns (ncols a multiple of 32), diagonal at column diag_col0 + i;
  // the square case is ncols == n, diag_col0 == 0.
  // np = 1 (static control, pegncde_build_adj_static): `snap` is the adjacency [B, n, n] and only its plane `a` = A is written, one
  // 4-KB tile per 32x32 block and one slab per graph; the tables of piece 0 are filled (the caller copies them to every piece)
  __shared__ __align__(16) float tile[4096];   // the tile in its final element order
  __shared__ float tcol[8][3][32];             // per-warp column sums of the time channel of (b,c,d)
  // blockIdx.y walks `gridDim.y` cubic pieces starting at piece0; the reference-layout source holds in_Tm1 pieces per
  // graph (== Tm1 for a whole path, == the count of a streamed range: pegncde_pack_adj_range)
  const int b = blockIdx.z, iv = piece0 + blockIdx.y;
  const int nt = npad >> 5;                       // row tiles
  const int ncpad = peg_npad(ncols), ntc = ncpad >> 5;   // column tiles per row of tiles
  const int ct = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t slab = ((size_t)b * Tm1 + iv);
  const size_t in_slab = (size_t)b * in_Tm1 + blockIdx.y;
  const float* src[4] = {ca, cb, cc, cd};  // (a,b,c,d) order
  float tsum[3] = {0.f, 0.f, 0.f};
  float dt = 1.f, dtp = 1.f;
  if (snap && np == 4) {
    const float* tb = ts + (size_t)b * (Tm1 + 1);
    dt = tb[iv + 1] - tb[iv];
    dtp = iv > 0 ? tb[iv] - tb[iv - 1] : dt;
  }
  for (int rt = 0; rt < nt; ++rt) {
    const size_t tile_base = (np == 4 ? slab : (size_t)b) * np * (size_t)npad * ncpad + ((size_t)rt * ntc + ct) * (1024 * np);
    if (tiled_in) {
      for (int idx = threadIdx.x; idx < 256 * np; idx += 256)
        *reinterpret_cast<float4*>(&tile[4 * idx]) = *reinterpret_cast<const float4*>(tiled_in + tile_base + 4 * idx);
      __syncthreads();
    }
    for (int idx = threadIdx.x; idx < 1024; idx += 256) {
      const int r = idx >> 5, c = idx & 31;      // r is warp-uniform, c == lane
      const int i = rt * 32 + r, k = ct * 32 + c;
      float hv[4] = {0.f, 0.f, 0.f, 0.f};
      if (np == 1 && i < n && k < ncols) {
        hv[0] = __ldg(snap + ((size_t)b * n + i) * (size_t)ncols + k);
      } else if (snap && i < n && k < ncols) {
        const float* Ab = snap + ((size_t)b * (Tm1 + 1) * n + i) * (size_t)ncols + k;
        const size_t knot = (size_t)n * ncols;
        const float y0 = __ldg(Ab + (size_t)iv * knot), y1 = __ldg(Ab + (size_t)(iv + 1) * knot);
        const float yp = iv > 0 ? __ldg(Ab + (size_t)(iv - 1) * knot) : 0.f;
        hermite_piece(y0, y1, yp, iv == 0, dt, dtp, hv);
      }
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        if (p >= np) break;
        float v = 0.f;
        const int to = (int)peg_tile_off(r, c, p, 1, np);   // offset inside the tile
        if (i < n && k < ncols) {
          if (tiled_in) {
            v = tile[to];
          } else if (snap) {
            v = hv[p];
          } else {
            const float2 tv = __ldg(reinterpret_cast<const float2*>(src[p]) + (in_slab * n + i) * (size_t)ncols + k);
            v = tv.y;
            if (p > 0) tsum[p - 1] += tv.x;
          }
          if (diag != nullptr && diag_col0 >= 0 && k == diag_col0 + i) diag[(slab * 4 + p) * n + i] = v;
        }
        if (!tiled_in) tile[to] = v;
      }
    }
    __syncthreads();
    if (!tiled_in) {
      for (int idx = threadIdx.x; idx < 256 * np; idx += 256)
        *reinterpret_cast<float4*>(adj_coef + tile_base + 4 * idx) = *reinterpret_cast<const float4*>(&tile[4 * idx]);
    }
    __syncthreads();
  }
  if (!tiled_in && !snap) {   // tch[b,iv,p,k] = mean over all rows of the time channel
#pragma unroll
    for (int p = 0; p < 3; ++p) tcol[warp][p][lane] = tsum[p];
    __syncthreads();
    if (threadIdx.x < 96) {
      const int p = threadIdx.x >> 5, k = ct * 32 + lane;
      float t = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) t += tcol[w8][p][lane];
      if (k < ncols) tch[(slab * 3 + p) * ncols + k] = t / (float)n;
    }
  }
}

// Row sums of the four tiled planes, deterministic: one block per 32-row tile walks the column tiles in order
// (fixed-order warp reductions, no float atomics), so the packed control -- and every accept / reject decision of an
// adaptive solve built on it -- is reproducible run to run.  grid (nt, T-1, B), block 256.  np = 1: the single plane of a static
// control (one slab per graph, sums of piece `piece0` of the tables), in the same order as plane `a` of a dense one.
__global__ void __launch_bounds__(256) k_adj_rowsums(const float* __restrict__ adj_coef, int n, int npad, int Tm1, int piece0,
                                                     float* __restrict__ rowsum, int ncpad, int np) {
  __shared__ __align__(16) float tile[4096];
  const int b = blockIdx.z, iv = piece0 + blockIdx.y, rt = blockIdx.x;
  const int nt = ncpad >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;   // nt = column tiles (ncpad == npad for a square path)
  const size_t slab = (size_t)b * Tm1 + iv;
  const float* base = adj_coef + (np == 4 ? slab : (size_t)b) * np * (size_t)npad * ncpad + (size_t)rt * nt * (1024 * np);
  float acc[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) acc[p][rr] = 0.f;
  for (int ct = 0; ct < nt; ++ct) {
    for (int idx = threadIdx.x; idx < 256 * np; idx += 256)
      *reinterpret_cast<float4*>(&tile[4 * idx]) = *reinterpret_cast<const float4*>(base + (size_t)ct * (1024 * np) + 4 * idx);
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
        if (p < np) acc[p][rr] += warp_sum(tile[peg_tile_off(4 * warp + rr, lane, p, 1, np)]);
    __syncthreads();
  }
  if (lane == 0) {
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int i = rt * 32 + 4 * warp + rr;
        if (i < n && p < np) rowsum[(slab * 4 + p) * n + i] = acc[p][rr];
      }
  }
}

// total[slab][p] = sum_i rowsum[slab][p][i] in a fixed order.  grid (4 * pieces, B), block 256.
__global__ void __launch_bounds__(256) k_adj_totals(const float* __restrict__ rowsum, int n, int Tm1, int piece0,
                                                    float* __restrict__ total) {
  __shared__ float sh[33];
  const size_t idx = ((size_t)blockIdx.y * Tm1 + piece0) * 4 + blockIdx.x;   // (slab, plane)
  const float* r = rowsum + idx * n;
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) acc += r[i];
  const float t = block_sum(acc, sh);
  if (threadIdx.x == 0) total[idx] = t;
}

// max |entry| of each of the four planes of one cubic piece.  grid (tile chunks, pieces, B), block 256; fmaxf is order
// independent, so the atomicMax on the bit pattern (non-negative floats order like unsigned integers) is reproducible.
// np = 1: the single plane of a static control (slab b), written to slot `a` of piece `piece0`.
__global__ void __launch_bounds__(256) k_adj_absmax(const float* __restrict__ adj_coef, int npad, int Tm1, int piece0,
                                                    float* __restrict__ absmax, int ncpad, int np) {
  __shared__ float sh[8][4];
  const int b = blockIdx.z, iv = piece0 + blockIdx.y;
  const int ntiles = (npad >> 5) * (ncpad >> 5), warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t slab = (size_t)b * Tm1 + iv;
  const float4* base = reinterpret_cast<const float4*>(adj_coef + (np == 4 ? slab : (size_t)b) * np * (size_t)npad * ncpad);
  float mx[4] = {0.f, 0.f, 0.f, 0.f};
  // a tile is 1024 float4: index i -> plane (i >> 7) & 3   ([g][plane][m][lane] with 4 floats per lane)
  for (int t = blockIdx.x; t < ntiles; t += gridDim.x)
    for (int i = threadIdx.x; i < 256 * np; i += 256) {
      const float4 v = __ldg(base + (size_t)t * (256 * np) + i);
      const int q = np == 4 ? (i >> 7) & 3 : 0;       // warp-uniform per iteration? i = tid + 256 k: (i >> 7) & 3 depends on tid >> 7 -> two values per block
      const float m = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));
#pragma unroll
      for (int qq = 0; qq < 4; ++qq) mx[qq] = (q == qq) ? fmaxf(mx[qq], m) : mx[qq];
    }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float m = warp_max(mx[q]);
    if (lane == 0) sh[warp][q] = m;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    float m = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) m = fmaxf(m, sh[w8][threadIdx.x]);
    atomicMax(reinterpret_cast<unsigned int*>(absmax + slab * 4 + threadIdx.x), __float_as_uint(m));
  }
}

__global__ void k_fill_tch_unit(float* __restrict__ tch, int n, size_t slabs) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= slabs * 3 * n) return;
  const int p = (idx / n) % 3;
  tch[idx] = p == 0 ? 1.f : 0.f;
}

// Column sums of the four tiled planes (directed fusion layer: layers.py:256-345 uses jnp.sum(., axis=0)), deterministic:
// one block per 32-column tile walks the row tiles in order; thread (warp w, lane c) keeps rows 4w..4w+3 of column c.
// grid (nt, T-1, B), block 256.  np = 1: the single plane of a static control (slab b), written to slot `a` of piece blockIdx.y.
__global__ void __launch_bounds__(256) k_adj_colsums(const float* __restrict__ adj_coef, int n, int npad, int Tm1,
                                                     float* __restrict__ colsum, int np) {
  __shared__ __align__(16) float tile[4096];
  __shared__ float part[8][4][32];
  const int b = blockIdx.z, iv = blockIdx.y, ct = blockIdx.x;
  const int nt = npad >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t slab = (size_t)b * Tm1 + iv;
  const float* base = adj_coef + (np == 4 ? slab : (size_t)b) * np * (size_t)npad * npad;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int rt = 0; rt < nt; ++rt) {
    for (int idx = threadIdx.x; idx < 256 * np; idx += 256)
      *reinterpret_cast<float4*>(&tile[4 * idx]) = *reinterpret_cast<const float4*>(base + ((size_t)rt * nt + ct) * (1024 * np) + 4 * idx);
    __syncthreads();
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
        if (p < np) acc[p] += tile[peg_tile_off(4 * warp + rr, lane, p, 1, np)];
    __syncthreads();
  }
#pragma unroll
  for (int p = 0; p < 4; ++p) part[warp][p][lane] = acc[p];
  __syncthreads();
  if (warp < np) {   // plane = warp, column = lane: add the 8 row groups in a fixed order
    float t = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) t += part[w8][warp][lane];
    const int k = ct * 32 + lane;
    if (k < n) colsum[(slab * 4 + warp) * n + k] = t;
  }
}

// =====================================================================================
// row-sharded mode: the per-layer exchange over peer memory (PegShard in pegncde.h)
// =====================================================================================
#define PEG_MAX_WORLD 8
struct ShardXchg {
  void* vt_hi[PEG_MAX_WORLD];        // peer bases of the V^T halves (bytes), copied from the host tables of PegShard
  void* vt_lo[PEG_MAX_WORLD];
  int32_t* vexp[PEG_MAX_WORLD];
  float* colsum[PEG_MAX_WORLD];
  uint32_t* flags[PEG_MAX_WORLD];
  int rank, world;
  uint32_t epoch;            // value raised in the peers' flags by this exchange (plus *epoch_base when that is set)
  const uint32_t* epoch_base;   // nullable device word: exchanges completed by earlier calls / graph replays (even)
  size_t half_bytes;         // bytes of one epoch-parity half of a V^T buffer
  int push_vt;               // 0: only the column sums travel (no V^T in this exchange)
  int rows;                  // B * d rows of V^T
  size_t pitch_bytes;        // row pitch of V^T in bytes (= n_glob * element size)
  size_t col0_bytes, slice_bytes;   // this rank's columns of every row
  int vexp_half, vexp_stride, blk0, nblk_loc, B;   // block exponents: [2][B * vexp_stride], this rank owns blocks [blk0, blk0 + nblk_loc)
  int push_vexp;
  const float* cs_src[2];    // local column-sum vectors (nullable), cs_len floats each
  float* cs_dst[2];          // where the rank-ordered sums go (k_shard_wait)
  int cs_len;
  size_t cs_half;            // floats of one epoch-parity half of the column-sum slots = world * 2 * cs_cap
  size_t cs_cap;             // floats reserved per (rank, vector)
  unsigned int* ticket;      // local arrival counter of k_shard_push (self-resetting)
};

// Copies this rank's slice of V^T (both parts), its block exponents and its column-sum vectors into every peer's buffers with
// 128-bit stores over NVLink, then raises flags[rank] = epoch on every peer (release at system scope).  grid (blocks, world - 1... the
// local copy needs no transfer: the producers wrote the local buffer in place), block 256.  blockIdx.y = peer slot.
__global__ void __launch_bounds__(256) k_shard_push(const ShardXchg x) {
  const int par = (int)(x.epoch & 1u);
  const int peer = blockIdx.y;                  // every rank, including this one (column sums go to the own slot too)
  const bool remote = peer != x.rank;
  if (x.push_vt && remote) {
    const char* src_hi = (const char*)x.vt_hi[x.rank] + par * x.half_bytes, *src_lo = (const char*)x.vt_lo[x.rank] + par * x.half_bytes;
    char* dst_hi = (char*)x.vt_hi[peer] + par * x.half_bytes, *dst_lo = (char*)x.vt_lo[peer] + par * x.half_bytes;
    const size_t v16 = x.slice_bytes / 16;      // the slice is a multiple of 128 nodes x >= 2 bytes
    const size_t total = (size_t)x.rows * v16;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
      const size_t r = i / v16, c = i - r * v16;
      const size_t off = r * x.pitch_bytes + x.col0_bytes + c * 16;
      *reinterpret_cast<uint4*>(dst_hi + off) = *reinterpret_cast<const uint4*>(src_hi + off);
      *reinterpret_cast<uint4*>(dst_lo + off) = *reinterpret_cast<const uint4*>(src_lo + off);
    }
    if (x.push_vexp && blockIdx.x == 0) {
      const int32_t* s = x.vexp[x.rank] + (size_t)par * x.vexp_half;
      int32_t* d = x.vexp[peer] + (size_t)par * x.vexp_half;
      for (int i = threadIdx.x; i < x.B * x.nblk_loc; i += blockDim.x) {
        const int b = i / x.nblk_loc, k = i - b * x.nblk_loc;
        d[(size_t)b * x.vexp_stride + x.blk0 + k] = s[(size_t)b * x.vexp_stride + x.blk0 + k];
      }
    }
  }
  if (blockIdx.x == 0) {
    for (int v = 0; v < 2; ++v) {
      if (!x.cs_src[v]) continue;
      float* d = x.colsum[peer] + (size_t)par * x.cs_half + ((size_t)x.rank * 2 + v) * x.cs_cap;
      for (int i = threadIdx.x; i < x.cs_len; i += blockDim.x) d[i] = x.cs_src[v][i];
    }
  }
  // all blocks of this launch done -> publish
  __threadfence_system();
  __syncthreads();
  __shared__ bool last;
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(x.ticket, 1u);
    last = (t == gridDim.x * gridDim.y - 1u);
    if (last) *x.ticket = 0u;
  }
  __syncthreads();
  if (last) {
    __threadfence_system();
    const uint32_t epoch = x.epoch + (x.epoch_base ? *reinterpret_cast<const volatile uint32_t*>(x.epoch_base) : 0u);
    for (int q = threadIdx.x; q < x.world; q += blockDim.x) {
      volatile uint32_t* f = x.flags[q] + x.rank;
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(epoch) : "memory");
    }
  }
}

// Waits until every rank has raised this exchange's epoch in the local flags, then adds the column-sum slots in rank order
// (deterministic) into the local vectors.  One block.  A peer that never arrives (an error on another rank) must not hang the
// GPU: after ~2 s of spinning the kernel gives up and records the failure in the error word flags[world] (checked by the host).
__global__ void __launch_bounds__(256) k_shard_wait(const ShardXchg x) {
  const int par = (int)(x.epoch & 1u);
  __shared__ int ok;
  if (threadIdx.x == 0) ok = 1;
  __syncthreads();
  if (threadIdx.x < x.world) {
    const uint32_t epoch = x.epoch + (x.epoch_base ? *reinterpret_cast<const volatile uint32_t*>(x.epoch_base) : 0u);
    const uint32_t* f = x.flags[x.rank] + threadIdx.x;
    const long long t0 = clock64();
    uint32_t v;
    while (true) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
      if ((int32_t)(v - epoch) >= 0) break;
      if (clock64() - t0 > 4000000000ll) { ok = 0; x.flags[x.rank][x.world] = 1u; break; }
      __nanosleep(200);
    }
  }
  __syncthreads();
  if (!ok) return;
  for (int v = 0; v < 2; ++v) {
    if (!x.cs_dst[v]) continue;
    const float* base = x.colsum[x.rank] + (size_t)par * x.cs_half + (size_t)v * x.cs_cap;
    for (int i = threadIdx.x; i < x.cs_len; i += blockDim.x) {
      float t = 0.f;
      for (int q = 0; q < x.world; ++q) t += __ldcg(base + (size_t)q * 2 * x.cs_cap + i);
      x.cs_dst[v][i] = t;
    }
  }
}

// end of an API call in graph-replayable mode: the epoch base moves past this call's exchanges
__global__ void k_epoch_advance(uint32_t* base, uint32_t count) { *base += count; }

// x coeffs: d,c,b,a each [B,T-1,n,e,2] -> x_coef [B,T-1,3,n,2e] (b,c,d)
__global__ void k_pack_x(const float* __restrict__ cd, const float* __restrict__ cc, const float* __restrict__ cb,
                         int n, int e2, size_t slabs, float* __restrict__ x_coef) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t per = (size_t)n * e2;
  if (idx >= slabs * per) return;
  const size_t slab = idx / per, r = idx % per;
  x_coef[(slab * 3 + 0) * per + r] = cb[idx];
  x_coef[(slab * 3 + 1) * per + r] = cc[idx];
  x_coef[(slab * 3 + 2) * per + r] = cd[idx];
}

// =====================================================================================
// per-stage scalars and O(n) vectors (control interpolation of everything that is not
// the n x n planes themselves: row sums, diagonals, totals are linear in the planes)
// =====================================================================================
struct PrepArgs {
  PegControl ctl;
  const float* params;
  Model model;
  int n_glob;   // node count the 1/n, 1/n^2 factors refer to (== n unless row-sharded)
  int B, n, e, T;
  float t;
  const float* t_dev;    // nullable: per-graph stage time = t_dev[b] + tcoef * dt_dev[b] (batched adaptive steps)
  const float* dt_dev;
  float tcoef;
  StageScalars* sc;
  float* svec;
};

// grid (ceil(max(n, n*2e/.. )/256), B): every block redoes the (tiny) interval search, then handles 256 nodes
__global__ void __launch_bounds__(256) k_stage_prep(PrepArgs a) {
  __shared__ float sh[40];
  __shared__ StageScalars S;
  const int b = blockIdx.y, tid = threadIdx.x;
  const int n = a.n, L = a.model.L, Tm1 = a.T - 1;
  const float* ts = a.ctl.ts + (size_t)b * a.T;
  const float tq = a.t_dev ? a.t_dev[b] + a.tcoef * a.dt_dev[b] : a.t;      // the stage time of this graph
  // index = clip(searchsorted(ts, t, 'left') - 1, 0, T-2)  (diffrax CubicInterpolation._interpret_t)
  float cnt = 0.f;
  for (int i = tid; i < a.T; i += blockDim.x) cnt += (ts[i] < tq) ? 1.f : 0.f;
  cnt = block_sum(cnt, sh);
  int iv = (int)(cnt + 0.5f) - 1;
  iv = max(0, min(iv, a.T - 2));
  const float s = tq - ts[iv];
  const float wA[4] = {1.f, s, s * s, s * s * s};
  const float wD[4] = {0.f, 1.f, 2.f * s, 3.f * s * s};
  const size_t slab = (size_t)b * Tm1 + iv;
  const float* tot = a.ctl.adj_total + slab * 4;
  const float totA = wA[0] * tot[0] + wA[1] * tot[1] + wA[2] * tot[2] + wA[3] * tot[3];
  const float totD = wD[1] * tot[1] + wD[2] * tot[2] + wD[3] * tot[3];
  const float inv_n = 1.f / (float)a.n_glob, inv_n2 = inv_n * inv_n;
  if (tid == 0 && blockIdx.x == 0) {
    S.interval = iv;
    S.s = s;
    for (int p = 0; p < 4; ++p) { S.wA[p] = wA[p]; S.wD[p] = wD[p]; }
    S.totA = totA;
    S.totD = totD;
    for (int p = 0; p < 4; ++p) S.amax[p] = a.ctl.adj_absmax ? a.ctl.adj_absmax[slab * 4 + p] : 0.f;
    for (int l = 0; l < L; ++l) {
      const float* f = a.params + a.model.layer[l].fus_off;
      S.kappa[l] = (f[12] + f[13]) * totA * inv_n2;
    }
    a.sc[b] = S;
  }
  float* sv = a.svec + (size_t)b * svec_stride(n, L, a.e);
  const float* rs = a.ctl.adj_rowsum + slab * 4 * n;
  const float* dg = a.ctl.adj_diag + slab * 4 * n;
  const float* tc = a.ctl.tch_coef + slab * 3 * n;
  const float* cs = a.model.directed ? a.ctl.adj_colsum + slab * 4 * n : nullptr;
  for (int i = blockIdx.x * blockDim.x + tid; i < n; i += gridDim.x * blockDim.x) {
    const float rA = wA[0] * rs[i] + wA[1] * rs[n + i] + wA[2] * rs[2 * n + i] + wA[3] * rs[3 * n + i];
    const float rD = wD[1] * rs[n + i] + wD[2] * rs[2 * n + i] + wD[3] * rs[3 * n + i];
    const float dA = wA[0] * dg[i] + wA[1] * dg[n + i] + wA[2] * dg[2 * n + i] + wA[3] * dg[3 * n + i];
    const float dD = wD[1] * dg[n + i] + wD[2] * dg[2 * n + i] + wD[3] * dg[3 * n + i];
    sv[svec_rA(n, L) + i] = rA;
    sv[svec_rD(n, L) + i] = rD;
    sv[svec_dgA(n, L) + i] = dA;
    sv[svec_dgD(n, L) + i] = dD;
    float cA = 0.f, cD = 0.f;
    if (cs) {
      cA = wA[0] * cs[i] + wA[1] * cs[n + i] + wA[2] * cs[2 * n + i] + wA[3] * cs[3 * n + i];
      cD = wD[1] * cs[n + i] + wD[2] * cs[2 * n + i] + wD[3] * cs[3 * n + i];
      sv[svec_cA(n, L) + i] = cA;
      sv[svec_cD(n, L) + i] = cD;
    }
    for (int l = 0; l < L; ++l) {
      const float* f = a.params + a.model.layer[l].fus_off;
      if (!cs) {   // ConvEquivFusionLayer (layers.py:102-160): row sums only
        sv[svec_v(n, l) + i] = f[4] * dA + f[5] * dD + (f[10] * rA + f[11] * rD) * inv_n + (f[14] * totA + f[15] * totD) * inv_n2;
        sv[svec_r(n, l) + i] = (f[6] * rA + f[7] * rD) * inv_n;
        sv[svec_c(n, l) + i] = (f[8] * rA + f[9] * rD) * inv_n;
      } else {     // ConvEquivFusionDirectedLayer (layers.py:256-345); f[16..21] = param4', param5', param6'
        // term 6 / 6': diag(colsum), diag(rowsum); term 4: colsum_i on row i; term 4': rowsum(A)_j, colsum(A')_j (reference quirk:
        // axis=0 for the derivative) on column j; term 5: colsum_j; term 5': rowsum_j
        sv[svec_v(n, l) + i] = f[4] * dA + f[5] * dD + (f[10] * cA + f[11] * cD) * inv_n + (f[20] * rA + f[21] * rD) * inv_n +
                               (f[14] * totA + f[15] * totD) * inv_n2;
        sv[svec_r(n, l) + i] = (f[6] * cA + f[7] * cD) * inv_n;
        sv[svec_c(n, l) + i] = (f[16] * rA + f[17] * cD) * inv_n + (f[8] * cA + f[9] * cD) * inv_n + (f[18] * rA + f[19] * rD) * inv_n;
      }
    }
    sv[svec_tg(n, L) + i] = tc[i] + s * (2.f * tc[n + i] + 3.f * s * tc[2 * n + i]);
  }
  if (a.e > 0) {
    const int e2 = 2 * a.e;
    const size_t per = (size_t)n * e2;
    const float* xc = a.ctl.x_coef + slab * 3 * per;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + tid; i < per; i += (size_t)gridDim.x * blockDim.x)
      sv[svec_xd(n, L) + i] = xc[i] + s * (2.f * xc[per + i] + 3.f * s * xc[2 * per + i]);
  }
}

// =====================================================================================
// Runge-Kutta linear combinations: out = sum_j c[j] * x[j]   (stage inputs, y update,
// adjoint stage cotangents).  float4-vectorised; count multiple of 4.
// =====================================================================================
struct CombArgs {
  const float* x[8];
  float c[8];
  int cnt;
  float* out;
  size_t count4;
  // batched adaptive steps: every graph has its own step size -- coefficients c[j], j >= 1, are multiplied by gscale[graph]
  const float* gscale;   // nullable [B]
  size_t per_graph4;     // float4 elements per graph
};
__global__ void __launch_bounds__(256) k_rk_combine(CombArgs a) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.count4) return;
  const float gs = a.gscale ? a.gscale[i / a.per_graph4] : 1.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (j < a.cnt) {
      const float4 v = reinterpret_cast<const float4*>(a.x[j])[i];
      const float c = (j > 0 && a.gscale) ? a.c[j] * gs : a.c[j];
      acc.x = fmaf(c, v.x, acc.x);
      acc.y = fmaf(c, v.y, acc.y);
      acc.z = fmaf(c, v.z, acc.z);
      acc.w = fmaf(c, v.w, acc.w);
    }
  }
  reinterpret_cast<float4*>(a.out)[i] = acc;
}

// =====================================================================================
// Scaled error norm of adaptive step-size control (diffrax PIDController: rms_norm(err / (atol + rtol max(|y0|,|y1|))),
// also the three norms of the initial-step heuristic):  out[b] = sum_i ((x - x2) / (atol + rtol max(|s0|, |s1|)))^2.
// One block per graph, fixed summation order (deterministic accept / reject decisions).  grid (B), block 1024.
// =====================================================================================
__global__ void __launch_bounds__(1024) k_scaled_sumsq(const float* __restrict__ x, const float* __restrict__ x2,
                                                       const float* __restrict__ s0, const float* __restrict__ s1,
                                                       float rtol, float atol, size_t per_graph, float* __restrict__ out) {
  __shared__ float sh[33];
  const size_t base = (size_t)blockIdx.x * per_graph;
  float acc = 0.f;
  for (size_t i = threadIdx.x; i < per_graph; i += blockDim.x) {
    const float a = fabsf(s0[base + i]);
    const float m = s1 ? fmaxf(a, fabsf(s1[base + i])) : a;
    const float v = (x[base + i] - (x2 ? x2[base + i] : 0.f)) / (atol + rtol * m);
    acc = fmaf(v, v, acc);
  }
  const float tot = block_sum(acc, sh);
  if (threadIdx.x == 0) out[blockIdx.x] = tot;
}

// =====================================================================================
// Batched adaptive step-size control on the device (diffrax PIDController(rtol, atol) with its defaults pcoeff = 0, icoeff = 1,
// dcoeff = 0 + _clip_to_end, call site src/models/graph_neural_cde.py:53-54,86-104): every trajectory of the batch keeps its own
// (tprev, tnext), accepted-step table and dense-output bookkeeping in device memory, so a batch advances with ONE step launch per
// attempt and no host round trip per step.
// =====================================================================================
struct AdaptState {        // one per trajectory (PegAdaptState in pegncde.h)
  float tprev, tnext;      // the step that is being / will be attempted
  int done, nacc, attempts, rejected;
  int mi;                  // next save time to emit
  int mi0, mi1;            // save indices emitted by the step just accepted: [mi0, mi1)
  int keep;                // decision for the step just attempted
  float h;                 // its size
  int overflow;            // the accepted-step table is full (the host grows it)
};

// one thread per trajectory: decide, record, choose the next step
__global__ void k_adapt_decide(AdaptState* st, const float* __restrict__ sumsq, int B, float nh, float t1, float safety, float factormin,
                               float factormax, float inv_order, const float* __restrict__ save_ts, int M, int cap,
                               float* __restrict__ step_tab /* [B][cap+1] */, int* __restrict__ sample_step /* [M][B] */,
                               float* __restrict__ sample_theta /* [M][B] */, float* __restrict__ dt_out /* [B] next h */,
                               float* __restrict__ t_out /* [B] next tprev */) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  AdaptState s = st[b];
  s.keep = 0; s.mi0 = s.mi1 = s.mi;
  if (!s.done && !s.overflow) {
    const float h = s.tnext - s.tprev;
    const float err = sqrtf(sumsq[b] / nh);
    const bool keep = err < 1.0f;
    float inv = 1.0f / err;
    if (!isfinite(inv)) inv = isnan(inv) ? 1.0f : 3.402823466e+38f;
    float factor = safety * powf(inv, inv_order);
    factor = fminf(fmaxf(factor, keep ? 1.0f : factormin), factormax);
    const float dt_new = h * factor;
    s.attempts += 1;
    s.h = h;
    float tprev_new = s.tprev;
    if (keep) {
      if (s.nacc >= cap) { s.overflow = 1; s.attempts -= 1; }
      else {
        s.keep = 1;
        while (s.mi1 < M && save_ts[s.mi1] <= s.tnext) {
          const float theta = fminf(fmaxf((save_ts[s.mi1] - s.tprev) / h, 0.f), 1.f);
          sample_step[(size_t)s.mi1 * B + b] = s.nacc;
          sample_theta[(size_t)s.mi1 * B + b] = theta;
          s.mi1 += 1;
        }
        s.mi = s.mi1;
        s.nacc += 1;
        step_tab[(size_t)b * (cap + 1) + s.nacc] = s.tnext;
        tprev_new = s.tnext;
      }
    } else {
      s.rejected += 1;
    }
    if (!s.overflow) {
      float tn = tprev_new + dt_new;
      if (tn > t1 - 1e-6f) tn = keep ? t1 : tprev_new + 0.5f * (t1 - tprev_new);     // diffrax _clip_to_end (fp32 times)
      s.tprev = tprev_new;
      s.tnext = tn;
      if (keep && tprev_new >= t1) s.done = 1;
    }
  }
  st[b] = s;
  t_out[b] = s.tprev;
  dt_out[b] = (s.done || s.overflow) ? 0.f : s.tnext - s.tprev;
}

// elementwise: dense-output samples of the accepted step, then y <- y1, k1 <- k7 (FSAL) and the checkpoint, per trajectory
__global__ void __launch_bounds__(256) k_adapt_apply(const AdaptState* __restrict__ st, int B, size_t per_graph4, int cap,
                                                     float4* __restrict__ y, const float4* __restrict__ y1, float4* __restrict__ k1,
                                                     const float4* __restrict__ k7, const float4* __restrict__ kst /* [5][B][nh] */,
                                                     float4* __restrict__ y_ckpt /* [B][cap+1][nh] */, float4* __restrict__ ys_save /* [M][B][nh] */,
                                                     const float* __restrict__ sample_theta) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * per_graph4) return;
  const int b = (int)(i / per_graph4);
  const size_t e = i - (size_t)b * per_graph4;
  const AdaptState s = st[b];
  if (!s.keep) return;
  const float4 yv = y[i], k1v = k1[i], k7v = k7[i];
  if (s.mi1 > s.mi0) {
    float4 ks[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) ks[q] = kst[(size_t)q * B * per_graph4 + i];
    for (int m = s.mi0; m < s.mi1; ++m) {
      const float th = sample_theta[(size_t)m * B + b];
      // Tsit5 dense-output weights b_i(theta) (the expanded Horner form of pegncde_tsit5_dense_weights)
      const float r[7][4] = {{1.0f, -2.763706197274826f, 2.9132554618219126f, -1.0530884977290216f},
                             {0.0f, 0.13169999999999998f, -0.2234f, 0.1017f},
                             {0.0f, 3.9302962368947516f, -5.941033872131505f, 2.490627285651253f},
                             {0.0f, -12.411077166933676f, 30.33818863028232f, -16.548102889244902f},
                             {0.0f, 37.50931341651104f, -88.1789048947664f, 47.37952196281928f},
                             {0.0f, -27.896526289197286f, 65.09189467479366f, -34.87065786149661f},
                             {0.0f, 1.5f, -4.0f, 2.5f}};
      float w[7];
#pragma unroll
      for (int q = 0; q < 7; ++q) w[q] = s.h * (th * (r[q][0] + th * (r[q][1] + th * (r[q][2] + th * r[q][3]))));
      float4 o = yv;
      auto axpy = [&](float c, const float4& v) { o.x = fmaf(c, v.x, o.x); o.y = fmaf(c, v.y, o.y); o.z = fmaf(c, v.z, o.z); o.w = fmaf(c, v.w, o.w); };
      axpy(w[0], k1v);
#pragma unroll
      for (int q = 0; q < 5; ++q) axpy(w[q + 1], ks[q]);
      axpy(w[6], k7v);
      ys_save[((size_t)m * B + b) * per_graph4 + e] = o;
    }
  }
  const float4 ynew = y1[i];
  y[i] = ynew;
  k1[i] = k7v;
  y_ckpt[((size_t)b * (cap + 1) + s.nacc) * per_graph4 + e] = ynew;
}

// =====================================================================================
// RMSNorm -> Linear  (layers.py:45-46): M = (w_n * z * rsqrt(mean z^2 + eps) + b_n) W^T + b
// The norm is linear in z up to the per-node scale, so it moves to the epilogue:
//     M[node][o] = rinv[node] * sum_k z[node][k] (w_n[k] W[o][k])  +  (sum_k b_n[k] W[o][k] + b[o])
// -> one pass over Z (sum z^2 is accumulated while the K chunks stream through), a plain 128 x 64 x d_in GEMM
// with 8 x 4 outputs per thread, and a fused epilogue that also emits V^T hi/lo and the column sums.
// grid (ceil(n/128), ceil(dout/64), B), block 256
// =====================================================================================
constexpr int NL_BM = 128, NL_BN = 64, NL_BK = 32;
__global__ void __launch_bounds__(256) k_norm_linear(const float* __restrict__ Z, int n, int din, int dout,
                                                     const float* __restrict__ W, const float* __restrict__ bias,
                                                     const float* __restrict__ nw, const float* __restrict__ nb,
                                                     float* __restrict__ M, float* __restrict__ Nout, ProducerOut po) {
  __shared__ bool is_last;
  __shared__ __align__(16) float zt[NL_BK][NL_BM + 4];   // [k][node]  raw input chunk
  __shared__ __align__(16) float wt[NL_BK][NL_BN + 4];   // [k][out]   W * norm weight
  __shared__ float rinv_s[NL_BM];
  __shared__ float cvec_s[NL_BN];
  const int tid = threadIdx.x;
  const int b = blockIdx.z, node0 = blockIdx.x * NL_BM, o0 = blockIdx.y * NL_BN;
  const float* Zb = Z + (size_t)b * n * din;
  const int ty = tid >> 4, tx = tid & 15;       // compute mapping: rows 8ty..8ty+7, cols 4tx..4tx+3
  const int zr = tid >> 1, zk = (tid & 1) * 16; // Z loader: row zr, 16 consecutive k
  const int wo = tid >> 2, wk = (tid & 3) * 8;  // W loader: out wo, 8 consecutive k
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float sumsq = 0.f, cpart = 0.f;
  const bool zrow_ok = node0 + zr < n, wrow_ok = o0 + wo < dout;
  for (int k0 = 0; k0 < din; k0 += NL_BK) {
    {
      float4 z4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = k0 + zk + 4 * u;
        z4[u] = (zrow_ok && k < din) ? *reinterpret_cast<const float4*>(Zb + (size_t)(node0 + zr) * din + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      float4 w4[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int k = k0 + wk + 4 * u;
        w4[u] = (wrow_ok && k < din) ? *reinterpret_cast<const float4*>(W + (size_t)(o0 + wo) * din + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float zz[4] = {z4[u].x, z4[u].y, z4[u].z, z4[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          sumsq = fmaf(zz[e], zz[e], sumsq);
          zt[zk + 4 * u + e][zr] = zz[e];
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float ww[4] = {w4[u].x, w4[u].y, w4[u].z, w4[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int k = k0 + wk + 4 * u + e;
          const float sw = k < din ? nw[k] : 0.f, sb = k < din ? nb[k] : 0.f;
          cpart = fmaf(sb, ww[e], cpart);
          wt[wk + 4 * u + e][wo] = ww[e] * sw;
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NL_BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&zt[k][8 * ty]);
      const float4 a1 = *reinterpret_cast<const float4*>(&zt[k][8 * ty + 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&wt[k][4 * tx]);
      const float aa[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  // per-node rsqrt(mean z^2 + eps) (2 loader threads per row) and the constant vector (4 loader threads per out)
  sumsq += __shfl_xor_sync(0xffffffffu, sumsq, 1);
  cpart += __shfl_xor_sync(0xffffffffu, cpart, 1);
  cpart += __shfl_xor_sync(0xffffffffu, cpart, 2);
  if ((tid & 1) == 0) rinv_s[zr] = rsqrtf(sumsq / (float)din + 1e-5f);
  if ((tid & 3) == 0) cvec_s[wo] = cpart + (wrow_ok ? bias[o0 + wo] : 0.f);
  __syncthreads();
  if (Nout != nullptr && blockIdx.y == 0 && zrow_ok) {   // normalised input (needed by the weight gradient)
    float* Nb = Nout + ((size_t)b * n + node0 + zr) * din;
    const float* Zr = Zb + (size_t)(node0 + zr) * din;
    const float ri = rinv_s[zr];
    for (int k = (tid & 1) * 4; k < din; k += 8) {
      const float4 z4 = *reinterpret_cast<const float4*>(Zr + k);
      const float4 s4 = *reinterpret_cast<const float4*>(nw + k), t4 = *reinterpret_cast<const float4*>(nb + k);
      *reinterpret_cast<float4*>(Nb + k) = make_float4(z4.x * ri * s4.x + t4.x, z4.y * ri * s4.y + t4.y, z4.z * ri * s4.z + t4.z, z4.w * ri * s4.w + t4.w);
    }
  }
  float* Mb = M + (size_t)b * n * dout;
  const int oc = o0 + 4 * tx;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int node = node0 + 8 * ty + i;
    const float ri = rinv_s[8 * ty + i];
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = (node < n && oc + j < dout) ? fmaf(ri, acc[i][j], cvec_s[4 * tx + j]) : 0.f;
    if (node >= n) continue;
    if (oc + 3 < dout) {
      *reinterpret_cast<float4*>(Mb + (size_t)node * dout + oc) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (oc + j < dout) Mb[(size_t)node * dout + oc + j] = acc[i][j];
    }
  }
  // ---- fused producer outputs (acc now holds M, zero outside [0,n) x [0,dout)) ----
  if (po.Thi != nullptr) {
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      const int nodeq = node0 + 8 * ty + 4 * hh;   // 4 consecutive nodes -> one float4 along the node axis of V^T
      if (nodeq < po.npad) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (oc + j >= dout) continue;
          const size_t o = ((size_t)b * dout + oc + j) * po.npad + nodeq;
          store_vt4(po, o, acc[4 * hh][j], acc[4 * hh + 1][j], acc[4 * hh + 2][j], acc[4 * hh + 3][j]);
        }
      }
    }
  }
  if (po.cb != nullptr) {
    // partial column sums over this block's 128 nodes: reduce the 16 thread rows through smem (zt is free now)
    float (*r0)[NL_BM + 4] = zt;                                  // rows 0..15  : plain sums   [ty][col]
    float (*r1)[NL_BM + 4] = reinterpret_cast<float (*)[NL_BM + 4]>(&zt[16][0]);   // rows 16..31 : weighted sums
    const float* vb = po.vec ? po.vec + (size_t)b * po.vec_stride : nullptr;
    float t0[4] = {0.f, 0.f, 0.f, 0.f}, t1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int node = node0 + 8 * ty + i;
      const float vv = (vb && node < n) ? vb[node] : 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) { t0[j] += acc[i][j]; t1[j] = fmaf(vv, acc[i][j], t1[j]); }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) { r0[ty][4 * tx + j] = t0[j]; r1[ty][4 * tx + j] = t1[j]; }
    __syncthreads();
    const int chunks = gridDim.x;
    if (tid < NL_BN && o0 + tid < dout) {
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int k = 0; k < 16; ++k) { s0 += r0[k][tid]; s1 += r1[k][tid]; }
      float* part = po.partial + (((size_t)b * chunks + blockIdx.x) * 2) * dout;
      part[o0 + tid] = s0;
      part[dout + o0 + tid] = s1;
    }
    finalize_colsums(po, b, chunks, dout, o0, NL_BN, po.tickets + (size_t)b * gridDim.y + blockIdx.y, &is_last);
  }
}

// =====================================================================================
// column reductions: cb[b][0][c] = sum_i V[b,i,c] ; cb[b][1][c] = sum_i vec[b][i] V[b,i,c]
// grid (ceil(d/32), ceil(n/CS_ROWS), B), block (32, 8).  Deterministic: every block writes its partial sums,
// the last block to finish (per column block) adds them in a fixed order; the ticket counter resets itself.
// =====================================================================================
constexpr int CS_ROWS = 256;

__global__ void __launch_bounds__(256) k_colsums(const float* __restrict__ V, int n, int d,
                                                 const float* __restrict__ vec, size_t vec_stride,
                                                 float* __restrict__ cb, float* __restrict__ partial,
                                                 unsigned int* __restrict__ tickets) {
  __shared__ float s0[8][33], s1[8][33];
  __shared__ bool is_last;
  const int b = blockIdx.z, c = blockIdx.x * 32 + threadIdx.x;
  const int r0 = blockIdx.y * CS_ROWS, r1 = min(n, r0 + CS_ROWS);
  const int chunks = gridDim.y;
  const float* Vb = V + (size_t)b * n * d;
  const float* vb = vec ? vec + (size_t)b * vec_stride : nullptr;
  float a0 = 0.f, a1 = 0.f;
  if (c < d) {
    for (int i = r0 + threadIdx.y; i < r1; i += 8) {
      const float v = Vb[(size_t)i * d + c];
      a0 += v;
      if (vb) a1 = fmaf(vb[i], v, a1);
    }
  }
  s0[threadIdx.y][threadIdx.x] = a0;
  s1[threadIdx.y][threadIdx.x] = a1;
  __syncthreads();
  float* part = partial + (((size_t)b * chunks + blockIdx.y) * 2) * d;
  if (threadIdx.y == 0 && c < d) {
#pragma unroll
    for (int k = 1; k < 8; ++k) { a0 += s0[k][threadIdx.x]; a1 += s1[k][threadIdx.x]; }
    part[c] = a0;
    part[d + c] = a1;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && threadIdx.y == 0) {
    unsigned int* tk = tickets + (size_t)b * gridDim.x + blockIdx.x;
    const unsigned int t = atomicAdd(tk, 1u);
    is_last = (t == (unsigned int)chunks - 1u);
    if (is_last) *tk = 0u;
  }
  __syncthreads();
  if (is_last && threadIdx.y == 0 && c < d) {
    __threadfence();
    float t0 = 0.f, t1 = 0.f;
    for (int k = 0; k < chunks; ++k) {
      const float* pk = partial + (((size_t)b * chunks + k) * 2) * d;
      t0 += __ldcg(pk + c);
      t1 += __ldcg(pk + d + c);
    }
    cb[((size_t)b * 2 + 0) * d + c] = t0;
    cb[((size_t)b * 2 + 1) * d + c] = t1;
  }
}

// =====================================================================================
// The matrix-free equivariant contraction (never builds the n x n fused adjacency):
//   forward  (NACC=1): OUT = V(1+v) + X V + Y^T V + rowc (1^T V) + 1 (vec^T V + kappa 1^T V)
//       with X = (1+p1_0) A_s + (1+p1_1) A'_s,  Y = p2_0 A_s + p2_1 A'_s   (layers.py:114-160)
//   backward (NACC=4): separate products A V, A'V, A^T V, A'^T V so the same pass also
//       yields the Frobenius products that are the gradients of param1 / param2.
// A_s and A'_s are formed on the fly from the four cubic-coefficient planes.
// grid (ceil(n/64), ceil(d/64), B), block 256; thread tile 4x4
// =====================================================================================

constexpr int CT_TI = 64, CT_TC = 64, CT_KC = 16, CT_LD = CT_TI + 4;

// Epilogue of the contraction for row gi, columns gc..gc+3 (shared by k_dual_contract and k_sparse_contract in peg_sparse.cuh).
// acc[.][i] = the products of this row (forward: [0] = X V + Y^T V; backward: A V, A'V, A^T V, A'^T V), ss / tt = the column sums
// 1^T V / vec^T V of these columns, Vb = V of graph b, alpha..delta = 1 + p1_0, 1 + p1_1, p2_0, p2_1.  Writes OUT; backward: adds the param1 / param2
// Frobenius-product terms of this row to g4.
template <int NACC, int R>
__device__ __forceinline__ void contract_epilogue4(const ContractArgs& a, int b, int gi, int gc, const float* __restrict__ sv, const float* Vb,
                                                   const float (&acc)[NACC][R][4], int i, const float (&ss)[4], const float (&tt)[4],
                                                   float kappa, float alpha, float beta, float gamma, float delta, float (&g4)[4]) {
  const int n = a.n, d = a.d;
  const float vi = 1.f + sv[a.v_off + gi];
  const float rc = sv[a.rowc_off + gi];
  const float tg = a.scale_tg ? sv[a.tg_off + gi] : 1.f;
  const float4 vin = *reinterpret_cast<const float4*>(Vb + (size_t)gi * d + gc);
  const float vv[4] = {vin.x, vin.y, vin.z, vin.w};
  float o[4];
  if (NACC == 1) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float val = vv[j] * vi + acc[0][i][j] + rc * ss[j] + tt[j] + kappa * ss[j];
      if (a.relu) val = fmaxf(val, 0.f);
      o[j] = val * tg;
    }
  } else {
    const float4 m4 = *reinterpret_cast<const float4*>(a.Mref + ((size_t)b * n + gi) * d + gc);
    const float mm[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      // acc[0]=A V, acc[1]=A'V, acc[2]=A^T V, acc[3]=A'^T V   (V = cotangent of the layer output)
      o[j] = vv[j] * vi + alpha * acc[2][i][j] + beta * acc[3][i][j] + gamma * acc[0][i][j] +
             delta * acc[1][i][j] + rc * ss[j] + tt[j] + kappa * ss[j];
      g4[0] = fmaf(acc[2][i][j], mm[j], g4[0]);  // d/d param1[0] = <A^T g, M>
      g4[1] = fmaf(acc[3][i][j], mm[j], g4[1]);  // d/d param1[1] = <A'^T g, M>
      g4[2] = fmaf(acc[0][i][j], mm[j], g4[2]);  // d/d param2[0] = <A g, M>
      g4[3] = fmaf(acc[1][i][j], mm[j], g4[3]);  // d/d param2[1] = <A' g, M>
    }
  }
  *reinterpret_cast<float4*>(a.out + ((size_t)b * n + gi) * d + gc) = make_float4(o[0], o[1], o[2], o[3]);
}

// STAT: static control (ContractArgs.stat): one plane per graph, read for every piece; planes b, c, d are exact zeros, so the
// arithmetic below is the dense control's on the snapshots [A] * T and the result is the same bit for bit
template <int NACC, bool STAT = false>
__global__ void __launch_bounds__(256) k_dual_contract(ContractArgs a) {
  constexpr int NS = (NACC == 1) ? 2 : 4;
  __shared__ __align__(16) float S[NS][CT_KC][CT_LD];
  __shared__ __align__(16) float Vs[CT_KC][CT_TC];
  __shared__ float red[40];
  const int tid = threadIdx.x;
  const int b = blockIdx.z, i0 = blockIdx.x * CT_TI, c0 = blockIdx.y * CT_TC;
  const int n = a.n, d = a.d;
  const StageScalars sc = a.sc[b];
  const float alpha = 1.f + a.fus[0], beta = 1.f + a.fus[1], gamma = a.fus[2], delta = a.fus[3];
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
  const int npad = a.ldn, nt = npad >> 5;
  const float* P = a.planes + (size_t)b * a.graph_stride + (STAT ? 0 : (size_t)sc.interval * 4 * npad * npad);
  constexpr int NPL = STAT ? 1 : 4;
  const float* Vb = a.V + (size_t)b * n * d;

  float acc[NACC][4][4];
#pragma unroll
  for (int q = 0; q < NACC; ++q)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[q][i][j] = 0.f;

  const int ty = tid >> 4, tx = tid & 15;
  // direct tile: element (row i, col k);  transposed tile: element (row k, col i)
  const int drow = tid >> 2, dkq = tid & 3;
  const int tkr = tid >> 4, tiq = tid & 15;

  for (int k0 = 0; k0 < n; k0 += CT_KC) {
    {  // direct part
      const int gi = i0 + drow, gk = k0 + 4 * dkq;
      float4 p[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) p[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gi < npad && gk < npad) {   // padding is zero-filled by the pack pre-pass
#pragma unroll
        for (int q = 0; q < NPL; ++q) p[q] = *reinterpret_cast<const float4*>(P + peg_tile_off(gi, gk, q, nt, NPL));
      }
      float x0[4], x1[4];
      const float* pf = reinterpret_cast<const float*>(p);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool ok = (gk + j) < n;
        const float e0 = pf[0 * 4 + j], e1 = pf[1 * 4 + j], e2 = pf[2 * 4 + j], e3 = pf[3 * 4 + j];
        x0[j] = ok ? (wx[0] * e0 + wx[1] * e1 + wx[2] * e2 + wx[3] * e3) : 0.f;
        x1[j] = ok ? (wy[0] * e0 + wy[1] * e1 + wy[2] * e2 + wy[3] * e3) : 0.f;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        S[0][4 * dkq + j][drow] = x0[j];
        if (NACC == 4) S[1][4 * dkq + j][drow] = x1[j];
      }
    }
    {  // transposed part
      const int gk = k0 + tkr, gi = i0 + 4 * tiq;
      float4 p[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) p[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gk < npad && gi < npad) {
#pragma unroll
        for (int q = 0; q < NPL; ++q) p[q] = *reinterpret_cast<const float4*>(P + peg_tile_off(gk, gi, q, nt, NPL));
      }
      const float* pf = reinterpret_cast<const float*>(p);
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
      *reinterpret_cast<float4*>(&S[NS / 2][tkr][4 * tiq]) = make_float4(y0[0], y0[1], y0[2], y0[3]);
      if (NACC == 4) *reinterpret_cast<float4*>(&S[3][tkr][4 * tiq]) = make_float4(y1[0], y1[1], y1[2], y1[3]);
    }
    {  // V chunk
      const int gk = k0 + tkr, gc = c0 + 4 * tiq;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gk < n && gc < d) v = *reinterpret_cast<const float4*>(Vb + (size_t)gk * d + gc);
      *reinterpret_cast<float4*>(&Vs[tkr][4 * tiq]) = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < CT_KC; ++k) {
      const float4 v4 = *reinterpret_cast<const float4*>(&Vs[k][4 * tx]);
      const float vv[4] = {v4.x, v4.y, v4.z, v4.w};
      if (NACC == 1) {
        const float4 s0 = *reinterpret_cast<const float4*>(&S[0][k][4 * ty]);
        const float4 s1 = *reinterpret_cast<const float4*>(&S[1][k][4 * ty]);
        const float aa[4] = {s0.x + s1.x, s0.y + s1.y, s0.z + s1.z, s0.w + s1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[0][i][j] = fmaf(aa[i], vv[j], acc[0][i][j]);
      } else {
#pragma unroll
        for (int q = 0; q < NACC; ++q) {
          const float4 s0 = *reinterpret_cast<const float4*>(&S[q][k][4 * ty]);
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
  const float* sv = a.svec + (size_t)b * a.sv_stride;
  const float* cb0 = a.colbuf + ((size_t)b * 2 + 0) * d;
  const float* cb1 = a.colbuf + ((size_t)b * 2 + 1) * d;
  const float kappa = sc.kappa[a.layer];
  const int gc = c0 + 4 * tx;
  float g4[4] = {0.f, 0.f, 0.f, 0.f};
  if (gc < d) {
    const float4 s4 = *reinterpret_cast<const float4*>(cb0 + gc);
    const float4 t4 = *reinterpret_cast<const float4*>(cb1 + gc);
    const float ss[4] = {s4.x, s4.y, s4.z, s4.w}, tt[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gi = i0 + 4 * ty + i;
      if (gi >= n) continue;
      contract_epilogue4<NACC, 4>(a, b, gi, gc, sv, Vb, acc, i, ss, tt, kappa, alpha, beta, gamma, delta, g4);
    }
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
// CDE wrapper (cde_wrapper_vector_field.py:21-25): dy[n,m] = sum_j out[n, m*2e + j] xd[n, j]
// =====================================================================================
__global__ void __launch_bounds__(256) k_wrapper_fwd(const float* __restrict__ OL, const float* __restrict__ svec,
                                                     size_t sv_stride, size_t xd_off, int n, int h, int e2, int B,
                                                     float* __restrict__ dy) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * n * h) return;
  const int m = idx % h;
  const size_t bn = idx / h;
  const int i = bn % n, b = bn / n;
  const float* xd = svec + (size_t)b * sv_stride + xd_off + (size_t)i * e2;
  const float* o = OL + bn * (size_t)h * e2 + (size_t)m * e2;
  float acc = 0.f;
  for (int j = 0; j < e2; ++j) acc = fmaf(o[j], xd[j], acc);
  dy[idx] = acc;
}

// cotangent of the last layer's output: OLbar[n, m*2e+j] = tg_n kbar[n,m] xd[n,j]   (e2 == 0: tg_n kbar[n,m])
__global__ void __launch_bounds__(256) k_wrapper_bwd(const float* __restrict__ kbar, const float* __restrict__ svec,
                                                     size_t sv_stride, size_t xd_off, size_t tg_off, int n, int h,
                                                     int e2, int B, float* __restrict__ OLbar) {
  const int dL = e2 > 0 ? h * e2 : h;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * n * dL) return;
  const int col = idx % dL;
  const size_t bn = idx / dL;
  const int i = bn % n, b = bn / n;
  const float* sv = svec + (size_t)b * sv_stride;
  const float tg = sv[tg_off + i];
  if (e2 > 0) {
    const int m = col / e2, j = col - m * e2;
    OLbar[idx] = tg * kbar[bn * h + m] * sv[xd_off + (size_t)i * e2 + j];
  } else {
    OLbar[idx] = tg * kbar[idx];
  }
}

// Top layer of a VJP without the CDE wrapper (e = 0), tensor-core path: ONE kernel instead of k_wrapper_bwd -> k_colsums ->
// k_block_exponent -> k_split_transpose.  A CTA owns a 128-node block with ALL d columns (d <= 256) in shared memory:
//   Obar = tg (.) kbar (written out), its block exponent (fp16x2 operands), V^T hi / lo in the contraction's operand format
//   (lane = node: coalesced), and the deterministic column sums 1^T Obar, r^T Obar (partials per block, last block adds them in
//   block order).  grid (ceil(rows_pad / 128), B), block 256, dynamic smem 128 * (d + 1) floats.
__global__ void __launch_bounds__(256) k_top_producer(const float* __restrict__ kbar, const float* __restrict__ svec, size_t sv_stride,
                                                      size_t tg_off, int n, int d, float* __restrict__ Obar, const ProducerOut po) {
  extern __shared__ __align__(16) float tp_tile[];     // [128][d + 1]
  __shared__ float bmax_s[8];
  __shared__ bool is_last;
  const int b = blockIdx.y, blk = blockIdx.x, i0 = blk * 128, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int pitch = d + 1, c4n = d >> 2;
  const float* sv = svec + (size_t)b * sv_stride;
  const float4* src = reinterpret_cast<const float4*>(kbar + (size_t)b * n * d);
  float4* dst = reinterpret_cast<float4*>(Obar + (size_t)b * n * d);
  float mx = 0.f;
  for (int idx = tid; idx < 128 * c4n; idx += 256) {
    const int r = idx / c4n, c4 = idx - r * c4n, i = i0 + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < n) {
      const float tg = sv[tg_off + i];
      const float4 k = __ldg(src + (size_t)i * c4n + c4);
      v = make_float4(tg * k.x, tg * k.y, tg * k.z, tg * k.w);
      dst[(size_t)i * c4n + c4] = v;
    }
    float* t = tp_tile + r * pitch + 4 * c4;
    t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
    mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  mx = warp_max(mx);
  if (lane == 0) bmax_s[warp] = mx;
  __syncthreads();
  float vscale = 1.f;
  if (po.t16 == PEG_FMT_FP16X2) {
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) mx = fmaxf(mx, bmax_s[w8]);
    const int e = block_exponent(mx);
    vscale = exp2_int(e);
    if (tid == 0) po.vexp[(size_t)b * po.vexp_stride + po.blk0 + blk] = e;
  }
  // V^T: warp w owns columns w, w + 8, ...; a lane owns nodes lane, lane + 32, ... of the block (odd pitch: conflict-free column walk)
  for (int c = warp; c < d; c += 8) {
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int r = lane + 32 * rr;
      if (i0 + r >= po.rows_pad) continue;
      const size_t o = ((size_t)b * d + c) * po.npad + po.col0 + i0 + r;
      const float v = tp_tile[r * pitch + c];
      if (po.t16 == PEG_FMT_FP16X2) store_vt_f16(po, o, v * vscale);
      else store_vt(po, o, v);
    }
  }
  // column sums over this block's nodes, rows in ascending order
  const int chunks = gridDim.x;
  const float* vb = po.vec ? po.vec + (size_t)b * po.vec_stride : nullptr;
  float* part = po.partial + (((size_t)b * chunks + blk) * 2) * d;
  for (int c = tid; c < d; c += 256) {
    float s0 = 0.f, s1 = 0.f;
    for (int r = 0; r < 128; ++r) {
      const float v = tp_tile[r * pitch + c];
      s0 += v;
      if (vb && i0 + r < n) s1 = fmaf(vb[i0 + r], v, s1);
    }
    part[c] = s0;
    part[d + c] = s1;
  }
  finalize_colsums(po, b, chunks, d, 0, d, po.tickets + b, &is_last);
}

// cotangent of control_data.derivative(t): g_xd[n,j] = sum_m tg_n kbar[n,m] OL[n, m*2e+j]  (OL = unscaled last-layer output)
__global__ void __launch_bounds__(256) k_wrapper_xbar(const float* __restrict__ kbar, const float* __restrict__ OLtg,
                                                      int n, int h, int e2, int B, float* __restrict__ gxd) {
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * n * e2) return;
  const int j = idx % e2;
  const size_t bn = idx / e2;
  float acc = 0.f;
  for (int m = 0; m < h; ++m) acc = fmaf(kbar[bn * h + m], OLtg[bn * (size_t)h * e2 + (size_t)m * e2 + j], acc);
  gxd[idx] = acc;
}

// cotangent of the node-signal coefficient path (TGB models learn it: tgb_graph_neural_cde.py:118-137).  X'(t) = b + s (2 c + 3 s d)
// on the stage's cubic piece, so g_b += g_xd, g_c += 2 s g_xd, g_d += 3 s^2 g_xd on that piece.  Stages run one after the
// other on the stream, so plain read-modify-write is race free.  g_xcoef [B, T-1, 3, n, 2e]
__global__ void __launch_bounds__(256) k_xcoef_accum(const float* __restrict__ gxd, const StageScalars* __restrict__ sc, int n,
                                                     int e2, int Tm1, int B, float* __restrict__ g_xcoef) {
  const size_t per = (size_t)n * e2;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * per) return;
  const int b = (int)(idx / per);
  const size_t i = idx % per;
  const float s = sc[b].s, g = gxd[idx];
  float* slab = g_xcoef + ((size_t)b * Tm1 + sc[b].interval) * 3 * per;
  slab[i] += g;
  slab[per + i] += 2.f * s * g;
  slab[2 * per + i] += 3.f * s * s * g;
}

// =====================================================================================
// gradients of param3..param8 of one layer: O(n d) dot products against row sums /
// diagonals / totals.  grid (ceil(n/8), B), block 256 (one warp per node)
// =====================================================================================
struct FusGradArgs {
  const float* G;      // cotangent of the layer output [B,n,d]
  const float* M;      // [B,n,d]
  const float* cbM;    // [B][2][d] : [0] = 1^T M
  const float* cbG;    // [B][2][d] : [0] = 1^T G
  const StageScalars* sc;
  const float* svec;
  size_t sv_stride;
  int n, d, L;
  int directed;
  float* g_fus;
};
__global__ void __launch_bounds__(256) k_fusion_vec_grads(FusGradArgs a) {
  __shared__ float sh[8][16];
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  const int n = a.n, d = a.d;
  const float* sv = a.svec + (size_t)b * a.sv_stride;
  const float* sM = a.cbM + (size_t)b * 2 * d;
  const float* sG = a.cbG + (size_t)b * 2 * d;
  float part[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) part[k] = 0.f;
  if (i < n) {
    const float* g = a.G + ((size_t)b * n + i) * d;
    const float* m = a.M + ((size_t)b * n + i) * d;
    float q = 0.f, u = 0.f, w = 0.f;
    for (int c = lane; c < d; c += 32) {
      const float gv = g[c], mv = m[c];
      q = fmaf(gv, mv, q);
      u = fmaf(gv, sM[c], u);
      w = fmaf(mv, sG[c], w);
    }
    q = warp_sum(q); u = warp_sum(u); w = warp_sum(w);
    const float rA = sv[svec_rA(n, a.L) + i], rD = sv[svec_rD(n, a.L) + i];
    const float dA = sv[svec_dgA(n, a.L) + i], dD = sv[svec_dgD(n, a.L) + i];
    part[0] = dA * q; part[1] = dD * q;      // param3
    part[8] = q;                              // param8 (* tot / n^2)
    if (!a.directed) {
      part[2] = rA * u; part[3] = rD * u;      // param4 (/n)
      part[4] = rA * w; part[5] = rD * w;      // param5 (/n)
      part[6] = rA * q; part[7] = rD * q;      // param6 (/n)
    } else {
      const float cA = sv[svec_cA(n, a.L) + i], cD = sv[svec_cD(n, a.L) + i];
      part[2] = cA * u; part[3] = cD * u;      // param4: colsum_i (1^T M) on row i
      part[4] = cA * w; part[5] = cD * w;      // param5: colsum_j on column j
      part[6] = cA * q; part[7] = cD * q;      // param6: diag(colsum)
      part[10] = rA * w; part[11] = cD * w;    // param4': rowsum(A)_j, colsum(A')_j on column j
      part[12] = rA * w; part[13] = rD * w;    // param5': rowsum_j on column j
      part[14] = rA * q; part[15] = rD * q;    // param6': diag(rowsum)
    }
  }
  if (blockIdx.x == 0 && warp == 0) {        // param7: tot_A / n^2 * (1^T G . 1^T M), once per graph
    float t = 0.f;
    for (int c = lane; c < d; c += 32) t = fmaf(sG[c], sM[c], t);
    part[9] = warp_sum(t);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 16; ++k) sh[warp][k] = part[k];
  }
  __syncthreads();
  if (a.directed && threadIdx.x >= 10 && threadIdx.x < 16) {   // param4', param5', param6' live at g_fus[16..21]
    float t = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) t += sh[w8][threadIdx.x];
    atomicAdd(a.g_fus + 16 + (threadIdx.x - 10), t / (float)n);
  }
  if (threadIdx.x < 10) {
    float t = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) t += sh[w8][threadIdx.x];
    const StageScalars sc = a.sc[b];
    const float inv_n = 1.f / (float)n, inv_n2 = inv_n * inv_n;
    const int k = threadIdx.x;
    if (k < 2) atomicAdd(a.g_fus + 4 + k, t);
    else if (k < 4) atomicAdd(a.g_fus + 6 + (k - 2), t * inv_n);
    else if (k < 6) atomicAdd(a.g_fus + 8 + (k - 4), t * inv_n);
    else if (k < 8) atomicAdd(a.g_fus + 10 + (k - 6), t * inv_n);
    else if (k == 8) {
      atomicAdd(a.g_fus + 14, t * sc.totA * inv_n2);
      atomicAdd(a.g_fus + 15, t * sc.totD * inv_n2);
    } else if (blockIdx.x == 0) {
      atomicAdd(a.g_fus + 12, t * sc.totA * inv_n2);
      atomicAdd(a.g_fus + 13, t * sc.totA * inv_n2);
    }
  }
}

// =====================================================================================
// backward of Linear + RMSNorm wrt the layer input (and the norm affine parameters):
//   Nbar = Mbar W ;  Zbar = rinv w Nbar - z rinv^3 <w Nbar, z>/din ;  optional ReLU mask (z > 0)
// grid (ceil(n/32), B), block 256: warp ty owns nodes 4ty..4ty+3, lane tx owns columns 4tx..4tx+3 (+128 if din > 128)
// =====================================================================================
__global__ void __launch_bounds__(256) k_linear_bwd(const float* __restrict__ Mbar, const float* __restrict__ W,
                                                    const float* __restrict__ Z, const float* __restrict__ nw,
                                                    int n, int din, int dout, int relu_mask,
                                                    float* __restrict__ Zbar, float* __restrict__ g_nw,
                                                    float* __restrict__ g_nb, ProducerOut po) {
  __shared__ bool is_last;
  __shared__ __align__(16) float mt[32][36];        // [k (dout chunk)][node]
  __shared__ __align__(16) float wsm[32][PEG_MAX_H]; // [k][c]
  __shared__ float gsw[PEG_MAX_H], gsb[PEG_MAX_H];
  const int tid = threadIdx.x, b = blockIdx.y, node0 = blockIdx.x * 32;
  const int ty = tid >> 5, tx = tid & 31;
  constexpr int REPS = PEG_MAX_H / 128;
  float acc[REPS][4][4];
#pragma unroll
  for (int r = 0; r < REPS; ++r)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[r][i][j] = 0.f;
  for (int c = tid; c < din; c += 256) { gsw[c] = 0.f; gsb[c] = 0.f; }
  const float* Mb = Mbar + (size_t)b * n * dout;
  for (int o0 = 0; o0 < dout; o0 += 32) {
    {  // Mbar chunk: 32 nodes x 32 k, thread -> node tid/8, 4 consecutive k
      const int r = tid >> 3, kq = (tid & 7) * 4;
      const int node = node0 + r;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int o = o0 + kq + u;
        mt[kq + u][r] = (node < n && o < dout) ? Mb[(size_t)node * dout + o] : 0.f;
      }
    }
    for (int idx = tid; idx < 32 * (din >> 2); idx += 256) {   // W chunk: 32 rows x din, float4
      const int k = idx / (din >> 2), c4 = idx - k * (din >> 2);
      const int o = o0 + k;
      const float4 w4 = (o < dout) ? *reinterpret_cast<const float4*>(W + (size_t)o * din + 4 * c4) : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(&wsm[k][4 * c4]) = w4;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < 32; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&mt[k][4 * ty]);
      const float aa[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
      for (int r = 0; r < REPS; ++r) {
        const int c = 4 * tx + 128 * r;
        if (c < din) {
          const float4 b4 = *reinterpret_cast<const float4*>(&wsm[k][c]);
          const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[r][i][j] = fmaf(aa[i], bb[j], acc[r][i][j]);
        }
      }
    }
    __syncthreads();
  }
  // norm backward: one warp holds complete rows of its 4 nodes
  float gw[REPS][4], gb[REPS][4];
#pragma unroll
  for (int r = 0; r < REPS; ++r)
#pragma unroll
    for (int j = 0; j < 4; ++j) { gw[r][j] = 0.f; gb[r][j] = 0.f; }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int node = node0 + 4 * ty + i;
    const bool ok = node < n;
    float z[REPS][4];
    float ss = 0.f, dot = 0.f;
#pragma unroll
    for (int r = 0; r < REPS; ++r) {
      const int c = 4 * tx + 128 * r;
      float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (ok && c < din) z4 = *reinterpret_cast<const float4*>(Z + ((size_t)b * n + node) * din + c);
      z[r][0] = z4.x; z[r][1] = z4.y; z[r][2] = z4.z; z[r][3] = z4.w;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ss = fmaf(z[r][j], z[r][j], ss);
        if (c < din) dot = fmaf(nw[c + j] * acc[r][i][j], z[r][j], dot);
      }
    }
    ss = warp_sum(ss);
    dot = warp_sum(dot);
    const float rinv = rsqrtf(ss / (float)din + 1e-5f);
    const float coef = rinv * rinv * rinv * dot / (float)din;
    if (ok) {
#pragma unroll
      for (int r = 0; r < REPS; ++r) {
        const int c = 4 * tx + 128 * r;
        if (c < din) {
          float zb[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            zb[j] = rinv * nw[c + j] * acc[r][i][j] - z[r][j] * coef;
            if (relu_mask && !(z[r][j] > 0.f)) zb[j] = 0.f;
            gw[r][j] = fmaf(acc[r][i][j] * z[r][j], rinv, gw[r][j]);
            gb[r][j] += acc[r][i][j];
          }
          *reinterpret_cast<float4*>(Zbar + ((size_t)b * n + node) * din + c) = make_float4(zb[0], zb[1], zb[2], zb[3]);
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[r][i][j] = zb[j];   // keep Zbar for the fused producer outputs below
        }
      }
    } else {
#pragma unroll
      for (int r = 0; r < REPS; ++r)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[r][i][j] = 0.f;
    }
  }
#pragma unroll
  for (int r = 0; r < REPS; ++r) {
    const int c = 4 * tx + 128 * r;
    if (c < din) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { atomicAdd(&gsw[c + j], gw[r][j]); atomicAdd(&gsb[c + j], gb[r][j]); }
    }
  }
  __syncthreads();
  for (int c = tid; c < din; c += 256) {
    atomicAdd(g_nw + c, gsw[c]);
    atomicAdd(g_nb + c, gsb[c]);
  }
  // ---- fused producer outputs: Zbar is the operand V of the next (lower) layer's adjoint contraction ----
  if (po.Thi != nullptr) {
    const int nodeq = node0 + 4 * ty;
    if (nodeq < po.npad) {
#pragma unroll
      for (int r = 0; r < REPS; ++r) {
        const int c = 4 * tx + 128 * r;
        if (c >= din) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const size_t o = ((size_t)b * din + c + j) * po.npad + nodeq;
          store_vt4(po, o, acc[r][0][j], acc[r][1][j], acc[r][2][j], acc[r][3][j]);
        }
      }
    }
  }
  if (po.cb != nullptr) {
    __syncthreads();   // gsw / gsb have been flushed: reuse them as the column accumulators of this block
    for (int c = tid; c < din; c += 256) { gsw[c] = 0.f; gsb[c] = 0.f; }
    __syncthreads();
    const float* vb = po.vec ? po.vec + (size_t)b * po.vec_stride : nullptr;
    float v4[4] = {0.f, 0.f, 0.f, 0.f};
    if (vb) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { const int node = node0 + 4 * ty + i; v4[i] = node < n ? vb[node] : 0.f; }
    }
    // deterministic order: warp ty adds its 4-node partial in turn
    for (int turn = 0; turn < 8; ++turn) {
      if (ty == turn) {
#pragma unroll
        for (int r = 0; r < REPS; ++r) {
          const int c = 4 * tx + 128 * r;
          if (c < din) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              gsw[c + j] += acc[r][0][j] + acc[r][1][j] + acc[r][2][j] + acc[r][3][j];
              gsb[c + j] += v4[0] * acc[r][0][j] + v4[1] * acc[r][1][j] + v4[2] * acc[r][2][j] + v4[3] * acc[r][3][j];
            }
          }
        }
      }
      __syncthreads();
    }
    const int chunks = gridDim.x;
    float* part = po.partial + (((size_t)b * chunks + blockIdx.x) * 2) * din;
    for (int c = tid; c < din; c += 256) { part[c] = gsw[c]; part[din + c] = gsb[c]; }
    finalize_colsums(po, b, chunks, din, 0, din, po.tickets + b, &is_last);
  }
}

// =====================================================================================
// weight / bias gradient: Wbar[o][c] += sum_nodes Mbar[node][o] N[node][c] ; bbar[o] += sum Mbar[node][o]
// nodes = all B*n rows, split over gridDim.z.  grid (ceil(dout/64), ceil(din/64), KS), block 256
// =====================================================================================
__global__ void __launch_bounds__(256) k_weight_grad(const float* __restrict__ Mbar, const float* __restrict__ N,
                                                     size_t rows, int din, int dout, int rows_per_slice,
                                                     float* __restrict__ gW, float* __restrict__ gb) {
  __shared__ __align__(16) float ms[16][68];
  __shared__ __align__(16) float ns[16][68];
  const int tid = threadIdx.x, o0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
  const size_t r_begin = (size_t)blockIdx.z * rows_per_slice;
  const size_t r_end = min(rows, r_begin + (size_t)rows_per_slice);
  const int ty = tid >> 4, tx = tid & 15;
  const int lk = tid >> 4, lq = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float bsum = 0.f;
  for (size_t k0 = r_begin; k0 < r_end; k0 += 16) {
    const size_t row = k0 + lk;
    {   // din, dout are multiples of 4 (check_dims): one 128-bit load / store per operand
      const int o = o0 + 4 * lq, c = c0 + 4 * lq;
      const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(&ms[lk][4 * lq]) = (row < r_end && o < dout) ? __ldg(reinterpret_cast<const float4*>(Mbar + row * dout + o)) : zero4;
      *reinterpret_cast<float4*>(&ns[lk][4 * lq]) = (row < r_end && c < din) ? __ldg(reinterpret_cast<const float4*>(N + row * din + c)) : zero4;
    }
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
    if (blockIdx.y == 0 && tid < 64) {
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
  if (blockIdx.y == 0 && tid < 64 && o0 + tid < dout) atomicAdd(gb + o0 + tid, bsum);
}

// elementwise ReLU mask on a cotangent: out = (z > 0) ? g : 0
__global__ void __launch_bounds__(256) k_axpy(float* __restrict__ y, const float* __restrict__ x, float a, size_t cnt) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < cnt) y[i] = fmaf(a, x[i], y[i]);
}

}  // namespace peg
