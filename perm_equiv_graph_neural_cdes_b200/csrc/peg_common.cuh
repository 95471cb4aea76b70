// Shared device/host definitions for the pegncde sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/pegncde.h"

#define PEG_MAX_LAYERS 8
#define PEG_MAX_H 256      // widest hidden state / layer input
#define PEG_MAX_T 4096

namespace peg {

struct LayerDesc {
  int din, dout;
  long long w_off, b_off, nw_off, nb_off, fus_off;  // float offsets into the packed params
};

struct Model {
  int L;
  int directed;  // ConvEquivFusionDirectedLayer: fusion block of 22 scalars (param4', 5', 6' appended)
  int P;  // total parameter count
  int dmax;
  LayerDesc layer[PEG_MAX_LAYERS];
};

// Per-graph, per-stage scalars (device, in workspace).  One per graph of the batch.
struct StageScalars {
  int interval;     // cubic piece index
  float s;          // t - ts[interval]
  float wA[4];      // A_s   = sum_p wA[p] * plane_p   (a,b,c,d) -> (1, s, s^2, s^3)
  float wD[4];      // A'_s  = sum_p wD[p] * plane_p            -> (0, 1, 2s, 3s^2)
  float totA, totD; // sum(A_s), sum(A'_s)
  float kappa[PEG_MAX_LAYERS];  // (p7_0 + p7_1) * totA / n^2   (reference quirk: both use sum(A))
  float amax[4];    // max |entry| of the four planes of this cubic piece (0 when the control carries no adj_absmax)
  float pad[2];
};

// Per-graph stage vectors live in one float array `svec` laid out as
//   [b][ (3*L + 1) * n + n * 2e ]  =  v_l[n], r_l[n], c_l[n] for l < L ; tg[n] ; xd[n, 2e]
// plus rA, rD, dgA, dgD, cA, cD [6][n] (needed by the fusion-parameter gradients; cA, cD = column sums, directed only).
__host__ __device__ inline size_t svec_stride(int n, int L, int e) {
  return (size_t)(3 * L + 1 + 6) * n + (size_t)n * 2 * e;
}
__host__ __device__ inline size_t svec_v(int n, int l) { return (size_t)(3 * l + 0) * n; }
__host__ __device__ inline size_t svec_r(int n, int l) { return (size_t)(3 * l + 1) * n; }
__host__ __device__ inline size_t svec_c(int n, int l) { return (size_t)(3 * l + 2) * n; }
__host__ __device__ inline size_t svec_tg(int n, int L) { return (size_t)(3 * L) * n; }
__host__ __device__ inline size_t svec_rA(int n, int L) { return (size_t)(3 * L + 1) * n; }
__host__ __device__ inline size_t svec_rD(int n, int L) { return (size_t)(3 * L + 2) * n; }
__host__ __device__ inline size_t svec_dgA(int n, int L) { return (size_t)(3 * L + 3) * n; }
__host__ __device__ inline size_t svec_dgD(int n, int L) { return (size_t)(3 * L + 4) * n; }
__host__ __device__ inline size_t svec_cA(int n, int L) { return (size_t)(3 * L + 5) * n; }   // column sums (directed layer only)
__host__ __device__ inline size_t svec_cD(int n, int L) { return (size_t)(3 * L + 6) * n; }
__host__ __device__ inline size_t svec_xd(int n, int L) { return (size_t)(3 * L + 7) * n; }

// ---- HBM layout of the cubic-coefficient planes (adjacency channel) -----------------------------------
// One slab = the four planes (a,b,c,d) of one cubic piece of one graph, npad x npad with npad = n rounded
// up to 32 (zero padded).  The slab is stored as 32x32 tiles of 16 KB: [row tile][col tile] -> [g][plane][m][lane][e]
// where the 32x32 plane tile is cut into 8x8 micro tiles of 4x4 floats, micro tile (rq, cq) sits on
// diagonal s = (rq - cq) & 7, g = s >> 2, lane = ((s & 3) << 3) | cq, m = row inside the micro tile,
// e = column inside the micro tile.  Consequences (both are what the converters of peg_tc.cu need):
//   * a warp-level 128-bit load of (g, plane, m) is 512 contiguous bytes, and a whole item is 4 x 16 KB blocks;
//   * every thread ends up holding a full 4x4 micro tile of all four planes, so the transposed orientation
//     is free in registers, and both orientations store bank-conflict-free into the swizzled operand tiles.
// A static control (PegControl.adj_static) stores ONE plane per graph in the same order with np = 1: 4-KB tiles
// [g][m][lane][e], so a warp-level 128-bit load is still 512 contiguous bytes.
__host__ __device__ inline int peg_npad(int n) { return (n + 31) / 32 * 32; }
__host__ __device__ inline size_t peg_tile_off(int i, int k, int q, int nt, int np = 4) {
  const int rt = i >> 5, ct = k >> 5, r = i & 31, c = k & 31;
  const int rq = r >> 2, m = r & 3, cq = c >> 2, e = c & 3;
  const int s = (rq - cq) & 7, g = s >> 2, lane = ((s & 3) << 3) | cq;
  return ((size_t)rt * nt + ct) * (1024 * np) + (size_t)(((g * np + q) * 4 + m) * 128 + lane * 4 + e);
}

// Tsit5 tableau (Tsitouras 2011) -- the tableau behind diffrax.Tsit5.
struct Tsit5 {
  double c[7];
  double a[7][6];
  double b[7];
  double berr[7];
};
inline const Tsit5& tsit5() {
  static const Tsit5 t = {
      {0.0, 0.161, 0.327, 0.9, 0.9800255409045097, 1.0, 1.0},
      {{0, 0, 0, 0, 0, 0},
       {0.161, 0, 0, 0, 0, 0},
       {-0.008480655492356989, 0.335480655492357, 0, 0, 0, 0},
       {2.8971530571054935, -6.359448489975075, 4.3622954328695815, 0, 0, 0},
       {5.325864828439257, -11.748883564062828, 7.4955393428898365, -0.09249506636175525, 0, 0},
       {5.86145544294642, -12.92096931784711, 8.159367898576159, -0.071584973281401, -0.028269050394068383, 0},
       {0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081,
        2.324710524099774}},
      {0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081, 2.324710524099774,
       0.0},
      {-0.00178001105222577714, -0.0008164344596567469, 0.007880878010261995, -0.1447110071732629,
       0.5823571654525552, -0.45808210592918697, 0.015151515151515152}};
  return t;
}

// arguments of the matrix-free contraction (CUDA-core kernel in peg_kernels.cuh, tcgen05 kernel in peg_tc.cu)
struct ContractArgs {
  const float* planes;   // adj_coef, or adj_static for a static control
  size_t graph_stride;   // floats per graph = (T-1)*4*n*ldn (static: ldn*ldn)
  int stat;              // static control: `planes` holds one plane per graph that serves every piece (A_s = a, A'_s = 0)
  const StageScalars* sc;
  const float* svec;
  size_t sv_stride;
  size_t rowc_off;       // offset in svec of the per-row coefficient of (1^T V): r_l (fwd) / c_l (bwd)
  size_t v_off;          // offset of v_l
  size_t tg_off;
  const float* fus;      // 16 fusion scalars of this layer
  const float* V;        // [B,n,d]
  const float* Mref;     // bwd only: M_l [B,n,d]
  const float* colbuf;   // [B][2][d]
  const float* cbM;      // bwd, tensor-core path only (nullable): [B][2][d] column sums of M -> the epilogue also emits the
                         // param3..8 gradients (otherwise k_fusion_vec_grads does)
  float* out;            // [B,n,d]
  float* g_fus;          // bwd only: gradient of the 16 fusion scalars (atomicAdd)
  int n, ldn /* = npad */, d, layer, L;
  int relu, scale_tg;
  int vt_ready;          // the producer kernel already wrote V^T hi/lo (tensor-core path skips its own transpose pass)
  // row-sharded mode (PegShard): n / ldn are this rank's rows, the K dimension runs over all ldk = n_glob columns, the transposed
  // products read the rank's rows of the TRANSPOSED path (planes_t) like direct ones.  Whole graph on one GPU: planes_t = nullptr,
  // ldk = ldn, n_glob = n, row_block0 = 0.
  const float* planes_t;
  int ldk, n_glob, row_block0;
};

struct Bump {
  char* base;
  size_t off;
  explicit Bump(void* p) : base((char*)p), off(0) {}
  template <typename T>
  T* take(size_t count) {
    off = (off + 255) & ~(size_t)255;
    T* r = base ? (T*)(base + off) : nullptr;
    off += count * sizeof(T);
    return r;
  }
};


// ---- device helpers shared by the CUDA-core kernels (peg_kernels.cuh) and the tensor-core kernels (peg_tc.cu) ----
#ifdef __CUDACC__
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// sum over the whole block (blockDim.x * blockDim.y threads, multiple of 32, <= 1024); result valid in all threads
__device__ __forceinline__ float block_sum(float v, float* sh /* >= 33 floats */) {
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nw = (blockDim.x * blockDim.y + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if ((tid & 31) == 0) sh[tid >> 5] = v;
  __syncthreads();
  if (tid < 32) {
    float x = tid < nw ? sh[tid] : 0.f;
    x = warp_sum(x);
    if (tid == 0) sh[32] = x;
  }
  __syncthreads();
  return sh[32];
}

// Fused-epilogue outputs of the kernels that PRODUCE the operand V of the next contraction:
//   * V^T split into tf32 hi / lo, [B][d][npad] (the TMA-loaded K-major B operand of peg_tc.cu), zero padded;
//   * column sums cb[b][0][c] = sum_i V[b,i,c], cb[b][1][c] = sum_i vec[b][i] V[b,i,c], reduced deterministically:
//     every block writes its partial, the last block of a column group (ticket) adds them in block order.
// Operand formats of the tcgen05 contraction (peg_tc.cu).  All three split x = hi + lo and run hi*hi + lo*hi + hi*lo with fp32 accumulation.
enum { PEG_FMT_TF32X3 = 0,   // tf32 parts in fp32 words, kind::tf32
       PEG_FMT_BF16X2 = 1,   // bf16 parts, kind::f16; no range management, 16 mantissa bits
       PEG_FMT_FP16X2 = 2 }; // fp16 parts, kind::f16, 22 mantissa bits; block floating point: V^T carries one power-of-two scale per
                             // 128-node block (vexp), the interpolated adjacency one scale per launch (from the plane maxima)
struct ProducerOut {
  float* Thi;             // nullable; fmt 0: fp32 words holding tf32-rounded values, fmt 1 / 2: packed bf16 / fp16 (same buffer)
  float* Tlo;
  int npad;
  int t16;                // operand format of the contraction that will read V^T (PEG_FMT_*)
  int* vexp;              // fmt 2: [B][vexp_stride] power-of-two exponent of every 128-node block: V^T holds V * 2^vexp
  int vexp_stride;
  int col0, blk0;         // row-sharded mode: this rank's rows are columns [col0, col0 + rows_pad) of V^T, blocks from blk0 (else 0, 0)
  int rows_pad;           // padded local row count (== npad unless row-sharded)
  float* cb;              // nullable
  float* partial;         // [B][chunks][2][d]
  unsigned int* tickets;  // self-resetting, one per (b, column group)
  const float* vec;       // nullable; per-graph stride vec_stride
  size_t vec_stride;
};

__device__ __forceinline__ float tf32_round(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

__device__ __forceinline__ unsigned short bf16_bits_rn(float x) {
  unsigned short r;
  asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ unsigned short f16_bits_rn(float x) {
  unsigned short r;
  asm("cvt.rn.f16.f32 %0, %1;" : "=h"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float f16_bits_to_f32(unsigned short h) {
  float r;
  asm("cvt.f32.f16 %0, %1;" : "=f"(r) : "h"(h));
  return r;
}
// Block exponent of the fp16x2 format: the power of two that brings a block whose largest magnitude is `amax` into [2^14, 2^15)
// (fp16 overflows at 65504), clamped so that 2^e and 2^-e stay normal fp32 numbers; an all-zero block gets the largest exponent.
#define PEG_VEXP_MAX 60
__device__ __forceinline__ int block_exponent(float amax) {
  if (!(amax > 0.f)) return PEG_VEXP_MAX;
  const int e = 14 - ((int)((__float_as_uint(amax) >> 23) & 0xffu) - 127);
  return max(-PEG_VEXP_MAX, min(PEG_VEXP_MAX, e));
}
__device__ __forceinline__ float exp2_int(int e) { return __uint_as_float((uint32_t)(e + 127) << 23); }   // e in [-126, 127]
// one element of V^T in the fp16x2 format: `vs` = v * 2^(block exponent)
__device__ __forceinline__ void store_vt_f16(const ProducerOut& po, size_t o, float vs) {
  const unsigned short h = f16_bits_rn(vs);
  reinterpret_cast<unsigned short*>(po.Thi)[o] = h;
  float lo_ = vs - f16_bits_to_f32(h);
  reinterpret_cast<unsigned short*>(po.Tlo)[o] = f16_bits_rn(lo_);
}
// max over the warp of a non-negative value
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// one element of V^T (hi + lo parts) at element offset o of the [B][d][npad] operand arrays, in the format the contraction reads
// (tf32 or bf16 parts; the fp16x2 format needs the block scale: store_vt_f16)
__device__ __forceinline__ void store_vt(const ProducerOut& po, size_t o, float v) {
  if (po.t16) {
    const unsigned short h = bf16_bits_rn(v);
    reinterpret_cast<unsigned short*>(po.Thi)[o] = h;
    reinterpret_cast<unsigned short*>(po.Tlo)[o] = bf16_bits_rn(v - __uint_as_float((uint32_t)h << 16));
  } else {
    const float h = tf32_round(v);
    po.Thi[o] = h;
    po.Tlo[o] = v - h;
  }
}
// four consecutive elements along the node axis (o multiple of 4)
__device__ __forceinline__ void store_vt4(const ProducerOut& po, size_t o, float v0, float v1, float v2, float v3) {
  if (po.t16) {
    const uint32_t h0 = bf16_bits_rn(v0), h1 = bf16_bits_rn(v1), h2 = bf16_bits_rn(v2), h3 = bf16_bits_rn(v3);
    const uint32_t l0 = bf16_bits_rn(v0 - __uint_as_float(h0 << 16)), l1 = bf16_bits_rn(v1 - __uint_as_float(h1 << 16));
    const uint32_t l2 = bf16_bits_rn(v2 - __uint_as_float(h2 << 16)), l3 = bf16_bits_rn(v3 - __uint_as_float(h3 << 16));
    *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(po.Thi) + o) = make_uint2(h0 | (h1 << 16), h2 | (h3 << 16));
    *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(po.Tlo) + o) = make_uint2(l0 | (l1 << 16), l2 | (l3 << 16));
  } else {
    const float h0 = tf32_round(v0), h1 = tf32_round(v1), h2 = tf32_round(v2), h3 = tf32_round(v3);
    *reinterpret_cast<float4*>(po.Thi + o) = make_float4(h0, h1, h2, h3);
    *reinterpret_cast<float4*>(po.Tlo + o) = make_float4(v0 - h0, v1 - h1, v2 - h2, v3 - h3);
  }
}

// called by ALL threads of the block after this block's partial sums for columns [c0, c0+ncols) have been written
// to partial[b][chunk][*][c]; `is_last` must be a __shared__ bool.
__device__ __forceinline__ void finalize_colsums(const ProducerOut& po, int b, int chunks, int d, int c0, int ncols,
                                                 unsigned int* ticket, bool* is_last) {
  __threadfence();
  __syncthreads();
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    *is_last = (t == (unsigned int)chunks - 1u);
    if (*is_last) *ticket = 0u;
  }
  __syncthreads();
  if (*is_last) {
    __threadfence();
    for (int c = tid; c < ncols; c += blockDim.x * blockDim.y) {
      if (c0 + c >= d) continue;
      float t0 = 0.f, t1 = 0.f;
      for (int k = 0; k < chunks; ++k) {
        const float* pk = po.partial + (((size_t)b * chunks + k) * 2) * d;
        t0 += __ldcg(pk + c0 + c);
        t1 += __ldcg(pk + d + c0 + c);
      }
      po.cb[((size_t)b * 2 + 0) * d + c0 + c] = t0;
      po.cb[((size_t)b * 2 + 1) * d + c0 + c] = t1;
    }
  }
}

#endif  // __CUDACC__

}  // namespace peg
