// tcgen05 (5th-gen tensor core) implementation of the matrix-free equivariant contraction.
// Declarations only; the kernels live in peg_tc.cu.
#pragma once
#include <atomic>
#include <cstdio>

#include "peg_common.cuh"

#define PEG_TRY(expr)            \
  do {                           \
    int _rc = (expr);            \
    if (_rc != PEG_OK) return _rc; \
  } while (0)

namespace peg {

// operand buffers the tensor-core path needs in the caller's workspace
struct TcWs {
  float* Vt_hi;  // [B][dmax][npad]  V^T, high part (K-major B operand): tf32-rounded fp32 words, or packed bf16 (tc_fmt16)
  float* Vt_lo;  // [B][dmax][npad]  residual V - high part, same format
  float* partial;  // [B][4][n][dmax] split-K accumulators (grids far smaller than the GPU)
  int npad;
  int fmt;          // operand format of this call (PEG_FMT_*), set by make_ctx from the flags and the control
  int* vexp;        // [B][vexp_stride] block exponents of V^T (fp16x2 format)
  unsigned int* vmax;   // [2][B][vexp_stride] scratch of k_block_exponent (maxima, arrival counters), zero between launches
  int vexp_stride;  // = ceil(ldk / 128)
  int ldk;          // row pitch of V^T in elements = padded GLOBAL node count (== npad unless row-sharded)
  int col0, blk0;   // row-sharded mode: this rank's rows are columns [col0, col0 + npad) of V^T (else 0)
};

// per-layer tf32 hi/lo copies of the Linear weights (built once per API call by tc_prep_weights):
//   Wn = W diag(norm.weight)  [dout][din]  (B operand of RMSNorm -> Linear; the norm scale rides in the epilogue)
//   cvec[o] = sum_k norm.bias[k] W[o][k] + bias[o]
struct TcLinear {
  float* Wn_hi[PEG_MAX_LAYERS];
  float* Wn_lo[PEG_MAX_LAYERS];
  float* cvec[PEG_MAX_LAYERS];
  float* Wt_hi[PEG_MAX_LAYERS];   // W^T [din][dout] (B operand of the Linear backward: Nbar = Mbar W)
  float* Wt_lo[PEG_MAX_LAYERS];
  bool ready;   // carved (tensor-core flag set)
};

void tc_carve(Bump& bp, const PegDims& d, int dmax, TcWs& w);
void tc_carve_linear(Bump& bp, const PegDims& d, const Model& m, TcLinear& w);
bool tc_linear_supported(int din, int dout);
// splits the weights of every layer (enqueue only); call once per API entry before the first evaluation
int tc_prep_weights(cudaStream_t st, const Model& m, const float* params, const TcLinear& w);
// M = rmsnorm(Z) W^T + b on tcgen05 (3xTF32), fused producer outputs as k_norm_linear (peg_kernels.cuh)
bool tc_norm_linear_full_columns(int dout);   // one CTA holds every output column of its 128 nodes (it can emit fp16x2 V^T)
// backward of Linear + RMSNorm wrt the layer input on tcgen05, epilogue as k_linear_bwd (peg_kernels.cuh).  With gW (only where
// tc_linear_bwd_fuses_weight_grad) it also accumulates gW += Mbar^T N and gb += 1^T Mbar; otherwise Nout (nullable) receives the
// normalised input N for tc_weight_grad.
int tc_linear_bwd(cudaStream_t st, const PegDims& d, const TcLinear& w, int layer, const float* Mbar, const float* Z,
                  const float* nw, const float* nb, int din, int dout, int relu_mask, float* Zbar, float* g_nw, float* g_nb,
                  float* gW, float* gb, float* Nout, const ProducerOut& po);
bool tc_linear_bwd_supported(int din, int dout);
bool tc_linear_bwd_fuses_weight_grad(const PegDims& d, int din, int dout);
// Wbar += Mbar^T N, bbar += 1^T Mbar over all rows, on tcgen05 (both operands transposed in the loaders); the shapes of
// tc_linear_bwd_supported
int tc_weight_grad(cudaStream_t st, const PegDims& d, const float* Mbar, const float* N, size_t rows, int din, int dout, float* gW,
                   float* gb);
int tc_norm_linear(cudaStream_t st, const PegDims& d, const TcLinear& w, int layer, const float* Z, int din, int dout, float* M,
                   const ProducerOut& po);
bool tc_supported(const PegDims& d, int dcols);
int tc_fmt(const PegDims& d, bool have_absmax);   // operand format of the contraction (PEG_FMT_*)
int tc_convert_v(cudaStream_t st, const PegDims& d, const TcWs& w, const ContractArgs& a);
int tc_contract(cudaStream_t st, const PegDims& d, const TcWs& w, const ContractArgs& a, bool bwd);
void set_last_cuda(int err);   // records a cudaError_t for pegncde_last_cuda_error() (defined in pegncde.cu)

// Kernel attributes are per function AND device: `done` holds one bit per device on which `set(dev)` has succeeded, so each device
// is configured once per process, also when one process drives several GPUs or calls in from several threads.
template <typename F>
int once_per_device(std::atomic<unsigned>& done, F set) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_last_cuda((int)cudaGetLastError()); return PEG_ERR_CUDA; }
  const unsigned bit = 1u << (dev & 31);
  if ((done.load(std::memory_order_acquire) & bit) != 0u) return PEG_OK;
  const cudaError_t e = set(dev);
  if (e != cudaSuccess) { set_last_cuda((int)e); (void)cudaGetLastError(); return PEG_ERR_CUDA; }
  done.fetch_or(bit, std::memory_order_release);
  return PEG_OK;
}

// raises the dynamic-smem limit of a kernel to the device's opt-in maximum
template <typename K>
int optin_smem(K kernel, std::atomic<unsigned>& done) {
  return once_per_device(done, [kernel](int dev) {
    int lim = 0;
    cudaDeviceGetAttribute(&lim, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, kernel) == cudaSuccess) lim -= (int)fa.sharedSizeBytes;   // static smem counts against the limit
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
    if (e != cudaSuccess) fprintf(stderr, "pegncde: cudaFuncSetAttribute(smem %d) failed: %s\n", lim, cudaGetErrorString(e));
    return e;
  });
}

// allows a kernel cluster sizes beyond the portable 8 CTAs
template <typename K>
int optin_nonportable_cluster(K kernel, std::atomic<unsigned>& done) {
  return once_per_device(done, [kernel](int) { return cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); });
}

}  // namespace peg
