// XLA FFI shim over the C-ABI (include/pegncde.h): what a JAX host registers with jax.ffi so that
// `fused_diffeqsolve` is an XLA custom call on the CUDA platform.
//
// Handlers: PegPackAdj, PegPackX (control pre-pass), PegVfFwd, PegVfVjp (the ODETerm callable and its VJP), PegStepFwd (one Tsit5
// step for the adaptive loop), PegSolveFwd, PegSolveBwd (the whole fixed-step solve and its exact adjoint).
// STATUS: NOT BUILT OR RUN IN THIS REPOSITORY'S IMAGE.  jax / jaxlib (and therefore xla/ffi/api/ffi.h) are not
// installed and cannot be installed here (no network); this file documents the binding exactly as a maintainer
// with a JAX environment would compile it:
//   g++ -O2 -shared -fPIC -I$(python -c "import jax; print(jax.ffi.include_dir())") -I../../include -I$CUDA_HOME/include
//       pegncde_ffi.cc -L.. -lpegncde -L$CUDA_HOME/lib64 -lcudart -o libpegncde_ffi.so        (one command line)
// What IS checked here (tests/test_host.py): the file compiles against a MOCK of the FFI API (tests/mock_xla_ffi) that
// type-checks every handler against its binding and against the prototypes of pegncde.h.
// Everything it calls is exercised on B200 through the same C-ABI from the torch/ctypes host (tests/).
#include <cstdint>

#include <cuda_runtime_api.h>   // cudaStream_t, cudaMemsetAsync

#include "pegncde.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

static PegDims dims_of(int32_t B, int32_t n, int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d{B, n, (n + 31) / 32 * 32, h, e, L, T, flags};
  return d;
}
// Batching rule: the handlers are registered with vmap_method="broadcast_all", so under jax.vmap(model)
// (src/configs/loss_configs.py:44) every operand arrives with one more leading axis and the custom call runs ONCE for the whole
// batch.  The attribute B is the un-vmapped batch; the effective PegDims.B is read off the state buffer [.., n, h].
template <typename Buf>
static int32_t batch_of(const Buf& y, int32_t n, int32_t h) { return (int32_t)(y.element_count() / ((size_t)n * h)); }
static PegControl control_of(const float* ts, const float* adj_coef, const float* adj_rowsum, const float* adj_diag, const float* adj_total,
                             const float* tch_coef, const float* x_coef, const float* adj_absmax) {
  PegControl c{ts, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef, x_coef, /*adj_colsum=*/nullptr, adj_absmax, /*shard=*/nullptr,
               /*sparse=*/nullptr};   // the handlers take dense planes only
  return c;
}

// Control-path pre-pass, once per batch (src/engine/trainer_pgt.py:201-207 hands the model the reference-layout arrays):
// operands: d, c, b, a  each [B, T-1, n, n, 2]  ->  results: adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef (PegControl fields)
static ffi::Error PackAdjImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> cd, ffi::Buffer<ffi::F32> cc, ffi::Buffer<ffi::F32> cb,
                              ffi::Buffer<ffi::F32> ca, ffi::ResultBuffer<ffi::F32> adj_coef,
                              ffi::ResultBuffer<ffi::F32> adj_rowsum, ffi::ResultBuffer<ffi::F32> adj_diag,
                              ffi::ResultBuffer<ffi::F32> adj_total, ffi::ResultBuffer<ffi::F32> tch_coef,
                              ffi::ResultBuffer<ffi::F32> adj_absmax, int32_t B, int32_t n,
                              int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  B = (int32_t)(adj_total->element_count() / ((size_t)(T - 1) * 4));
  PegDims d = dims_of(B, n, h, e, L, T, flags);
  // (the pack kernel writes the zero padding of the ldn x ldn tiles itself: uninitialised result buffers are fine)
  int rc = pegncde_pack_adj(stream, &d, cd.typed_data(), cc.typed_data(), cb.typed_data(), ca.typed_data(),
                            adj_coef->typed_data(), adj_rowsum->typed_data(), adj_diag->typed_data(),
                            adj_total->typed_data(), tch_coef->typed_data());
  if (rc == PEG_OK) rc = pegncde_adj_absmax(stream, &d, 0, T - 1, adj_coef->typed_data(), adj_absmax->typed_data());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

// operands: d, c, b, a  each [B, T-1, n, e, 2]  ->  result: x_coef [B, T-1, 3, n, 2e]
static ffi::Error PackXImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> cd, ffi::Buffer<ffi::F32> cc, ffi::Buffer<ffi::F32> cb,
                            ffi::Buffer<ffi::F32> ca, ffi::ResultBuffer<ffi::F32> x_coef, int32_t B, int32_t n, int32_t h,
                            int32_t e, int32_t L, int32_t T, int32_t flags) {
  B = (int32_t)(x_coef->element_count() / ((size_t)(T - 1) * 3 * n * 2 * e));
  PegDims d = dims_of(B, n, h, e, L, T, flags);
  const int rc = pegncde_pack_x(stream, &d, cd.typed_data(), cc.typed_data(), cb.typed_data(), ca.typed_data(), x_coef->typed_data());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

// operands: params, ts, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef, x_coef, step_ts(host attr), y0
// results:  y_ckpt [S+1,B,n,h], stage_store, workspace (XLA-allocated scratch results)
static ffi::Error SolveFwdImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> ts,
                               ffi::Buffer<ffi::F32> adj_coef, ffi::Buffer<ffi::F32> adj_rowsum,
                               ffi::Buffer<ffi::F32> adj_diag, ffi::Buffer<ffi::F32> adj_total,
                               ffi::Buffer<ffi::F32> tch_coef, ffi::Buffer<ffi::F32> x_coef, ffi::Buffer<ffi::F32> adj_absmax,
                               ffi::Buffer<ffi::F32> y0,
                               ffi::ResultBuffer<ffi::F32> y_ckpt, ffi::ResultBuffer<ffi::F32> stage_store,
                               ffi::ResultBuffer<ffi::U8> workspace, ffi::Span<const float> step_ts, int32_t B, int32_t n,
                               int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d = dims_of(batch_of(y0, n, h), n, h, e, L, T, flags);
  PegControl c = control_of(ts.typed_data(), adj_coef.typed_data(), adj_rowsum.typed_data(), adj_diag.typed_data(), adj_total.typed_data(),
                            tch_coef.typed_data(), e > 0 ? x_coef.typed_data() : nullptr, adj_absmax.typed_data());
  const int32_t steps = (int32_t)step_ts.size() - 1;
  const int rc = pegncde_solve_fwd(stream, &d, &c, params.typed_data(), step_ts.begin(), steps, y0.typed_data(), nullptr,
                                   y_ckpt->typed_data(), stage_store->element_count() ? stage_store->typed_data() : nullptr,
                                   workspace->typed_data(), workspace->element_count());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

static ffi::Error SolveBwdImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> ts,
                               ffi::Buffer<ffi::F32> adj_coef, ffi::Buffer<ffi::F32> adj_rowsum,
                               ffi::Buffer<ffi::F32> adj_diag, ffi::Buffer<ffi::F32> adj_total,
                               ffi::Buffer<ffi::F32> tch_coef, ffi::Buffer<ffi::F32> x_coef, ffi::Buffer<ffi::F32> adj_absmax,
                               ffi::Buffer<ffi::F32> y_ckpt,
                               ffi::Buffer<ffi::F32> stage_store, ffi::Buffer<ffi::F32> g_ckpt,
                               ffi::ResultBuffer<ffi::F32> g_y0, ffi::ResultBuffer<ffi::F32> g_params,
                               ffi::ResultBuffer<ffi::U8> workspace, ffi::Span<const float> step_ts, int32_t B, int32_t n,
                               int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d = dims_of(batch_of(*g_y0, n, h), n, h, e, L, T, flags);
  PegControl c = control_of(ts.typed_data(), adj_coef.typed_data(), adj_rowsum.typed_data(), adj_diag.typed_data(), adj_total.typed_data(),
                            tch_coef.typed_data(), e > 0 ? x_coef.typed_data() : nullptr, adj_absmax.typed_data());
  const int32_t steps = (int32_t)step_ts.size() - 1;
  cudaMemsetAsync(g_params->typed_data(), 0, g_params->element_count() * sizeof(float), stream);
  // the cotangent of the saved trajectory arrives as g_ckpt [S+1,B,n,h] (its last slab is the cotangent of y(T))
  const int rc = pegncde_solve_bwd(stream, &d, &c, params.typed_data(), step_ts.begin(), steps, y_ckpt.typed_data(),
                                   stage_store.element_count() ? stage_store.typed_data() : nullptr, nullptr,
                                   g_ckpt.typed_data(), /*g_stage=*/nullptr, g_y0->typed_data(), g_params->typed_data(), /*g_xcoef=*/nullptr,
                                   workspace->typed_data(), workspace->element_count());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

// The ODETerm callable itself, vf(t, y, args) (src/models/vector_fields/perm_equiv_graph_vector_field.py:85-129): what the Equinox
// module FusedPermEquivGraphVectorField calls when a stock diffrax solver drives it stage by stage.  t is a host scalar attribute
// of the call in eager mode and a [1] operand under jit (diffrax traces t): the operand form is the one bound here.
static ffi::Error VfFwdImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> ts, ffi::Buffer<ffi::F32> adj_coef,
                            ffi::Buffer<ffi::F32> adj_rowsum, ffi::Buffer<ffi::F32> adj_diag, ffi::Buffer<ffi::F32> adj_total,
                            ffi::Buffer<ffi::F32> tch_coef, ffi::Buffer<ffi::F32> x_coef, ffi::Buffer<ffi::F32> adj_absmax,
                            ffi::Buffer<ffi::F32> y, ffi::ResultBuffer<ffi::F32> dy, ffi::ResultBuffer<ffi::U8> workspace, float t,
                            int32_t B, int32_t n, int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d = dims_of(batch_of(y, n, h), n, h, e, L, T, flags);
  PegControl c = control_of(ts.typed_data(), adj_coef.typed_data(), adj_rowsum.typed_data(), adj_diag.typed_data(), adj_total.typed_data(),
                            tch_coef.typed_data(), e > 0 ? x_coef.typed_data() : nullptr, adj_absmax.typed_data());
  const int rc = pegncde_vf_fwd(stream, &d, &c, params.typed_data(), t, y.typed_data(), dy->typed_data(), workspace->typed_data(),
                                workspace->element_count());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

static ffi::Error VfVjpImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> ts, ffi::Buffer<ffi::F32> adj_coef,
                            ffi::Buffer<ffi::F32> adj_rowsum, ffi::Buffer<ffi::F32> adj_diag, ffi::Buffer<ffi::F32> adj_total,
                            ffi::Buffer<ffi::F32> tch_coef, ffi::Buffer<ffi::F32> x_coef, ffi::Buffer<ffi::F32> adj_absmax,
                            ffi::Buffer<ffi::F32> y, ffi::Buffer<ffi::F32> g_dy, ffi::ResultBuffer<ffi::F32> g_y,
                            ffi::ResultBuffer<ffi::F32> g_params, ffi::ResultBuffer<ffi::U8> workspace, float t, int32_t B, int32_t n,
                            int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d = dims_of(batch_of(y, n, h), n, h, e, L, T, flags);
  PegControl c = control_of(ts.typed_data(), adj_coef.typed_data(), adj_rowsum.typed_data(), adj_diag.typed_data(), adj_total.typed_data(),
                            tch_coef.typed_data(), e > 0 ? x_coef.typed_data() : nullptr, adj_absmax.typed_data());
  cudaMemsetAsync(g_params->typed_data(), 0, g_params->element_count() * sizeof(float), stream);
  const int rc = pegncde_vf_vjp(stream, &d, &c, params.typed_data(), t, y.typed_data(), g_dy.typed_data(), g_y->typed_data(),
                                g_params->typed_data(), /*g_xdot=*/nullptr, workspace->typed_data(), workspace->element_count());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

// One Tsit5 step with its error estimate and all seven slopes: the body of the jax.lax.while_loop of the adaptive solve
// (src/models/graph_neural_cde.py:86-104; the PID controller arithmetic stays in jnp on scalars).
static ffi::Error StepFwdImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> params, ffi::Buffer<ffi::F32> ts, ffi::Buffer<ffi::F32> adj_coef,
                              ffi::Buffer<ffi::F32> adj_rowsum, ffi::Buffer<ffi::F32> adj_diag, ffi::Buffer<ffi::F32> adj_total,
                              ffi::Buffer<ffi::F32> tch_coef, ffi::Buffer<ffi::F32> x_coef, ffi::Buffer<ffi::F32> adj_absmax,
                              ffi::Buffer<ffi::F32> y, ffi::Buffer<ffi::F32> k1_in, ffi::ResultBuffer<ffi::F32> k1,
                              ffi::ResultBuffer<ffi::F32> y1, ffi::ResultBuffer<ffi::F32> y_err, ffi::ResultBuffer<ffi::F32> k7,
                              ffi::ResultBuffer<ffi::F32> k_stages, ffi::ResultBuffer<ffi::U8> workspace, float t, float dt, int32_t k1_valid,
                              int32_t B, int32_t n, int32_t h, int32_t e, int32_t L, int32_t T, int32_t flags) {
  PegDims d = dims_of(batch_of(y, n, h), n, h, e, L, T, flags);
  PegControl c = control_of(ts.typed_data(), adj_coef.typed_data(), adj_rowsum.typed_data(), adj_diag.typed_data(), adj_total.typed_data(),
                            tch_coef.typed_data(), e > 0 ? x_coef.typed_data() : nullptr, adj_absmax.typed_data());
  if (k1_valid) cudaMemcpyAsync(k1->typed_data(), k1_in.typed_data(), k1_in.element_count() * sizeof(float), cudaMemcpyDeviceToDevice, stream);
  const int rc = pegncde_step_fwd(stream, &d, &c, params.typed_data(), t, dt, y.typed_data(), k1->typed_data(), k1_valid, y1->typed_data(),
                                  y_err->typed_data(), k7->typed_data(), k_stages->typed_data(), workspace->typed_data(), workspace->element_count());
  if (rc != PEG_OK) return ffi::Error(ffi::ErrorCode::kInternal, pegncde_strerror(rc));
  return ffi::Error::Success();
}

#define PEG_BIND_COMMON()                                                                                         \
  ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>()
#define PEG_DIM_ATTRS()                                                                                           \
  Attr<int32_t>("B").Attr<int32_t>("n").Attr<int32_t>("h").Attr<int32_t>("e").Attr<int32_t>("L").Attr<int32_t>("T").Attr<int32_t>("flags")
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegPackAdj, PackAdjImpl,
                              PEG_BIND_COMMON()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>()
                                  .PEG_DIM_ATTRS());
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegPackX, PackXImpl,
                              PEG_BIND_COMMON()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>()
                                  .PEG_DIM_ATTRS());
#define PEG_CONTROL_ARGS() /* params, ts, adj_coef, adj_rowsum, adj_diag, adj_total, tch_coef, x_coef, adj_absmax */                        \
  Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()                 \
      .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()            \
      .Arg<ffi::Buffer<ffi::F32>>()
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegVfFwd, VfFwdImpl,
                              PEG_BIND_COMMON().PEG_CONTROL_ARGS().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<float>("t").PEG_DIM_ATTRS());
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegVfVjp, VfVjpImpl,
                              PEG_BIND_COMMON().PEG_CONTROL_ARGS().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<float>("t").PEG_DIM_ATTRS());
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegStepFwd, StepFwdImpl,
                              PEG_BIND_COMMON().PEG_CONTROL_ARGS().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<float>("t").Attr<float>("dt").Attr<int32_t>("k1_valid").PEG_DIM_ATTRS());
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegSolveFwd, SolveFwdImpl,
                              PEG_BIND_COMMON()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<ffi::Span<const float>>("step_ts")
                                  .Attr<int32_t>("B").Attr<int32_t>("n").Attr<int32_t>("h").Attr<int32_t>("e")
                                  .Attr<int32_t>("L").Attr<int32_t>("T").Attr<int32_t>("flags"));
XLA_FFI_DEFINE_HANDLER_SYMBOL(PegSolveBwd, SolveBwdImpl,
                              PEG_BIND_COMMON()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::U8>>()
                                  .Attr<ffi::Span<const float>>("step_ts")
                                  .Attr<int32_t>("B").Attr<int32_t>("n").Attr<int32_t>("h").Attr<int32_t>("e")
                                  .Attr<int32_t>("L").Attr<int32_t>("T").Attr<int32_t>("flags"));
