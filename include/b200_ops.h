/* b200_ops.h -- C ABI of the B200-native op-kernel layer (libb200tf.so).
 *
 * This is the drop-in boundary described in SURVEY.md section 8(b): plain pointers, sizes and
 * ints only; no C++ or torch types cross it.  Every entry point sits where the reference's GPU
 * op kernels call into StreamExecutor (tensorflow/stream_executor/stream.h: ThenBlasGemm :1154,
 * ThenConvolveWithAlgorithm, ThenMemcpy :1482-1529, ThenMemZero :1531, ThenRecordEvent :214,
 * BlockHostUntilDone :1591) or launch their own CUDA kernels; each declaration cites the
 * reference code it replaces.  The thin OpKernel wrappers in
 * simple_tensorflow_b200/csrc/tensorflow/core/kernels/ are the only intended callers.
 *
 * Conventions
 *   - All data pointers are DEVICE pointers unless the name ends in _host.
 *   - `stream` is a cudaStream_t / CUstream passed as void* (NULL = legacy default stream).
 *     Every op only ENQUEUES work and returns (gpu_device.cc:337-399 contract); nothing in an op
 *     entry point synchronises the device.
 *   - Return value: 0 on success, otherwise a tensorflow::error::Code value
 *     (tensorflow/core/lib/core/error_codes.proto): 3 INVALID_ARGUMENT, 8 RESOURCE_EXHAUSTED,
 *     12 UNIMPLEMENTED, 13 INTERNAL.  b200_last_error() returns the message for the calling
 *     thread; the wrapper turns both into a tensorflow::Status.
 *   - dtype arguments use tensorflow::DataType numbering (framework/types.proto).
 *   - Tensors are dense row-major (framework/tensor_types.h:25-28); images are NHWC, filters HWIO.
 *   - There is NO CPU fallback: without a CUDA device every compute entry point returns
 *     13 INTERNAL.
 */
#ifndef B200_OPS_H_
#define B200_OPS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_API __attribute__((visibility("default")))

/* tensorflow::error::Code subset */
enum {
  B200_OK = 0,
  B200_INVALID_ARGUMENT = 3,
  B200_RESOURCE_EXHAUSTED = 8,
  B200_FAILED_PRECONDITION = 9,
  B200_UNIMPLEMENTED = 12,
  B200_INTERNAL = 13,
  B200_UNAVAILABLE = 14
};

/* tensorflow::DataType subset (framework/types.proto:13-40) */
enum {
  B200_DT_FLOAT = 1,
  B200_DT_INT32 = 3,
  B200_DT_INT64 = 9,
  B200_DT_BFLOAT16 = 14,
  B200_DT_HALF = 19      /* IEEE fp16: b200_cast only; the ops take it through fp32 (half_ops.cc) */
};

/* ------------------------------------------------------------------ library / device */
B200_API const char* b200_version(void);
B200_API const char* b200_last_error(void);
/* Number of CUDA devices visible (0 without a GPU; never fails). */
B200_API int b200_device_count(void);
B200_API int b200_set_device(int ordinal);
/* Kernels launched by this library in the calling process since load (all threads). */
B200_API uint64_t b200_launch_count(void);
/* Gradient exchanges issued by this process since load: launches of the NVLink peer-memory
 * all-reduce kernel (b200_peer_all_reduce) and NCCL all-reduce calls (b200_nccl_all_reduce*).
 * bench.py reads it around the timed region to say which exchange actually ran (the device falls
 * back to NCCL when the peer arena cannot be mapped).  No reference counterpart: the reference
 * ships no collective (third_party/nccl.BUILD has no call sites). */
B200_API void b200_collective_counts(uint64_t* peer_launches, uint64_t* nccl_calls);
/* Measurement hook for bench.py's roofline: between begin and end every tensor-core GEMM launch
 * (MatMul, BatchMatMul, the conv GEMMs) is bracketed by CUDA events on its own stream;
 * end() waits for them and returns the summed device time, launch count and 2*M*N*K FLOPs. */
/* 1 while a b200_profile_begin/end pass is active (the executor then bypasses captured graphs, whose
 * launches carry no per-launch events). */
B200_API int b200_profile_active(void);
/* Adds n to the launch counter: a replayed CUDA graph launches the kernels of the captured step
 * without passing through the b200_* entry points that count them. */
B200_API void b200_note_launches(uint64_t n);
/* The same for the gradient-exchange counters of b200_collective_counts. */
B200_API void b200_note_collectives(uint64_t peer_launches, uint64_t nccl_calls);
/* Step-level CUDA graphs (the executor captures one Session.Run plan, keyed like the reference's
 * executor cache, direct_session.cc:918-936): capture everything the b200_* calls enqueue on
 * `stream` between begin and end (relaxed mode), instantiate, replay.  end returns the executable
 * graph or, on failure, B200_INTERNAL with the stream back in normal mode. */
B200_API int b200_stream_begin_capture(void* stream);
B200_API int b200_stream_end_capture(void* stream, void** graph_exec);
B200_API int b200_graph_launch(void* graph_exec, void* stream);
B200_API int b200_graph_destroy(void* graph_exec);
B200_API int b200_profile_begin(void);
B200_API int b200_profile_end(double* gemm_ms_total, uint64_t* gemm_launches,
                              double* gemm_flops_total);
/* MatMul/Conv precision for DT_FLOAT: 0 = single-pass TF32 tensor cores (default; inputs are
 * truncated to 10 mantissa bits by the MMA, fp32 accumulate), 1 = SIMT fp32 FMA (IEEE fp32
 * products, the reference Eigen path's arithmetic).  Shapes the TMA path cannot address
 * (leading dimension not a multiple of 16 bytes) always use the SIMT kernel. */
B200_API int b200_set_matmul_precision(int mode);
B200_API int b200_get_matmul_precision(void);

/* ------------------------------------------------------------------ StreamExecutor-level shim
 * Mirrors Stream / StreamExecutor members the reference's GPU device uses
 * (stream_executor/stream.h:116,189,214,1482-1531,1591; stream_executor_pimpl.h:110,191). */
B200_API int b200_stream_create(void** stream);
/* high_priority != 0: the device's highest stream priority (the reference creates all streams at
 * default priority; the collective stream wants its few CTAs scheduled ahead of queued GEMMs). */
B200_API int b200_stream_create_with_priority(void** stream, int high_priority);
B200_API int b200_stream_destroy(void* stream);
B200_API int b200_stream_synchronize(void* stream);          /* BlockHostUntilDone */
B200_API int b200_stream_wait_event(void* stream, void* event);
/* Run fn(arg) on a driver thread once everything enqueued on `stream` so far has completed
 * (Stream::ThenDoHostCallback, stream_executor/stream.h:1624).  fn must not call CUDA. */
B200_API int b200_stream_add_host_callback(void* stream, void (*fn)(void*), void* arg); /* ThenWaitFor */
B200_API int b200_event_create(void** event);
B200_API int b200_event_destroy(void* event);
B200_API int b200_event_record(void* event, void* stream);   /* ThenRecordEvent */
B200_API int b200_event_synchronize(void* event);
B200_API int b200_event_query(void* event);                  /* 0 done, 1 pending, <0 error */
B200_API int b200_event_elapsed_ms(void* start, void* stop, float* ms);
B200_API int b200_malloc(void** dptr, size_t bytes);         /* AllocateArray */
B200_API int b200_free(void* dptr);
B200_API int b200_host_malloc(void** hptr, size_t bytes);    /* HostMemoryAllocate (pinned) */
B200_API int b200_host_free(void* hptr);
B200_API int b200_memcpy_h2d_async(void* dst, const void* src_host, size_t bytes, void* stream);
B200_API int b200_memcpy_d2h_async(void* dst_host, const void* src, size_t bytes, void* stream);
B200_API int b200_memcpy_d2d_async(void* dst, const void* src, size_t bytes, void* stream);
B200_API int b200_memset_async(void* dst, int byte_value, size_t bytes, void* stream); /* ThenMemZero */
B200_API int b200_mem_info(size_t* free_bytes, size_t* total_bytes);

/* ------------------------------------------------------------------ MatMul / BatchMatMul
 * Replaces LaunchMatMul<GPUDevice,T,true>::launch -> ThenBlasGemm (core/kernels/matmul_op.cc:162-203).
 * a is [m,k] (or [k,m] when transpose_a), b is [k,n] (or [n,k] when transpose_b), c is [m,n];
 * same argument meaning as the op attrs (core/ops/math_ops.cc:1033-1040).  m,n,k > 0: the
 * zero-size rules of MatMulOp::Compute (matmul_op.cc:240-253) stay in the OpKernel wrapper.
 * dtype: DT_FLOAT (tf32 tensor cores, fp32 accumulate) or DT_BFLOAT16 (fp32 accumulate).
 * workspace (optional, may be NULL/0): b200_matmul_workspace_bytes() bytes of device scratch let
 * shapes with few output tiles (e.g. dW = X^T dY, 1024x1024 output, K = 4096) split K across
 * SMs; partial sums are added in a fixed order, so results do not depend on scheduling.  The
 * OpKernel wrapper obtains it with allocate_temp, as the reference's GPU conv kernels do. */
B200_API size_t b200_matmul_workspace_bytes(int dtype, int64_t m, int64_t n, int64_t k);
B200_API int b200_matmul(int dtype, const void* a, const void* b, void* c, int64_t m, int64_t n,
                         int64_t k, int transpose_a, int transpose_b, void* workspace,
                         size_t workspace_bytes, void* stream);
/* MatMul with the element-wise op that follows it in the graph applied in the GEMM epilogue
 * (accumulator still in registers, one HBM write instead of three round trips):
 *   bias != NULL                -> BiasAdd   (bias [n], bias_op.cc:62-117 semantics)
 *   relu != 0                   -> Relu      (relu_op_functor.h:28-38), after the bias
 *   relu_grad_features != NULL  -> ReluGrad  c = (a.b) * (features > 0), features [m, n]
 *                                  (relu_op_functor.h:44-57); exclusive with relu
 * Used by the executor's MatMul+BiasAdd(+Relu) / MatMul+ReluGrad rewrite (the role the
 * reference gives its GraphOptimizer, direct_session.cc:1051); op boundaries in the user's graph
 * are unchanged and results are identical to running the ops one by one. */
B200_API int b200_fused_matmul(int dtype, const void* a, const void* b, void* c, int64_t m,
                               int64_t n, int64_t k, int transpose_a, int transpose_b,
                               const void* bias, int relu, const void* relu_grad_features,
                               void* stream);
/* The same with optional scratch (b200_matmul_workspace_bytes): lets a bias / relu-tailed product
 * with few output tiles split K; the tail is then applied by the ordered reduction pass. */
B200_API int b200_fused_matmul_ws(int dtype, const void* a, const void* b, void* c, int64_t m,
                                  int64_t n, int64_t k, int transpose_a, int transpose_b,
                                  const void* bias, int relu, const void* relu_grad_features,
                                  void* workspace, size_t workspace_bytes, void* stream);
/* Two independent products with the arguments of b200_fused_matmul_ws each (one dtype), computed
 * as two b200_fused_matmul_ws calls would compute them, bit for bit.  When both run on the tensor
 * cores with the same tile config and one is K-major x K-major (dX = dY W^T: transpose_b) while
 * the other is MN-major x MN-major (dW = X^T dY: transpose_a), they share one persistent launch:
 * the second product's operand fill and main loop hide the first one's epilogue, and the CTA
 * pairs one product would leave idle get work.  Otherwise they run one after the other.
 * workspace (optional): b200_matmul_pair_workspace_bytes() bytes; product 0's split-K scratch
 * (b200_matmul_workspace_bytes of its shape) sits at offset 0, product 1's at the next 256-byte
 * boundary after it. */
B200_API size_t b200_matmul_pair_workspace_bytes(int dtype, int64_t m0, int64_t n0, int64_t k0,
                                                 int64_t m1, int64_t n1, int64_t k1);
B200_API int b200_matmul_pair(int dtype, const void* a0, const void* b0, void* c0, int64_t m0,
                              int64_t n0, int64_t k0, int transpose_a0, int transpose_b0,
                              const void* bias0, int relu0, const void* relu_grad_features0,
                              const void* a1, const void* b1, void* c1, int64_t m1, int64_t n1,
                              int64_t k1, int transpose_a1, int transpose_b1, const void* bias1,
                              int relu1, const void* relu_grad_features1, void* workspace,
                              size_t workspace_bytes, void* stream);
/* Replaces LaunchBatchMatMul<GPUDevice,Scalar>::Launch -> ThenBlasGemmBatchedWithScratch
 * (core/kernels/batch_matmul_op_impl.h:297-363).  x is [batch,m,k] (or [batch,k,m] when adj_x),
 * y is [batch,k,n] (or [batch,n,k] when adj_y); strided, no pointer arrays, no scratch. */
B200_API int b200_batch_matmul(int dtype, const void* x, const void* y, void* out, int64_t batch,
                               int64_t m, int64_t n, int64_t k, int adj_x, int adj_y,
                               void* stream);

/* ------------------------------------------------------------------ BiasAdd / BiasAddGrad
 * BiasGPU<T>::compute, NHWC (core/kernels/bias_op_gpu.cu.cc:69-88; op bias_op.cc:43-117):
 * out[r, c] = in[r, c] + bias[c], rows = prod(leading dims); out may alias in. */
B200_API int b200_bias_add(int dtype, const void* in, const void* bias, void* out, int64_t rows,
                           int64_t channels, void* stream);
/* BiasGradGPU<T>::compute, NHWC (bias_op_gpu.cu.cc:189-242; op bias_op.cc:171-227):
 * out[c] = sum_r out_backprop[r, c]; fp32 accumulation, deterministic two-stage reduction
 * (no atomics).  workspace: b200_bias_add_grad_workspace_bytes() bytes of device scratch. */
B200_API size_t b200_bias_add_grad_workspace_bytes(int dtype, int64_t rows, int64_t channels);
B200_API int b200_bias_add_grad(int dtype, const void* out_backprop, void* out, int64_t rows,
                                int64_t channels, void* workspace, size_t workspace_bytes,
                                void* stream);
/* data_format = NCHW, native (no layout change): BiasGPU<T>::compute's BiasNCHWKernel
 * (bias_op_gpu.cu.cc:56-63,80-86) and BiasGradGPU's BiasGradNCHW_SharedAtomics (:140-188,225-233).
 * The tensor is [batch, channels, image] with image = prod(dims after the channel dimension), so
 * 3-D, 4-D and 5-D NCHW inputs (bias_op.cc:75-107) are one call.  out may alias in.  The
 * gradient is a two-stage ordered reduction (no atomics, bit-reproducible); workspace:
 * b200_bias_add_grad_nchw_workspace_bytes() bytes of device scratch. */
B200_API int b200_bias_add_nchw(int dtype, const void* in, const void* bias, void* out,
                                int64_t batch, int64_t channels, int64_t image, void* stream);
B200_API size_t b200_bias_add_grad_nchw_workspace_bytes(int dtype, int64_t batch,
                                                        int64_t channels, int64_t image);
B200_API int b200_bias_add_grad_nchw(int dtype, const void* out_backprop, void* out,
                                     int64_t batch, int64_t channels, int64_t image,
                                     void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ Relu / ReluGrad
 * functor::Relu / functor::ReluGrad (core/kernels/relu_op_functor.h:28-60):
 * y = max(x, 0);  dx = g * (f > 0) with f the Relu input or output.  In-place allowed. */
B200_API int b200_relu(int dtype, const void* features, void* activations, int64_t n,
                       void* stream);
B200_API int b200_relu_grad(int dtype, const void* gradients, const void* features,
                            void* backprops, int64_t n, void* stream);
/* backprops = ReluGrad(gradients, features) and bias_grad = BiasAddGrad(backprops) in ONE pass over
 * [rows, channels]: the pair a convolution / dense layer's backward pass runs back to back
 * (relu_op.h:62-94 then bias_op.cc:171-227); `backprops` may alias `gradients`.  Created by the
 * executor's rewrite (`_ReluGradBiasAddGrad`); workspace from the _workspace_bytes call. */
B200_API size_t b200_relu_grad_bias_grad_workspace_bytes(int dtype, int64_t rows, int64_t channels);
B200_API int b200_relu_grad_bias_grad(int dtype, const void* gradients, const void* features,
                                      void* backprops, void* bias_grad, int64_t rows,
                                      int64_t channels, void* workspace, size_t workspace_bytes,
                                      void* stream);

/* ------------------------------------------------------------------ Softmax / LogSoftmax
 * SoftmaxEigenImpl (core/kernels/softmax_op_functor.h:43-99): rank-2 [rows, cols];
 * softmax = exp(x - max) * (1 / sum);  log variant = x - max - log(sum exp(x - max)). */
B200_API int b200_softmax(int dtype, const void* logits, void* out, int64_t rows, int64_t cols,
                          int log_softmax, void* stream);
/* XentEigenImpl (core/kernels/xent_op.h:47-113): loss[r] = sum_c labels*(log sum exp - (x-max)),
 * backprop = softmax - labels. */
B200_API int b200_softmax_xent(int dtype, const void* logits, const void* labels, void* loss,
                               void* backprop, int64_t rows, int64_t cols, void* stream);
/* Same, with the backprop output multiplied by a DEVICE scalar before it is stored (the
 * `backprop * grad_loss` Mul that nn_grad.py:323-333 emits right behind the op, folded in by the
 * executor when grad_loss is a scalar constant).  fp32 only; NULL scale == b200_softmax_xent. */
B200_API int b200_softmax_xent_scaled(int dtype, const void* logits, const void* labels, void* loss,
                                      void* backprop, int64_t rows, int64_t cols,
                                      const float* backprop_scale, void* stream);

/* ------------------------------------------------------------------ MaxPool / MaxPoolGrad (NHWC)
 * MaxPoolForwardNHWC (core/kernels/maxpooling_op_gpu.cu.cc:93-129) with the CPU kernel's
 * semantics (pooling_ops_common.h:204-238): padded cells never participate.
 * pad_top/pad_left are the "before" paddings from GetWindowedOutputSize. */
B200_API int b200_max_pool(int dtype, const void* in, void* out, int64_t batch, int64_t in_h,
                           int64_t in_w, int64_t channels, int64_t out_h, int64_t out_w,
                           int window_h, int window_w, int stride_h, int stride_w, int pad_top,
                           int pad_left, void* stream);
/* MaxPoolingGradOp (core/kernels/maxpooling_op.cc:230-306,117-178): gradient goes to the first
 * maximum of each window in row-major scan order; gather formulation, no atomics. */
B200_API int b200_max_pool_grad(int dtype, const void* orig_in, const void* orig_out,
                                const void* grad, void* in_backprop, int64_t batch, int64_t in_h,
                                int64_t in_w, int64_t channels, int64_t out_h, int64_t out_w,
                                int window_h, int window_w, int stride_h, int stride_w,
                                int pad_top, int pad_left, void* stream);
/* MaxPoolGrad -> ReluGrad -> BiasAddGrad of a conv / bias / relu / pool block in one pass
 * (maxpooling_op.cc:230-306 + relu_op.h:70-98 + bias_op.cc:171-227; the executor's
 * `_MaxPoolGradReluGradBiasAddGrad` rewrite).  orig_in is the pool's input = the Relu output = the
 * ReluGrad's features.  backprops = ReluGrad(MaxPoolGrad(orig_in, ., grad), orig_in), bias_grad =
 * its sum over N, H, W (ordered, no atomics).  Returns B200_UNIMPLEMENTED when the windows do not
 * tile the input or the channel count has no flat 16-byte mapping (workspace_bytes() == 0): the
 * caller then runs b200_max_pool_grad and b200_relu_grad_bias_grad. */
B200_API size_t b200_max_pool_grad_relu_bias_grad_workspace_bytes(
    int dtype, int64_t batch, int64_t in_h, int64_t in_w, int64_t channels, int64_t out_h,
    int64_t out_w, int window_h, int window_w, int stride_h, int stride_w, int pad_top, int pad_left);
B200_API int b200_max_pool_grad_relu_bias_grad(
    int dtype, const void* orig_in, const void* grad, void* backprops, void* bias_grad,
    int64_t batch, int64_t in_h, int64_t in_w, int64_t channels, int64_t out_h, int64_t out_w,
    int window_h, int window_w, int stride_h, int stride_w, int pad_top, int pad_left,
    void* workspace, size_t workspace_bytes, void* stream);


/* ------------------------------------------------------------------ Cast / ArgMax (bit-exact)
 * CastOp (core/kernels/cast_op.cc, cast_op.h:93-141): float->bfloat16 TRUNCATES the low 16 bits
 * (framework/bfloat16.cc:20-31), bfloat16->float shifts; int32/int64/float conversions follow
 * C++ static_cast. */
B200_API int b200_cast(int src_dtype, int dst_dtype, const void* in, void* out, int64_t n,
                       void* stream);
/* ArgOp<..., ArgMax> (core/kernels/argmax_op.cc:44-98): input viewed as [outer, axis, inner],
 * output int64 [outer, inner]; lowest index wins ties. */
B200_API int b200_argmax(int dtype, const void* in, int64_t* out, int64_t outer, int64_t axis_size,
                         int64_t inner, void* stream);

/* ------------------------------------------------------------------ Conv2D family (NHWC, HWIO)
 * Geometry is what Conv2DOp::Compute / ConvBackpropComputeDimensions derive
 * (core/kernels/conv_ops.cc:267-380, conv_grad_ops.cc:37-126): out size and the "before"
 * paddings come from GetWindowedOutputSizeVerbose (framework/common_shape_fns.cc:19-56). */
typedef struct b200_conv2d_geometry {
  int64_t batch, in_h, in_w, in_c;      /* input  [batch, in_h, in_w, in_c]        */
  int64_t filter_h, filter_w, out_c;    /* filter [filter_h, filter_w, in_c, out_c] */
  int64_t out_h, out_w;                 /* output [batch, out_h, out_w, out_c]      */
  int32_t stride_h, stride_w;
  int32_t pad_top, pad_left;
} b200_conv2d_geometry;

/* Scratch needed by any of the three conv entry points for this geometry (may be 0). */
B200_API size_t b200_conv2d_workspace_bytes(int dtype, const b200_conv2d_geometry* g, int which);
/* which: 0 forward, 1 backprop-input, 2 backprop-filter */

/* Replaces LaunchConv2DOp<GPUDevice,T>::launch (core/kernels/conv_ops.cc:433-720). */
B200_API int b200_conv2d(int dtype, const void* input, const void* filter, void* output,
                         const b200_conv2d_geometry* g, void* workspace, size_t workspace_bytes,
                         void* stream);
/* out = [relu](conv2d(input, filter) + bias[k]) in one pass: the tail the executor's rewrite of
 * Conv2D -> BiasAdd (-> Relu) chains asks for (`_FusedConv2D`; what later TensorFlow's remapper
 * does).  Replaces LaunchConv2DOp (conv_ops.cc:433-720) + BiasOp (bias_op.cc:62-117) +
 * ReluOp (relu_op.h:34-60) launched back to back; same arithmetic, same workspace as b200_conv2d. */
B200_API int b200_fused_conv2d(int dtype, const void* input, const void* filter, const void* bias,
                               int relu, void* output, const b200_conv2d_geometry* geom,
                               void* workspace, size_t workspace_bytes, void* stream);
/* Replaces Conv2DSlowBackpropInputOp<GPUDevice,T> (core/kernels/conv_grad_input_ops.cc:533-917). */
B200_API int b200_conv2d_backprop_input(int dtype, const void* filter, const void* out_backprop,
                                        void* in_backprop, const b200_conv2d_geometry* g,
                                        void* workspace, size_t workspace_bytes, void* stream);
/* Replaces Conv2DSlowBackpropFilterOp<GPUDevice,T> (core/kernels/conv_grad_filter_ops.cc:361-738). */
B200_API int b200_conv2d_backprop_filter(int dtype, const void* input, const void* out_backprop,
                                         void* filter_backprop, const b200_conv2d_geometry* g,
                                         void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------ graph glue (SURVEY 8f rank 1)
 * ApplyGradientDescent (core/kernels/training_ops.cc:410-412): var -= alpha * delta; alpha is a
 * DEVICE scalar of the same dtype, as in the reference's GPU functor (training_ops_gpu.cu.cc). */
B200_API int b200_apply_gradient_descent(int dtype, void* var, const void* alpha,
                                         const void* delta, int64_t n, void* stream);
/* The same update for `count` variables in one launch (host arrays of device pointers / element
 * counts).  Element-wise identical to `count` calls of b200_apply_gradient_descent. */
B200_API int b200_apply_gradient_descent_multi(int dtype, int count, void* const* vars_host,
                                               const void* const* alphas_host,
                                               const void* const* deltas_host,
                                               const int64_t* n_host, void* stream);
/* Mul (core/kernels/cwise_op_mul_1.cc) for the two shapes gradient graphs need: same-shape, or
 * y a DEVICE scalar broadcast over x (y_is_scalar != 0). */
B200_API int b200_mul(int dtype, const void* x, const void* y, void* out, int64_t n,
                      int y_is_scalar, void* stream);
/* out[b][col][row] = in[b][row][col]: the NCHW <-> NHWC layout change the reference's GPU kernels do
 * around cuDNN (core/kernels/conv_ops.cc:558-612,712-719, conv_2d.h NHWCToNCHW / NCHWToNHWC); here
 * it lets NCHW graphs use the NHWC-native kernels.  batch <= 65535, rows <= 2 M. */
B200_API int b200_batched_transpose(int dtype, const void* in, void* out, int64_t batch,
                                    int64_t rows, int64_t cols, void* stream);
/* Add (core/kernels/cwise_op_add_1.cc), same two shapes. */
B200_API int b200_add(int dtype, const void* x, const void* y, void* out, int64_t n,
                      int y_is_scalar, void* stream);
/* AddN (core/kernels/aggregate_ops.cc:153-176) for n_inputs <= 8. */
B200_API int b200_add_n(int dtype, const void* const* inputs_host, int n_inputs, void* out,
                        int64_t n, void* stream);
/* out = in * scale (used for the mean-loss gradient and the 1/p replica average). */
B200_API int b200_scale(int dtype, const void* in, float scale, void* out, int64_t n,
                        void* stream);
/* out[0] = sum(in[0..n)) * scale; fp32, deterministic (loss reduction: Mean/Sum glue). */
B200_API int b200_reduce_sum(int dtype, const void* in, float scale, void* out, int64_t n,
                             void* stream);
/* Sum / Mean over one contiguous run of axes: `in` viewed as [outer, reduce, inner],
 * out[o, i] = scale * sum_r in[o, r, i]; fp32 accumulation, fixed order, float / bfloat16.
 * Replaces ReductionOp<GPUDevice, T, SumReducer / MeanReducer> for the axis patterns that
 * collapse to one reduced run (core/kernels/reduction_ops_common.h ReductionHelper::Simplify,
 * reduction_ops_sum.cc, reduction_ops_mean.cc). */
B200_API int b200_reduce(int dtype, const void* in, void* out, int64_t outer, int64_t reduce,
                         int64_t inner, float scale, void* stream);

/* ------------------------------------------------------------------ replica data-parallel
 * One NCCL all-reduce (sum) over a contiguous gradient arena on the compute stream
 * (SURVEY.md 8e).  The reference has no collective op (third_party/nccl.BUILD has no call
 * sites); this replaces its tower pattern _Send/_Recv + AddN (aggregate_ops.cc:153-176).
 * libnccl is dlopen()ed on first use; unique-id exchange is the host's job. */
B200_API int b200_nccl_unique_id(void* id128_host);  /* writes 128 bytes */
B200_API int b200_nccl_comm_init_rank(void** comm, int nranks, const void* id128_host, int rank);
B200_API int b200_nccl_comm_destroy(void* comm);
/* average != 0 -> ncclAvg (sum / ranks) so a gradient mean needs no separate scale kernel.
 * Calls between group_start / group_end are aggregated by NCCL into ONE collective launch, so a
 * set of gradient tensors is reduced without packing them into a staging buffer. */
B200_API int b200_nccl_group_start(void);
B200_API int b200_nccl_group_end(void);
B200_API int b200_nccl_all_reduce(int dtype, const void* sendbuf, void* recvbuf, int64_t count,
                                  int average, void* comm, void* stream);
B200_API int b200_nccl_all_reduce_sum(int dtype, const void* sendbuf, void* recvbuf,
                                      int64_t count, void* comm, void* stream);
B200_API int b200_nccl_comm_user_rank(void* comm, int* rank);
/* ncclAllGather of `bytes_per_rank` bytes (device buffers); used to exchange IPC handles. */
B200_API int b200_nccl_all_gather_bytes(const void* sendbuf, void* recvbuf, int64_t bytes_per_rank,
                                        void* comm, void* stream);

/* ------------------------------------------------------------------ NVLink peer memory
 * A peer arena is one device buffer per rank, mapped into every rank of the communicator with
 * CUDA IPC (one process per GPU).  b200_peer_all_reduce is an in-place fp32 all-reduce over the
 * same byte range of every rank's arena, done by ONE kernel with peer loads over NVLink: the
 * gradient exchange of replica data-parallel training (SURVEY 8e; the reference does it with
 * _Send/_Recv + AddN, core/kernels/aggregate_ops.cc:153-176, common_runtime/gpu/gpu_util.cc:190-250).
 * Creation is collective over `nccl_comm` (handle exchange) and returns B200_UNAVAILABLE on every
 * rank when any rank cannot map its peers.  All ranks must issue the same sequence of
 * b200_peer_all_reduce calls.  max_ctas <= 0: the default grid (64 CTAs of 256 threads, which fit
 * on SMs next to resident GEMM CTAs). */
B200_API int b200_peer_arena_create(void* nccl_comm, int rank, int nranks, size_t data_bytes,
                                    void** arena);
/* What the last arena created in this process runs on: "nvls" (NVSwitch multicast memory, in-switch
 * reduction: nvls_allreduce.cu), "peer-ipc" (peer-mapped buffers, peer_allreduce.cu) or "none". */
B200_API const char* b200_peer_arena_backend(void);
/* 1 when the current device / driver can back an arena with NVSwitch multicast memory (and
 * B200TF_NVLS is not 0): what a front-end asks before it decides to bucket the gradient exchange
 * for overlap (simple_tensorflow_b200/ops.py apply_gradients).  No reference counterpart. */
B200_API int b200_nvls_supported(void);
B200_API int b200_peer_arena_destroy(void* arena);
B200_API void* b200_peer_arena_data(void* arena);
B200_API size_t b200_peer_arena_bytes(void* arena);
B200_API int b200_peer_all_reduce(void* arena, int dtype, size_t offset_bytes, int64_t count,
                                  int average, int max_ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_OPS_H_ */
