// MatMul / BatchMatMul for DEVICE_GPU on B200.
// Same validation, shape and zero-size rules as the reference's MatMulOp::Compute
// (core/kernels/matmul_op.cc:215-256) and BatchMatMul::Compute
// (core/kernels/batch_matmul_op_impl.h:367-434); the launch goes to b200_matmul /
// b200_batch_matmul instead of Stream::ThenBlasGemm (matmul_op.cc:179-195).
#include "tensorflow/core/kernels/gpu_kernel_util.h"

namespace tensorflow {

template <typename T>
class MatMulOp : public OpKernel {
 public:
  explicit MatMulOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_a", &transpose_a_));
    OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_b", &transpose_b_));
  }

  void Compute(OpKernelContext* ctx) override {
    const Tensor& a = ctx->input(0);
    const Tensor& b = ctx->input(1);
    OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(a.shape()),
                errors::InvalidArgument("In[0] is not a matrix"));
    OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(b.shape()),
                errors::InvalidArgument("In[1] is not a matrix"));
    const int a_contract = transpose_a_ ? 0 : 1;
    const int b_contract = transpose_b_ ? 1 : 0;
    OP_REQUIRES(ctx, a.dim_size(a_contract) == b.dim_size(b_contract),
                errors::InvalidArgument("Matrix size-incompatible: In[0]: ",
                                        a.shape().DebugString(), ", In[1]: ",
                                        b.shape().DebugString()));
    const int64 m = a.dim_size(1 - a_contract), k = a.dim_size(a_contract);
    const int64 n = b.dim_size(1 - b_contract);
    Tensor* out = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, TensorShape({m, n}), &out));
    if (out->NumElements() == 0) return;  // [0,x] or [x,0] operands: nothing to do
    void* stream = GetCudaStream(ctx);
    if (a.NumElements() == 0 || b.NumElements() == 0) {  // k == 0: zero-fill (:246-253)
      OP_REQUIRES_OK(ctx, FromAbi(b200_memset_async(out->raw_data(), 0, out->TotalBytes(), stream),
                                  "MatMul zero fill"));
      return;
    }
    const size_t ws_bytes = b200_matmul_workspace_bytes(AbiType<T>::v, m, n, k);
    Tensor scratch;
    if (ws_bytes > 0)  // split-K partial sums (stays alive until the stream passes it)
      OP_REQUIRES_OK(ctx, ctx->allocate_temp(DT_UINT8, TensorShape({(int64)ws_bytes}), &scratch));
    OP_REQUIRES_OK(ctx, FromAbi(b200_matmul(AbiType<T>::v, a.raw_data(), b.raw_data(),
                                            out->raw_data(), m, n, k, transpose_a_, transpose_b_,
                                            ws_bytes ? scratch.raw_data() : nullptr, ws_bytes,
                                            stream),
                                "Blas GEMM launch failed"));
  }

 private:
  bool transpose_a_;
  bool transpose_b_;
};

template <typename T>
class BatchMatMulOp : public OpKernel {
 public:
  explicit BatchMatMulOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    OP_REQUIRES_OK(ctx, ctx->GetAttr("adj_x", &adj_x_));
    OP_REQUIRES_OK(ctx, ctx->GetAttr("adj_y", &adj_y_));
  }

  void Compute(OpKernelContext* ctx) override {
    const Tensor& in0 = ctx->input(0);
    const Tensor& in1 = ctx->input(1);
    OP_REQUIRES(ctx, in0.dims() == in1.dims(),
                errors::InvalidArgument("In[0] and In[1] has different ndims: ",
                                        in0.shape().DebugString(), " vs. ",
                                        in1.shape().DebugString()));
    const int ndims = in0.dims();
    OP_REQUIRES(ctx, ndims >= 2,
                errors::InvalidArgument("In[0] and In[1] ndims must be >= 2: ", ndims));
    TensorShape out_shape;
    int64 batch = 1;
    for (int i = 0; i < ndims - 2; ++i) {  // batch dims must match exactly, no broadcasting
      OP_REQUIRES(ctx, in0.dim_size(i) == in1.dim_size(i),
                  errors::InvalidArgument("In[0].dim(", i, ") and In[1].dim(", i,
                                          ") must be the same: ", in0.shape().DebugString(),
                                          " vs ", in1.shape().DebugString()));
      out_shape.AddDim(in0.dim_size(i));
      batch *= in0.dim_size(i);
    }
    int64 d0 = in0.dim_size(ndims - 2), d1 = in0.dim_size(ndims - 1);
    int64 d2 = in1.dim_size(ndims - 2), d3 = in1.dim_size(ndims - 1);
    if (adj_x_) std::swap(d0, d1);
    if (adj_y_) std::swap(d2, d3);
    OP_REQUIRES(ctx, d1 == d2,
                errors::InvalidArgument("In[0] mismatch In[1] shape: ", d1, " vs. ", d2, ": ",
                                        in0.shape().DebugString(), " ", in1.shape().DebugString(),
                                        " ", adj_x_, " ", adj_y_));
    out_shape.AddDim(d0);
    out_shape.AddDim(d3);
    Tensor* out = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, out_shape, &out));
    if (out->NumElements() == 0) return;
    void* stream = GetCudaStream(ctx);
    if (in0.NumElements() == 0 || in1.NumElements() == 0) {
      OP_REQUIRES_OK(ctx, FromAbi(b200_memset_async(out->raw_data(), 0, out->TotalBytes(), stream),
                                  "BatchMatMul zero fill"));
      return;
    }
    OP_REQUIRES_OK(ctx, FromAbi(b200_batch_matmul(AbiType<T>::v, in0.raw_data(), in1.raw_data(),
                                                  out->raw_data(), batch, d0, d3, d1, adj_x_,
                                                  adj_y_, stream),
                                "Blas xGEMMBatched launch failed"));
  }

 private:
  bool adj_x_;
  bool adj_y_;
};

// _FusedMatMul: MatMul whose epilogue applies the BiasAdd / Relu / ReluGrad that followed it.
template <typename T>
class FusedMatMulOp : public OpKernel {
 public:
  explicit FusedMatMulOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_a", &transpose_a_));
    OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_b", &transpose_b_));
    std::vector<std::string> fused;
    OP_REQUIRES_OK(ctx, ctx->GetAttr("fused_ops", &fused));
    if (fused == std::vector<std::string>{"BiasAdd"}) mode_ = kBias;
    else if (fused == std::vector<std::string>{"BiasAdd", "Relu"}) mode_ = kBiasRelu;
    else if (fused == std::vector<std::string>{"ReluGrad"}) mode_ = kReluGrad;
    else
      OP_REQUIRES(ctx, false, errors::InvalidArgument("Unsupported fused_ops for _FusedMatMul"));
    OP_REQUIRES(ctx, ctx->num_inputs() == 3,
                errors::InvalidArgument("_FusedMatMul expects exactly one extra argument"));
  }

  void Compute(OpKernelContext* ctx) override {
    const Tensor& a = ctx->input(0);
    const Tensor& b = ctx->input(1);
    const Tensor& arg = ctx->input(2);
    OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(a.shape()),
                errors::InvalidArgument("In[0] is not a matrix"));
    OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(b.shape()),
                errors::InvalidArgument("In[1] is not a matrix"));
    const int a_contract = transpose_a_ ? 0 : 1;
    const int b_contract = transpose_b_ ? 1 : 0;
    OP_REQUIRES(ctx, a.dim_size(a_contract) == b.dim_size(b_contract),
                errors::InvalidArgument("Matrix size-incompatible: In[0]: ",
                                        a.shape().DebugString(), ", In[1]: ",
                                        b.shape().DebugString()));
    const int64 m = a.dim_size(1 - a_contract), k = a.dim_size(a_contract);
    const int64 n = b.dim_size(1 - b_contract);
    if (mode_ == kReluGrad) {
      OP_REQUIRES(ctx, arg.shape() == TensorShape({m, n}),
                  errors::InvalidArgument("Inputs must have the same size"));  // relu_op.h:48-60
    } else {
      OP_REQUIRES(ctx, TensorShapeUtils::IsVector(arg.shape()),
                  errors::InvalidArgument("Biases must be 1D: ", arg.shape().DebugString()));
      OP_REQUIRES(ctx, arg.dim_size(0) == n,
                  errors::InvalidArgument("Must provide as many biases as the last dimension of "
                                          "the input tensor: ", arg.shape().DebugString(),
                                          " vs. ", TensorShape({m, n}).DebugString()));
    }
    Tensor* out = nullptr;
    OP_REQUIRES_OK(ctx, ctx->allocate_output(0, TensorShape({m, n}), &out));
    if (out->NumElements() == 0) return;
    void* stream = GetCudaStream(ctx);
    if (k == 0) {  // product is zero: run the tail on a zero matrix, op by op
      OP_REQUIRES_OK(ctx, FromAbi(b200_memset_async(out->raw_data(), 0, out->TotalBytes(), stream),
                                  "_FusedMatMul zero fill"));
      if (mode_ != kReluGrad)
        OP_REQUIRES_OK(ctx, FromAbi(b200_bias_add(AbiType<T>::v, out->raw_data(), arg.raw_data(),
                                                  out->raw_data(), m, n, stream), "BiasAdd"));
      if (mode_ == kBiasRelu)
        OP_REQUIRES_OK(ctx, FromAbi(b200_relu(AbiType<T>::v, out->raw_data(), out->raw_data(),
                                              m * n, stream), "Relu"));
      return;
    }
    // scratch lets a bias / relu-tailed product with few output tiles split K (the tail then
    // rides on the ordered reduction pass); allocate_temp like the plain MatMul does
    const size_t ws_bytes =
        mode_ == kReluGrad ? 0 : b200_matmul_workspace_bytes(AbiType<T>::v, m, n, k);
    Tensor scratch;
    if (ws_bytes > 0)
      OP_REQUIRES_OK(ctx, ctx->allocate_temp(DT_UINT8, TensorShape({static_cast<int64>(ws_bytes)}),
                                             &scratch));
    OP_REQUIRES_OK(ctx, FromAbi(b200_fused_matmul_ws(
                                    AbiType<T>::v, a.raw_data(), b.raw_data(), out->raw_data(), m,
                                    n, k, transpose_a_, transpose_b_,
                                    mode_ == kReluGrad ? nullptr : arg.raw_data(),
                                    mode_ == kBiasRelu, mode_ == kReluGrad ? arg.raw_data() : nullptr,
                                    ws_bytes ? scratch.raw_data() : nullptr, ws_bytes, stream),
                                "Blas GEMM launch failed"));
  }

 private:
  enum Mode { kBias, kBiasRelu, kReluGrad };
  bool transpose_a_;
  bool transpose_b_;
  Mode mode_ = kBias;
};

// _MatMulPair: two independent products (a dense layer's dX and dW), each checked and allocated
// as its own MatMul / _FusedMatMul would be, computed by one b200_matmul_pair call.
template <typename T>
class MatMulPairOp : public OpKernel {
 public:
  explicit MatMulPairOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    for (int q = 0; q < 2; ++q) {
      Product& p = p_[q];
      const std::string sfx = q == 0 ? "0" : "1";
      OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_a" + sfx, &p.ta));
      OP_REQUIRES_OK(ctx, ctx->GetAttr("transpose_b" + sfx, &p.tb));
      std::vector<std::string> fused;
      OP_REQUIRES_OK(ctx, ctx->GetAttr("fused_ops" + sfx, &fused));
      int64 num_args = 0;
      OP_REQUIRES_OK(ctx, ctx->GetAttr("num_args" + sfx, &num_args));
      if (fused.empty()) p.mode = kNone;
      else if (fused == std::vector<std::string>{"BiasAdd"}) p.mode = kBias;
      else if (fused == std::vector<std::string>{"BiasAdd", "Relu"}) p.mode = kBiasRelu;
      else if (fused == std::vector<std::string>{"ReluGrad"}) p.mode = kReluGrad;
      else
        OP_REQUIRES(ctx, false, errors::InvalidArgument("Unsupported fused_ops for _MatMulPair"));
      OP_REQUIRES(ctx, num_args == (p.mode == kNone ? 0 : 1),
                  errors::InvalidArgument("_MatMulPair: one extra argument per fused product"));
    }
  }

  void Compute(OpKernelContext* ctx) override {
    int next = 0;
    bool degenerate = false;
    for (int q = 0; q < 2; ++q) {
      Product& p = p_[q];
      const Tensor& a = ctx->input(next);
      const Tensor& b = ctx->input(next + 1);
      p.arg = p.mode == kNone ? nullptr : &ctx->input(next + 2);
      next += p.mode == kNone ? 2 : 3;
      OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(a.shape()),
                  errors::InvalidArgument("In[0] is not a matrix"));
      OP_REQUIRES(ctx, TensorShapeUtils::IsMatrix(b.shape()),
                  errors::InvalidArgument("In[1] is not a matrix"));
      const int a_contract = p.ta ? 0 : 1;
      const int b_contract = p.tb ? 1 : 0;
      OP_REQUIRES(ctx, a.dim_size(a_contract) == b.dim_size(b_contract),
                  errors::InvalidArgument("Matrix size-incompatible: In[0]: ",
                                          a.shape().DebugString(), ", In[1]: ",
                                          b.shape().DebugString()));
      p.a = &a;
      p.b = &b;
      p.m = a.dim_size(1 - a_contract);
      p.k = a.dim_size(a_contract);
      p.n = b.dim_size(1 - b_contract);
      if (p.mode == kReluGrad) {
        OP_REQUIRES(ctx, p.arg->shape() == TensorShape({p.m, p.n}),
                    errors::InvalidArgument("Inputs must have the same size"));
      } else if (p.mode != kNone) {
        OP_REQUIRES(ctx, TensorShapeUtils::IsVector(p.arg->shape()),
                    errors::InvalidArgument("Biases must be 1D: ", p.arg->shape().DebugString()));
        OP_REQUIRES(ctx, p.arg->dim_size(0) == p.n,
                    errors::InvalidArgument("Must provide as many biases as the last dimension of "
                                            "the input tensor: ", p.arg->shape().DebugString(),
                                            " vs. ", TensorShape({p.m, p.n}).DebugString()));
      }
      OP_REQUIRES_OK(ctx, ctx->allocate_output(q, TensorShape({p.m, p.n}), &p.out));
      degenerate = degenerate || p.out->NumElements() == 0 || p.k == 0;
    }
    void* stream = GetCudaStream(ctx);
    if (degenerate) {  // an empty output or k == 0: each product on its own, as its op does it
      for (const Product& p : p_) RunOne(ctx, p, stream);
      return;
    }
    const Product &p0 = p_[0], &p1 = p_[1];
    const size_t ws_bytes =
        b200_matmul_pair_workspace_bytes(AbiType<T>::v, p0.m, p0.n, p0.k, p1.m, p1.n, p1.k);
    Tensor scratch;
    if (ws_bytes > 0)
      OP_REQUIRES_OK(ctx, ctx->allocate_temp(DT_UINT8, TensorShape({static_cast<int64>(ws_bytes)}),
                                             &scratch));
    OP_REQUIRES_OK(ctx, FromAbi(b200_matmul_pair(
                                    AbiType<T>::v, p0.a->raw_data(), p0.b->raw_data(),
                                    p0.out->raw_data(), p0.m, p0.n, p0.k, p0.ta, p0.tb, p0.bias(),
                                    p0.mode == kBiasRelu, p0.features(), p1.a->raw_data(),
                                    p1.b->raw_data(), p1.out->raw_data(), p1.m, p1.n, p1.k, p1.ta,
                                    p1.tb, p1.bias(), p1.mode == kBiasRelu, p1.features(),
                                    ws_bytes ? scratch.raw_data() : nullptr, ws_bytes, stream),
                                "Blas GEMM launch failed"));
  }

 private:
  enum Mode { kNone, kBias, kBiasRelu, kReluGrad };
  struct Product {
    bool ta = false, tb = false;
    Mode mode = kNone;
    const Tensor *a = nullptr, *b = nullptr, *arg = nullptr;
    Tensor* out = nullptr;
    int64 m = 0, n = 0, k = 0;
    const void* bias() const { return mode == kBias || mode == kBiasRelu ? arg->raw_data() : nullptr; }
    const void* features() const { return mode == kReluGrad ? arg->raw_data() : nullptr; }
  };

  static void RunOne(OpKernelContext* ctx, const Product& p, void* stream) {
    if (p.out->NumElements() == 0) return;
    void* c = p.out->raw_data();
    if (p.k == 0) {  // product is zero: run the tail on a zero matrix, op by op
      OP_REQUIRES_OK(ctx, FromAbi(b200_memset_async(c, 0, p.out->TotalBytes(), stream),
                                  "_MatMulPair zero fill"));
      if (p.bias())
        OP_REQUIRES_OK(ctx, FromAbi(b200_bias_add(AbiType<T>::v, c, p.bias(), c, p.m, p.n, stream),
                                    "BiasAdd"));
      if (p.mode == kBiasRelu)
        OP_REQUIRES_OK(ctx, FromAbi(b200_relu(AbiType<T>::v, c, c, p.m * p.n, stream), "Relu"));
      return;
    }
    const size_t ws_bytes =
        p.mode == kReluGrad ? 0 : b200_matmul_workspace_bytes(AbiType<T>::v, p.m, p.n, p.k);
    Tensor scratch;
    if (ws_bytes > 0)
      OP_REQUIRES_OK(ctx, ctx->allocate_temp(DT_UINT8, TensorShape({static_cast<int64>(ws_bytes)}),
                                             &scratch));
    OP_REQUIRES_OK(ctx, FromAbi(b200_fused_matmul_ws(
                                    AbiType<T>::v, p.a->raw_data(), p.b->raw_data(), c, p.m, p.n,
                                    p.k, p.ta, p.tb, p.bias(), p.mode == kBiasRelu, p.features(),
                                    ws_bytes ? scratch.raw_data() : nullptr, ws_bytes, stream),
                                "Blas GEMM launch failed"));
  }

  Product p_[2];
};

#define REGISTER_GPU(T)                                                                        \
  REGISTER_KERNEL_BUILDER(Name("MatMul").Device(DEVICE_GPU).TypeConstraint<T>("T"),            \
                          MatMulOp<T>);                                                        \
  REGISTER_KERNEL_BUILDER(Name("BatchMatMul").Device(DEVICE_GPU).TypeConstraint<T>("T"),       \
                          BatchMatMulOp<T>);                                                   \
  REGISTER_KERNEL_BUILDER(Name("_FusedMatMul").Device(DEVICE_GPU).TypeConstraint<T>("T"),      \
                          FusedMatMulOp<T>);                                               \
  REGISTER_KERNEL_BUILDER(Name("_MatMulPair").Device(DEVICE_GPU).TypeConstraint<T>("T"),       \
                          MatMulPairOp<T>);
REGISTER_B200_FLOAT_TYPES(REGISTER_GPU)
#undef REGISTER_GPU

}  // namespace tensorflow
