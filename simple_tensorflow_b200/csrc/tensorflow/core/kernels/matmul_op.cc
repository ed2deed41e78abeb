// MatMul / BatchMatMul for DEVICE_GPU on B200.
// Same validation, shape and zero-size rules as the reference's MatMulOp::Compute
// (core/kernels/matmul_op.cc:215-256) and BatchMatMul::Compute
// (core/kernels/batch_matmul_op_impl.h:367-434); the launch goes to b200_fused_matmul_ws,
// b200_matmul_pair or b200_batch_matmul instead of Stream::ThenBlasGemm (matmul_op.cc:179-195).
#include "tensorflow/core/kernels/gpu_kernel_util.h"

namespace tensorflow {

// One dense product as MatMul, _FusedMatMul and each half of _MatMulPair compute it: attributes
// (`sfx` is a _MatMulPair product's attribute suffix), the reference's shape checks, output
// allocation, and the launch of a product that runs on its own.
template <typename T>
struct DenseProduct {
  enum Mode { kNone, kBias, kBiasRelu, kReluGrad };
  bool ta = false, tb = false;
  Mode mode = kNone;
  const Tensor *a = nullptr, *b = nullptr, *arg = nullptr;
  Tensor* out = nullptr;
  int64 m = 0, n = 0, k = 0;

  // `op` names the op in errors; MatMul has no fused_ops attribute.
  Status Init(OpKernelConstruction* ctx, const char* op, bool has_fused_ops,
              const std::string& sfx = "") {
    TF_RETURN_IF_ERROR(ctx->GetAttr("transpose_a" + sfx, &ta));
    TF_RETURN_IF_ERROR(ctx->GetAttr("transpose_b" + sfx, &tb));
    if (!has_fused_ops) return Status::OK();
    std::vector<std::string> fused;
    TF_RETURN_IF_ERROR(ctx->GetAttr("fused_ops" + sfx, &fused));
    if (fused.empty()) mode = kNone;
    else if (fused == std::vector<std::string>{"BiasAdd"}) mode = kBias;
    else if (fused == std::vector<std::string>{"BiasAdd", "Relu"}) mode = kBiasRelu;
    else if (fused == std::vector<std::string>{"ReluGrad"}) mode = kReluGrad;
    else return errors::InvalidArgument("Unsupported fused_ops for ", op);
    return Status::OK();
  }

  int num_inputs() const { return mode == kNone ? 2 : 3; }
  const void* bias() const { return mode == kBias || mode == kBiasRelu ? arg->raw_data() : nullptr; }
  const void* features() const { return mode == kReluGrad ? arg->raw_data() : nullptr; }
  // An empty output or k == 0: no GEMM, see RunAlone.
  bool degenerate() const { return out->NumElements() == 0 || k == 0; }

  // Checks inputs first, first + 1 (A, B) and, with a tail, first + 2; allocates output `index`.
  Status Prepare(OpKernelContext* ctx, int first, int index) {
    a = &ctx->input(first);
    b = &ctx->input(first + 1);
    arg = mode == kNone ? nullptr : &ctx->input(first + 2);
    if (!TensorShapeUtils::IsMatrix(a->shape()))
      return errors::InvalidArgument("In[0] is not a matrix");
    if (!TensorShapeUtils::IsMatrix(b->shape()))
      return errors::InvalidArgument("In[1] is not a matrix");
    const int a_contract = ta ? 0 : 1;
    const int b_contract = tb ? 1 : 0;
    if (a->dim_size(a_contract) != b->dim_size(b_contract))
      return errors::InvalidArgument("Matrix size-incompatible: In[0]: ", a->shape().DebugString(),
                                     ", In[1]: ", b->shape().DebugString());
    m = a->dim_size(1 - a_contract);
    k = a->dim_size(a_contract);
    n = b->dim_size(1 - b_contract);
    if (mode == kReluGrad) {
      if (arg->shape() != TensorShape({m, n}))
        return errors::InvalidArgument("Inputs must have the same size");  // relu_op.h:48-60
    } else if (mode != kNone) {
      if (!TensorShapeUtils::IsVector(arg->shape()))
        return errors::InvalidArgument("Biases must be 1D: ", arg->shape().DebugString());
      if (arg->dim_size(0) != n)
        return errors::InvalidArgument("Must provide as many biases as the last dimension of "
                                       "the input tensor: ", arg->shape().DebugString(), " vs. ",
                                       TensorShape({m, n}).DebugString());
    }
    return ctx->allocate_output(index, TensorShape({m, n}), &out);
  }

  Status RunAlone(OpKernelContext* ctx, const char* op, void* stream) const {
    if (out->NumElements() == 0) return Status::OK();  // [0,x] or [x,0] operands: nothing to do
    void* c = out->raw_data();
    if (k == 0) {  // product is zero (matmul_op.cc:246-253): run the tail on a zero matrix, op by op
      TF_RETURN_IF_ERROR(FromAbi(b200_memset_async(c, 0, out->TotalBytes(), stream),
                                 strings::StrCat(op, " zero fill").c_str()));
      if (bias())
        TF_RETURN_IF_ERROR(
            FromAbi(b200_bias_add(AbiType<T>::v, c, bias(), c, m, n, stream), "BiasAdd"));
      if (mode == kBiasRelu)
        TF_RETURN_IF_ERROR(FromAbi(b200_relu(AbiType<T>::v, c, c, m * n, stream), "Relu"));
      return Status::OK();
    }
    // split-K partial sums; the scratch stays alive until the stream passes it.  A bias / relu
    // tail then rides on the ordered reduction pass; a ReluGrad tail needs the unsplit sum.
    const size_t ws_bytes =
        mode == kReluGrad ? 0 : b200_matmul_workspace_bytes(AbiType<T>::v, m, n, k);
    Tensor scratch;
    if (ws_bytes > 0)
      TF_RETURN_IF_ERROR(
          ctx->allocate_temp(DT_UINT8, TensorShape({static_cast<int64>(ws_bytes)}), &scratch));
    return FromAbi(b200_fused_matmul_ws(AbiType<T>::v, a->raw_data(), b->raw_data(), c, m, n, k,
                                        ta, tb, bias(), mode == kBiasRelu, features(),
                                        ws_bytes ? scratch.raw_data() : nullptr, ws_bytes, stream),
                   "Blas GEMM launch failed");
  }
};

template <typename T>
class MatMulOp : public OpKernel {
 public:
  explicit MatMulOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    OP_REQUIRES_OK(ctx, p_.Init(ctx, "MatMul", false));
  }

  void Compute(OpKernelContext* ctx) override {
    DenseProduct<T> p = p_;  // this call's tensors and shapes; p_ keeps the attributes
    OP_REQUIRES_OK(ctx, p.Prepare(ctx, 0, 0));
    OP_REQUIRES_OK(ctx, p.RunAlone(ctx, "MatMul", GetCudaStream(ctx)));
  }

 private:
  DenseProduct<T> p_;
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
    OP_REQUIRES_OK(ctx, p_.Init(ctx, "_FusedMatMul", true));
    OP_REQUIRES(ctx, p_.mode != DenseProduct<T>::kNone,
                errors::InvalidArgument("Unsupported fused_ops for _FusedMatMul"));
    OP_REQUIRES(ctx, ctx->num_inputs() == 3,
                errors::InvalidArgument("_FusedMatMul expects exactly one extra argument"));
  }

  void Compute(OpKernelContext* ctx) override {
    DenseProduct<T> p = p_;
    OP_REQUIRES_OK(ctx, p.Prepare(ctx, 0, 0));
    OP_REQUIRES_OK(ctx, p.RunAlone(ctx, "_FusedMatMul", GetCudaStream(ctx)));
  }

 private:
  DenseProduct<T> p_;
};

// _MatMulPair: two independent products (a dense layer's dX and dW), each checked and allocated
// as its own MatMul / _FusedMatMul would be, computed by one b200_matmul_pair call.
template <typename T>
class MatMulPairOp : public OpKernel {
 public:
  explicit MatMulPairOp(OpKernelConstruction* ctx) : OpKernel(ctx) {
    for (int q = 0; q < 2; ++q) {
      const std::string sfx = q == 0 ? "0" : "1";
      OP_REQUIRES_OK(ctx, p_[q].Init(ctx, "_MatMulPair", true, sfx));
      int64 num_args = 0;
      OP_REQUIRES_OK(ctx, ctx->GetAttr("num_args" + sfx, &num_args));
      OP_REQUIRES(ctx, num_args == p_[q].num_inputs() - 2,
                  errors::InvalidArgument("_MatMulPair: one extra argument per fused product"));
    }
  }

  void Compute(OpKernelContext* ctx) override {
    DenseProduct<T> p0 = p_[0], p1 = p_[1];
    OP_REQUIRES_OK(ctx, p0.Prepare(ctx, 0, 0));
    OP_REQUIRES_OK(ctx, p1.Prepare(ctx, p0.num_inputs(), 1));
    void* stream = GetCudaStream(ctx);
    if (p0.degenerate() || p1.degenerate()) {  // each product on its own, as its op runs it
      OP_REQUIRES_OK(ctx, p0.RunAlone(ctx, "_MatMulPair", stream));
      OP_REQUIRES_OK(ctx, p1.RunAlone(ctx, "_MatMulPair", stream));
      return;
    }
    const size_t ws_bytes =
        b200_matmul_pair_workspace_bytes(AbiType<T>::v, p0.m, p0.n, p0.k, p1.m, p1.n, p1.k);
    Tensor scratch;
    if (ws_bytes > 0)
      OP_REQUIRES_OK(ctx, ctx->allocate_temp(DT_UINT8, TensorShape({static_cast<int64>(ws_bytes)}),
                                             &scratch));
    OP_REQUIRES_OK(ctx, FromAbi(b200_matmul_pair(
                                    AbiType<T>::v, p0.a->raw_data(), p0.b->raw_data(),
                                    p0.out->raw_data(), p0.m, p0.n, p0.k, p0.ta, p0.tb, p0.bias(),
                                    p0.mode == DenseProduct<T>::kBiasRelu, p0.features(),
                                    p1.a->raw_data(), p1.b->raw_data(), p1.out->raw_data(), p1.m,
                                    p1.n, p1.k, p1.ta, p1.tb, p1.bias(),
                                    p1.mode == DenseProduct<T>::kBiasRelu, p1.features(),
                                    ws_bytes ? scratch.raw_data() : nullptr, ws_bytes, stream),
                                "Blas GEMM launch failed"));
  }

 private:
  DenseProduct<T> p_[2];
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
