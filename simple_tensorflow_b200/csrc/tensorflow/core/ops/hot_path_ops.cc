// REGISTER_OP definitions of the hot path and its graph glue.  Signatures are the reference's
// (core/ops/math_ops.cc:52-58,1033-1040; nn_ops.cc:432-463,503-606,1264-1298,1550-1564,1673-1719;
// training_ops.cc ApplyGradientDescent; state_ops.cc VariableV2/Assign; array_ops.cc
// Const/Identity/Reshape/Placeholder/Shape; no_op.cc) with ONE additive change: `bfloat16` is
// appended to the allowed `T` lists (the reference allows DT_BFLOAT16 "only for cast ops",
// framework/types.proto:30) so BASELINE configs 4-5 (bf16 storage, fp32 accumulate) can be
// expressed.  Shape functions are not registered: shapes are checked by the kernels at run time.
#include "tensorflow/core/framework/op.h"

namespace tensorflow {

#define PADDING_ATTR "padding: {'SAME', 'VALID'}"
#define DATA_FORMAT_ATTR "data_format: {'NHWC', 'NCHW'} = 'NHWC'"

REGISTER_OP("MatMul")
    .Input("a: T").Input("b: T").Output("product: T")
    .Attr("transpose_a: bool = false").Attr("transpose_b: bool = false")
    .Attr("T: {half, float, double, int32, complex64, complex128, bfloat16}");

// Produced only by the executor's rewrite of MatMul+BiasAdd(+Relu) / MatMul+ReluGrad chains (the
// shape later TensorFlow's grappler remapper gives the same fusion): args[0] is the bias or the
// ReluGrad features; fused_ops is one of {BiasAdd}, {BiasAdd, Relu}, {ReluGrad}.
REGISTER_OP("_FusedMatMul")
    .Input("a: T").Input("b: T").Input("args: num_args * T").Output("product: T")
    .Attr("T: {float, bfloat16}").Attr("num_args: int >= 0")
    .Attr("transpose_a: bool = false").Attr("transpose_b: bool = false")
    .Attr("fused_ops: list(string)");

// Executor-internal (DirectSession::FuseSiblingMatMuls): two independent MatMul / _FusedMatMul
// products, each with the inputs and attrs of a _FusedMatMul (a plain MatMul has num_args = 0 and
// no fused_ops), computed by one persistent GEMM launch.
REGISTER_OP("_MatMulPair")
    .Input("a0: T").Input("b0: T").Input("args0: num_args0 * T")
    .Input("a1: T").Input("b1: T").Input("args1: num_args1 * T")
    .Output("product0: T").Output("product1: T")
    .Attr("T: {float, bfloat16}").Attr("num_args0: int >= 0").Attr("num_args1: int >= 0")
    .Attr("transpose_a0: bool = false").Attr("transpose_b0: bool = false")
    .Attr("transpose_a1: bool = false").Attr("transpose_b1: bool = false")
    .Attr("fused_ops0: list(string)").Attr("fused_ops1: list(string)");

REGISTER_OP("BatchMatMul")
    .Input("x: T").Input("y: T").Output("output: T")
    .Attr("T: {half, float, double, int32, complex64, complex128, bfloat16}")
    .Attr("adj_x: bool = false").Attr("adj_y: bool = false");

REGISTER_OP("Conv2D")
    .Input("input: T").Input("filter: T").Output("output: T")
    .Attr("T: {half, float, double, bfloat16}").Attr("strides: list(int)")
    .Attr("use_cudnn_on_gpu: bool = true").Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR);

// Produced only by the executor's rewrite of Conv2D -> BiasAdd (-> Relu) chains (NHWC):
// args[0] is the bias; fused_ops is {BiasAdd} or {BiasAdd, Relu}.
REGISTER_OP("_FusedConv2D")
    .Input("input: T").Input("filter: T").Input("args: num_args * T").Output("output: T")
    .Attr("T: {float, bfloat16}").Attr("num_args: int >= 0").Attr("strides: list(int)")
    .Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR).Attr("fused_ops: list(string)");

REGISTER_OP("Conv2DBackpropInput")
    .Input("input_sizes: int32").Input("filter: T").Input("out_backprop: T").Output("output: T")
    .Attr("T: {half, float, double, bfloat16}").Attr("strides: list(int)")
    .Attr("use_cudnn_on_gpu: bool = true").Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR);

REGISTER_OP("Conv2DBackpropFilter")
    .Input("input: T").Input("filter_sizes: int32").Input("out_backprop: T").Output("output: T")
    .Attr("T: {half, float, double, bfloat16}").Attr("strides: list(int)")
    .Attr("use_cudnn_on_gpu: bool = true").Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR);

REGISTER_OP("BiasAdd")
    .Attr("T: numbertype").Input("value: T").Input("bias: T").Attr(DATA_FORMAT_ATTR)
    .Output("output: T");

REGISTER_OP("BiasAddGrad")
    .Attr("T: numbertype").Input("out_backprop: T").Attr(DATA_FORMAT_ATTR).Output("output: T");

REGISTER_OP("Relu").Input("features: T").Output("activations: T").Attr("T: realnumbertype");

REGISTER_OP("ReluGrad")
    .Input("gradients: T").Input("features: T").Output("backprops: T").Attr("T: realnumbertype");

REGISTER_OP("Softmax").Input("logits: T").Output("softmax: T")
    .Attr("T: {half, float, double, bfloat16}");

REGISTER_OP("LogSoftmax").Input("logits: T").Output("logsoftmax: T")
    .Attr("T: {half, float, double, bfloat16}");

REGISTER_OP("SoftmaxCrossEntropyWithLogits")
    .Input("features: T").Input("labels: T").Output("loss: T").Output("backprop: T")
    .Attr("T: {half, float, double, bfloat16}");

// Executor-internal (direct_session.cc FuseXentScale): backprop is multiplied by a scalar.
REGISTER_OP("_ScaledSoftmaxCrossEntropyWithLogits")
    .Input("features: T").Input("labels: T").Input("backprop_scale: T")
    .Output("loss: T").Output("backprop: T").Attr("T: {float}");

REGISTER_OP("MaxPool")
    .Attr("T: {float, half, bfloat16} = DT_FLOAT")
    .Attr("ksize: list(int) >= 4").Attr("strides: list(int) >= 4")
    .Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR)
    .Input("input: T").Output("output: T");

REGISTER_OP("MaxPoolGrad")
    .Attr("ksize: list(int) >= 4").Attr("strides: list(int) >= 4")
    .Attr(PADDING_ATTR).Attr(DATA_FORMAT_ATTR)
    .Input("orig_input: T").Input("orig_output: T").Input("grad: T").Output("output: T")
    .Attr("T: {float, half, bfloat16} = DT_FLOAT");

REGISTER_OP("Cast").Input("x: SrcT").Output("y: DstT").Attr("SrcT: type").Attr("DstT: type");

REGISTER_OP("ArgMax")
    .Input("input: T").Input("dimension: Tidx").Output("output: int64")
    .Attr("T: numbertype").Attr("Tidx: {int32, int64} = DT_INT32");

// ---- graph glue (SURVEY 8f rank 1)
REGISTER_OP("AddN").Input("inputs: N * T").Output("sum: T").Attr("N: int >= 1")
    .Attr("T: numbertype").SetIsCommutative();

REGISTER_OP("Mul").Input("x: T").Input("y: T").Output("z: T").Attr("T: numbertype")
    .SetIsCommutative();
// math_ops.cc BINARY_MORE: "Add" (what a loaded model's bias / offset usually is)
REGISTER_OP("Add").Input("x: T").Input("y: T").Output("z: T").Attr("T: numbertype");

REGISTER_OP("Mean")
    .Input("input: T").Input("reduction_indices: Tidx").Output("output: T")
    .Attr("keep_dims: bool = false").Attr("T: numbertype")
    .Attr("Tidx: {int32, int64} = DT_INT32");

// Executor-internal (DirectSession::FuseReluGradBiasGrad): ReluGrad followed by an NHWC BiasAddGrad
// of its result, one pass over the tensor.
REGISTER_OP("_ReluGradBiasAddGrad")
    .Input("gradients: T").Input("features: T").Output("backprops: T").Output("bias_grad: T")
    .Attr("T: {float, bfloat16}");

// Executor-internal (DirectSession::FusePoolGradReluGradBiasGrad): MaxPoolGrad whose only reader
// is a `_ReluGradBiasAddGrad` that masks with the pool's own input (the Relu output).
REGISTER_OP("_MaxPoolGradReluGradBiasAddGrad")
    .Input("orig_input: T").Input("orig_output: T").Input("grad: T")
    .Output("backprops: T").Output("bias_grad: T")
    .Attr("ksize: list(int) >= 4").Attr("strides: list(int) >= 4")
    .Attr("padding: {'SAME', 'VALID'}").Attr(DATA_FORMAT_ATTR).Attr("T: {float, bfloat16}");

// math_ops.cc:1330-1343 ("Sum": same signature as "Mean")
REGISTER_OP("Sum")
    .Input("input: T").Input("reduction_indices: Tidx").Output("output: T")
    .Attr("keep_dims: bool = false").Attr("T: numbertype")
    .Attr("Tidx: {int32, int64} = DT_INT32");

REGISTER_OP("ApplyGradientDescent")
    .Input("var: Ref(T)").Input("alpha: T").Input("delta: T").Output("out: Ref(T)")
    .Attr("T: numbertype").Attr("use_locking: bool = false");

// Executor-internal (direct_session.cc FuseApplyGradientDescent): N updates, one launch.
REGISTER_OP("_MultiApplyGradientDescent")
    .Input("var: N * Ref(T)").Input("alpha: N * T").Input("delta: N * T")
    .Output("out: N * Ref(T)").Attr("N: int >= 1").Attr("T: {float, bfloat16}");

REGISTER_OP("VariableV2")
    .Output("ref: Ref(dtype)").Attr("shape: shape").Attr("dtype: type")
    .Attr("container: string = ''").Attr("shared_name: string = ''").SetIsStateful();

REGISTER_OP("Assign")
    .Input("ref: Ref(T)").Input("value: T").Output("output_ref: Ref(T)").Attr("T: type")
    .Attr("validate_shape: bool = true").Attr("use_locking: bool = true")
    .SetAllowsUninitializedInput();

REGISTER_OP("Const").Output("output: dtype").Attr("value: tensor").Attr("dtype: type");
REGISTER_OP("Identity").Input("input: T").Output("output: T").Attr("T: type");
REGISTER_OP("Reshape")
    .Input("tensor: T").Input("shape: Tshape").Output("output: T").Attr("T: type")
    .Attr("Tshape: {int32, int64} = DT_INT32");
REGISTER_OP("Placeholder").Output("output: dtype").Attr("dtype: type").Attr("shape: shape = {}");
REGISTER_OP("Shape").Input("input: T").Output("output: out_type").Attr("T: type")
    .Attr("out_type: {int32, int64} = DT_INT32");
REGISTER_OP("NoOp");

// ---- replica data-parallel (additive; the reference ships no collective op, SURVEY 8e):
// sums `data` element-wise across the replicas of the session's communicator, in place.
REGISTER_OP("B200AllReduce")
    .Input("data: Ref(T)").Output("out: Ref(T)").Attr("T: {float, bfloat16}")
    .Attr("scale: float = 1.0").SetIsStateful();

// Fused form for gradient sets: the N per-tensor all-reduces are grouped (ncclGroupStart/End)
// into ONE NCCL launch on the compute stream; `scale` = 1/replicas maps to ncclAvg.
REGISTER_OP("B200AllReduceN")
    .Input("inputs: N * T").Output("outputs: N * T").Attr("N: int >= 1")
    .Attr("T: {float, bfloat16}").Attr("scale: float = 1.0").SetIsStateful();

}  // namespace tensorflow
