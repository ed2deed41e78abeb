"""CPU-only checks of the host side: ABI surface, registries, NodeDef validation, gradient
graph construction, and that nothing silently falls back when there is no GPU."""
import os
import re
import subprocess

import numpy as np
import pytest

from simple_tensorflow_b200 import _lib, client, ops as tf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "b200_ops.h")).read()
    return sorted(set(re.findall(r"B200_API\s+[\w\s\*]+?\b(b200_\w+)\s*\(", text)))


def test_abi_header_matches_library_and_binding():
    declared = _header_symbols()
    assert len(declared) >= 50
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), "libb200tf.so does not export " + name
    assert sorted(_lib.SIGNATURES) == declared, set(_lib.SIGNATURES) ^ set(declared)
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH]).decode()
    exported = sorted(set(re.findall(r"\bT (b200_\w+)", out)))
    assert exported == declared, set(exported) ^ set(declared)


def test_c_api_header_matches_framework_library():
    # every TF_* / B200TF_* function the C API header declares is exported by
    # libb200tf_framework.so, nothing else is, and the Python binding only names real functions
    text = open(os.path.join(ROOT, "simple_tensorflow_b200", "csrc", "tensorflow", "c",
                             "c_api.h")).read()
    declared = sorted(set(re.findall(r"TF_CAPI_EXPORT\s+extern\s+[\w\s\*]+?\b((?:B200)?TF_\w+)\s*\(", text)))
    assert len(declared) >= 50
    out = subprocess.check_output(["nm", "-D", "--defined-only", client.FRAMEWORK_PATH]).decode()
    exported = sorted(set(re.findall(r"\bT ((?:B200)?TF_\w+)", out)))
    assert exported == declared, set(exported) ^ set(declared)
    assert set(client._SIGS) <= set(declared), set(client._SIGS) - set(declared)


def test_no_vendor_gemm_or_dnn_libraries_linked():
    for path in (_lib.LIB_PATH, client.FRAMEWORK_PATH):
        out = subprocess.check_output(["ldd", path]).decode().lower()
        for banned in ("cublas", "cudnn", "cutlass", "cufft", "libtorch", "libc10"):
            assert banned not in out, (path, banned)
    syms = subprocess.check_output(["nm", "-D", "--undefined-only", _lib.LIB_PATH]).decode()
    assert "cublas" not in syms.lower() and "cudnn" not in syms.lower()


def test_product_code_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "simple_tensorflow_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cc", ".cu", ".h", ".cuh")):
                text = open(os.path.join(base, f), errors="replace").read()
                assert "oracle_bind" not in text and "liboracle" not in text, os.path.join(base, f)
    # developer tools are not test infrastructure either: only tests/, smoke() and bench.py's CPU
    # legs may use the oracle
    for f in os.listdir(os.path.join(ROOT, "tools")):
        if f.endswith(".py"):
            text = open(os.path.join(ROOT, "tools", f)).read()
            assert "oracle_bind" not in text and "liboracle" not in text, f


def test_library_loads_without_gpu_and_fails_loudly():
    lib = _lib.load()
    assert lib.b200_version().startswith(b"b200tf")
    if lib.b200_device_count() > 0:
        pytest.skip("GPU present")
    rc = lib.b200_matmul(_lib.DT_FLOAT, 16, 16, 16, 4, 4, 4, 0, 0, None, 0, None)
    assert rc == 13 and b"no CUDA device" in lib.b200_last_error()  # INTERNAL, no CPU fallback
    assert lib.b200_relu(_lib.DT_FLOAT, 16, 16, 4, None) == 13
    with pytest.raises(client.OpError) as e:
        client.Session(client.Graph())
    assert e.value.error_code == 5 and "no CPU fallback" in e.value.message


def test_workspace_queries_are_host_only():
    lib = _lib.load()
    # dW of the MLP (1024x1024 out, K=4096) wants split-K scratch; the forward GEMM does not
    assert lib.b200_matmul_workspace_bytes(_lib.DT_FLOAT, 1024, 1024, 4096) > 0
    assert lib.b200_matmul_workspace_bytes(_lib.DT_FLOAT, 4096, 1024, 1024) == 0
    assert lib.b200_bias_add_grad_workspace_bytes(_lib.DT_FLOAT, 4096, 1024) >= 1024 * 4
    g = _lib.ConvGeometry(512, 14, 14, 32, 5, 5, 64, 14, 14, 1, 1, 2, 2)
    import ctypes
    ws = lib.b200_conv2d_workspace_bytes(_lib.DT_FLOAT, ctypes.byref(g), 2)
    patches = 512 * 196 * 800 * 4
    if lib.b200_device_count() > 0:
        # with a device the halo-tile filter gradient runs: no patch matrix, one fp32 partial
        # filter gradient per slice (conv_halo_wgrad.cu)
        assert 0 < ws < patches and ws % (5 * 5 * 32 * 64 * 4) == 0, ws
    else:
        # without one the filter-gradient path materialises the patch matrix
        assert ws >= patches, ws


def test_registries_hold_the_hot_path():
    ops_ = set(client.registered_ops())
    for name in ["MatMul", "BatchMatMul", "Conv2D", "Conv2DBackpropInput", "Conv2DBackpropFilter",
                 "BiasAdd", "BiasAddGrad", "Relu", "ReluGrad", "Softmax", "LogSoftmax", "MaxPool",
                 "MaxPoolGrad", "Cast", "ArgMax", "SoftmaxCrossEntropyWithLogits",
                 "ApplyGradientDescent", "AddN", "VariableV2", "Assign"]:
        assert name in ops_
    kernels = client.registered_kernels()
    assert kernels.count("MatMul:GPU:") == 3  # float + bfloat16 + half (fp32 adaptor) registrations
    assert all(k.split(":")[1] == "GPU" for k in kernels), "a CPU kernel would be a fallback"


def test_node_def_validation_errors():
    g = client.Graph()
    x = g.create_op("Placeholder", [], {"dtype": ("type", tf.float32)}, "x").outputs[0]
    with pytest.raises(client.OpError) as e:  # op not registered
        g.create_op("NotAnOp", [], {}, "n")
    assert e.value.error_code == 5
    with pytest.raises(client.OpError) as e:  # missing required attr
        g.create_op("Conv2D", [x, x], {"T": ("type", tf.float32), "padding": "SAME"}, "c")
    assert e.value.error_code == 3 and "strides" in e.value.message
    with pytest.raises(client.OpError) as e:  # attr value outside the allowed list
        g.create_op("MatMul", [x, x], {"T": ("type", tf.int64)}, "m")
    assert e.value.error_code == 3 and "allowed values" in e.value.message
    with pytest.raises(client.OpError) as e:  # wrong attr kind
        g.create_op("MatMul", [x, x], {"T": ("type", tf.float32), "transpose_a": 3}, "m2")
    assert e.value.error_code == 3
    with pytest.raises(client.OpError) as e:  # ksize needs >= 4 entries
        g.create_op("MaxPool", [x], {"ksize": ("ints", [1, 2]), "strides": ("ints", [1, 2, 2, 1]),
                                     "padding": "SAME"}, "p")
    assert "at least minimum" in e.value.message
    ok = g.create_op("MatMul", [x, x], {"T": ("type", tf.float32)}, "ok")  # defaults applied
    assert ok.outputs[0].dtype == tf.float32
    again = g.create_op("MatMul", [x, x], {"T": ("type", tf.float32)}, "ok")  # uniquified
    assert again.name == "ok_1"


def test_gradient_graph_matches_reference_rules():
    tf.reset_default_graph()
    x = tf.placeholder(tf.float32, [8, 16], "x")
    lab = tf.placeholder(tf.float32, [8, 4], "labels")
    W = tf.Variable(np.zeros((16, 4), np.float32), name="W")
    b = tf.Variable(np.zeros(4, np.float32), name="b")
    logits = tf.bias_add(tf.matmul(x, W), b)
    loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(logits, lab))
    dW, db, dx = tf.gradients(loss, [W, b, x])
    # math_grad.py:774-794: d/dW of x*W is MatMul(x, grad, transpose_a=True)
    assert dW.op.type == "MatMul" and dW.op.attrs["transpose_a"] and not dW.op.attrs["transpose_b"]
    assert dW.op.inputs[0].name == "x:0"
    # nn_grad.py:180-204
    assert db.op.type == "BiasAddGrad"
    assert dx.op.type == "MatMul" and dx.op.attrs["transpose_b"]
    assert tf.gradients(loss, [lab]) == [None]
    train = tf.GradientDescentOptimizer(0.1).minimize(loss)
    assert train.type == "NoOp" and len(train.control_inputs) == 2
    assert {c.type for c in train.control_inputs} == {"ApplyGradientDescent"}


def _mlp(widths):
    tf.reset_default_graph()
    x = tf.placeholder(tf.float32, [8, widths[0]], "x")
    lab = tf.placeholder(tf.float32, [8, widths[-1]], "labels")
    Ws = [tf.Variable(np.zeros((a, b), np.float32), name="W%d" % i)
          for i, (a, b) in enumerate(zip(widths[:-1], widths[1:]))]
    Bs = [tf.Variable(np.zeros(b, np.float32), name="b%d" % i) for i, b in enumerate(widths[1:])]
    h = x
    for i, (w, b) in enumerate(zip(Ws, Bs)):
        h = tf.bias_add(tf.matmul(h, w), b)
        if i < len(Ws) - 1:
            h = tf.relu(h)
    return tf.reduce_mean(tf.softmax_cross_entropy_with_logits(h, lab)), Ws, Bs


def test_replica_gradient_exchange_graph():
    # num_replicas > 1: gradients go through B200AllReduceN (scale 1/p) before the updates;
    # default = one collective over everything, bucket_bytes = size-capped buckets filled in the
    # order backprop emits the gradients (last layer first)
    loss, Ws, Bs = _mlp([64, 512, 512, 16])
    train = tf.GradientDescentOptimizer(0.1).minimize(loss, Ws + Bs, num_replicas=4)
    g = tf.get_default_graph()
    ars = [op for op in g.operations if op.type == "B200AllReduceN"]
    assert len(ars) == 1 and len(ars[0].inputs) == 6
    assert abs(ars[0].attrs["scale"] - 0.25) < 1e-9
    applies = [op for op in g.operations if op.type == "ApplyGradientDescent"]
    assert len(applies) == 6 and all(a.inputs[2].op is ars[0] for a in applies)
    # every variable is updated with ITS reduced gradient
    for a in applies:
        var = a.inputs[0].op.name
        src = ars[0].inputs[a.inputs[2].index].op
        assert (src.type == "BiasAddGrad") == var.startswith("b")
    assert train.type == "NoOp"

    loss, Ws, Bs = _mlp([64, 512, 512, 16])
    tf.GradientDescentOptimizer(0.1).minimize(loss, Ws + Bs, num_replicas=2,
                                              bucket_bytes=256 * 1024)
    ars = [op for op in tf.get_default_graph().operations if op.type == "B200AllReduceN"]
    # layer 2 (512x16 = 32 KB + bias) is too small to close a bucket: it rides with layer 1
    # (512x512 = 1 MB), layer 0 (64x512 = 128 KB + bias) is the tail
    sizes = [[int(np.prod(g.shapes[i.name])) for i in op.inputs] for op in ars
             for g in [tf.get_default_graph()]]
    assert sizes == [[16, 512 * 16, 512, 512 * 512], [512, 64 * 512]], sizes
    order = [op.inputs[0].op.name for op in ars]
    assert order[0].startswith("BiasAddGrad")        # the last layer's gradients come first

    # one replica: no collective at all
    loss, Ws, Bs = _mlp([8, 8])
    tf.GradientDescentOptimizer(0.1).minimize(loss)
    assert not [op for op in tf.get_default_graph().operations if op.type.startswith("B200AllReduce")]


def test_reference_style_names_build_the_same_graph():
    # simple_tensorflow_b200.compat: tf.nn.* / tf.train.* / named-argument xent as in nn_ops.py
    import simple_tensorflow_b200.compat as tfc
    tfc.reset_default_graph()
    x = tfc.placeholder(tfc.float32, [8, 16])
    y = tfc.placeholder(tfc.float32, [8, 4])
    W = tfc.Variable(np.zeros((16, 4), np.float32))
    b = tfc.Variable(np.zeros(4, np.float32))
    logits = tfc.nn.bias_add(tfc.matmul(tfc.nn.relu(x), W), b)
    loss = tfc.reduce_mean(tfc.nn.softmax_cross_entropy_with_logits(labels=y, logits=logits))
    train = tfc.train.GradientDescentOptimizer(0.1).minimize(loss)
    types = [op.type for op in tfc.get_default_graph().operations]
    for t in ("Relu", "MatMul", "BiasAdd", "SoftmaxCrossEntropyWithLogits", "Mean", "BiasAddGrad",
              "ApplyGradientDescent"):
        assert t in types, t
    assert train.type == "NoOp"
    with pytest.raises(ValueError):   # positional arguments are refused, like the reference
        tfc.nn.softmax_cross_entropy_with_logits(logits, y)
    # the labels really are the second kernel input
    xent = [op for op in tfc.get_default_graph().operations
            if op.type == "SoftmaxCrossEntropyWithLogits"][0]
    assert xent.inputs[0].name == logits.name and xent.inputs[1].name == y.name


def test_host_tensor_roundtrip():
    a = np.arange(24, dtype=np.float32).reshape(2, 3, 4)
    t = client.HostTensor.from_numpy(a)
    assert t.shape == (2, 3, 4) and t.dtype == tf.float32
    np.testing.assert_array_equal(t.numpy(), a)
    i = client.HostTensor.from_numpy(np.array([1, 2, 3], np.int64))
    assert i.dtype == tf.int64 and i.numpy().tolist() == [1, 2, 3]
