"""GPU: graphs built through the Python front-end -> C API -> DirectSession-contract executor ->
OpKernel wrappers -> C ABI kernels, checked against the oracle chained on the CPU.
Covers BASELINE configs 1-3 at reduced batch (full sizes run in bench.py and in the
property tests of test_ops_gpu.py)."""
import numpy as np
import pytest

from simple_tensorflow_b200 import client, ops as tf

pytestmark = pytest.mark.gpu


def test_direct_session_minus_ax_known_answers():
    # core/common_runtime/direct_session_test.cc:54-137: a=[[3,2],[-1,0]], x=[[1],[1]]; y=a*x=5,-1;
    # y_neg... we run y = a*x and z = a*y (17, ... uses a*(a*x)): a*[5,-1] = [13,-5]
    tf.reset_default_graph()
    a = tf.constant(np.array([[3, 2], [-1, 0]], np.float32))
    x = tf.placeholder(tf.float32, [2, 1], "x")
    y = tf.matmul(a, x, name="y")
    z = tf.matmul(a, y, name="z")
    with client.Session(tf.get_default_graph()) as sess:
        yv, zv = sess.run([y, z], {x: np.array([[1], [1]], np.float32)})
        np.testing.assert_array_equal(yv.ravel(), [5.0, -1.0])
        np.testing.assert_array_equal(zv.ravel(), [13.0, -5.0])
        # feeding an intermediate tensor prunes its producer (direct_session_test.cc TestFeed)
        zv2 = sess.run(z, {y: np.array([[1], [2]], np.float32)})
        np.testing.assert_array_equal(zv2.ravel(), [7.0, -1.0])
        st = sess.last_run_stats()
        assert st["kernels_launched"] >= 1 and st["h2d_bytes"] == 8


def test_single_matmul_128_config1(oracle, rng):
    # BASELINE config 1: single MatMul 128x128 fp32 through the session
    a = rng.randn(128, 128).astype(np.float32)
    b = rng.randn(128, 128).astype(np.float32)
    tf.reset_default_graph()
    pa, pb = tf.placeholder(tf.float32, [128, 128]), tf.placeholder(tf.float32, [128, 128])
    c = tf.matmul(pa, pb)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(c, {pa: a, pb: b})
    ref = oracle.matmul(a, b)
    assert np.abs(got - ref).max() / np.abs(ref).max() < 3e-3


def _mlp_reference(oracle, x, labels, ws, bs, lr):
    acts, pres = [x], []
    for i, (w, b) in enumerate(zip(ws, bs)):
        pre = oracle.bias_add(oracle.matmul(acts[-1], w), b)
        pres.append(pre)
        acts.append(oracle.relu(pre) if i < len(ws) - 1 else pre)
    lvec, bp = oracle.softmax_xent(acts[-1], labels)
    g = bp / np.float32(x.shape[0])
    new_ws, new_bs = [None] * len(ws), [None] * len(ws)
    for i in reversed(range(len(ws))):
        new_bs[i] = oracle.apply_gradient_descent(bs[i], lr, oracle.bias_add_grad(g))
        new_ws[i] = oracle.apply_gradient_descent(ws[i], lr, oracle.matmul(acts[i], g, True, False))
        if i > 0:
            g = oracle.relu_grad(oracle.matmul(g, ws[i], False, True), acts[i])
    return float(lvec.mean()), new_ws, new_bs


def test_mlp_training_step_config2_reduced(oracle, rng):
    B, D = 512, 256
    x = rng.uniform(-1, 1, (B, D)).astype(np.float32)
    labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
    ws = [(rng.randn(D, D) / np.sqrt(D)).astype(np.float32) for _ in range(3)]
    bs = [np.full(D, 0.1, np.float32) for _ in range(3)]
    tf.reset_default_graph()
    xp, lp = tf.placeholder(tf.float32, [B, D]), tf.placeholder(tf.float32, [B, D])
    Ws = [tf.Variable(w, name="W%d" % i) for i, w in enumerate(ws)]
    Bs = [tf.Variable(b, name="b%d" % i) for i, b in enumerate(bs)]
    h = xp
    for i in range(3):
        h = tf.bias_add(tf.matmul(h, Ws[i]), Bs[i])
        if i < 2:
            h = tf.relu(h)
    loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(h, lp))
    train = tf.GradientDescentOptimizer(0.5).minimize(loss)
    with client.Session(tf.get_default_graph()) as sess:
        sess.run(tf.global_variables_initializer())
        got_loss, _ = sess.run([loss, train], {xp: x, lp: labels})
        got_ws = sess.run([v.ref for v in Ws])
        got_bs = sess.run([v.ref for v in Bs])
        loss2 = sess.run(loss, {xp: x, lp: labels})
    ref_loss, ref_ws, ref_bs = _mlp_reference(oracle, x, labels, ws, bs, 0.5)
    assert abs(got_loss - ref_loss) < 1e-2 * abs(ref_loss)
    for g, r in zip(got_ws + got_bs, ref_ws + ref_bs):
        assert np.abs(g - r).max() / np.abs(r).max() < 1e-2
    assert loss2 < got_loss  # one SGD step on the same batch reduces the loss


@pytest.mark.parametrize("exact_fp32", [False, True])
def test_lenet_training_step_config3_reduced(oracle, rng, exact_fp32):
    # exact_fp32=True runs the GEMMs on the IEEE-fp32 SIMT kernel: element-wise comparison.
    # Default TF32 mode: a pre-activation within TF32 rounding of zero may flip its ReLU mask
    # relative to the fp32 oracle, which moves single entries of a small-batch weight gradient by
    # O(1) of their size; the comparison there is in Frobenius norm (still <= 1e-2 relative).
    from simple_tensorflow_b200 import _lib
    assert _lib.load().b200_set_matmul_precision(1 if exact_fp32 else 0) == 0
    try:
        _lenet_step(oracle, rng, exact_fp32)
    finally:
        _lib.load().b200_set_matmul_precision(0)


def _lenet_step(oracle, rng, exact_fp32):
    B = 8
    x = rng.uniform(0, 1, (B, 28, 28, 1)).astype(np.float32)
    labels = np.eye(10, dtype=np.float32)[rng.randint(0, 10, B)]
    w1 = (rng.randn(5, 5, 1, 32) * 0.1).astype(np.float32)
    w2 = (rng.randn(5, 5, 32, 64) * 0.05).astype(np.float32)
    w3 = (rng.randn(7 * 7 * 64, 128) * 0.02).astype(np.float32)
    w4 = (rng.randn(128, 10) * 0.1).astype(np.float32)
    b1, b2 = np.full(32, 0.1, np.float32), np.full(64, 0.1, np.float32)
    b3, b4 = np.full(128, 0.1, np.float32), np.full(10, 0.1, np.float32)
    lr = 0.1
    tf.reset_default_graph()
    xp, lp = tf.placeholder(tf.float32, [B, 28, 28, 1]), tf.placeholder(tf.float32, [B, 10])
    V = {n: tf.Variable(v, name=n) for n, v in dict(w1=w1, w2=w2, w3=w3, w4=w4, b1=b1, b2=b2,
                                                    b3=b3, b4=b4).items()}
    c1 = tf.relu(tf.bias_add(tf.conv2d(xp, V["w1"], [1, 1, 1, 1], "SAME"), V["b1"]))
    p1 = tf.max_pool(c1, [1, 2, 2, 1], [1, 2, 2, 1], "SAME")
    c2 = tf.relu(tf.bias_add(tf.conv2d(p1, V["w2"], [1, 1, 1, 1], "SAME"), V["b2"]))
    p2 = tf.max_pool(c2, [1, 2, 2, 1], [1, 2, 2, 1], "SAME")
    flat = tf.reshape(p2, [B, 7 * 7 * 64])
    f1 = tf.relu(tf.bias_add(tf.matmul(flat, V["w3"]), V["b3"]))
    logits = tf.bias_add(tf.matmul(f1, V["w4"]), V["b4"])
    loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(logits, lp))
    train = tf.GradientDescentOptimizer(lr).minimize(loss)
    with client.Session(tf.get_default_graph()) as sess:
        sess.run(tf.global_variables_initializer())
        got_loss, _ = sess.run([loss, train], {xp: x, lp: labels})
        got = dict(zip(V, sess.run([V[n].ref for n in V])))
        pred = sess.run(tf.argmax(logits, 1), {xp: x, lp: labels})

    o = oracle
    a1 = o.relu(o.bias_add(o.conv2d(x, w1, (1, 1), "SAME"), b1))
    q1 = o.max_pool(a1, (2, 2), (2, 2), "SAME")
    a2 = o.relu(o.bias_add(o.conv2d(q1, w2, (1, 1), "SAME"), b2))
    q2 = o.max_pool(a2, (2, 2), (2, 2), "SAME")
    fl = q2.reshape(B, -1)
    g1 = o.relu(o.bias_add(o.matmul(fl, w3), b3))
    lg = o.bias_add(o.matmul(g1, w4), b4)
    lvec, bp = o.softmax_xent(lg, labels)
    d = bp / np.float32(B)
    ref = {"b4": o.apply_gradient_descent(b4, lr, o.bias_add_grad(d)),
           "w4": o.apply_gradient_descent(w4, lr, o.matmul(g1, d, True, False))}
    d = o.relu_grad(o.matmul(d, w4, False, True), g1)
    ref["b3"] = o.apply_gradient_descent(b3, lr, o.bias_add_grad(d))
    ref["w3"] = o.apply_gradient_descent(w3, lr, o.matmul(fl, d, True, False))
    d = o.matmul(d, w3, False, True).reshape(q2.shape)
    d = o.relu_grad(o.max_pool_grad(a2, d, (2, 2), (2, 2), "SAME"), a2)
    ref["b2"] = o.apply_gradient_descent(b2, lr, o.bias_add_grad(d))
    ref["w2"] = o.apply_gradient_descent(w2, lr, o.conv2d_backprop_filter(q1, w2.shape, d, (1, 1), "SAME"))
    d = o.conv2d_backprop_input(q1.shape, w2, d, (1, 1), "SAME")
    d = o.relu_grad(o.max_pool_grad(a1, d, (2, 2), (2, 2), "SAME"), a1)
    ref["b1"] = o.apply_gradient_descent(b1, lr, o.bias_add_grad(d))
    ref["w1"] = o.apply_gradient_descent(w1, lr, o.conv2d_backprop_filter(x, w1.shape, d, (1, 1), "SAME"))
    assert abs(got_loss - lvec.mean()) < 1e-2 * abs(lvec.mean())
    if exact_fp32:
        errs = {n: float(np.abs(got[n] - ref[n]).max() / np.abs(ref[n]).max()) for n in V}
        assert all(e < 1e-3 for e in errs.values()), errs
    else:
        errs = {n: float(np.linalg.norm((got[n] - ref[n]).ravel()) / np.linalg.norm(ref[n].ravel()))
                for n in V}
        assert all(e < 1e-2 for e in errs.values()), errs
    assert pred.dtype == np.int64 and pred.shape == (B,)


def test_vgg_style_training_step_config5_reduced(oracle, rng):
    # BASELINE config 5's graph shape (8 x Conv2D 3x3 SAME + ReLU in four blocks with 2x2 pools,
    # then a classifier), reduced to batch 4 / 16x16 inputs, fp32 graph: one fwd+bwd+SGD step vs
    # the oracle.  The first layer (C=3) takes the patch-matrix path, the other seven the
    # TMA-im2col implicit GEMM (forward, input gradient and filter gradient).
    B, H = 4, 16
    widths = [(3, 32), (32, 32), (32, 64), (64, 64), (64, 64), (64, 64), (64, 96), (96, 96)]
    pool_after = {1, 3, 5, 7}
    x = rng.uniform(-1, 1, (B, H, H, 3)).astype(np.float32)
    labels = np.eye(10, dtype=np.float32)[rng.randint(0, 10, B)]
    ws = [(rng.randn(3, 3, ci, co) * np.sqrt(2.0 / (9 * ci))).astype(np.float32) for ci, co in widths]
    bs = [np.full(co, 0.05, np.float32) for _, co in widths]
    wf = (rng.randn(96, 10) * 0.1).astype(np.float32)
    bf = np.zeros(10, np.float32)
    lr = 0.05
    tf.reset_default_graph()
    xp, lp = tf.placeholder(tf.float32, [B, H, H, 3]), tf.placeholder(tf.float32, [B, 10])
    Wv = [tf.Variable(w, name="w%d" % i) for i, w in enumerate(ws)]
    Bv = [tf.Variable(b, name="b%d" % i) for i, b in enumerate(bs)]
    Wf, Bf = tf.Variable(wf, name="wf"), tf.Variable(bf, name="bf")
    h = xp
    for i in range(8):
        h = tf.relu(tf.bias_add(tf.conv2d(h, Wv[i], [1, 1, 1, 1], "SAME"), Bv[i]))
        if i in pool_after:
            h = tf.max_pool(h, [1, 2, 2, 1], [1, 2, 2, 1], "SAME")
    logits = tf.bias_add(tf.matmul(tf.reshape(h, [B, 96]), Wf), Bf)
    loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(logits, lp))
    train = tf.GradientDescentOptimizer(lr).minimize(loss)
    with client.Session(tf.get_default_graph()) as sess:
        sess.run(tf.global_variables_initializer())
        got_loss, _ = sess.run([loss, train], {xp: x, lp: labels})
        got_w = sess.run([v.ref for v in Wv] + [Wf.ref])
        got_b = sess.run([v.ref for v in Bv] + [Bf.ref])

    o = oracle
    acts, pre_pool, inputs = [], [], []
    a = x
    for i in range(8):
        inputs.append(a)
        a = o.relu(o.bias_add(o.conv2d(a, ws[i], (1, 1), "SAME"), bs[i]))
        acts.append(a)
        if i in pool_after:
            pre_pool.append(a)
            a = o.max_pool(a, (2, 2), (2, 2), "SAME")
    flat = a.reshape(B, 96)
    lg = o.bias_add(o.matmul(flat, wf), bf)
    lvec, bp = o.softmax_xent(lg, labels)
    d = bp / np.float32(B)
    ref_w, ref_b = [None] * 9, [None] * 9
    ref_b[8] = o.apply_gradient_descent(bf, lr, o.bias_add_grad(d))
    ref_w[8] = o.apply_gradient_descent(wf, lr, o.matmul(flat, d, True, False))
    d = o.matmul(d, wf, False, True).reshape(a.shape)
    for i in reversed(range(8)):
        if i in pool_after:
            d = o.max_pool_grad(acts[i], d, (2, 2), (2, 2), "SAME")
        d = o.relu_grad(d, acts[i])
        ref_b[i] = o.apply_gradient_descent(bs[i], lr, o.bias_add_grad(d))
        ref_w[i] = o.apply_gradient_descent(
            ws[i], lr, o.conv2d_backprop_filter(inputs[i], ws[i].shape, d, (1, 1), "SAME"))
        if i > 0:
            d = o.conv2d_backprop_input(inputs[i].shape, ws[i], d, (1, 1), "SAME")
    assert abs(got_loss - lvec.mean()) < 1e-2 * abs(lvec.mean())
    # The bar is on the updated values (1e-2 relative, Frobenius: TF32 may flip single ReLU masks at
    # this batch size, see the LeNet test); the update itself -- after eight TF32 layers of
    # backprop -- is additionally held to 8 % so that a wrong gradient cannot hide behind lr
    # (at batch 4 a handful of flipped ReLU masks move the first layer's gradient by ~5 %:
    # tests/workloads.py::KernelRounding explains the sqrt(flip fraction) law).
    for name, got, ref, old in ([("w%d" % i, got_w[i], ref_w[i], (ws + [wf])[i]) for i in range(9)] +
                                [("b%d" % i, got_b[i], ref_b[i], (bs + [bf])[i]) for i in range(9)]):
        upd_ref = (ref - old).ravel().astype(np.float64)
        upd_got = (got - old).ravel().astype(np.float64)
        assert np.linalg.norm(upd_got - upd_ref) <= 8e-2 * max(np.linalg.norm(upd_ref), 1e-12), name
        assert np.linalg.norm((got - ref).ravel()) <= 1e-2 * np.linalg.norm(ref.ravel()), name


def test_fusion_rewrite_matches_unfused(oracle, rng, monkeypatch):
    # MatMul+BiasAdd+Relu and MatMul+ReluGrad chains run as _FusedMatMul (fewer launches), with
    # results identical (same GEMM, same fp32 tail) to the op-by-op execution.
    B, D = 512, 256
    x = rng.uniform(-1, 1, (B, D)).astype(np.float32)
    labels = np.eye(D, dtype=np.float32)[rng.randint(0, D, B)]
    ws = [(rng.randn(D, D) / np.sqrt(D)).astype(np.float32) for _ in range(3)]

    def run(disable):
        if disable:
            monkeypatch.setenv("B200TF_DISABLE_FUSION", "1")
        else:
            monkeypatch.delenv("B200TF_DISABLE_FUSION", raising=False)
        tf.reset_default_graph()
        xp, lp = tf.placeholder(tf.float32, [B, D]), tf.placeholder(tf.float32, [B, D])
        Ws = [tf.Variable(w, name="W%d" % i) for i, w in enumerate(ws)]
        Bs = [tf.Variable(np.full(D, 0.1, np.float32), name="b%d" % i) for i in range(3)]
        h = xp
        for i in range(3):
            h = tf.bias_add(tf.matmul(h, Ws[i]), Bs[i])
            if i < 2:
                h = tf.relu(h)
        loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(h, lp))
        train = tf.GradientDescentOptimizer(0.5).minimize(loss)
        with client.Session(tf.get_default_graph()) as sess:
            sess.run(tf.global_variables_initializer())
            lv, _ = sess.run([loss, train], {xp: x, lp: labels})
            stats = sess.last_run_stats()
            return lv, sess.run([v.ref for v in Ws + Bs]), stats

    l0, v0, s0 = run(disable=True)
    l1, v1, s1 = run(disable=False)
    assert s1["nodes_executed"] < s0["nodes_executed"]
    assert s1["kernels_launched"] < s0["kernels_launched"]
    # same arithmetic; only the split-K choice (hence fp32 summation order) of small GEMMs differs
    assert abs(l0 - l1) <= 1e-5 * abs(l0)
    for a, b in zip(v0, v1):  # weights are O(0.1): a different fp32 summation order moves them by ~1e-5
        np.testing.assert_allclose(a, b, rtol=1e-4, atol=5e-5)


@pytest.mark.parametrize("hw,ksize", [((12, 12), 2), ((9, 9), 2)])
def test_pool_grad_relu_grad_bias_grad_rewrite(rng, monkeypatch, hw, ksize):
    # conv -> bias -> relu -> max_pool: the backward tail MaxPoolGrad -> ReluGrad -> BiasAddGrad
    # runs as one `_MaxPoolGradReluGradBiasAddGrad` node (one kernel when the windows tile the
    # input -- 12x12 -- and the two-kernel composition when they do not -- 9x9 VALID); same values
    # as the op-by-op execution, the bias gradient up to its summation order
    B, C, K = 6, 32, 64
    x = rng.uniform(-1, 1, (B, hw[0], hw[1], C)).astype(np.float32)
    w = (rng.randn(3, 3, C, K) * 0.1).astype(np.float32)
    b = (rng.randn(K) * 0.1).astype(np.float32)

    def run(disable):
        if disable:
            monkeypatch.setenv("B200TF_DISABLE_FUSION", "1")
        else:
            monkeypatch.delenv("B200TF_DISABLE_FUSION", raising=False)
        tf.reset_default_graph()
        xp = tf.placeholder(tf.float32, list(x.shape))
        wv, bv = tf.Variable(w, name="w"), tf.Variable(b, name="b")
        a = tf.relu(tf.bias_add(tf.conv2d(xp, wv, [1, 1, 1, 1], "SAME"), bv))
        p = tf.max_pool(a, [1, ksize, ksize, 1], [1, ksize, ksize, 1], "VALID")
        loss = tf.reduce_sum(tf.multiply(p, p))
        gx, gw, gb = tf.gradients(loss, [xp, wv, bv])
        with client.Session(tf.get_default_graph()) as sess:
            sess.run(tf.global_variables_initializer())
            out = sess.run([gx, gw, gb], {xp: x})
            return out, sess.last_run_stats()

    ref, s0 = run(disable=True)
    got, s1 = run(disable=False)
    assert s1["nodes_executed"] < s0["nodes_executed"]
    np.testing.assert_allclose(got[2], ref[2], rtol=1e-5, atol=1e-5)
    # dY is bit-identical, so the convolution gradients are too
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1], ref[1])


def test_xent_scale_rewrite_is_bit_exact(rng, monkeypatch):
    # xent -> Mul(backprop, 1/N) (the gradient of a mean loss) runs as one scaled xent kernel:
    # (softmax - labels) is rounded to fp32 and then multiplied, exactly like the two-op form
    B, C = 300, 1000
    logits = rng.uniform(-3, 3, (B, C)).astype(np.float32)
    labels = np.eye(C, dtype=np.float32)[rng.randint(0, C, B)]

    def run(disable):
        if disable:
            monkeypatch.setenv("B200TF_DISABLE_FUSION", "1")
        else:
            monkeypatch.delenv("B200TF_DISABLE_FUSION", raising=False)
        tf.reset_default_graph()
        xp, lp = tf.placeholder(tf.float32, [B, C]), tf.placeholder(tf.float32, [B, C])
        h = tf.identity(xp)
        loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(h, lp))
        (dlogits,) = tf.gradients(loss, [h])
        with client.Session(tf.get_default_graph()) as sess:
            out = sess.run([loss, dlogits], {xp: logits, lp: labels})
            return out, sess.last_run_stats()["nodes_executed"]

    (l0, g0), n0 = run(disable=True)
    (l1, g1), n1 = run(disable=False)
    assert n1 == n0 - 1  # the Mul is gone
    np.testing.assert_array_equal(g0, g1)
    assert l0 == l1
    p = np.exp(logits - logits.max(1, keepdims=True))
    ref = (p / p.sum(1, keepdims=True) - labels) / B
    np.testing.assert_allclose(g1, ref, rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("adj_x", [False, True])
@pytest.mark.parametrize("adj_y", [False, True])
def test_batch_matmul_gradients(oracle, rng, adj_x, adj_y):
    # math_grad.py:871-894 through the graph: d/dx, d/dy of sum(w * BatchMatMul(x, y)) vs the oracle
    b, m, k, n = 3, 40, 24, 56
    x = rng.randn(*((b, k, m) if adj_x else (b, m, k))).astype(np.float32)
    y = rng.randn(*((b, n, k) if adj_y else (b, k, n))).astype(np.float32)
    w = rng.randn(b, m, n).astype(np.float32)
    tf.reset_default_graph()
    xp, yp = tf.placeholder(tf.float32, list(x.shape)), tf.placeholder(tf.float32, list(y.shape))
    z = tf.batch_matmul(xp, yp, adj_x, adj_y)
    loss = tf.reduce_mean(tf.multiply(z, tf.constant(w)))
    gx, gy = tf.gradients(loss, [xp, yp])
    with client.Session(tf.get_default_graph()) as sess:
        got_z, got_gx, got_gy = sess.run([z, gx, gy], {xp: x, yp: y})
    ref_z = oracle.batch_matmul(x, y, adj_x, adj_y)
    g = w / np.float32(w.size)
    xm = np.swapaxes(x, 1, 2) if adj_x else x           # [b, m, k]
    ym = np.swapaxes(y, 1, 2) if adj_y else y           # [b, k, n]
    dxm = np.einsum("bmn,bkn->bmk", g.astype(np.float64), ym.astype(np.float64))
    dym = np.einsum("bmk,bmn->bkn", xm.astype(np.float64), g.astype(np.float64))
    ref_gx = np.swapaxes(dxm, 1, 2) if adj_x else dxm
    ref_gy = np.swapaxes(dym, 1, 2) if adj_y else dym
    assert np.abs(got_z - ref_z).max() / np.abs(ref_z).max() < 3e-3
    assert np.abs(got_gx - ref_gx).max() / np.abs(ref_gx).max() < 3e-3
    assert np.abs(got_gy - ref_gy).max() / np.abs(ref_gy).max() < 3e-3


def test_nchw_graph_matches_nhwc_graph(rng):
    # data_format="NCHW" (GPU-only in the reference: conv_ops.cc:758-763, bias_op.cc:242-299,
    # maxpooling_op.cc:341-404): the convolution transposes in and out of the NHWC kernels, BiasAdd /
    # BiasAddGrad / MaxPool(+Grad) run natively on the NCHW planes.  Same arithmetic per element, so
    # a NCHW conv -> bias -> relu -> pool block matches the NHWC one bit for bit; only the bias
    # gradient is summed in another (fixed) order
    B, H, W, C, K = 3, 12, 10, 32, 64
    x = rng.uniform(-1, 1, (B, H, W, C)).astype(np.float32)
    w = (rng.randn(3, 3, C, K) * 0.1).astype(np.float32)
    b = rng.randn(K).astype(np.float32)

    def run(fmt):
        tf.reset_default_graph()
        nchw = fmt == "NCHW"
        xin = np.ascontiguousarray(x.transpose(0, 3, 1, 2)) if nchw else x
        xp = tf.placeholder(tf.float32, list(xin.shape))
        wv, bv = tf.Variable(w, name="w"), tf.Variable(b, name="b")
        st = [1, 1, 2, 1] if nchw else [1, 2, 1, 1]          # stride 2 along H, 1 along W
        c = tf.conv2d(xp, wv, st, "SAME", data_format=fmt)
        a = tf.relu(tf.bias_add(c, bv, data_format=fmt))
        ks = [1, 1, 2, 2] if nchw else [1, 2, 2, 1]
        p = tf.max_pool(a, ks, ks, "SAME", data_format=fmt)
        loss = tf.reduce_mean(tf.multiply(p, p))
        gx, gw, gb = tf.gradients(loss, [xp, wv, bv])
        with client.Session(tf.get_default_graph()) as sess:
            sess.run(tf.global_variables_initializer())
            out = sess.run([p, gx, gw, gb], {xp: xin})
        if nchw:
            out[0] = out[0].transpose(0, 2, 3, 1)
            out[1] = out[1].transpose(0, 2, 3, 1)
        return out

    ref, got = run("NHWC"), run("NCHW")
    assert ref[0].shape == (B, 3, 5, K)  # conv stride 2 along H, then the 2x2 pool
    for r, g in zip(ref[:3], got[:3]):
        np.testing.assert_array_equal(r, g)
    np.testing.assert_allclose(got[3], ref[3], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("shape", [(6, 5, 4), (2, 3, 4, 6, 10), (3, 8, 7, 9)])
def test_nchw_bias_add_any_rank(rng, shape):
    # GetBiasValueDims (bias_op.cc:140-150): channel = dims - 3, every dimension before it is batch
    x = rng.uniform(-1, 1, shape).astype(np.float32)
    b = rng.uniform(-1, 1, shape[-3]).astype(np.float32)
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, list(shape))
    bv = tf.Variable(b, name="b")
    y = tf.bias_add(xp, bv, data_format="NCHW")
    loss = tf.reduce_sum(tf.multiply(y, y))
    gx, gb = tf.gradients(loss, [xp, bv])
    with client.Session(tf.get_default_graph()) as sess:
        sess.run(tf.global_variables_initializer())
        yv, gxv, gbv = sess.run([y, gx, gb], {xp: x})
    ref = x + b[:, None, None]
    np.testing.assert_array_equal(yv, ref)
    np.testing.assert_allclose(gxv, 2 * ref, rtol=1e-6)
    axes = tuple(i for i in range(len(shape)) if i != len(shape) - 3)
    np.testing.assert_allclose(gbv, (2 * ref.astype(np.float64)).sum(axes), rtol=1e-5, atol=1e-5)


def test_reference_style_script_runs():
    # simple_tensorflow_b200.compat: the names of a TensorFlow-1.0 script (tf.nn.*, tf.train.*,
    # tf.Session() on the default graph); uniform logits -> loss = log(4)
    import simple_tensorflow_b200.compat as tfc
    tfc.reset_default_graph()
    x = tfc.placeholder(tfc.float32, [8, 16])
    y = tfc.placeholder(tfc.float32, [8, 4])
    W = tfc.Variable(np.full((16, 4), 0.1, np.float32))
    b = tfc.Variable(np.zeros(4, np.float32))
    logits = tfc.nn.bias_add(tfc.matmul(tfc.nn.relu(x), W), b)
    loss = tfc.reduce_mean(tfc.nn.softmax_cross_entropy_with_logits(labels=y, logits=logits))
    train = tfc.train.GradientDescentOptimizer(0.1).minimize(loss)
    with tfc.Session() as sess:
        sess.run(tfc.global_variables_initializer())
        xv = np.ones((8, 16), np.float32)
        yv = np.eye(4, dtype=np.float32)[np.arange(8) % 4]
        l0, _ = sess.run([loss, train], {x: xv, y: yv})
        l1 = sess.run(loss, {x: xv, y: yv})
    assert abs(l0 - np.log(4)) < 1e-5 and l1 <= l0 + 1e-6


def test_all_reduce_n_single_replica(rng):
    # without a communicator the op is an identity (times scale): the N>1 path runs in bench.py
    a = rng.randn(1000).astype(np.float32)
    b = rng.randn(33, 7).astype(np.float32)
    tf.reset_default_graph()
    pa, pb = tf.placeholder(tf.float32, [1000]), tf.placeholder(tf.float32, [33, 7])
    ra, rb = tf.all_reduce_n([tf.identity(pa), tf.identity(pb)], scale=0.5)
    with client.Session(tf.get_default_graph()) as sess:
        ga, gb = sess.run([ra, rb], {pa: a, pb: b})
    np.testing.assert_array_equal(ga, a * np.float32(0.5))
    np.testing.assert_array_equal(gb, b * np.float32(0.5))


def test_staged_feeds_match_host_feeds(oracle, rng):
    # Session.stage(): the copy runs on the host_to_device stream, Run() only orders behind it
    a = rng.uniform(-1, 1, (300, 128)).astype(np.float32)
    b = rng.uniform(-1, 1, (128, 64)).astype(np.float32)
    tf.reset_default_graph()
    pa, pb = tf.placeholder(tf.float32, [300, 128]), tf.placeholder(tf.float32, [128, 64])
    c = tf.relu(tf.matmul(pa, pb))
    axis = tf.placeholder(tf.int32, [])
    am = tf.get_default_graph().create_op("ArgMax", [c, axis], {"T": ("type", tf.float32)},
                                          "am").outputs[0]
    with client.Session(tf.get_default_graph()) as sess:
        host = sess.run(c, {pa: a, pb: b})
        sa, sb = sess.stage(a), sess.stage(client.HostTensor.from_numpy(b))
        assert sa.shape == (300, 128) and sa.nbytes == a.nbytes
        staged = sess.run(c, {pa: sa, pb: sb})
        np.testing.assert_array_equal(host, staged)
        # a staged tensor stays valid device memory: feed it again, mixed with a host feed
        again = sess.run(c, {pa: sa, pb: b})
        np.testing.assert_array_equal(host, again)
        assert sess.last_run_stats()["h2d_bytes"] == b.nbytes
        # pipelined use: stage the next input before running the current one
        nxt = sess.stage(a * 2)
        cur = sess.run(c, {pa: sa, pb: sb})
        np.testing.assert_array_equal(host, cur)
        np.testing.assert_array_equal(sess.run(c, {pa: nxt, pb: sb}),
                                      sess.run(c, {pa: a * 2, pb: b}))
        # HostMemory consumers (ArgMax's `dimension`) cannot take a device-resident feed
        with pytest.raises(client.OpError) as e:
            sess.run(am, {pa: sa, pb: sb, axis: sess.stage(np.int32(1))})
        assert e.value.error_code == 3 and "host memory" in e.value.message
    ref = oracle.relu(oracle.matmul(a, b))
    assert np.abs(host - ref).max() / np.abs(ref).max() < 3e-3


def test_schedule_is_a_valid_order_for_out_of_order_graphs(rng):
    # the list scheduler must respect data AND control edges whatever the construction order
    tf.reset_default_graph()
    v = tf.Variable(np.zeros(4, np.float32), name="v")
    one = tf.constant(np.ones(4, np.float32))
    with_init = tf.get_default_graph().create_op(
        "Identity", [v.ref], {"T": ("type", tf.float32)}, "read_after_init",
        control_inputs=[v.initializer])
    out = tf.add_n([with_init.outputs[0], one])
    with client.Session(tf.get_default_graph()) as sess:
        np.testing.assert_array_equal(sess.run(out), np.ones(4, np.float32))


def test_session_error_behaviour(rng):
    tf.reset_default_graph()
    x = tf.placeholder(tf.float32, [4, 3], "x")
    w = tf.Variable(np.ones((5, 2), np.float32), name="w")
    y = tf.matmul(x, w, name="bad_matmul")
    with client.Session(tf.get_default_graph()) as sess:
        with pytest.raises(client.OpError) as e:  # placeholder not fed (constant_op.cc)
            sess.run(y)
        assert e.value.error_code in (3, 9)
        with pytest.raises(client.OpError) as e:  # variable read before its initializer ran
            sess.run(y, {x: np.ones((4, 3), np.float32)})
        assert e.value.error_code == 9 and "uninitialized" in e.value.message
        sess.run(tf.global_variables_initializer())
        with pytest.raises(client.OpError) as e:  # matmul_op.cc:228-232
            sess.run(y, {x: np.ones((4, 3), np.float32)})
        assert e.value.error_code == 3 and "Matrix size-incompatible" in e.value.message
        assert "bad_matmul" in e.value.message
        # the session stays usable after a failed step
        w2 = sess.run(w.ref)
        np.testing.assert_array_equal(w2, np.ones((5, 2), np.float32))


def test_bf16_graph_additive_dtype(oracle, rng):
    # BASELINE config 4's dtype: bf16 storage, fp32 accumulate (additive T extension)
    B, D = 256, 128
    x = oracle.truncate_to_bf16(rng.uniform(-1, 1, (B, D)).astype(np.float32))
    w = oracle.truncate_to_bf16((rng.randn(D, D) / np.sqrt(D)).astype(np.float32))
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, [B, D])
    h = tf.relu(tf.matmul(tf.cast(xp, tf.bfloat16), tf.constant(w, tf.bfloat16)))
    out = tf.cast(h, tf.float32)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(out, {xp: x})
    ref = oracle.relu(oracle.matmul(x, w))
    assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-2


@pytest.mark.parametrize("bf16", [False, True])
def test_sum_and_mean_reductions(oracle, rng, bf16):
    # reduction_ops_common.h patterns that collapse to one reduced run: full, rows, columns,
    # middle axes, negative indices, keep_dims; VERDICT r1 "Sum is not registered, Mean all dims only"
    x = rng.uniform(-1, 1, (6, 5, 7, 4)).astype(np.float32)
    if bf16:
        x = oracle.truncate_to_bf16(x)
    cases = [(None, False), ([0, 1, 2, 3], True), (3, False), (-1, True), (0, False), ([0, 1], False),
             ([1, 2], False), ([1, 2], True), ([2, 3], False), ([-3, -2], False)]
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, list(x.shape), "x")
    src = tf.cast(xp, tf.bfloat16) if bf16 else xp
    outs = []
    for axis, keep in cases:
        for fn in (tf.reduce_sum, tf.reduce_mean):
            y = fn(src, axis, keep)
            outs.append(tf.cast(y, tf.float32) if bf16 else y)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(outs, {xp: x})
    it = iter(got)
    for axis, keep in cases:
        ax = None if axis is None else tuple(axis) if isinstance(axis, list) else axis
        for fn in (np.sum, np.mean):
            ref = fn(x.astype(np.float64), axis=ax, keepdims=keep)
            g = next(it)
            assert g.shape == ref.shape, (axis, keep, g.shape, ref.shape)
            np.testing.assert_allclose(g, ref, rtol=1e-2 if bf16 else 1e-5, atol=1e-2 if bf16 else 1e-5)


def test_reduce_sum_middle_axis_with_more_than_65535_outer_rows(rng):
    # [70000, 10, 3] reduced over axis 1 collapses to outer = 70000, inner = 3: more outer rows than
    # one grid dimension holds
    x = rng.uniform(-1, 1, (70000, 10, 3)).astype(np.float32)
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, list(x.shape), "x")
    y = tf.reduce_sum(xp, 1)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(y, {xp: x})
    ref = x.astype(np.float64).sum(1)
    assert got.shape == ref.shape
    assert (np.abs(got - ref) <= 1e-5 * np.abs(x).astype(np.float64).sum(1)).all()


def test_alternating_reduction_axes_are_rejected(rng):
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, [3, 4, 5], "x")
    y = tf.reduce_sum(xp, [0, 2])
    with client.Session(tf.get_default_graph()) as sess:
        with pytest.raises(client.OpError) as e:
            sess.run(y, {xp: np.ones((3, 4, 5), np.float32)})
        assert e.value.error_code == 12  # Unimplemented


def test_add_n_more_than_eight_inputs(rng):
    # aggregate_ops.cc:60-130 handles any N (unrolled by 8)
    xs = [rng.randn(33, 17).astype(np.float32) for _ in range(19)]
    tf.reset_default_graph()
    ps = [tf.placeholder(tf.float32, [33, 17]) for _ in xs]
    y = tf.add_n(ps)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(y, dict(zip(ps, xs)))
    ref = xs[0].copy()
    for a in xs[1:]:
        ref = ref + a          # left to right in fp32, like the kernel
    np.testing.assert_array_equal(got, ref)


@pytest.mark.parametrize("relu", [False, True])
def test_fused_matmul_with_few_tiles_splits_k(oracle, rng, relu):
    # LeNet fc1's shape (512 x 1024 x 3136): 8 pair tiles for 74 pairs -> the fused MatMul+BiasAdd
    # (+Relu) splits K and its tail rides on the ordered reduction pass; same result as op by op
    x = rng.uniform(-1, 1, (512, 3136)).astype(np.float32)
    w = (rng.randn(3136, 1024) / 56.0).astype(np.float32)
    b = rng.uniform(-0.5, 0.5, 1024).astype(np.float32)
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float32, [512, 3136], "x")
    y = tf.bias_add(tf.matmul(xp, tf.constant(w)), tf.constant(b))
    if relu:
        y = tf.relu(y)
    with client.Session(tf.get_default_graph()) as sess:
        got = sess.run(y, {xp: x})
        assert sess.last_run_stats()["kernels_launched"] == 2  # split GEMM + reduction with the tail
    ref = oracle.bias_add(oracle.matmul(x, w), b)
    if relu:
        ref = oracle.relu(ref)
    assert np.abs(got - ref).max() / np.abs(ref).max() < 3e-3
    if relu:
        assert got.min() >= 0.0


def _h(a):
    """fp32 values that survive a float -> half -> float round trip (the half parity inputs)."""
    return np.asarray(a, np.float32).astype(np.float16)


def test_half_hot_path_ops_vs_oracle(oracle, rng):
    # DT_HALF for the ops the reference registers half GPU kernels for (matmul_op.cc:301-332,
    # conv_ops.cc:758-763, maxpooling_op.cc:646-651, bias_op.cc:242-299): oracle on the fp16-rounded
    # inputs, reference tolerance for half 1e-3 (python/framework/test_util.py:515-523) relative to
    # the output scale
    x = _h(rng.uniform(-1, 1, (64, 96)))
    w = _h(rng.randn(96, 48) / 10.0)
    b = _h(rng.uniform(-0.5, 0.5, 48))
    img = _h(rng.uniform(-1, 1, (3, 12, 12, 32)))
    flt = _h(rng.randn(3, 3, 32, 32) / 17.0)
    cb = _h(rng.uniform(-0.5, 0.5, 32))
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float16, [64, 96], "x")
    ip = tf.placeholder(tf.float16, [3, 12, 12, 32], "img")
    dense = tf.relu(tf.bias_add(tf.matmul(xp, tf.constant(w, tf.float16)), tf.constant(b, tf.float16)))
    conv = tf.bias_add(tf.conv2d(ip, tf.constant(flt, tf.float16), [1, 1, 1, 1], "SAME"),
                       tf.constant(cb, tf.float16))
    pool = tf.max_pool(conv, [1, 2, 2, 1], [1, 2, 2, 1], "VALID")
    sm = tf.softmax(tf.matmul(xp, tf.constant(w, tf.float16)))
    back = tf.cast(dense, tf.float32)
    with client.Session(tf.get_default_graph()) as sess:
        got_dense, got_conv, got_pool, got_sm, got_back = sess.run(
            [dense, conv, pool, sm, back], {xp: x, ip: img})
    assert got_dense.dtype == np.float16 and got_pool.dtype == np.float16
    f = lambda a: np.asarray(a, np.float32)
    ref_dense = oracle.relu(oracle.bias_add(oracle.matmul(f(x), f(w)), f(b)))
    ref_conv = oracle.bias_add(oracle.conv2d(f(img), f(flt), (1, 1), "SAME"), f(cb))
    ref_pool = oracle.max_pool(_h(ref_conv).astype(np.float32), (2, 2), (2, 2), "VALID")
    ref_sm = oracle.softmax(_h(oracle.matmul(f(x), f(w))).astype(np.float32))
    for got, ref in ((got_dense, ref_dense), (got_conv, ref_conv), (got_sm, ref_sm)):
        assert np.abs(f(got) - ref).max() <= 2e-3 * max(np.abs(ref).max(), 1.0)
    # pooling a half tensor is exact given the same conv output bits
    np.testing.assert_array_equal(got_pool, oracle.max_pool(f(got_conv), (2, 2), (2, 2), "VALID").astype(np.float16))
    assert np.abs(f(got_pool) - ref_pool).max() <= 2e-3 * np.abs(ref_pool).max()
    np.testing.assert_array_equal(got_back, f(got_dense))  # Cast half -> float is exact


def test_half_conv_gradients_vs_oracle(oracle, rng):
    x = _h(rng.uniform(-1, 1, (2, 10, 10, 32)))
    flt = _h(rng.randn(3, 3, 32, 32) / 17.0)
    dy = _h(rng.uniform(-1, 1, (2, 10, 10, 32)))
    tf.reset_default_graph()
    xp = tf.placeholder(tf.float16, list(x.shape), "x")
    dp = tf.placeholder(tf.float16, list(dy.shape), "dy")
    fc = tf.constant(flt, tf.float16)
    g = tf.get_default_graph()
    attrs = {"T": ("type", tf.float16), "strides": ("list(int)", [1, 1, 1, 1]),
             "padding": ("string", "SAME"), "data_format": ("string", "NHWC")}
    y = tf.conv2d(xp, fc, [1, 1, 1, 1], "SAME")
    conv_op = y.op
    dx, dw = tf._GRAD["Conv2D"](conv_op, dp)
    with client.Session(g) as sess:
        got_dx, got_dw = sess.run([dx, dw], {xp: x, dp: dy})
    f = lambda a: np.asarray(a, np.float32)
    ref_dx = oracle.conv2d_backprop_input(x.shape, f(flt), f(dy), (1, 1), "SAME")
    ref_dw = oracle.conv2d_backprop_filter(f(x), flt.shape, f(dy), (1, 1), "SAME")
    assert got_dx.dtype == np.float16 and got_dw.dtype == np.float16
    assert np.abs(f(got_dx) - ref_dx).max() <= 2e-3 * np.abs(ref_dx).max()
    assert np.abs(f(got_dw) - ref_dw).max() <= 2e-3 * np.abs(ref_dw).max()


def test_stream_host_callback_runs_after_enqueued_work():
    # Stream::ThenDoHostCallback (stream_executor/stream.h:1624) -> b200_stream_add_host_callback
    import ctypes
    from simple_tensorflow_b200 import _lib
    L = _lib.load()
    stream = ctypes.c_void_p()
    assert L.b200_stream_create(ctypes.byref(stream)) == 0
    dev = ctypes.c_void_p()
    assert L.b200_malloc(ctypes.byref(dev), 1 << 20) == 0
    seen = []
    CB = ctypes.CFUNCTYPE(None, ctypes.c_void_p)
    cb = CB(lambda arg: seen.append(arg))
    assert L.b200_memset_async(dev, 0, 1 << 20, stream) == 0
    assert L.b200_stream_add_host_callback(stream, ctypes.cast(cb, ctypes.c_void_p), ctypes.c_void_p(42)) == 0
    assert L.b200_stream_synchronize(stream) == 0
    assert seen == [42]
    assert L.b200_stream_add_host_callback(stream, None, None) != 0  # null callback is rejected
    L.b200_free(dev)
    L.b200_stream_destroy(stream)


def _resident_training_losses(steps, graph_env, monkeypatch):
    """Train the small resident-input MLP for `steps` Session.Run calls; -> (losses, W after)."""
    import importlib
    if graph_env is None:
        monkeypatch.delenv("B200TF_CUDA_GRAPH", raising=False)
    else:
        monkeypatch.setenv("B200TF_CUDA_GRAPH", graph_env)
    r = np.random.RandomState(5)
    B, D = 256, 128
    x = r.uniform(-1, 1, (B, D)).astype(np.float32)
    labels = np.eye(D, dtype=np.float32)[r.randint(0, D, B)]
    w = (r.randn(D, D) / np.sqrt(D)).astype(np.float32)
    tf.reset_default_graph()
    X, L_ = tf.Variable(x, name="x"), tf.Variable(labels, name="l")
    W1, W2 = tf.Variable(w, name="w1"), tf.Variable(w.T.copy(), name="w2")
    b1 = tf.Variable(np.full(D, 0.1, np.float32), name="b1")
    h = tf.relu(tf.bias_add(tf.matmul(X.ref, W1), b1))
    loss = tf.reduce_mean(tf.softmax_cross_entropy_with_logits(tf.matmul(h, W2), L_.ref))
    train = tf.GradientDescentOptimizer(0.5).minimize(loss, [W1, W2, b1])
    losses, launches = [], []
    with client.Session(tf.get_default_graph()) as sess:
        sess.run(tf.global_variables_initializer())
        for _ in range(steps):
            losses.append(float(sess.run([loss, train])[0]))
            launches.append(sess.last_run_stats()["kernels_launched"])
        w_after = sess.run(W1.ref)
        # a different plan (fetch only) after the captured one still sees the trained variable
        loss_only = float(sess.run(loss))
    return losses, w_after, launches, loss_only


def test_step_level_cuda_graph_replays_the_step_bit_exactly(monkeypatch):
    # SURVEY 8f rank 3: a plan without feeds is captured into a CUDA graph on its third run and
    # replayed; results and the reported launch count must be those of the un-captured executor
    plain = _resident_training_losses(8, "0", monkeypatch)
    graph = _resident_training_losses(8, None, monkeypatch)
    assert plain[0] == graph[0], (plain[0], graph[0])
    np.testing.assert_array_equal(plain[1], graph[1])
    assert graph[2][0] == graph[2][-1] > 0          # replays report the captured launch count
    assert plain[2] == graph[2]
    assert plain[3] == graph[3]
    assert graph[0][-1] < graph[0][0]                # and the model did train
