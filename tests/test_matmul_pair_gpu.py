"""b200_matmul_pair and the executor's _MatMulPair rewrite against the two products run apart.

A dense layer's input gradient dX = dY W^T (K-major x K-major, often with a ReluGrad tail) and its
weight gradient dW = X^T dY (MN-major x MN-major, often split over K) share one persistent GEMM
launch.  Each product keeps its tile order, split plan and fused tail, so every output must be
bit-identical to its own b200_fused_matmul_ws call (fp32 compared through uint32 views, bf16 as raw
bits).  Each case also asserts the b200_launch_count() delta: one GEMM launch plus one reduction
per split product when paired, the two separate launches' count when the pair falls back.
"""
import numpy as np
import pytest
import torch

import abi_util as au
import workloads as W
from simple_tensorflow_b200 import client, ops as tf

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    assert au.lib().b200_device_count() >= 1


def raw_bits(t):
    torch.cuda.synchronize()
    if t.dtype == torch.bfloat16:
        return t.view(torch.int16).cpu().numpy()
    return t.view(torch.int32).cpu().numpy()


def layer_products(rng, batch, d_in, d_out, bf16, dx_tail="relu_grad", dw_tail=None):
    """(dX, dW) product descriptions of one dense layer: x [batch, d_in], w [d_in, d_out]."""
    def t(shape, lo=-1.0, hi=1.0):
        return au.dev(rng.uniform(lo, hi, shape).astype(np.float32), bf16)
    dy, x, w = t((batch, d_out)), t((batch, d_in)), t((d_in, d_out))
    dx = dict(a=dy, b=w, m=batch, n=d_in, k=d_out, ta=0, tb=1, bias=None, relu=0, features=None)
    dw = dict(a=x, b=dy, m=d_in, n=d_out, k=batch, ta=1, tb=0, bias=None, relu=0, features=None)
    for p, tail in ((dx, dx_tail), (dw, dw_tail)):
        if tail == "relu_grad":
            f = rng.uniform(-1, 1, (p["m"], p["n"])).astype(np.float32)
            f[::7, ::5] = 0.0
            p["features"] = au.dev(f, bf16)
        elif tail == "bias_relu":
            p["bias"], p["relu"] = t((p["n"],)), 1
    return dx, dw


def ptr(t):
    return None if t is None else t.data_ptr()


def run_separate(p, bf16):
    """The product as its own MatMul / _FusedMatMul op computes it: workspace unless ReluGrad."""
    L = au.lib()
    out = au.empty((p["m"], p["n"]), au.tdt(bf16), fill=float("nan"))
    nb = 0 if p["features"] is not None else L.b200_matmul_workspace_bytes(
        au.cdt(bf16), p["m"], p["n"], p["k"])
    scratch = au.ws(nb)
    au.call(L.b200_fused_matmul_ws, au.cdt(bf16), p["a"].data_ptr(), p["b"].data_ptr(),
            out.data_ptr(), p["m"], p["n"], p["k"], p["ta"], p["tb"], ptr(p["bias"]), p["relu"],
            ptr(p["features"]), scratch.data_ptr() if nb else None, nb, au.stream())
    return out


def run_pair(p0, p1, bf16):
    L = au.lib()
    outs = [au.empty((p["m"], p["n"]), au.tdt(bf16), fill=float("nan")) for p in (p0, p1)]
    nb = L.b200_matmul_pair_workspace_bytes(au.cdt(bf16), p0["m"], p0["n"], p0["k"],
                                            p1["m"], p1["n"], p1["k"])
    scratch = au.ws(nb)
    args = []
    for p, o in zip((p0, p1), outs):
        args += [p["a"].data_ptr(), p["b"].data_ptr(), o.data_ptr(), p["m"], p["n"], p["k"],
                 p["ta"], p["tb"], ptr(p["bias"]), p["relu"], ptr(p["features"])]
    au.call(L.b200_matmul_pair, au.cdt(bf16), *args, scratch.data_ptr() if nb else None, nb,
            au.stream())
    return outs


# (batch, d_in, d_out, bf16, dX tail, dW tail, launches of the two separate calls, paired)
CASES = {
    # the bench MLP's hidden layer: dX with ReluGrad (64 items), dW split 4 (64 items) + reduce
    "mlp_layer": (4096, 1024, 1024, False, "relu_grad", None, 3, True),
    "mlp_layer_bf16": (4096, 1024, 1024, True, "relu_grad", None, 3, True),
    # LeNet fc1: dX 512 x 3136 x 1024 split 2 + reduce, dW 3136 x 1024 x 512 unsplit
    "lenet_fc1": (512, 3136, 1024, False, None, None, 3, True),
    # the 512 x 256 layers of test_session_gpu.py::test_fusion_rewrite_matches_unfused
    "small_layer": (512, 256, 256, False, "relu_grad", None, 3, True),
    "small_layer_bf16": (512, 256, 256, True, "relu_grad", None, 3, True),
    # ragged: M, N not multiples of 256, K (300 and 600) not multiples of BK = 32
    "ragged": (600, 392, 300, False, "relu_grad", None, 3, True),
    # dX takes 256-wide pair tiles, dW (N = 200) 128-wide ones: two launches as before
    "configs_differ": (600, 392, 200, False, "relu_grad", None, 3, False),
    # a bias + relu tail on dX: both products split, the tail rides on dX's reduction
    "bias_relu_tail": (512, 256, 256, False, "bias_relu", None, 4, True),
}


@pytest.mark.parametrize("swap", [False, True], ids=["dx_first", "dw_first"])
@pytest.mark.parametrize("case", list(CASES))
def test_pair_is_the_two_products_bit_for_bit(rng, case, swap):
    batch, d_in, d_out, bf16, dx_tail, dw_tail, n_sep, paired = CASES[case]
    dx, dw = layer_products(rng, batch, d_in, d_out, bf16, dx_tail, dw_tail)
    p0, p1 = (dw, dx) if swap else (dx, dw)
    (want0, n0) = au.launches(run_separate, p0, bf16)
    (want1, n1) = au.launches(run_separate, p1, bf16)
    assert n0 + n1 == n_sep
    (got0, got1), n_pair = au.launches(run_pair, p0, p1, bf16)
    assert n_pair == (n_sep - 1 if paired else n_sep)
    np.testing.assert_array_equal(raw_bits(got0), raw_bits(want0))
    np.testing.assert_array_equal(raw_bits(got1), raw_bits(want1))


def test_pair_without_workspace_runs_unsplit(rng):
    # no scratch: neither product splits, so the pair is a single launch
    dx, dw = layer_products(rng, 4096, 1024, 1024, False)
    L = au.lib()
    outs = [au.empty((p["m"], p["n"])) for p in (dx, dw)]
    args = []
    for p, o in zip((dx, dw), outs):
        args += [p["a"].data_ptr(), p["b"].data_ptr(), o.data_ptr(), p["m"], p["n"], p["k"],
                 p["ta"], p["tb"], ptr(p["bias"]), p["relu"], ptr(p["features"])]
    _, n = au.launches(au.call, L.b200_matmul_pair, au.cdt(False), *args, None, 0, au.stream())
    assert n == 1
    want = [au.empty((p["m"], p["n"])) for p in (dx, dw)]
    for p, o in zip((dx, dw), want):
        au.call(L.b200_fused_matmul_ws, au.cdt(False), p["a"].data_ptr(), p["b"].data_ptr(),
                o.data_ptr(), p["m"], p["n"], p["k"], p["ta"], p["tb"], None, 0,
                ptr(p["features"]), None, 0, au.stream())
    for g, w in zip(outs, want):
        np.testing.assert_array_equal(raw_bits(g), raw_bits(w))


def _layer_session(rng, fetch):
    B, D, O = 1024, 512, 512
    x = rng.uniform(-1, 1, (B, D)).astype(np.float32)
    dy = rng.uniform(-1, 1, (B, O)).astype(np.float32)
    w = rng.uniform(-1, 1, (D, O)).astype(np.float32)
    tf.reset_default_graph()
    X, DY, Wt = tf.constant(x), tf.constant(dy), tf.constant(w)
    g = tf.get_default_graph()
    dx = g.create_op("ReluGrad", [tf.matmul(DY, Wt, transpose_b=True), tf.relu(X)],
                     {"T": ("type", tf.float32)}, "ReluGrad").outputs[0]
    dw = tf.matmul(X, DY, transpose_a=True)
    names = {"dx": dx, "dw": dw}
    with client.Session(tf.get_default_graph()) as sess:
        out = sess.run([names[f] for f in fetch])
        return out, sess.last_run_stats()["kernels_launched"]


def test_session_groups_a_layers_dx_and_dw_bit_for_bit():
    both, n_both = _layer_session(np.random.RandomState(3), ["dw", "dx"])
    (dw,), n_dw = _layer_session(np.random.RandomState(3), ["dw"])
    (dx,), n_dx = _layer_session(np.random.RandomState(3), ["dx"])
    np.testing.assert_array_equal(both[0].view(np.uint32), dw.view(np.uint32))
    np.testing.assert_array_equal(both[1].view(np.uint32), dx.view(np.uint32))
    # one GEMM launch instead of two; relu(X) and dW's split-K reduction run either way
    assert n_both == n_dw + n_dx - 1


def test_full_size_mlp_step_launches():
    w = W.get("mlp")
    B = w.build(num_replicas=1, seed=1234, resident=True)
    with client.Session(B.tf.get_default_graph()) as sess:
        sess.run(B.tf.global_variables_initializer())
        for _ in range(3):
            sess.run(list(B.resident))
        assert sess.last_run_stats()["kernels_launched"] == 15


def _degenerate_graph(case):
    """Fetches and numpy results of a graph whose products have k == 0 or an empty output."""
    rng = np.random.RandomState(5)
    a, b = np.zeros((4, 0), np.float32), np.zeros((0, 3), np.float32)
    if case == "matmul_k0":
        return [tf.matmul(tf.constant(a), tf.constant(b))], [a @ b]
    if case == "bias_relu_k0":  # _FusedMatMul: the tail runs on a zero product
        bias = np.array([0.5, -0.25, 0.0], np.float32)
        y = tf.relu(tf.bias_add(tf.matmul(tf.constant(a), tf.constant(b)), tf.constant(bias)))
        return [y], [np.maximum(np.broadcast_to(bias, (4, 3)), 0)]
    # _MatMulPair: X [0, 5] feeds X W (empty output) and dW = X^T dY (k == 0, zero-filled).  The
    # constants come first: a product pairs only with one whose inputs exist at its place.
    x, dy = np.zeros((0, 5), np.float32), np.zeros((0, 3), np.float32)
    w = rng.uniform(-1, 1, (5, 3)).astype(np.float32)
    X, Wt, DY = tf.constant(x), tf.constant(w), tf.constant(dy)
    return [tf.matmul(X, Wt), tf.matmul(X, DY, transpose_a=True)], [x @ w, x.T @ dy]


# case -> how many nodes fewer the fused graph runs than the op-by-op one
DEGENERATE = {"matmul_k0": 0, "bias_relu_k0": 2, "pair": 1}


@pytest.mark.parametrize("case", list(DEGENERATE))
def test_session_degenerate_products_match_unfused(case, monkeypatch):
    def run(disable):
        if disable:
            monkeypatch.setenv("B200TF_DISABLE_FUSION", "1")
        else:
            monkeypatch.delenv("B200TF_DISABLE_FUSION", raising=False)
        tf.reset_default_graph()
        fetches, want = _degenerate_graph(case)
        with client.Session(tf.get_default_graph()) as sess:
            return sess.run(fetches), want, sess.last_run_stats()["nodes_executed"]

    got, want, nodes = run(disable=False)
    ref, _, ref_nodes = run(disable=True)
    assert ref_nodes - nodes == DEGENERATE[case]
    for g, r, w in zip(got, ref, want):
        assert g.shape == w.shape
        np.testing.assert_array_equal(g, w)
        np.testing.assert_array_equal(g.view(np.uint32), r.view(np.uint32))
