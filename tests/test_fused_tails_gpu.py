"""Fused entry points against their unfused composition, through the C ABI (include/b200_ops.h).

The header promises that every fused entry point gives the same results as running the ops one by
one.  For fp32 that is checked bit for bit (`.view(np.uint32)`, so -0 and +0 differ) against the
library's own composition with the same workspace choice: the tile configuration depends only on
the shape and on whether scratch is present, split-K partials are added in ascending split order
either way, and each tail is one fp32 add and / or a select.  bf16 ReluGrad is bit-exact too
(masking by 0 / 1 commutes with rounding); a bf16 bias / relu tail rounds once where the
composition rounds twice, so those are checked against the fp32 oracle on bf16-truncated inputs.

Every case also records the b200_launch_count() delta and asserts the count its path implies in the
code, so that a case cannot pass on a path other than the one it is named for.
"""
import numpy as np
import pytest

import abi_util as au

pytestmark = pytest.mark.gpu

TOL = 1e-2          # bf16 parity bar (inputs truncated to bf16, fp32 oracle)
TOL_TF32 = 3e-3     # single-pass TF32 tensor-core paths
TOL_EXACT = 1e-5    # CUDA-core fp32 and reduction paths


@pytest.fixture(scope="module", autouse=True)
def _device():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    assert au.lib().b200_device_count() >= 1


def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def assert_same_bits(got, want):
    assert got.shape == want.shape
    np.testing.assert_array_equal(bits(got), bits(want))


def map_launches(n, bf16=False, aligned=True):
    """Kernels an element-wise map of n elements launches (elementwise.cu launch_map): a 16-byte
    vector kernel over the whole vectors, a scalar kernel over the rest."""
    width = 8 if bf16 else 4
    nvec = n // width if aligned else 0
    return int(nvec > 0) + int(nvec * width < n)


def f64_matmul(a, b, ta=False, tb=False):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return (a.T if ta else a) @ (b.T if tb else b)


def mixed_features(rng, m, n):
    """ReluGrad features whose sign alternates by column (and flips every other row), with exact
    zeros and -0: the two bf16 halves of every 32-bit word get different masks."""
    f = rng.uniform(0.1, 1.0, (m, n)).astype(np.float32)
    sign = np.where((np.arange(n)[None, :] + np.arange(m)[:, None]) % 2 == 0, 1.0, -1.0)
    f = (f * sign).astype(np.float32)
    f[::5, ::3] = 0.0
    f[2::7, 1::4] = -0.0
    return f


def operands(rng, m, n, k, ta=False, tb=False, bf16=False, oracle=None):
    a = rng.uniform(-1, 1, (k, m) if ta else (m, k)).astype(np.float32)
    b = rng.uniform(-1, 1, (n, k) if tb else (k, n)).astype(np.float32)
    bias = rng.uniform(-1, 1, n).astype(np.float32)
    if bf16:
        a, b, bias = (oracle.truncate_to_bf16(v) for v in (a, b, bias))
    return a, b, bias


# =============================================================================== fused MatMul
# (m, n, k): full tiles; ragged; CTA-pair tiles with an 8-column last tile
FUSED_SHAPES = [(512, 384, 256), (200, 136, 72), (512, 520, 260)]


@pytest.mark.parametrize("m,n,k", FUSED_SHAPES + [(200, 130, 256)])
def test_fused_matmul_fp32_is_the_composition_bit_for_bit(oracle, rng, m, n, k):
    # (200, 130, 256) with B stored [N, K]: N % 4 != 0, so C and the features cannot be TMA maps;
    # the direct-store epilogue runs with scalar bias and scalar feature loads
    tb = n % 4 != 0
    a, b, bias = operands(rng, m, n, k, tb=tb)
    feat = mixed_features(rng, m, n)
    plain, nl = au.launches(au.matmul, a, b, tb=tb, use_workspace=False)
    assert nl == 1
    assert au.rel_err(plain, oracle.matmul(a, b, False, tb)) < TOL_TF32
    with_bias = au.bias_add(plain, bias)
    for kw, want in [(dict(bias=bias), with_bias),
                     (dict(bias=bias, relu=True), au.relu(with_bias)),
                     (dict(features=feat), au.relu_grad(plain, feat))]:
        got, nl = au.launches(au.fused_matmul, a, b, tb=tb, **kw)
        assert nl == 1, kw  # the tail is in the GEMM epilogue
        assert_same_bits(got, want)
        assert_same_bits(au.fused_matmul(a, b, tb=tb, **kw), got)  # run to run


@pytest.mark.parametrize("ta", [False, True])
@pytest.mark.parametrize("tb", [False, True])
@pytest.mark.parametrize("m,n,k", [(512, 384, 256), (200, 136, 72)])
def test_fused_matmul_relu_grad_transposed_operands(oracle, rng, m, n, k, ta, tb):
    a, b, _ = operands(rng, m, n, k, ta, tb)
    feat = mixed_features(rng, m, n)
    plain = au.matmul(a, b, ta, tb, use_workspace=False)
    got, nl = au.launches(au.fused_matmul, a, b, ta, tb, features=feat)
    assert nl == 1
    assert_same_bits(got, au.relu_grad(plain, feat))
    assert au.rel_err(got, oracle.relu_grad(oracle.matmul(a, b, ta, tb), feat)) < TOL_TF32


@pytest.mark.parametrize("m,n,k", FUSED_SHAPES)
def test_fused_matmul_unaligned_bias_takes_the_scalar_bias_loads(rng, m, n, k):
    # a bias pointer one element past a 16-byte boundary: bias_vec = 0, per-column loads
    a, b, bias = operands(rng, m, n, k)
    want = au.bias_add(au.matmul(a, b, use_workspace=False), bias)
    for relu in (False, True):
        got, nl = au.launches(au.fused_matmul_ws, a, b, bias=bias, relu=relu, workspace_bytes=0,
                              bias_offset=1)
        assert nl == 1
        assert_same_bits(got, au.relu(want) if relu else want)


@pytest.mark.parametrize("m,n,k,tb", [(512, 384, 256, False), (200, 136, 72, False),
                                      (512, 520, 256, False), (512, 520, 260, False),
                                      (200, 130, 256, True)])
def test_fused_matmul_bf16(oracle, rng, m, n, k, tb):
    # (512, 520, 260): a 520-byte row of A is no multiple of 16 bytes, so TMA cannot address it and
    # the product runs on the CUDA cores, followed by the tail kernels (as MatMul + BiasAdd would)
    tensor = (k * 2) % 16 == 0 and ((k if tb else n) * 2) % 16 == 0
    a, b, bias = operands(rng, m, n, k, tb=tb, bf16=True, oracle=oracle)
    feat = oracle.truncate_to_bf16(mixed_features(rng, m, n))
    plain, nl = au.launches(au.matmul, a, b, tb=tb, bf16=True, use_workspace=False)
    assert nl == 1
    ref = oracle.matmul(a, b, False, tb)
    relu_n = map_launches(m * n, bf16=True)
    # ReluGrad: the mask commutes with the one rounding to bf16 -> bit-exact, half-words included
    got, nl = au.launches(au.fused_matmul, a, b, tb=tb, features=feat, bf16=True)
    assert nl == (1 if tensor else 1 + relu_n)
    assert_same_bits(got, au.relu_grad(plain, feat, bf16=True))
    assert (got[feat <= 0] == 0).all()
    assert au.rel_err(got, oracle.relu_grad(ref, feat)) < TOL
    # bias / bias + relu: one rounding (fused) vs two (composition) -> against the oracle
    ref_b = oracle.bias_add(ref, bias)
    got, nl = au.launches(au.fused_matmul, a, b, tb=tb, bias=bias, bf16=True)
    assert nl == (1 if tensor else 2)
    assert au.rel_err(got, ref_b) < TOL
    got, nl = au.launches(au.fused_matmul, a, b, tb=tb, bias=bias, relu=True, bf16=True)
    assert nl == (1 if tensor else 2 + relu_n)
    assert au.rel_err(got, oracle.relu(ref_b)) < TOL
    assert (got >= 0).all()
    assert_same_bits(au.fused_matmul(a, b, tb=tb, bias=bias, relu=True, bf16=True), got)


@pytest.mark.parametrize("m,n,k", [(512, 4, 1024),    # 4-output head: matrix-vector
                                   (2, 1024, 512),    # batch-2 dense layer: vector-matrix
                                   (16, 16, 64)])     # M*N*K < 32^3: tiny
def test_fused_matmul_uses_the_kernel_matmul_uses(oracle, rng, m, n, k):
    # MatMul sends these shapes to the exact-fp32 CUDA-core kernels; the fused form must too, so
    # that fusing a BiasAdd / Relu / ReluGrad into the product never changes its value
    a, b, bias = operands(rng, m, n, k)
    feat = mixed_features(rng, m, n)
    plain, nl = au.launches(au.matmul, a, b, use_workspace=False)
    assert nl == 1
    assert au.rel_err(plain, f64_matmul(a, b)) < TOL_EXACT
    with_bias = au.bias_add(plain, bias)
    relu_n = map_launches(m * n)
    for kw, want, tail in [(dict(bias=bias), with_bias, 1),
                           (dict(bias=bias, relu=True), au.relu(with_bias), 1 + relu_n),
                           (dict(features=feat), au.relu_grad(plain, feat), relu_n)]:
        got, nl = au.launches(au.fused_matmul, a, b, **kw)
        assert_same_bits(got, want)
        assert nl == 1 + tail, kw  # CUDA-core GEMM, then the tail kernels


# =============================================================================== split-K
SPLIT_SHAPES = [
    (128, 64, 16384, False),   # one output tile, 64 splits: the generic reducer
    (200, 136, 8192, False),   # ragged M and N, more than 16 splits
    (256, 130, 8192, True),    # N % 4 != 0: direct partial stores, generic reducer
    (512, 1024, 3136, False),  # LeNet fc1: 9 splits, the flat reducer
]


@pytest.mark.parametrize("m,n,k,tb", SPLIT_SHAPES)
def test_split_k_fused_tail_is_the_composition_bit_for_bit(rng, m, n, k, tb):
    a, b, bias = operands(rng, m, n, k, tb=tb)
    L = au.lib()
    assert L.b200_matmul_workspace_bytes(au.cdt(False), m, n, k) > 0  # this shape splits K
    plain, nl = au.launches(au.matmul, a, b, tb=tb)
    assert nl == 2  # split GEMM + ordered reduction
    ref = f64_matmul(a, b, False, tb)
    assert au.rel_err(plain, ref) < TOL_TF32
    with_bias = au.bias_add(plain, bias)
    for relu in (False, True):
        got, nl = au.launches(au.fused_matmul_ws, a, b, tb=tb, bias=bias, relu=relu)
        assert nl == 2  # the tail rides on the reduction pass
        assert_same_bits(got, au.relu(with_bias) if relu else with_bias)
        assert_same_bits(au.fused_matmul_ws(a, b, tb=tb, bias=bias, relu=relu), got)
    assert_same_bits(au.matmul(a, b, tb=tb), plain)


def test_split_k_bf16(oracle, rng):
    m, n, k = 256, 256, 8192
    a, b, bias = operands(rng, m, n, k, bf16=True, oracle=oracle)
    ref = f64_matmul(a, b)
    got, nl = au.launches(au.matmul, a, b, bf16=True)
    assert nl == 2
    assert au.rel_err(got, ref) < TOL
    for relu in (False, True):
        got, nl = au.launches(au.fused_matmul_ws, a, b, bias=bias, relu=relu, bf16=True)
        assert nl == 2
        want = ref + bias
        assert au.rel_err(got, np.maximum(want, 0) if relu else want) < TOL
        if relu:
            assert (got >= 0).all()


@pytest.mark.parametrize("splits", range(2, 17))
def test_split_k_flat_reducer_every_split_count(rng, splits):
    # the launcher lowers the split count until the partials fit the scratch it was given: a
    # workspace of exactly s * M * N * 4 bytes gives s splits (for s <= 16, 512 K blocks in chunks of
    # ceil(512 / s) make exactly s non-empty splits), i.e. the flat reducer instantiated for s
    m, n, k = 128, 64, 16384
    a, b, bias = operands(rng, m, n, k)
    nb = splits * m * n * 4
    plain, nl = au.launches(au.matmul, a, b, workspace_bytes=nb)
    assert nl == 2
    assert au.rel_err(plain, f64_matmul(a, b)) < TOL_TF32
    want = au.relu(au.bias_add(plain, bias))
    got, nl = au.launches(au.fused_matmul_ws, a, b, bias=bias, relu=True, workspace_bytes=nb)
    assert nl == 2
    assert_same_bits(got, want)


# =============================================================================== fused Conv2D
# (input, filter, strides, padding, kernels of the plain convolution, tail in its epilogue, tol)
CONV_CASES = [
    # C_in = 1, unit stride: the lane-per-filter conv_c1 kernel (IEEE fp32)
    ((5, 13, 11, 1), (5, 5, 1, 64), (1, 1), "SAME", 1, True, TOL_EXACT),
    ((9, 7, 30, 1), (3, 3, 1, 96), (1, 1), "SAME", 1, True, TOL_EXACT),
    # C_in <= 4: conv_small_cin_fwd_kernel, 5x5x1 / 3x3x3 specialisations, generic 16 and 4
    # filters per thread
    ((3, 11, 9, 1), (5, 5, 1, 32), (2, 2), "SAME", 1, True, TOL_EXACT),
    ((2, 12, 12, 3), (3, 3, 3, 64), (1, 1), "SAME", 1, True, TOL_EXACT),
    ((2, 6, 7, 2), (7, 5, 2, 32), (1, 2), "SAME", 1, True, TOL_EXACT),
    ((2, 8, 8, 4), (3, 3, 4, 12), (1, 1), "VALID", 1, True, TOL_EXACT),
    # halo tile (conv_halo.cu): several bands, asymmetric SAME, a ragged second N block
    ((2, 40, 70, 32), (3, 3, 32, 32), (1, 1), "SAME", 1, True, TOL_TF32),
    ((5, 11, 13, 32), (2, 4, 32, 96), (1, 1), "SAME", 1, True, TOL_TF32),
    ((2, 8, 8, 64), (1, 3, 64, 320), (1, 1), "SAME", 1, True, TOL_TF32),
    # implicit GEMM (strided), then BiasAdd / Relu kernels
    ((2, 15, 13, 32), (3, 3, 32, 16), (2, 2), "SAME", 1, False, TOL_TF32),
    # patch matrix (im2col + CUDA-core GEMM: N = 10 cannot be a TMA operand), then the tail
    ((2, 10, 10, 6), (3, 3, 6, 10), (1, 1), "SAME", 2, False, TOL_EXACT),
    # pointwise: plain GEMM on the input, then the tail
    ((3, 12, 12, 16), (1, 1, 16, 24), (1, 1), "VALID", 1, False, TOL_TF32),
]


def conv_tail_launches(out_size, relu, bf16=False):
    # b200_bias_add is one kernel (vector or scalar), b200_relu a map
    return 1 + (map_launches(out_size, bf16) if relu else 0)


@pytest.mark.parametrize("shape,fshape,strides,padding,conv_n,epilogue,tol", CONV_CASES)
def test_fused_conv2d_fp32_is_the_composition_bit_for_bit(oracle, rng, shape, fshape, strides,
                                                           padding, conv_n, epilogue, tol):
    x = rng.rand(*shape).astype(np.float32) - 0.5
    f = rng.rand(*fshape).astype(np.float32) - 0.5
    bias = rng.uniform(-1, 1, fshape[3]).astype(np.float32)
    plain, nl = au.launches(au.conv2d, x, f, strides, padding, oracle)
    assert nl == conv_n
    ref = oracle.conv2d(x, f, strides, padding)
    with_bias = au.bias_add(plain, bias)
    for relu in (False, True):
        got, nl = au.launches(au.fused_conv2d, x, f, bias, relu, strides, padding, oracle)
        want = au.relu(with_bias) if relu else with_bias
        assert_same_bits(got, want)
        expect = conv_n if epilogue else conv_n + conv_tail_launches(got.size, relu)
        assert nl == expect, relu
        ref_t = oracle.bias_add(ref, bias)
        assert au.rel_err(got, oracle.relu(ref_t) if relu else ref_t) < tol
        assert_same_bits(au.fused_conv2d(x, f, bias, relu, strides, padding, oracle), got)
    # no tail at all: the plain convolution
    assert_same_bits(au.fused_conv2d(x, f, None, False, strides, padding, oracle), plain)


@pytest.mark.parametrize("shape,fshape,strides,conv_n,epilogue", [
    ((2, 40, 70, 64), (3, 3, 64, 64), (1, 1), 1, True),     # halo tile
    ((2, 15, 13, 64), (3, 3, 64, 16), (2, 2), 1, False),    # implicit GEMM, then the tail
])
def test_fused_conv2d_bf16(oracle, rng, shape, fshape, strides, conv_n, epilogue):
    x = oracle.truncate_to_bf16(rng.rand(*shape).astype(np.float32) - 0.5)
    f = oracle.truncate_to_bf16((rng.rand(*fshape).astype(np.float32) - 0.5) * 0.2)
    bias = oracle.truncate_to_bf16(rng.uniform(-1, 1, fshape[3]).astype(np.float32))
    ref = oracle.bias_add(oracle.conv2d(x, f, strides, "SAME"), bias)
    for relu in (False, True):
        got, nl = au.launches(au.fused_conv2d, x, f, bias, relu, strides, "SAME", oracle, bf16=True)
        expect = conv_n if epilogue else conv_n + conv_tail_launches(got.size, relu, True)
        assert nl == expect
        assert au.rel_err(got, oracle.relu(ref) if relu else ref) < TOL
        if relu:
            assert (got >= 0).all()


def test_fused_conv2d_relu_without_bias_is_rejected(oracle, rng):
    x = rng.rand(2, 8, 8, 32).astype(np.float32)
    f = rng.rand(3, 3, 32, 32).astype(np.float32)
    with pytest.raises(au._lib.B200Error) as e:
        au.fused_conv2d(x, f, None, True, (1, 1), "SAME", oracle)
    assert e.value.code == 3  # INVALID_ARGUMENT


# =============================================================================== ReluGrad + BiasAddGrad
BIG_ROWS = 512 * 28 * 28  # LeNet conv1's backward pass: the grid reaches its 4 * SM-count cap
RGBG_CASES = (
    # (channels, bf16, flat path): G = channels / (16 bytes) a power of two <= 32
    [(c, False, True) for c in (4, 32, 64, 128)] + [(c, True, True) for c in (8, 64, 256)] +
    [(12, False, False), (1000, False, False), (1030, False, False), (24, True, False)])
RGBG_PARAMS = [(rows,) + case for case in RGBG_CASES
               for rows in ((1, 7, BIG_ROWS) if case[0] <= 256 else (1, 7, 3000))]


def rgbg_inputs(rng, rows, c, bf16, oracle):
    if rows >= 100000:  # quarter integers: exact in bf16, cheap to draw
        g = (rng.randint(-8, 8, (rows, c)).astype(np.float32) / 4).astype(np.float32)
    else:
        g = rng.uniform(-1, 1, (rows, c)).astype(np.float32)
    f = mixed_features(rng, rows, c)
    if bf16:
        g, f = oracle.truncate_to_bf16(g), oracle.truncate_to_bf16(f)
    return g, f


def check_bias_grad(got, dy, bf16):
    ref = dy.astype(np.float64).sum(0)
    bound = TOL_EXACT * np.abs(dy).astype(np.float64).sum(0) + 1e-30
    if bf16:
        bound = bound + 2.0 ** -8 * np.abs(ref)  # the one rounding of the result
    assert (np.abs(got - ref) <= bound).all()


@pytest.mark.parametrize("rows,channels,bf16,flat", RGBG_PARAMS)
def test_relu_grad_bias_grad_is_the_composition_bit_for_bit(oracle, rng, rows, channels, bf16, flat):
    g, f = rgbg_inputs(rng, rows, channels, bf16, oracle)
    (dy, db), nl = au.launches(au.relu_grad_bias_grad, g, f, bf16=bf16)
    # flat: one pass; otherwise b200_relu_grad (a map) + b200_bias_add_grad (one kernel)
    assert nl == (1 if flat else map_launches(g.size, bf16) + 1)
    want_dy = au.relu_grad(g, f, bf16=bf16)
    assert_same_bits(dy, want_dy)
    assert (dy[f <= 0] == 0).all()
    assert_same_bits(db, au.bias_add_grad(want_dy, bf16=bf16))
    check_bias_grad(db, dy, bf16)
    assert_same_bits(au.relu_grad_bias_grad(g, f, bf16=bf16)[1], db)  # ordered: run to run


@pytest.mark.parametrize("channels,bf16", [(32, False), (12, False), (64, True), (24, True)])
def test_relu_grad_bias_grad_aliased_and_unaligned(oracle, rng, channels, bf16):
    rows = 3001
    g, f = rgbg_inputs(rng, rows, channels, bf16, oracle)
    want_dy = au.relu_grad(g, f, bf16=bf16)
    dy, db = au.relu_grad_bias_grad(g, f, bf16=bf16)
    # backprops written over the gradients (the ABI allows it): same bits
    (dy_a, db_a), _ = au.launches(au.relu_grad_bias_grad, g, f, bf16=bf16, alias=True)
    assert_same_bits(dy_a, dy)
    assert_same_bits(db_a, db)
    # pointers one element past a 16-byte boundary: the two library kernels, each on its scalar
    # path (2 launches); same bits as that composition
    (dy_o, db_o), nl = au.launches(au.relu_grad_bias_grad, g, f, bf16=bf16, offset=1)
    assert nl == 2
    assert_same_bits(dy_o, want_dy)
    assert_same_bits(db_o, au.bias_add_grad(want_dy, bf16=bf16, offset=1))
    check_bias_grad(db_o, dy_o, bf16)


@pytest.mark.parametrize("channels,bf16", [(32, False), (12, False), (64, True)])
def test_relu_grad_bias_grad_zero_rows(channels, bf16):
    dy, db = au.relu_grad_bias_grad(np.zeros((0, channels), np.float32),
                                    np.zeros((0, channels), np.float32), bf16=bf16)
    assert dy.shape == (0, channels)
    assert_same_bits(db, np.zeros(channels, np.float32))  # +0, not NaN / -0


@pytest.mark.parametrize("channels", [32, 12])
def test_relu_grad_bias_grad_special_values(rng, channels):
    # where features <= 0 the result is g * 0: NaN for +-inf / NaN, -0 for negative g
    rows = 1024
    g = rng.uniform(-1, 1, (rows, channels)).astype(np.float32)
    f = rng.uniform(-1, 1, (rows, channels)).astype(np.float32)
    f[:, 1] = -1.0
    f[:, 2] = 0.0
    f[:, 3] = -0.0
    g[::3, 1] = np.inf
    g[1::3, 1] = -np.inf
    g[2::3, 2] = np.nan
    g[:, 3] = -np.abs(g[:, 3])
    g[::2, 0] = -0.0
    want_dy = au.relu_grad(g, f)
    dy, db = au.relu_grad_bias_grad(g, f)
    assert_same_bits(dy, want_dy)
    assert_same_bits(db, au.bias_add_grad(want_dy))
    assert np.isnan(dy[np.arange(rows) % 3 != 2, 1]).all() and np.isnan(dy[2::3, 2]).all()
    assert (bits(dy[:, 3]) == 0x80000000).all()


# =============================================================================== scaled cross-entropy
XENT_COLS = [4, 128, 132, 256, 512, 1024, 1022, 1030, 3000]
XENT_ROWS = [1, 7, 300, 4096]


def xent_inputs(rng, rows, cols):
    x = (rng.randn(rows, cols) * 2).astype(np.float32)
    lab = rng.rand(rows, cols).astype(np.float32) ** 4  # soft labels
    lab /= lab.sum(1, keepdims=True)
    lab[1::3] *= np.float32(0.7)  # rows whose labels sum to 0.7
    return x, lab.astype(np.float32)


def xent_f64(x, lab):
    x = x.astype(np.float64)
    s = x - x.max(1, keepdims=True)
    lse = np.log(np.exp(s).sum(1, keepdims=True))
    return (lab * (lse - s)).sum(1), np.exp(s - lse) - lab


@pytest.mark.parametrize("rows", XENT_ROWS)
@pytest.mark.parametrize("cols", XENT_COLS)
def test_softmax_xent_scaled_is_the_composition_bit_for_bit(rng, rows, cols):
    x, lab = xent_inputs(rng, rows, cols)
    loss, bp = au.softmax_xent(x, lab)
    (loss0, bp0), nl = au.launches(au.softmax_xent_scaled, x, lab, None)
    assert nl == 1
    assert_same_bits(loss0, loss)  # NULL scale == b200_softmax_xent
    assert_same_bits(bp0, bp)
    rloss, rbp = xent_f64(x, lab)
    np.testing.assert_allclose(loss, rloss, rtol=1e-5, atol=1e-5)
    for scale in (1.0 / rows, 0.5, -2.0):
        (sloss, sbp), nl = au.launches(au.softmax_xent_scaled, x, lab, scale)
        assert nl == 1
        assert_same_bits(sloss, loss)  # the loss does not depend on the scale
        assert_same_bits(sbp, au.mul_scalar(bp, scale))
        np.testing.assert_allclose(sbp, rbp * scale, rtol=1e-4, atol=1e-6 * abs(scale))


@pytest.mark.parametrize("cols", [128, 1024, 3000])
def test_softmax_xent_scaled_unaligned_logits(rng, cols):
    # logits one element past a 16-byte boundary: the scalar row-per-warp / block kernels
    rows = 300
    x, lab = xent_inputs(rng, rows, cols)
    loss, bp = au.softmax_xent_scaled(x, lab, None, offset=1)
    (sloss, sbp), nl = au.launches(au.softmax_xent_scaled, x, lab, 0.25, offset=1)
    assert nl == 1
    assert_same_bits(sloss, loss)
    assert_same_bits(sbp, au.mul_scalar(bp, 0.25))
    rloss, rbp = xent_f64(x, lab)
    np.testing.assert_allclose(sloss, rloss, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(sbp, rbp * 0.25, rtol=1e-4, atol=1e-6)


def test_softmax_xent_scaled_bf16_is_unimplemented(rng):
    x, lab = xent_inputs(rng, 8, 64)
    with pytest.raises(au._lib.B200Error) as e:
        au.softmax_xent_scaled(x, lab, 0.5, bf16=True)
    assert e.value.code == 12  # UNIMPLEMENTED


# =============================================================================== Sum / Mean
REDUCE_SHAPES = [(1, 1_000_003, 1), (4096, 1024, 1), (1, 4096, 1024), (33, 17, 31), (512, 196, 64),
                 (65535, 3, 5), (70000, 10, 3), (5, 0, 1), (5, 0, 7)]


@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("shape", REDUCE_SHAPES)
def test_reduce_vs_f64(oracle, rng, shape, bf16):
    x = rng.uniform(-1, 1, shape).astype(np.float32)
    if bf16:
        x = oracle.truncate_to_bf16(x)
    x64 = x.astype(np.float64)
    for scale in (1.0, 1.0 / max(shape[1], 1)):
        got, nl = au.launches(au.reduce, x, scale, bf16)
        assert nl == 1
        ref = x64.sum(1) * np.float32(scale)
        bound = TOL_EXACT * np.abs(x64).sum(1) * scale
        if bf16:
            bound = bound + 2.0 ** -8 * np.abs(ref)
        assert got.shape == ref.shape
        assert (np.abs(got - ref) <= bound).all(), np.abs(got - ref).max()
        assert_same_bits(au.reduce(x, scale, bf16), got)
    if shape[1] == 0:
        assert_same_bits(got, np.zeros(got.shape, np.float32))
