"""Test-side helpers that drive the C ABI (include/b200_ops.h) with numpy in / numpy out.

torch is used only as the device-memory allocator and for host<->device copies; every compute
call goes through libb200tf.so via ctypes, on torch's current CUDA stream.
"""
import ctypes

import numpy as np
import torch

from simple_tensorflow_b200 import _lib

DT = {np.dtype(np.float32): _lib.DT_FLOAT, np.dtype(np.int32): _lib.DT_INT32,
      np.dtype(np.int64): _lib.DT_INT64}
BF16 = "bf16"


def lib():
    return _lib.load()


def stream():
    return torch.cuda.current_stream().cuda_stream


def dev(a, bf16=False):
    """numpy -> CUDA tensor (bf16=True: fp32 values are converted with TRUNCATION, like Cast)."""
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if bf16:
        assert t.dtype == torch.float32
        bits = (t.view(torch.int32) >> 16).to(torch.int16)
        t = bits.view(torch.bfloat16)
    return t


def host(t):
    torch.cuda.synchronize()
    if t.dtype == torch.bfloat16:
        return t.float().cpu().numpy()
    return t.cpu().numpy()


def empty(shape, dtype=torch.float32, fill=None):
    t = torch.empty(tuple(int(s) for s in shape), dtype=dtype, device="cuda")
    if fill is not None and t.numel():
        t.fill_(fill)
    return t


def ws(nbytes):
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device="cuda")


def call(fn, *args):
    rc = fn(*args)
    if rc != 0:
        raise _lib.B200Error(rc, lib().b200_last_error().decode())


def tdt(bf16):
    return torch.bfloat16 if bf16 else torch.float32


def cdt(bf16):
    return _lib.DT_BFLOAT16 if bf16 else _lib.DT_FLOAT


def launches(fn, *args, **kwargs):
    """(fn(*args, **kwargs), kernels libb200tf.so launched during the call)."""
    L = lib()
    before = L.b200_launch_count()
    r = fn(*args, **kwargs)
    return r, L.b200_launch_count() - before


def offset_copy(a, bf16=False, offset=0):
    """Device copy of `a` that starts `offset` elements into its allocation (offset 1: a pointer
    that is NOT 16-byte aligned, every element still inside the allocation).  Returns (tensor, ptr)."""
    flat = np.ascontiguousarray(a, np.float32).ravel()
    t = dev(np.concatenate([np.zeros(offset, np.float32), flat]), bf16)
    return t, t.data_ptr() + offset * t.element_size()


def matmul(a, b, ta=False, tb=False, bf16=False, use_workspace=True, workspace_bytes=None):
    """workspace_bytes: scratch size to pass (default: what b200_matmul_workspace_bytes asks for)."""
    L = lib()
    m = a.shape[1] if ta else a.shape[0]
    k = a.shape[0] if ta else a.shape[1]
    n = b.shape[0] if tb else b.shape[1]
    da, db = dev(a, bf16), dev(b, bf16)
    out = empty((m, n), tdt(bf16), fill=float("nan"))
    nb = L.b200_matmul_workspace_bytes(cdt(bf16), m, n, k) if use_workspace else 0
    if workspace_bytes is not None:
        nb = workspace_bytes
    w = ws(nb)
    call(L.b200_matmul, cdt(bf16), da.data_ptr(), db.data_ptr(), out.data_ptr(), m, n, k, int(ta),
         int(tb), w.data_ptr() if nb else None, nb, stream())
    return host(out)


def fused_matmul(a, b, ta=False, tb=False, bias=None, relu=False, features=None, bf16=False):
    L = lib()
    m = a.shape[1] if ta else a.shape[0]
    k = a.shape[0] if ta else a.shape[1]
    n = b.shape[0] if tb else b.shape[1]
    da, db = dev(a, bf16), dev(b, bf16)
    dbias = dev(bias, bf16) if bias is not None else None
    dfeat = dev(features, bf16) if features is not None else None
    out = empty((m, n), tdt(bf16), fill=float("nan"))
    call(L.b200_fused_matmul, cdt(bf16), da.data_ptr(), db.data_ptr(), out.data_ptr(), m, n, k,
         int(ta), int(tb), dbias.data_ptr() if dbias is not None else None, int(relu),
         dfeat.data_ptr() if dfeat is not None else None, stream())
    return host(out)


def fused_matmul_ws(a, b, ta=False, tb=False, bias=None, relu=False, features=None, bf16=False,
                    workspace_bytes=None, bias_offset=0):
    """b200_fused_matmul_ws.  workspace_bytes: None = b200_matmul_workspace_bytes, 0 = no scratch.
    bias_offset: elements between the bias allocation and the pointer passed (1: unaligned bias)."""
    L = lib()
    m = a.shape[1] if ta else a.shape[0]
    k = a.shape[0] if ta else a.shape[1]
    n = b.shape[0] if tb else b.shape[1]
    da, db = dev(a, bf16), dev(b, bf16)
    pbias = None
    if bias is not None:
        dbias, pbias = offset_copy(bias, bf16, bias_offset)
    dfeat = dev(features, bf16) if features is not None else None
    out = empty((m, n), tdt(bf16), fill=float("nan"))
    nb = L.b200_matmul_workspace_bytes(cdt(bf16), m, n, k) if workspace_bytes is None else workspace_bytes
    w = ws(nb)
    call(L.b200_fused_matmul_ws, cdt(bf16), da.data_ptr(), db.data_ptr(), out.data_ptr(), m, n, k,
         int(ta), int(tb), pbias, int(relu), dfeat.data_ptr() if dfeat is not None else None,
         w.data_ptr() if nb else None, nb, stream())
    return host(out)


def batch_matmul(x, y, adj_x=False, adj_y=False, bf16=False):
    L = lib()
    batch = x.shape[0]
    m = x.shape[2] if adj_x else x.shape[1]
    k = x.shape[1] if adj_x else x.shape[2]
    n = y.shape[1] if adj_y else y.shape[2]
    dx, dy = dev(x, bf16), dev(y, bf16)
    out = empty((batch, m, n), tdt(bf16), fill=float("nan"))
    call(L.b200_batch_matmul, cdt(bf16), dx.data_ptr(), dy.data_ptr(), out.data_ptr(), batch, m, n,
         k, int(adj_x), int(adj_y), stream())
    return host(out)


def bias_add(x, b, bf16=False):
    dx, db = dev(x, bf16), dev(b, bf16)
    out = torch.empty_like(dx)
    call(lib().b200_bias_add, cdt(bf16), dx.data_ptr(), db.data_ptr(), out.data_ptr(),
         x.size // max(b.size, 1), b.size, stream())
    return host(out)


def bias_add_grad(g, bf16=False, offset=0):
    """offset: elements between the gradient's allocation and the pointer passed."""
    L = lib()
    c = g.shape[-1]
    rows = g.size // max(c, 1)
    dg, pg = offset_copy(g, bf16, offset)
    out = empty((c,), tdt(bf16), fill=float("nan"))
    nb = L.b200_bias_add_grad_workspace_bytes(cdt(bf16), rows, c)
    w = ws(nb)
    call(L.b200_bias_add_grad, cdt(bf16), pg, out.data_ptr(), rows, c, w.data_ptr(), nb, stream())
    return host(out)


def relu_grad_bias_grad(g, f, bf16=False, offset=0, alias=False):
    """b200_relu_grad_bias_grad on [rows, channels] = g.shape -> (backprops, bias_grad).
    offset: elements between each allocation and the pointer passed; alias: backprops written over
    the gradients buffer."""
    L = lib()
    c = g.shape[-1]
    rows = g.size // max(c, 1)
    dg, pg = offset_copy(g, bf16, offset)
    df, pf = offset_copy(f, bf16, offset)
    if alias:
        dbp, pbp = dg, pg
    else:
        dbp = empty((g.size + offset,), tdt(bf16), fill=float("nan"))
        pbp = dbp.data_ptr() + offset * dbp.element_size()
    out = empty((c,), tdt(bf16), fill=float("nan"))
    nb = L.b200_relu_grad_bias_grad_workspace_bytes(cdt(bf16), rows, c)
    w = ws(nb)
    call(L.b200_relu_grad_bias_grad, cdt(bf16), pg, pf, pbp, out.data_ptr(), rows, c, w.data_ptr(),
         nb, stream())
    return host(dbp)[offset:].reshape(g.shape), host(out)


def bias_add_nchw(x, b, bf16=False):
    """x: [batch dims..., C, H, W] (GetBiasValueDims, bias_op.cc:140-150)."""
    c, image = x.shape[-3], x.shape[-2] * x.shape[-1]
    batch = x.size // max(c * image, 1)
    dx, db = dev(x, bf16), dev(b, bf16)
    out = torch.empty_like(dx)
    call(lib().b200_bias_add_nchw, cdt(bf16), dx.data_ptr(), db.data_ptr(), out.data_ptr(), batch,
         c, image, stream())
    return host(out)


def bias_add_grad_nchw(g, bf16=False):
    L = lib()
    c, image = g.shape[-3], g.shape[-2] * g.shape[-1]
    batch = g.size // max(c * image, 1)
    dg = dev(g, bf16)
    out = empty((c,), tdt(bf16), fill=float("nan"))
    nb = L.b200_bias_add_grad_nchw_workspace_bytes(cdt(bf16), batch, c, image)
    w = ws(nb)
    call(L.b200_bias_add_grad_nchw, cdt(bf16), dg.data_ptr(), out.data_ptr(), batch, c, image,
         w.data_ptr(), nb, stream())
    return host(out)


def relu(x, bf16=False):
    dx = dev(x, bf16)
    out = torch.empty_like(dx)
    call(lib().b200_relu, cdt(bf16), dx.data_ptr(), out.data_ptr(), x.size, stream())
    return host(out)


def relu_grad(g, f, bf16=False):
    dg, df = dev(g, bf16), dev(f, bf16)
    out = torch.empty_like(dg)
    call(lib().b200_relu_grad, cdt(bf16), dg.data_ptr(), df.data_ptr(), out.data_ptr(), g.size,
         stream())
    return host(out)


def softmax(x, log=False, bf16=False):
    dx = dev(x, bf16)
    out = torch.empty_like(dx)
    call(lib().b200_softmax, cdt(bf16), dx.data_ptr(), out.data_ptr(), x.shape[0], x.shape[1],
         int(log), stream())
    return host(out)


def softmax_xent(logits, labels, bf16=False):
    dl, dlab = dev(logits, bf16), dev(labels, bf16)
    loss = empty((logits.shape[0],), tdt(bf16), fill=float("nan"))
    bp = torch.empty_like(dl)
    call(lib().b200_softmax_xent, cdt(bf16), dl.data_ptr(), dlab.data_ptr(), loss.data_ptr(),
         bp.data_ptr(), logits.shape[0], logits.shape[1], stream())
    return host(loss), host(bp)


def softmax_xent_scaled(logits, labels, scale, bf16=False, offset=0):
    """b200_softmax_xent_scaled; scale: a float (uploaded as a device scalar) or None (NULL).
    offset: elements between the logits allocation and the pointer passed."""
    rows, cols = logits.shape
    dl, pl = offset_copy(logits, bf16, offset)
    dlab = dev(labels, bf16)
    dsc = dev(np.array([scale], np.float32)) if scale is not None else None
    loss = empty((rows,), tdt(bf16), fill=float("nan"))
    bp = empty((rows, cols), tdt(bf16), fill=float("nan"))
    call(lib().b200_softmax_xent_scaled, cdt(bf16), pl, dlab.data_ptr(), loss.data_ptr(),
         bp.data_ptr(), rows, cols, dsc.data_ptr() if dsc is not None else None, stream())
    return host(loss), host(bp)


def mul_scalar(x, y, bf16=False):
    """b200_mul with y a device scalar broadcast over x."""
    dx, dy = dev(x, bf16), dev(np.array([y], np.float32), bf16)
    out = empty(x.shape, tdt(bf16), fill=float("nan"))
    call(lib().b200_mul, cdt(bf16), dx.data_ptr(), dy.data_ptr(), out.data_ptr(), x.size, 1,
         stream())
    return host(out)


def reduce(x, scale=1.0, bf16=False):
    """b200_reduce over axis 1 of x viewed as [outer, reduce, inner] -> [outer, inner]."""
    outer, red, inner = x.shape
    dx = dev(x, bf16) if x.size else ws(16)
    out = empty((outer, inner), tdt(bf16), fill=float("nan"))
    call(lib().b200_reduce, cdt(bf16), dx.data_ptr(), out.data_ptr(), outer, red, inner, scale,
         stream())
    return host(out)


def max_pool(x, ksize, strides, padding, oracle, bf16=False):
    n, h, w, c = x.shape
    oh, ow, pt, pl = pool_geometry(x.shape, ksize, strides, padding)
    dx = dev(x, bf16)
    out = empty((n, oh, ow, c), tdt(bf16), fill=float("nan"))
    call(lib().b200_max_pool, cdt(bf16), dx.data_ptr(), out.data_ptr(), n, h, w, c, oh, ow,
         ksize[0], ksize[1], strides[0], strides[1], pt, pl, stream())
    return host(out)


def max_pool_grad(x, grad, ksize, strides, padding, oracle, bf16=False):
    n, h, w, c = x.shape
    oh, ow, pt, pl = pool_geometry(x.shape, ksize, strides, padding)
    dx, dg = dev(x, bf16), dev(grad, bf16)
    out = empty(x.shape, tdt(bf16), fill=float("nan"))
    call(lib().b200_max_pool_grad, cdt(bf16), dx.data_ptr(), None, dg.data_ptr(), out.data_ptr(), n,
         h, w, c, oh, ow, ksize[0], ksize[1], strides[0], strides[1], pt, pl, stream())
    return host(out)


def max_pool_grad_relu_bias_grad(x, grad, ksize, strides, padding, bf16=False):
    """Returns (backprops, bias_grad), or None when the geometry is outside the fused kernel."""
    L = lib()
    n, h, w, c = x.shape
    oh, ow, pt, pl = pool_geometry(x.shape, ksize, strides, padding)
    geo = (n, h, w, c, oh, ow, ksize[0], ksize[1], strides[0], strides[1], pt, pl)
    nb = L.b200_max_pool_grad_relu_bias_grad_workspace_bytes(cdt(bf16), *geo)
    if nb == 0:
        return None
    dx, dg = dev(x, bf16), dev(grad, bf16)
    out = empty(x.shape, tdt(bf16), fill=float("nan"))
    db = empty((c,), tdt(bf16), fill=float("nan"))
    wk = ws(nb)
    call(L.b200_max_pool_grad_relu_bias_grad, cdt(bf16), dx.data_ptr(), dg.data_ptr(), out.data_ptr(),
         db.data_ptr(), *geo, wk.data_ptr(), nb, stream())
    return host(out), host(db)


def cast(x, src, dst):
    """src/dst: numpy dtypes or the string 'bf16' (bf16 travels as uint16 bit patterns)."""
    L = lib()
    code = lambda d: _lib.DT_BFLOAT16 if d == BF16 else DT[np.dtype(d)]
    tdst = torch.int16 if dst == BF16 else {np.float32: torch.float32, np.int32: torch.int32,
                                            np.int64: torch.int64}[dst]
    dx = torch.from_numpy(np.ascontiguousarray(x).view(np.int16) if src == BF16
                          else np.ascontiguousarray(x)).cuda()
    out = torch.empty(x.shape, dtype=tdst, device="cuda")
    call(L.b200_cast, code(src), code(dst), dx.data_ptr(), out.data_ptr(), x.size, stream())
    r = host(out)
    return r.view(np.uint16) if dst == BF16 else r


def argmax(x, axis):
    axis = axis % x.ndim
    outer = int(np.prod(x.shape[:axis], dtype=np.int64))
    inner = int(np.prod(x.shape[axis + 1:], dtype=np.int64))
    dx = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    out = torch.full(x.shape[:axis] + x.shape[axis + 1:], -1, dtype=torch.int64, device="cuda")
    call(lib().b200_argmax, DT[x.dtype], dx.data_ptr(), out.data_ptr(), outer, x.shape[axis], inner,
         stream())
    return host(out)


def windowed(in_size, filt, stride, padding):
    """SAME / VALID output size and leading pad, restated here from the documented rule
    (core/framework/common_shape_fns.cc:19-47) INDEPENDENTLY of the oracle and of the product's
    padding.h, so that the raw C-ABI tests do not take their geometry from the thing they check:
    VALID: out = ceil((in - filt + 1) / stride), no padding;  SAME: out = ceil(in / stride),
    total pad = max((out - 1) * stride + filt - in, 0), the smaller half goes in front."""
    if padding == "VALID":
        return -(-(in_size - filt + 1) // stride), 0
    out = -(-in_size // stride)
    total = max((out - 1) * stride + filt - in_size, 0)
    return out, total // 2


def _geom(oracle, in_shape, filter_shape, strides, padding):
    n, h, w, c = in_shape
    r, s, c2, k = filter_shape
    assert c == c2
    oh, pt = windowed(h, r, strides[0], padding)
    ow, pl = windowed(w, s, strides[1], padding)
    return _lib.ConvGeometry(n, h, w, c, r, s, k, oh, ow, strides[0], strides[1], pt, pl)


def pool_geometry(in_shape, ksize, strides, padding):
    n, h, w, c = in_shape
    oh, pt = windowed(h, ksize[0], strides[0], padding)
    ow, pl = windowed(w, ksize[1], strides[1], padding)
    return oh, ow, pt, pl


def conv2d(x, f, strides, padding, oracle, bf16=False):
    L = lib()
    g = _geom(oracle, x.shape, f.shape, strides, padding)
    dx, df = dev(x, bf16), dev(f, bf16)
    out = empty((g.batch, g.out_h, g.out_w, g.out_c), tdt(bf16), fill=float("nan"))
    nb = L.b200_conv2d_workspace_bytes(cdt(bf16), ctypes.byref(g), 0)
    w = ws(nb)
    call(L.b200_conv2d, cdt(bf16), dx.data_ptr(), df.data_ptr(), out.data_ptr(), ctypes.byref(g),
         w.data_ptr(), nb, stream())
    return host(out)


def fused_conv2d(x, f, bias, relu, strides, padding, oracle, bf16=False):
    """b200_fused_conv2d (bias may be None) with the workspace b200_conv2d would get."""
    L = lib()
    g = _geom(oracle, x.shape, f.shape, strides, padding)
    dx, df = dev(x, bf16), dev(f, bf16)
    dbias = dev(bias, bf16) if bias is not None else None
    out = empty((g.batch, g.out_h, g.out_w, g.out_c), tdt(bf16), fill=float("nan"))
    nb = L.b200_conv2d_workspace_bytes(cdt(bf16), ctypes.byref(g), 0)
    w = ws(nb)
    call(L.b200_fused_conv2d, cdt(bf16), dx.data_ptr(), df.data_ptr(),
         dbias.data_ptr() if dbias is not None else None, int(relu), out.data_ptr(),
         ctypes.byref(g), w.data_ptr(), nb, stream())
    return host(out)


def conv2d_backprop_input(in_shape, f, dy, strides, padding, oracle, bf16=False):
    L = lib()
    g = _geom(oracle, in_shape, f.shape, strides, padding)
    df, ddy = dev(f, bf16), dev(dy, bf16)
    out = empty(in_shape, tdt(bf16), fill=float("nan"))
    nb = L.b200_conv2d_workspace_bytes(cdt(bf16), ctypes.byref(g), 1)
    w = ws(nb)
    call(L.b200_conv2d_backprop_input, cdt(bf16), df.data_ptr(), ddy.data_ptr(), out.data_ptr(),
         ctypes.byref(g), w.data_ptr(), nb, stream())
    return host(out)


def conv2d_backprop_filter(x, filter_shape, dy, strides, padding, oracle, bf16=False):
    L = lib()
    g = _geom(oracle, x.shape, filter_shape, strides, padding)
    dx, ddy = dev(x, bf16), dev(dy, bf16)
    out = empty(filter_shape, tdt(bf16), fill=float("nan"))
    nb = L.b200_conv2d_workspace_bytes(cdt(bf16), ctypes.byref(g), 2)
    w = ws(nb)
    call(L.b200_conv2d_backprop_filter, cdt(bf16), dx.data_ptr(), ddy.data_ptr(), out.data_ptr(),
         ctypes.byref(g), w.data_ptr(), nb, stream())
    return host(out)


def rel_err(got, ref):
    """max |got - ref| / max |ref| : the 'relative fp32' measure of the 1e-2 parity bar."""
    ref = np.asarray(ref, np.float64)
    got = np.asarray(got, np.float64)
    denom = max(float(np.max(np.abs(ref))) if ref.size else 0.0, 1e-30)
    return float(np.max(np.abs(got - ref))) / denom if ref.size else 0.0
