"""numpy front-end to the CPU oracle (oracle/oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; the product package never does (tests/test_abi.py greps for that).
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
# Same source built with -ffp-contract=fast (FMA): the CPU ARM bench.py times, never the checker.
ORACLE_FAST_SO = os.path.join(ORACLE_DIR, "_build", "liboracle_fast.so")

i64 = ctypes.c_int64
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_u16p = np.ctypeslib.ndpointer(dtype=np.uint16, flags="C_CONTIGUOUS")


class ConvGeom(ctypes.Structure):
    _fields_ = [("batch", i64), ("in_h", i64), ("in_w", i64), ("in_c", i64),
                ("filter_h", i64), ("filter_w", i64), ("out_c", i64),
                ("out_h", i64), ("out_w", i64),
                ("stride_h", ctypes.c_int32), ("stride_w", ctypes.c_int32),
                ("pad_top", ctypes.c_int32), ("pad_left", ctypes.c_int32)]


_lib = None
_libs = {}
_kind = "exact"


def _host_cpu():
    """What oracle/Makefile writes to _build/host.txt: CPU model + md5 of the ISA flags line."""
    try:
        out = subprocess.run(
            ["sh", "-c", '(grep -m1 "model name" /proc/cpuinfo; grep -m1 "^flags" /proc/cpuinfo | md5sum)'],
            capture_output=True, text=True, timeout=10).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def build():
    """(Re)build oracle/_build/liboracle.so when it is missing, older than its source, or was
    compiled (-march=native) on a different CPU model than the one we are running on.  In a
    read-only tree (a benchmark run from an installed checkout) the rebuild goes to a temporary
    directory instead."""
    global ORACLE_SO, ORACLE_FAST_SO
    src = os.path.join(ORACLE_DIR, "oracle.c")
    build_dir = os.path.dirname(ORACLE_SO)
    stamp = os.path.join(build_dir, "host.txt")
    built_on = open(stamp).read().strip() if os.path.exists(stamp) else None
    foreign = built_on is not None and built_on != _host_cpu()
    stale = any((not os.path.exists(so)) or
                (os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(so))
                for so in (ORACLE_SO, ORACLE_FAST_SO))
    if not (stale or foreign):
        return
    writable = os.access(build_dir if os.path.isdir(build_dir) else ORACLE_DIR, os.W_OK)
    if not writable:
        tmp = tempfile.mkdtemp(prefix="oracle-")
        atexit.register(shutil.rmtree, tmp, True)
        for f in ("Makefile", "oracle.c"):
            shutil.copy(os.path.join(ORACLE_DIR, f), tmp)
        subprocess.check_call(["make", "-C", tmp], stdout=subprocess.DEVNULL)
        ORACLE_SO = os.path.join(tmp, "_build", "liboracle.so")
        ORACLE_FAST_SO = os.path.join(tmp, "_build", "liboracle_fast.so")
        return
    if foreign:
        subprocess.check_call(["make", "-C", ORACLE_DIR, "clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", ORACLE_DIR], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        _lib = _libs.get(_kind)
    if _lib is None:
        build()
        L = ctypes.CDLL(ORACLE_FAST_SO if _kind == "fast" else ORACLE_SO)
        L.oracle_num_threads.restype = ctypes.c_int
        L.oracle_windowed_output_size.argtypes = [i64, i64, i64, ctypes.c_int] + \
            [ctypes.POINTER(i64)] * 3
        L.oracle_windowed_output_size.restype = ctypes.c_int
        L.oracle_matmul_f32.argtypes = [_f32p, _f32p, _f32p, i64, i64, i64, ctypes.c_int,
                                        ctypes.c_int]
        L.oracle_batch_matmul_f32.argtypes = [_f32p, _f32p, _f32p, i64, i64, i64, i64,
                                              ctypes.c_int, ctypes.c_int]
        L.oracle_bias_add_f32.argtypes = [_f32p, _f32p, _f32p, i64, i64]
        L.oracle_bias_add_grad_f32.argtypes = [_f32p, _f32p, i64, i64]
        L.oracle_relu_f32.argtypes = [_f32p, _f32p, i64]
        L.oracle_relu_grad_f32.argtypes = [_f32p, _f32p, _f32p, i64]
        L.oracle_softmax_f32.argtypes = [_f32p, _f32p, i64, i64, ctypes.c_int]
        L.oracle_softmax_xent_f32.argtypes = [_f32p, _f32p, _f32p, _f32p, i64, i64]
        L.oracle_max_pool_f32.argtypes = [_f32p, _f32p] + [i64] * 6 + [ctypes.c_int] * 6
        L.oracle_max_pool_grad_f32.argtypes = [_f32p, _f32p, _f32p] + [i64] * 6 + \
            [ctypes.c_int] * 6
        L.oracle_cast_f32_to_bf16.argtypes = [_f32p, _u16p, i64]
        L.oracle_cast_bf16_to_f32.argtypes = [_u16p, _f32p, i64]
        L.oracle_cast_f32_to_i32.argtypes = [_f32p, _i32p, i64]
        L.oracle_cast_i32_to_f32.argtypes = [_i32p, _f32p, i64]
        L.oracle_cast_i64_to_f32.argtypes = [_i64p, _f32p, i64]
        L.oracle_cast_f32_to_i64.argtypes = [_f32p, _i64p, i64]
        L.oracle_cast_i32_to_i64.argtypes = [_i32p, _i64p, i64]
        L.oracle_cast_i64_to_i32.argtypes = [_i64p, _i32p, i64]
        L.oracle_argmax_f32.argtypes = [_f32p, _i64p, i64, i64, i64]
        L.oracle_argmax_i32.argtypes = [_i32p, _i64p, i64, i64, i64]
        L.oracle_conv2d_f32.argtypes = [_f32p, _f32p, _f32p, ctypes.POINTER(ConvGeom)]
        L.oracle_conv2d_backprop_input_f32.argtypes = [_f32p, _f32p, _f32p,
                                                       ctypes.POINTER(ConvGeom)]
        L.oracle_conv2d_backprop_filter_f32.argtypes = [_f32p, _f32p, _f32p,
                                                        ctypes.POINTER(ConvGeom)]
        L.oracle_apply_gradient_descent_f32.argtypes = [_f32p, ctypes.c_float, _f32p, i64]
        _lib = _libs[_kind] = L
    return _lib


def select(kind):
    """"exact" (default): the bit-stable checker build.  "fast": the FMA build that bench.py's
    CPU arms time.  Returns the previous selection."""
    global _lib, _kind
    assert kind in ("exact", "fast")
    prev, _kind = _kind, kind
    _lib = None
    return prev


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def num_threads():
    return lib().oracle_num_threads()


def set_num_threads(n):
    L = lib()
    L.oracle_set_num_threads.argtypes = [ctypes.c_int]
    L.oracle_set_num_threads.restype = None
    L.oracle_set_num_threads(int(n))


def windowed_output_size(input_size, filter_size, stride, padding):
    """-> (output_size, pad_before, pad_after); padding is 'SAME' or 'VALID'."""
    o, b, a = i64(), i64(), i64()
    rc = lib().oracle_windowed_output_size(input_size, filter_size, stride,
                                           1 if padding == "SAME" else 0, o, b, a)
    if rc != 0:
        raise ValueError("invalid window arguments")
    return o.value, b.value, a.value


def matmul(a, b, transpose_a=False, transpose_b=False):
    a, b = _f32(a), _f32(b)
    m = a.shape[1] if transpose_a else a.shape[0]
    k = a.shape[0] if transpose_a else a.shape[1]
    n = b.shape[0] if transpose_b else b.shape[1]
    out = np.empty((m, n), np.float32)
    lib().oracle_matmul_f32(a, b, out, m, n, k, int(transpose_a), int(transpose_b))
    return out


def batch_matmul(x, y, adj_x=False, adj_y=False):
    x, y = _f32(x), _f32(y)
    batch = x.shape[0]
    m = x.shape[2] if adj_x else x.shape[1]
    k = x.shape[1] if adj_x else x.shape[2]
    n = y.shape[1] if adj_y else y.shape[2]
    out = np.empty((batch, m, n), np.float32)
    lib().oracle_batch_matmul_f32(x, y, out, batch, m, n, k, int(adj_x), int(adj_y))
    return out


def bias_add(x, bias):
    x, bias = _f32(x), _f32(bias)
    out = np.empty_like(x)
    lib().oracle_bias_add_f32(x, bias, out, x.size // max(bias.size, 1), bias.size)
    return out


def bias_add_grad(g):
    g = _f32(g)
    c = g.shape[-1]
    out = np.empty((c,), np.float32)
    lib().oracle_bias_add_grad_f32(g, out, g.size // max(c, 1), c)
    return out


def relu(x):
    x = _f32(x)
    out = np.empty_like(x)
    lib().oracle_relu_f32(x, out, x.size)
    return out


def relu_grad(g, f):
    g, f = _f32(g), _f32(f)
    out = np.empty_like(g)
    lib().oracle_relu_grad_f32(g, f, out, g.size)
    return out


def softmax(x, log=False):
    x = _f32(x)
    out = np.empty_like(x)
    lib().oracle_softmax_f32(x, out, x.shape[0], x.shape[1], int(log))
    return out


def softmax_xent(logits, labels):
    logits, labels = _f32(logits), _f32(labels)
    loss = np.empty((logits.shape[0],), np.float32)
    bp = np.empty_like(logits)
    lib().oracle_softmax_xent_f32(logits, labels, loss, bp, logits.shape[0], logits.shape[1])
    return loss, bp


def pool_geometry(in_shape, ksize, strides, padding):
    n, h, w, c = in_shape
    oh, pt, _ = windowed_output_size(h, ksize[0], strides[0], padding)
    ow, pl, _ = windowed_output_size(w, ksize[1], strides[1], padding)
    return oh, ow, pt, pl


def max_pool(x, ksize, strides, padding):
    x = _f32(x)
    n, h, w, c = x.shape
    oh, ow, pt, pl = pool_geometry(x.shape, ksize, strides, padding)
    out = np.empty((n, oh, ow, c), np.float32)
    lib().oracle_max_pool_f32(x, out, n, h, w, c, oh, ow, ksize[0], ksize[1], strides[0],
                              strides[1], pt, pl)
    return out


def max_pool_grad(x, grad, ksize, strides, padding):
    x, grad = _f32(x), _f32(grad)
    n, h, w, c = x.shape
    oh, ow, pt, pl = pool_geometry(x.shape, ksize, strides, padding)
    assert grad.shape == (n, oh, ow, c), (grad.shape, (n, oh, ow, c))
    out = np.empty_like(x)
    lib().oracle_max_pool_grad_f32(x, grad, out, n, h, w, c, oh, ow, ksize[0], ksize[1],
                                   strides[0], strides[1], pt, pl)
    return out


def cast_f32_to_bf16(x):
    x = _f32(x)
    out = np.empty(x.shape, np.uint16)
    lib().oracle_cast_f32_to_bf16(x, out, x.size)
    return out


def cast_bf16_to_f32(x):
    x = np.ascontiguousarray(x, np.uint16)
    out = np.empty(x.shape, np.float32)
    lib().oracle_cast_bf16_to_f32(x, out, x.size)
    return out


def truncate_to_bf16(x):
    """fp32 values that survive a float->bfloat16->float round trip (the bf16 parity inputs)."""
    return cast_bf16_to_f32(cast_f32_to_bf16(x))


_CASTS = {
    (np.float32, np.int32): "oracle_cast_f32_to_i32", (np.int32, np.float32): "oracle_cast_i32_to_f32",
    (np.int64, np.float32): "oracle_cast_i64_to_f32", (np.float32, np.int64): "oracle_cast_f32_to_i64",
    (np.int32, np.int64): "oracle_cast_i32_to_i64", (np.int64, np.int32): "oracle_cast_i64_to_i32",
}


def cast(x, dst):
    src = x.dtype.type
    x = np.ascontiguousarray(x)
    out = np.empty(x.shape, dst)
    getattr(lib(), _CASTS[(src, dst)])(x, out, x.size)
    return out


def argmax(x, axis):
    x = np.ascontiguousarray(x)
    axis = axis % x.ndim
    outer = int(np.prod(x.shape[:axis], dtype=np.int64))
    inner = int(np.prod(x.shape[axis + 1:], dtype=np.int64))
    out = np.empty(x.shape[:axis] + x.shape[axis + 1:], np.int64)
    if x.dtype == np.float32:
        lib().oracle_argmax_f32(x, out, outer, x.shape[axis], inner)
    elif x.dtype == np.int32:
        lib().oracle_argmax_i32(x, out, outer, x.shape[axis], inner)
    else:
        raise TypeError(x.dtype)
    return out


def conv_geometry(in_shape, filter_shape, strides, padding):
    """strides = [stride_h, stride_w] -> ConvGeom (out size / paddings per common_shape_fns.cc)."""
    n, h, w, c = in_shape
    r, s, c2, k = filter_shape
    assert c == c2, "input and filter must have the same depth"
    oh, pt, _ = windowed_output_size(h, r, strides[0], padding)
    ow, pl, _ = windowed_output_size(w, s, strides[1], padding)
    return ConvGeom(n, h, w, c, r, s, k, oh, ow, strides[0], strides[1], pt, pl)


def conv2d(x, f, strides, padding):
    x, f = _f32(x), _f32(f)
    g = conv_geometry(x.shape, f.shape, strides, padding)
    out = np.empty((g.batch, g.out_h, g.out_w, g.out_c), np.float32)
    lib().oracle_conv2d_f32(x, f, out, ctypes.byref(g))
    return out


def conv2d_backprop_input(in_shape, f, dy, strides, padding):
    f, dy = _f32(f), _f32(dy)
    g = conv_geometry(in_shape, f.shape, strides, padding)
    assert dy.shape == (g.batch, g.out_h, g.out_w, g.out_c), (dy.shape, g.out_h, g.out_w)
    out = np.empty(tuple(in_shape), np.float32)
    lib().oracle_conv2d_backprop_input_f32(f, dy, out, ctypes.byref(g))
    return out


def conv2d_backprop_filter(x, filter_shape, dy, strides, padding):
    x, dy = _f32(x), _f32(dy)
    g = conv_geometry(x.shape, filter_shape, strides, padding)
    assert dy.shape == (g.batch, g.out_h, g.out_w, g.out_c), (dy.shape, g.out_h, g.out_w)
    out = np.empty(tuple(filter_shape), np.float32)
    lib().oracle_conv2d_backprop_filter_f32(x, dy, out, ctypes.byref(g))
    return out


def apply_gradient_descent(var, alpha, delta):
    var = _f32(var).copy()
    lib().oracle_apply_gradient_descent_f32(var, alpha, _f32(delta), var.size)
    return var
