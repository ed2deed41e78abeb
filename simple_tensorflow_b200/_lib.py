"""ctypes binding of the C ABI declared in include/b200_ops.h (libb200tf.so).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C simple_tensorflow_b200/csrc``.
There is deliberately no fallback: if the shared object is missing, importing a symbol raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200tf.so")

# tensorflow::DataType numbering (framework/types.proto)
DT_FLOAT, DT_INT32, DT_INT64, DT_BFLOAT16 = 1, 3, 9, 14

c_void_p, c_int, c_int64, c_size_t, c_float = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_float)


class ConvGeometry(ctypes.Structure):
    """struct b200_conv2d_geometry (include/b200_ops.h)."""
    _fields_ = [
        ("batch", c_int64), ("in_h", c_int64), ("in_w", c_int64), ("in_c", c_int64),
        ("filter_h", c_int64), ("filter_w", c_int64), ("out_c", c_int64),
        ("out_h", c_int64), ("out_w", c_int64),
        ("stride_h", ctypes.c_int32), ("stride_w", ctypes.c_int32),
        ("pad_top", ctypes.c_int32), ("pad_left", ctypes.c_int32),
    ]


# name -> (restype, argtypes).  Must list EVERY symbol include/b200_ops.h declares
# (tests/test_abi.py parses the header and checks both directions).
SIGNATURES = {
    "b200_version": (ctypes.c_char_p, []),
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_device_count": (c_int, []),
    "b200_set_device": (c_int, [c_int]),
    "b200_launch_count": (ctypes.c_uint64, []),
    "b200_collective_counts": (None, [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64)]),
    "b200_profile_active": (c_int, []),
    "b200_note_launches": (None, [ctypes.c_uint64]),
    "b200_note_collectives": (None, [ctypes.c_uint64, ctypes.c_uint64]),
    "b200_stream_begin_capture": (c_int, [c_void_p]),
    "b200_stream_end_capture": (c_int, [c_void_p, ctypes.POINTER(c_void_p)]),
    "b200_graph_launch": (c_int, [c_void_p, c_void_p]),
    "b200_graph_destroy": (c_int, [c_void_p]),
    "b200_profile_begin": (c_int, []),
    "b200_profile_end": (c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64),
                                 ctypes.POINTER(ctypes.c_double)]),
    "b200_set_matmul_precision": (c_int, [c_int]),
    "b200_get_matmul_precision": (c_int, []),
    "b200_stream_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "b200_stream_create_with_priority": (c_int, [ctypes.POINTER(c_void_p), c_int]),
    "b200_stream_destroy": (c_int, [c_void_p]),
    "b200_stream_synchronize": (c_int, [c_void_p]),
    "b200_stream_wait_event": (c_int, [c_void_p, c_void_p]),
    "b200_stream_add_host_callback": (c_int, [c_void_p, c_void_p, c_void_p]),
    "b200_event_create": (c_int, [ctypes.POINTER(c_void_p)]),
    "b200_event_destroy": (c_int, [c_void_p]),
    "b200_event_record": (c_int, [c_void_p, c_void_p]),
    "b200_event_synchronize": (c_int, [c_void_p]),
    "b200_event_query": (c_int, [c_void_p]),
    "b200_event_elapsed_ms": (c_int, [c_void_p, c_void_p, ctypes.POINTER(c_float)]),
    "b200_malloc": (c_int, [ctypes.POINTER(c_void_p), c_size_t]),
    "b200_free": (c_int, [c_void_p]),
    "b200_host_malloc": (c_int, [ctypes.POINTER(c_void_p), c_size_t]),
    "b200_host_free": (c_int, [c_void_p]),
    "b200_memcpy_h2d_async": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200_memcpy_d2h_async": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200_memcpy_d2d_async": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200_memset_async": (c_int, [c_void_p, c_int, c_size_t, c_void_p]),
    "b200_mem_info": (c_int, [ctypes.POINTER(c_size_t), ctypes.POINTER(c_size_t)]),
    "b200_matmul_workspace_bytes": (c_size_t, [c_int, c_int64, c_int64, c_int64]),
    "b200_matmul": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                            c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "b200_fused_matmul": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                  c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "b200_fused_matmul_ws": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                  c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "b200_matmul_pair_workspace_bytes": (c_size_t, [c_int, c_int64, c_int64, c_int64, c_int64,
                                                    c_int64, c_int64]),
    "b200_matmul_pair": (c_int, [c_int]
                         + [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int, c_int,
                            c_void_p, c_int, c_void_p] * 2
                         + [c_void_p, c_size_t, c_void_p]),
    "b200_batch_matmul": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                  c_int64, c_int, c_int, c_void_p]),
    "b200_bias_add": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "b200_bias_add_grad_workspace_bytes": (c_size_t, [c_int, c_int64, c_int64]),
    "b200_bias_add_grad": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_void_p,
                                   c_size_t, c_void_p]),
    "b200_bias_add_nchw": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                   c_void_p]),
    "b200_bias_add_grad_nchw_workspace_bytes": (c_size_t, [c_int, c_int64, c_int64, c_int64]),
    "b200_bias_add_grad_nchw": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                        c_void_p, c_size_t, c_void_p]),
    "b200_relu": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200_relu_grad": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200_relu_grad_bias_grad_workspace_bytes": (c_size_t, [c_int, c_int64, c_int64]),
    "b200_relu_grad_bias_grad": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                         c_int64, c_void_p, c_size_t, c_void_p]),
    "b200_softmax": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p]),
    "b200_softmax_xent": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                  c_int64, c_void_p]),
    "b200_softmax_xent_scaled": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                  c_int64, c_void_p, c_void_p]),
    "b200_max_pool": (c_int, [c_int, c_void_p, c_void_p] + [c_int64] * 6 + [c_int] * 6
                      + [c_void_p]),
    "b200_max_pool_grad": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int64] * 6
                           + [c_int] * 6 + [c_void_p]),
    "b200_max_pool_grad_relu_bias_grad_workspace_bytes": (c_size_t, [c_int] + [c_int64] * 6 + [c_int] * 6),
    "b200_max_pool_grad_relu_bias_grad": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p] +
                                          [c_int64] * 6 + [c_int] * 6 +
                                          [c_void_p, c_size_t, c_void_p]),
    "b200_cast": (c_int, [c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200_argmax": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "b200_conv2d_workspace_bytes": (c_size_t, [c_int, ctypes.POINTER(ConvGeometry), c_int]),
    "b200_conv2d": (c_int, [c_int, c_void_p, c_void_p, c_void_p, ctypes.POINTER(ConvGeometry),
                            c_void_p, c_size_t, c_void_p]),
    "b200_fused_conv2d": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                  ctypes.POINTER(ConvGeometry), c_void_p, c_size_t, c_void_p]),
    "b200_conv2d_backprop_input": (c_int, [c_int, c_void_p, c_void_p, c_void_p,
                                           ctypes.POINTER(ConvGeometry), c_void_p, c_size_t,
                                           c_void_p]),
    "b200_conv2d_backprop_filter": (c_int, [c_int, c_void_p, c_void_p, c_void_p,
                                            ctypes.POINTER(ConvGeometry), c_void_p, c_size_t,
                                            c_void_p]),
    "b200_apply_gradient_descent": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64,
                                            c_void_p]),
    "b200_apply_gradient_descent_multi": (c_int, [c_int, c_int, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p]),
    "b200_mul": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "b200_batched_transpose": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "b200_add": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "b200_add_n": (c_int, [c_int, ctypes.POINTER(c_void_p), c_int, c_void_p, c_int64, c_void_p]),
    "b200_scale": (c_int, [c_int, c_void_p, c_float, c_void_p, c_int64, c_void_p]),
    "b200_reduce_sum": (c_int, [c_int, c_void_p, c_float, c_void_p, c_int64, c_void_p]),
    "b200_reduce": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_float, c_void_p]),
    "b200_nccl_unique_id": (c_int, [c_void_p]),
    "b200_nccl_comm_init_rank": (c_int, [ctypes.POINTER(c_void_p), c_int, c_void_p, c_int]),
    "b200_nccl_comm_destroy": (c_int, [c_void_p]),
    "b200_nccl_group_start": (c_int, []),
    "b200_nccl_group_end": (c_int, []),
    "b200_nccl_all_reduce": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "b200_nccl_all_reduce_sum": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "b200_nccl_comm_user_rank": (c_int, [c_void_p, ctypes.POINTER(c_int)]),
    "b200_nccl_all_gather_bytes": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "b200_peer_arena_create": (c_int, [c_void_p, c_int, c_int, c_size_t, ctypes.POINTER(c_void_p)]),
    "b200_peer_arena_backend": (ctypes.c_char_p, []),
    "b200_nvls_supported": (c_int, []),
    "b200_peer_arena_destroy": (c_int, [c_void_p]),
    "b200_peer_arena_data": (c_void_p, [c_void_p]),
    "b200_peer_arena_bytes": (c_size_t, [c_void_p]),
    "b200_peer_all_reduce": (c_int, [c_void_p, c_int, c_size_t, c_int64, c_int, c_int, c_void_p]),
}

_lib = None


class B200Error(RuntimeError):
    """A non-zero tensorflow::error::Code returned by the C ABI."""

    def __init__(self, code, message):
        super().__init__(f"[code {code}] {message}")
        self.code = code
        self.message = message


def load():
    """dlopen libb200tf.so (once) and attach the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (there is no CPU/PyTorch fallback for the B200 op kernels)")
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        if os.environ.get("B200TF_ALLOW_PARTIAL") == "1" and not hasattr(lib, name):
            continue  # developer probes against a partially built library only
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise B200Error(rc, load().b200_last_error().decode("utf-8", "replace"))
