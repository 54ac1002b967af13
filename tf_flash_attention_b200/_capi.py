"""ctypes binding of the C ABI declared in include/fa_b200.h.

Framework-neutral: everything here deals in raw pointers and sizes. The library is
built in-tree by ``tf_flash_attention_b200/csrc/Makefile`` (sm_100a only). There is
no fallback: if ``libfa_b200.so`` is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.abspath(os.path.dirname(__file__))
LIB_PATH = os.environ.get("FA_B200_LIB") or os.path.join(_HERE, "libfa_b200.so")  # env override: developer A/B builds

FA_F16, FA_F32, FA_F64, FA_BF16 = 0, 1, 2, 3
FA_RING_HANDLE_BYTES = 128
RULES = {"full": 0, "causal": 1, "local": 2}
SYNC_MODES = {"none_front": 0, "scale_front": 1, "scale_end": 2}

FA_OK = 0
FA_EINVAL_NULL = -1
FA_EINVAL_DTYPE = -2
FA_EINVAL_SEQ_DIMS = -3
FA_EINVAL_RULE = -4
FA_EINVAL_SYNC_MODE = -5
FA_EINVAL_WINDOW = -6
FA_EINVAL_STRIDE = -7
FA_EINVAL_SHAPE = -8
FA_EINVAL_WORKSPACE = -9
FA_EINVAL_RANK = -10
FA_EINVAL_CHANNEL = -11
FA_EINVAL_BATCH = -12
FA_EINVAL_SEQ_SHAPE = -13
FA_EINVAL_LAYOUT = -14
FA_ECUDA = -100
FA_LAYOUT_CHANNEL_FIRST, FA_LAYOUT_CHANNEL_LAST = 0, 1
FA_ENODEVICE = -101

PATH_NAMES = {0: "none", 1: "generic_simt", 2: "tcgen05_f16", 3: "tcgen05_f32_split", 4: "dmma_f64"}


class Problem(C.Structure):
    """Mirror of fa_problem_t."""
    _fields_ = [
        ("dtype", C.c_int32), ("seq_dims", C.c_int32), ("rule", C.c_int32),
        ("window_size", C.c_int32), ("log2_stride_size", C.c_int32), ("is_causal", C.c_int32),
        ("sync_mode", C.c_int32), ("d", C.c_int32), ("v_d", C.c_int32), ("layout", C.c_int32),
        ("batch", C.c_int64),
        ("q_shape", C.c_int32 * 2), ("k_shape", C.c_int32 * 2),
        ("q_index_base", C.c_int32), ("k_index_base", C.c_int32),
        ("q_full_len", C.c_int32), ("k_full_len", C.c_int32),
        ("accumulate", C.c_int32), ("heads", C.c_int32),
    ]


class FlashAttentionError(RuntimeError):
    """Raised for FA_ECUDA and friends (the reference raises tf.errors.InternalError)."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


class InvalidArgumentError(ValueError):
    """Raised for FA_EINVAL_* (the reference raises tf.errors.InvalidArgumentError)."""

    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make -C tf_flash_attention_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, i64 = C.c_void_p, C.c_size_t, C.c_int32, C.c_int64
    PP = C.POINTER(Problem)
    sig = {
        "fa_forward": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_backward": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_workspace_bytes": (sz, [PP, C.c_int]),
        "fa_estimate_forward_flops": (C.c_int, [PP, i32, C.POINTER(C.c_float)]),
        "fa_count_attended": (C.c_int, [PP, C.POINTER(i64)]),
        "fa_pattern_mask": (C.c_int, [PP, vp]),
        "fa_pattern_mask_fast": (C.c_int, [PP, i32, i32, vp]),
        "fa_orders": (C.c_int, [PP, vp, vp, vp]),
        "fa_classify_tiles": (C.c_int, [PP, i32, i32, vp]),
        "fa_check_forward_shapes": (C.c_int, [i32, i32, C.POINTER(i64), i32, C.POINTER(i64), i32,
                                              C.POINTER(i64), PP]),
        "fa_check_backward_shapes": (C.c_int, [i32] + [i32, C.POINTER(i64)] * 7 + [PP]),
        "fa_host_arena_bytes": (sz, [PP, C.c_int]),
        "fa_forward_host": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_backward_host": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_backward_host_resident": (C.c_int, [PP, vp, vp, vp, vp, vp, sz, vp]),
        "fa_step_host_arena_bytes": (sz, [PP]),
        "fa_forward_backward_host": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_partial_merge": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, C.c_int, vp]),
        "fa_partial_finalize": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp]),
        "fa_layout_transpose": (C.c_int, [C.c_int32, vp, vp, i64, i64, C.c_int32, C.c_int32, C.c_int, vp]),
        "fa_grad_accumulate": (C.c_int, [C.c_int32, vp, vp, i64, C.c_int, vp]),
        "fa_grad_finalize": (C.c_int, [C.c_int32, vp, vp, i64, vp]),
        "fa_backward_accumulate_supported": (C.c_int, [PP, i64]),
        "fa_backward_accumulate": (C.c_int, [PP, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, sz, vp]),
        "fa_strerror": (C.c_char_p, [C.c_int]),
        "fa_last_cuda_error": (C.c_int, []),
        "fa_last_path": (C.c_int, []),
        "fa_dispatch_path": (C.c_int, [PP, C.c_int, C.c_char_p, sz]),
        "fa_launch_count": (i64, [C.c_int]),
        "fa_set_path_override": (None, [C.c_int]),
        "fa_set_grad_precision": (C.c_int, [C.c_int]),
        "fa_kernel_timing": (None, [C.c_int]),
        "fa_kernel_timings": (C.c_int, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_float)]),
        "fa_version": (C.c_char_p, []),
        "fa_plan_stats": (C.c_int, [C.POINTER(C.c_uint64), C.c_int]),
        "fa_ring_create": (C.c_int, [i32, i32, sz, i32, C.POINTER(vp), vp]),
        "fa_ring_connect": (C.c_int, [vp, vp, vp]),
        "fa_ring_slot": (vp, [vp, i32]),
        "fa_ring_send": (C.c_int, [vp, i32, i32, C.POINTER(vp), C.POINTER(sz), i32, vp]),
        "fa_ring_recv_wait": (C.c_int, [vp, i32, vp]),
        "fa_ring_recv_release": (C.c_int, [vp, i32, vp]),
        "fa_ring_destroy": (C.c_int, [vp]),
        "fa_ring_causal_arena_bytes": (sz, [i32, i64, i32, i32, i32, i32, i32]),
        "fa_ring_causal_slot_bytes": (sz, [i32, i64, i32, i32, i32, i32]),
        "fa_ring_causal_forward": (C.c_int, [vp, i32, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "fa_ring_causal_backward": (C.c_int, [vp, vp, i32, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                              vp, sz, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, sorted(sig)


lib, EXPORTED_SYMBOLS = _load()


def strerror(status):
    return lib.fa_strerror(status).decode()


def check(status, what=""):
    if status == FA_OK:
        return
    msg = strerror(status)
    if status == FA_ECUDA:
        msg += f" [cudaError {lib.fa_last_cuda_error()}]"
    if what:
        msg = f"{what}: {msg}"
    if -99 <= status < 0:
        raise InvalidArgumentError(status, msg)
    raise FlashAttentionError(status, msg)


def _dims(shape):
    arr = (C.c_int64 * max(1, len(shape)))(*[int(s) for s in shape])
    return len(shape), arr


def make_problem(dtype_code, seq_dims, rule, sync_mode, q_shape, k_shape, v_shape,
                 window_size=1, log2_stride_size=0, is_causal=False):
    """Validates un-flattened TF-style shapes exactly as the reference forward OpKernel does
    (flash_attention_forward.cc:97-140) and returns a filled Problem."""
    p = Problem()
    p.dtype = dtype_code
    p.rule = RULES[rule]
    if sync_mode not in SYNC_MODES:
        raise InvalidArgumentError(FA_EINVAL_SYNC_MODE, f"Unsupported sync_mode: {sync_mode}")
    p.sync_mode = SYNC_MODES[sync_mode]
    p.window_size = int(window_size)
    p.log2_stride_size = int(log2_stride_size)
    p.is_causal = int(bool(is_causal))
    rq, dq = _dims(q_shape)
    rk, dk = _dims(k_shape)
    rv, dv = _dims(v_shape)
    check(lib.fa_check_forward_shapes(seq_dims, rq, dq, rk, dk, rv, dv, C.byref(p)), "shape check")
    return p


def check_backward_shapes(p, shapes):
    """shapes = (Q, K, V, O, l, m, dO) un-flattened; flash_attention_backward.cc:197-258."""
    args = []
    for s in shapes:
        r, d = _dims(s)
        args += [r, d]
    check(lib.fa_check_backward_shapes(p.seq_dims, *args, C.byref(p)), "shape check")


def dispatch_path(p, backward=False):
    """(kernel family name, reason) fa_forward / fa_backward will take for problem p (host only; fa_dispatch_path)."""
    buf = C.create_string_buffer(320)
    rc = lib.fa_dispatch_path(C.byref(p), int(backward), buf, len(buf))
    if rc < 0:
        check(rc, "fa_dispatch_path")
    return PATH_NAMES[rc], buf.value.decode()


def pattern_mask(p):
    import numpy as np
    q = int(np.prod([p.q_shape[i] for i in range(p.seq_dims)]))
    k = int(np.prod([p.k_shape[i] for i in range(p.seq_dims)]))
    out = np.zeros((q, k), dtype=np.uint8)
    check(lib.fa_pattern_mask(C.byref(p), out.ctypes.data), "fa_pattern_mask")
    return out.astype(bool)


def pattern_mask_fast(p, tile, resident_is_q):
    import numpy as np
    q = int(np.prod([p.q_shape[i] for i in range(p.seq_dims)]))
    k = int(np.prod([p.k_shape[i] for i in range(p.seq_dims)]))
    out = np.zeros((q, k), dtype=np.uint8)
    check(lib.fa_pattern_mask_fast(C.byref(p), tile, int(resident_is_q), out.ctypes.data), "fa_pattern_mask_fast")
    return out.astype(bool)


def orders(p):
    import numpy as np
    q = int(np.prod([p.q_shape[i] for i in range(p.seq_dims)]))
    k = int(np.prod([p.k_shape[i] for i in range(p.seq_dims)]))
    qo = np.zeros(q, dtype=np.int32)
    ko = np.zeros(k, dtype=np.int32)
    ref = np.zeros(2, dtype=np.int32)
    check(lib.fa_orders(C.byref(p), qo.ctypes.data, ko.ctypes.data, ref.ctypes.data), "fa_orders")
    return ref[: p.seq_dims].tolist(), qo, ko


def classify_tiles(p, tile_q, tile_k):
    import numpy as np
    q = int(np.prod([p.q_shape[i] for i in range(p.seq_dims)]))
    k = int(np.prod([p.k_shape[i] for i in range(p.seq_dims)]))
    nqt, nkt = -(-q // tile_q), -(-k // tile_k)
    out = np.zeros((nqt, nkt), dtype=np.uint8)
    check(lib.fa_classify_tiles(C.byref(p), tile_q, tile_k, out.ctypes.data), "fa_classify_tiles")
    return out


def count_attended(p):
    n = C.c_int64(0)
    check(lib.fa_count_attended(C.byref(p), C.byref(n)), "fa_count_attended")
    return n.value


def estimate_forward_flops(p, shared_mem_bytes=0):
    f = C.c_float(0)
    check(lib.fa_estimate_forward_flops(C.byref(p), shared_mem_bytes, C.byref(f)), "fa_estimate_forward_flops")
    return f.value


def kernel_timings(max_entries=4096):
    """[(kernel name, ms)] of every launch since fa_kernel_timing(1) / the last call."""
    names = (C.c_char_p * max_entries)()
    ms = (C.c_float * max_entries)()
    n = lib.fa_kernel_timings(max_entries, names, ms)
    return [(names[i].decode(), float(ms[i])) for i in range(n)]
