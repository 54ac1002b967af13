'''
Drop-in mirror of the reference's public module ``flash_attention/flash_attention.py``:
the same six entry points, argument names, defaults and return convention

  full_1d(Q, K, V, sync_mode='none_front', returning_l_m=False)          reference :80
  causal_1d(Q, K, V, sync_mode, returning_l_m=False)                      reference :122
  local_1d(Q, K, V, window_size, log2_stride_size, is_causal, sync_mode,  reference :163
           returning_l_m=False)
  full_2d / causal_2d / local_2d                                          reference :219,266,312

with the same channel-first layouts ``batch_shape + (channel, sequence...)``, the same
dtypes (float16 / float32 / float64; ``l`` is float32 for float16 inputs) plus bfloat16 for
torch tensors (``l`` float32, as for float16; NumPy has no bfloat16), and the
registered gradient (only ``dO`` is propagated; gradients of ``l`` and ``m`` are
ignored, reference :374-390).

TensorFlow is not available in this image, so tensors are ``torch`` CUDA tensors (device
memory + stream plumbing only; every computation happens in libfa_b200.so behind the C
ABI of include/fa_b200.h) or host ``numpy`` arrays (staged through the C ABI's host-buffer
entry points). The TensorFlow OpKernel shim that registers the reference's 30 ops on top
of the same C ABI lives in ``csrc/tf_ops`` (see INTEGRATION.md).

Masking rules and sync modes are documented in the reference module docstring
(reference :1-69); the attended pattern is bit-identical (tests/test_pattern_*.py).
'''
import ctypes as C

import numpy as np

from . import _capi

try:  # torch is plumbing (device memory, streams, autograd glue), not the product
    import torch
except Exception:  # pragma: no cover
    torch = None

_NP_DTYPES = {np.dtype(np.float16): _capi.FA_F16, np.dtype(np.float32): _capi.FA_F32,
              np.dtype(np.float64): _capi.FA_F64}
_NP_L_DTYPE = {_capi.FA_F16: np.float32, _capi.FA_F32: np.float32, _capi.FA_F64: np.float64}


def _torch_codes():
    return {torch.float16: _capi.FA_F16, torch.float32: _capi.FA_F32, torch.float64: _capi.FA_F64,
            torch.bfloat16: _capi.FA_BF16}


def _l_dtype(dtype):
    """dtype of ``l`` for inputs of `dtype`: float32 for the 16-bit types"""
    return torch.float32 if dtype in (torch.float16, torch.bfloat16) else dtype


def _is_torch(x):
    return torch is not None and isinstance(x, torch.Tensor)


def _dtype_code(x):
    if _is_torch(x):
        codes = _torch_codes()
        if x.dtype not in codes:
            raise _capi.InvalidArgumentError(-2, f"unsupported dtype {x.dtype}")
        return codes[x.dtype]
    dt = np.asarray(x).dtype
    if dt not in _NP_DTYPES:
        raise _capi.InvalidArgumentError(-2, f"unsupported dtype {dt}")
    return _NP_DTYPES[dt]


LAYOUTS = ('channel_first', 'channel_last')


def _cf_shape(shape, seq_dims):
    """channel-last outer + seq + (heads, channels) -> the channel-first shape outer + (heads, channels) + seq"""
    shape = tuple(shape)
    if len(shape) < seq_dims + 2:
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_RANK, "channel-last tensors are outer + sequence + (heads, channels)")
    n = len(shape)
    return shape[: n - seq_dims - 2] + shape[n - 2:] + shape[n - seq_dims - 2: n - 2]


def _problem(seq_dims, rule, Q, K, V, sync_mode, window_size=1, log2_stride_size=0, is_causal=False,
             layout='channel_first'):
    code = _dtype_code(Q)
    if _dtype_code(K) != code or _dtype_code(V) != code:
        raise _capi.InvalidArgumentError(-2, "Q, K and V must have the same dtype")
    if layout not in LAYOUTS:
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_LAYOUT, f"layout must be one of {LAYOUTS}")
    shapes = [tuple(x.shape) for x in (Q, K, V)]
    if layout == 'channel_last':
        shapes = [_cf_shape(sh, seq_dims) for sh in shapes]
    p = _capi.make_problem(code, seq_dims, rule, sync_mode, shapes[0], shapes[1], shapes[2],
                           window_size, log2_stride_size, is_causal)
    if layout == 'channel_last':
        p.layout = _capi.FA_LAYOUT_CHANNEL_LAST
        p.heads = int(Q.shape[-2])
    return p


def _out_shapes(p, Q, V):
    sd = p.seq_dims
    qs = tuple(Q.shape)
    if p.layout == _capi.FA_LAYOUT_CHANNEL_LAST:   # O: outer + seq + (heads, v_d); l, m: outer + (heads,) + seq
        outer, seq = qs[: len(qs) - sd - 2], qs[len(qs) - sd - 2: len(qs) - 2]
        return outer + seq + (qs[-2], p.v_d), outer + (qs[-2],) + seq
    batch, seq = qs[: len(qs) - sd - 1], qs[len(qs) - sd:]
    return batch + (p.v_d,) + seq, batch + seq


def _cl_to_cf(x, seq_dims):
    """channel-last tensor of any outer rank / 1-D or 2-D sequence -> channel-first, through the adapter kernel"""
    sh = tuple(x.shape)
    n = len(sh)
    outer, seq = sh[: n - seq_dims - 2], sh[n - seq_dims - 2: n - 2]
    y = from_channel_last(x.reshape((int(np.prod(outer, dtype=np.int64)), int(np.prod(seq, dtype=np.int64))) + sh[-2:]))
    return y.reshape(outer + sh[-2:] + seq)


def _cf_to_cl(x, seq_dims):
    sh = tuple(x.shape)
    n = len(sh)
    outer, hc, seq = sh[: n - seq_dims - 2], sh[n - seq_dims - 2: n - seq_dims], sh[n - seq_dims:]
    y = to_channel_last(x.reshape((int(np.prod(outer, dtype=np.int64)),) + hc + (int(np.prod(seq, dtype=np.int64)),)))
    return y.reshape(outer + seq + hc)


def _channel_first_problem(p):
    q = _capi.Problem.from_buffer_copy(p)
    q.layout, q.heads = _capi.FA_LAYOUT_CHANNEL_FIRST, 0
    return q


# ------------------------------------------------------------------------------------ #
# device path (torch CUDA tensors)
# ------------------------------------------------------------------------------------ #
_ws_cache = {}


def _workspace(nbytes, device):
    if nbytes == 0:
        return None, 0
    key = (device.index, torch.cuda.current_stream(device).cuda_stream)
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf, buf.numel()


def _forward_device(p, Q, K, V, out=None):
    if not Q.is_cuda:
        raise _capi.FlashAttentionError(-101, "torch inputs must live on a CUDA device (no CPU fallback)")
    Q, K, V = Q.contiguous(), K.contiguous(), V.contiguous()
    o_shape, lm_shape = _out_shapes(p, Q, V)
    l_dtype = _l_dtype(Q.dtype)
    if out is None:
        O = torch.empty(o_shape, dtype=Q.dtype, device=Q.device)
        l = torch.empty(lm_shape, dtype=l_dtype, device=Q.device)
        m = torch.empty(lm_shape, dtype=Q.dtype, device=Q.device)
    else:
        O, l, m = out
    with torch.cuda.device(Q.device):
        ws, ws_bytes = _workspace(_capi.lib.fa_workspace_bytes(C.byref(p), 0), Q.device)
        stream = torch.cuda.current_stream(Q.device).cuda_stream
        rc = _capi.lib.fa_forward(C.byref(p), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(),
                                  l.data_ptr(), m.data_ptr(), ws.data_ptr() if ws is not None else None,
                                  ws_bytes, stream)
    if rc == _capi.FA_EINVAL_LAYOUT and p.layout == _capi.FA_LAYOUT_CHANNEL_LAST and out is None:
        # no kernel reads this dtype / shape channel-last: the adapter pass either side of the channel-first op
        sd = p.seq_dims
        Oc, l, m = _forward_device(_channel_first_problem(p), *(_cl_to_cf(t, sd) for t in (Q, K, V)))
        return _cf_to_cl(Oc, sd), l, m
    _capi.check(rc, "fa_forward")
    return O, l, m


def _backward_device(p, Q, K, V, O, l, m, dO):
    Q, K, V, O, l, m, dO = (t.contiguous() for t in (Q, K, V, O, l, m, dO))
    shapes = [tuple(t.shape) for t in (Q, K, V, O, l, m, dO)]
    if p.layout == _capi.FA_LAYOUT_CHANNEL_LAST:
        shapes = [sh if i in (4, 5) else _cf_shape(sh, p.seq_dims) for i, sh in enumerate(shapes)]
    _capi.check_backward_shapes(p, shapes)
    dQ, dK, dV = torch.empty_like(Q), torch.empty_like(K), torch.empty_like(V)
    with torch.cuda.device(Q.device):
        ws, ws_bytes = _workspace(_capi.lib.fa_workspace_bytes(C.byref(p), 1), Q.device)
        stream = torch.cuda.current_stream(Q.device).cuda_stream
        rc = _capi.lib.fa_backward(C.byref(p), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(),
                                   l.data_ptr(), m.data_ptr(), dO.data_ptr(), dQ.data_ptr(), dK.data_ptr(),
                                   dV.data_ptr(), ws.data_ptr() if ws is not None else None, ws_bytes, stream)
    if rc == _capi.FA_EINVAL_LAYOUT and p.layout == _capi.FA_LAYOUT_CHANNEL_LAST:
        sd = p.seq_dims
        Qc, Kc, Vc, Oc, dOc = (_cl_to_cf(t, sd) for t in (Q, K, V, O, dO))
        return tuple(_cf_to_cl(g, sd) for g in _backward_device(_channel_first_problem(p), Qc, Kc, Vc, Oc, l, m, dOc))
    _capi.check(rc, "fa_backward")
    return dQ, dK, dV


if torch is not None:
    class _AttentionFn(torch.autograd.Function):
        """The registered gradient (reference: RegisterGradient on the 12 forward ops,
        flash_attention.py:392-471, fed by _compute_gradients :374-390)."""

        @staticmethod
        def forward(ctx, Q, K, V, p):
            O, l, m = _forward_device(p, Q, K, V)
            ctx.save_for_backward(Q, K, V, O, l, m)
            ctx.problem = p
            ctx.mark_non_differentiable(l, m)
            return O, l, m

        @staticmethod
        def backward(ctx, dO, _dl, _dm):
            Q, K, V, O, l, m = ctx.saved_tensors
            dQ, dK, dV = _backward_device(ctx.problem, Q, K, V, O, l, m, dO)
            return dQ, dK, dV, None


# ------------------------------------------------------------------------------------ #
# host path (numpy arrays): copies inside the C ABI call
# ------------------------------------------------------------------------------------ #
_arena = {}


def _device_arena(nbytes):
    if torch is None or not torch.cuda.is_available():
        raise _capi.FlashAttentionError(-101, "no CUDA device available (there is no CPU fallback)")
    buf = _arena.get("buf")
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        _arena["buf"] = buf
    return buf


def _forward_host(p, Q, K, V):
    Q, K, V = (np.ascontiguousarray(x) for x in (Q, K, V))
    o_shape, lm_shape = _out_shapes(p, Q, V)
    O = np.empty(o_shape, dtype=Q.dtype)
    l = np.empty(lm_shape, dtype=_NP_L_DTYPE[p.dtype])
    m = np.empty(lm_shape, dtype=Q.dtype)
    nbytes = _capi.lib.fa_host_arena_bytes(C.byref(p), 0)
    arena = _device_arena(nbytes)
    rc = _capi.lib.fa_forward_host(C.byref(p), Q.ctypes.data, K.ctypes.data, V.ctypes.data, O.ctypes.data,
                                   l.ctypes.data, m.ctypes.data, arena.data_ptr(), arena.numel(),
                                   torch.cuda.current_stream().cuda_stream)
    _capi.check(rc, "fa_forward_host")
    return O, l, m


def backward_host(p, Q, K, V, O, l, m, dO):
    """Host-buffer backward (numpy in, numpy out)."""
    Q, K, V, O, l, m, dO = (np.ascontiguousarray(x) for x in (Q, K, V, O, l, m, dO))
    _capi.check_backward_shapes(p, [x.shape for x in (Q, K, V, O, l, m, dO)])
    dQ, dK, dV = np.empty_like(Q), np.empty_like(K), np.empty_like(V)
    arena = _device_arena(_capi.lib.fa_host_arena_bytes(C.byref(p), 1))
    rc = _capi.lib.fa_backward_host(C.byref(p), Q.ctypes.data, K.ctypes.data, V.ctypes.data, O.ctypes.data,
                                    l.ctypes.data, m.ctypes.data, dO.ctypes.data, dQ.ctypes.data,
                                    dK.ctypes.data, dV.ctypes.data, arena.data_ptr(), arena.numel(),
                                    torch.cuda.current_stream().cuda_stream)
    _capi.check(rc, "fa_backward_host")
    return dQ, dK, dV


def _attend(p, Q, K, V, returning_l_m):
    if p.layout != _capi.FA_LAYOUT_CHANNEL_FIRST and not _is_torch(Q):
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_LAYOUT, "channel-last operands are torch CUDA tensors")
    if _is_torch(Q):
        if torch.is_grad_enabled() and (Q.requires_grad or K.requires_grad or V.requires_grad):
            results = _AttentionFn.apply(Q, K, V, p)
        else:
            results = _forward_device(p, Q, K, V)
    else:
        results = _forward_host(p, Q, K, V)
    return results if returning_l_m else results[0]


# ------------------------------------------------------------------------------------ #
# public API — same names, argument order and defaults as the reference
# ------------------------------------------------------------------------------------ #
# `layout` (keyword only, not in the reference): 'channel_last' takes Q, K, V as outer + sequence + (heads, channels) -
# what a projection produces - and returns O the same way (l, m: outer + (heads,) + sequence). The fp16 / bf16
# tensor-core kernels read and write that layout directly through their TMA descriptors (SURVEY.md section 8 f3); other dtypes /
# shapes go through the adapter kernel either side of the channel-first op.
def full_1d(Q, K, V, sync_mode='none_front', returning_l_m=False, *, layout='channel_first'):
    '''Full attention (no masking) on 1d sequences. Reference: flash_attention.py:80-119.'''
    return _attend(_problem(1, 'full', Q, K, V, sync_mode, layout=layout), Q, K, V, returning_l_m)


def causal_1d(Q, K, V, sync_mode, returning_l_m=False, *, layout='channel_first'):
    '''Causal attention on 1d sequences. Reference: flash_attention.py:122-160.'''
    return _attend(_problem(1, 'causal', Q, K, V, sync_mode, layout=layout), Q, K, V, returning_l_m)


def local_1d(Q, K, V, window_size, log2_stride_size, is_causal, sync_mode, returning_l_m=False, *,
             layout='channel_first'):
    '''Local attention on 1d sequences; window length 2*window_size-1, stride 2**log2_stride_size.
    Reference: flash_attention.py:163-216.'''
    return _attend(_problem(1, 'local', Q, K, V, sync_mode, window_size, log2_stride_size, is_causal, layout),
                   Q, K, V, returning_l_m)


def full_2d(Q, K, V, sync_mode='none_front', returning_l_m=False, *, layout='channel_first'):
    '''Full attention on 2d sequences. Reference: flash_attention.py:219-263.'''
    return _attend(_problem(2, 'full', Q, K, V, sync_mode, layout=layout), Q, K, V, returning_l_m)


def causal_2d(Q, K, V, sync_mode, returning_l_m=False, *, layout='channel_first'):
    '''Causal attention on 2d sequences (row-major order). Reference: flash_attention.py:266-309.'''
    return _attend(_problem(2, 'causal', Q, K, V, sync_mode, layout=layout), Q, K, V, returning_l_m)


def local_2d(Q, K, V, window_size, log2_stride_size, is_causal, sync_mode, returning_l_m=False, *,
             layout='channel_first'):
    '''Local attention on 2d sequences. Reference: flash_attention.py:312-370.'''
    return _attend(_problem(2, 'local', Q, K, V, sync_mode, window_size, log2_stride_size, is_causal, layout),
                   Q, K, V, returning_l_m)


# backward ops, callable directly like the reference's `_fa_kernel.*_attention_backward{1,2}d[_float16]`
def attention_backward(seq_dims, rule, Q, K, V, O, l, m, dO, sync_mode, window_size=1, log2_stride_size=0,
                       is_causal=False, *, layout='channel_first'):
    p = _problem(seq_dims, rule, Q, K, V, sync_mode, window_size, log2_stride_size, is_causal, layout)
    if _is_torch(Q):
        return _backward_device(p, Q, K, V, O, l, m, dO)
    return backward_host(p, Q, K, V, O, l, m, dO)


def forward_backward_host(seq_dims, rule, Q, K, V, dO, sync_mode, window_size=1, log2_stride_size=0, is_causal=False,
                          pipelined=True):
    """One training step on host (NumPy) buffers: forward, then the registered backward. Q, K, V and dO cross PCIe once
    on the way in, O, l, m, dQ, dK, dV once on the way out. `pipelined` (default): one `fa_forward_backward_host` call
    that overlaps uploads, kernels and downloads of successive batch chunks; otherwise `fa_forward_host` followed by
    `fa_backward_host_resident` in one arena (the forward's tensors stay on the device for the gradient).
    Returns (O, l, m, dQ, dK, dV)."""
    p = _problem(seq_dims, rule, Q, K, V, sync_mode, window_size, log2_stride_size, is_causal)
    Q, K, V, dO = (np.ascontiguousarray(x) for x in (Q, K, V, dO))
    o_shape, lm_shape = _out_shapes(p, Q, V)
    if tuple(dO.shape) != tuple(o_shape):
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_SEQ_SHAPE, f"dO has shape {dO.shape}, expected {o_shape}")
    O = np.empty(o_shape, dtype=Q.dtype)
    l = np.empty(lm_shape, dtype=_NP_L_DTYPE[p.dtype])
    m = np.empty(lm_shape, dtype=Q.dtype)
    dQ, dK, dV = np.empty_like(Q), np.empty_like(K), np.empty_like(V)
    stream = torch.cuda.current_stream().cuda_stream
    if pipelined:
        arena = _device_arena(_capi.lib.fa_step_host_arena_bytes(C.byref(p)))
        _capi.check(_capi.lib.fa_forward_backward_host(C.byref(p), Q.ctypes.data, K.ctypes.data, V.ctypes.data,
                                                       dO.ctypes.data, O.ctypes.data, l.ctypes.data, m.ctypes.data,
                                                       dQ.ctypes.data, dK.ctypes.data, dV.ctypes.data, arena.data_ptr(),
                                                       arena.numel(), stream), "fa_forward_backward_host")
        return O, l, m, dQ, dK, dV
    arena = _device_arena(_capi.lib.fa_host_arena_bytes(C.byref(p), 1))
    _capi.check(_capi.lib.fa_forward_host(C.byref(p), Q.ctypes.data, K.ctypes.data, V.ctypes.data, O.ctypes.data,
                                          l.ctypes.data, m.ctypes.data, arena.data_ptr(), arena.numel(), stream),
                "fa_forward_host")
    _capi.check(_capi.lib.fa_backward_host_resident(C.byref(p), dO.ctypes.data, dQ.ctypes.data, dK.ctypes.data,
                                                    dV.ctypes.data, arena.data_ptr(), arena.numel(), stream),
                "fa_backward_host_resident")
    return O, l, m, dQ, dK, dV


def estimate_forward_flops(seq_dims, rule, q_shape, k_shape, v_shape, dtype, sync_mode, window_size=1,
                           log2_stride_size=0, is_causal=False, shared_mem_bytes=0):
    '''The reference's Estimate{Full,Causal,Local}AttentionForward{1,2}dFlops ops
    (flash_attention.py:475-562, flash_attention_forward.cc:390-474), host only.'''
    code = _NP_DTYPES[np.dtype(dtype)]
    p = _capi.make_problem(code, seq_dims, rule, sync_mode, tuple(q_shape), tuple(k_shape), tuple(v_shape),
                           window_size, log2_stride_size, is_causal)
    return _capi.estimate_forward_flops(p, shared_mem_bytes)


def dispatch_path(seq_dims, rule, q_shape, k_shape, v_shape, dtype, sync_mode='none_front', window_size=1,
                  log2_stride_size=0, is_causal=False, backward=False):
    '''Which kernel family a call with these (channel-first) shapes takes, and - when it is the generic SIMT family -
    why the tensor-core kernels decline it (host only; `fa_dispatch_path`). Returns (name, reason).'''
    code = _NP_DTYPES[np.dtype(dtype)]
    p = _capi.make_problem(code, seq_dims, rule, sync_mode, tuple(q_shape), tuple(k_shape), tuple(v_shape),
                           window_size, log2_stride_size, is_causal)
    return _capi.dispatch_path(p, backward)


# ---- layout adapters (SURVEY.md section 8 f3: the step either side of the op) -----------------------------------
def from_channel_last(x):
    """[batch, seq, heads, channels] (torch CUDA tensor) -> the op's channel-first [batch, heads, channels, seq]."""
    return _layout(x, True)


def to_channel_last(x):
    """The op's channel-first [batch, heads, channels, seq] -> [batch, seq, heads, channels]."""
    return _layout(x, False)


def _layout(x, to_channel_first):
    import torch
    if not _is_torch(x) or not x.is_cuda:
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_NULL, "layout adapters take torch CUDA tensors (no CPU fallback)")
    if x.dim() != 4:
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_RANK, "expected a rank-4 tensor")
    codes = _torch_codes()
    if x.dtype not in codes:
        raise _capi.InvalidArgumentError(_capi.FA_EINVAL_DTYPE, f"unsupported dtype {x.dtype}")
    x = x.contiguous()
    if to_channel_first:
        b, s, h, c = x.shape
        y = torch.empty((b, h, c, s), dtype=x.dtype, device=x.device)
    else:
        b, h, c, s = x.shape
        y = torch.empty((b, s, h, c), dtype=x.dtype, device=x.device)
    _capi.check(_capi.lib.fa_layout_transpose(codes[x.dtype], x.data_ptr(), y.data_ptr(), b, s, h, c,
                                              int(to_channel_first), torch.cuda.current_stream(x.device).cuda_stream),
                "fa_layout_transpose")
    return y
