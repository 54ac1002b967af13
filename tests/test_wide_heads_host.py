"""Head widths above 256 channels, host only: which kernels serve them, what workspace they need, and where the grid
ends. No GPU is needed: fa_dispatch_path, fa_workspace_bytes and the argument checks of fa_forward / fa_backward run
on the host."""
import ctypes as C

import numpy as np
import pytest

from tf_flash_attention_b200 import _capi

WIDE_REASON = ("more than 256 channels: channel-sliced generic kernels (each CTA owns at most 256 output channels and "
               "recomputes S for them)")
GRID_REASON = "more than 256 channels: batch x tiles x channel slices exceeds a 31-bit grid"
ACC_BYTES = {_capi.FA_F16: 4, _capi.FA_F32: 4, _capi.FA_F64: 8}


def _problem(dtype, d, v_d, batch=2, q=300, k=300, rule="causal"):
    return _capi.make_problem(dtype, 1, rule, "none_front", (batch, d, q), (batch, d, k), (batch, v_d, k))


def _dispatch(p, backward):
    buf = C.create_string_buffer(320)
    rc = _capi.lib.fa_dispatch_path(C.byref(p), int(backward), buf, len(buf))
    return rc, buf.value.decode()


@pytest.mark.parametrize("dtype,d,v_d", [(dt, d, v_d) for dt in (_capi.FA_F16, _capi.FA_F32, _capi.FA_F64)
                                          for d, v_d in ((257, 257), (320, 64), (64, 520))]
                         + [(_capi.FA_F16, 1024, 1024), (_capi.FA_F32, 1024, 1024)])
def test_dispatch_names_the_wide_kernels(dtype, d, v_d):
    for rule in ("full", "causal", "local"):
        p = _problem(dtype, d, v_d, rule=rule)
        for backward in (False, True):
            assert _capi.dispatch_path(p, backward) == ("generic_simt", WIDE_REASON)


def test_reasons_at_and_below_256_channels_are_unchanged():
    p = _problem(_capi.FA_F32, 256, 256)
    assert _capi.dispatch_path(p) == ("generic_simt", "more than 64 channels: generic kernels")
    p = _problem(_capi.FA_F16, 256, 200)
    assert _capi.dispatch_path(p, True) == ("generic_simt", "more than 128 channels: generic kernels")


@pytest.mark.parametrize("dtype", [_capi.FA_F16, _capi.FA_F32, _capi.FA_F64], ids=["f16", "f32", "f64"])
def test_every_shape_the_reference_tiles_has_a_kernel(dtype):
    """Wherever the reference finds a key tile that fits shared memory (fa_estimate_forward_flops succeeds), a kernel
    family takes the problem, forward and backward."""
    rng = np.random.default_rng(dtype)
    widths = sorted(set(range(8, 2049, 61)) | {255, 256, 257, 851, 852, 1706, 1707, 1758, 1759, 2048}
                    | set(int(x) for x in rng.integers(1, 2049, 24)))
    flops = C.c_float(0)
    accepted = 0
    for d in widths:
        for v_d in widths[::3] + [d]:
            p = _problem(dtype, d, v_d, batch=3, q=70, k=90)
            if _capi.lib.fa_estimate_forward_flops(C.byref(p), 0, C.byref(flops)) != _capi.FA_OK:
                continue
            accepted += 1
            for backward in (False, True):
                rc, reason = _dispatch(p, backward)
                assert rc >= 1, f"d={d} v_d={v_d} backward={backward}: {rc} {reason}"
    assert accepted > 100


@pytest.mark.parametrize("dtype", [_capi.FA_F16, _capi.FA_F32, _capi.FA_F64], ids=["f16", "f32", "f64"])
@pytest.mark.parametrize("d,v_d", [(257, 257), (320, 64), (64, 520), (800, 800)])
def test_workspace_is_the_generic_statistics_only(dtype, d, v_d):
    """No workspace for the forward; the backward keeps the generic family's LSE + D rows and nothing per slice."""
    for batch, q in ((1, 1), (3, 333), (16, 4096)):
        p = _problem(dtype, d, v_d, batch=batch, q=q, k=200)
        assert _capi.lib.fa_workspace_bytes(C.byref(p), 0) == 0
        assert _capi.lib.fa_workspace_bytes(C.byref(p), 1) == 2 * batch * q * ACC_BYTES[dtype]


def test_grid_beyond_31_bits_is_a_shape_error():
    """batch x row tiles x channel slices must fit a 31-bit grid: beyond it the call is refused before any launch."""
    one = C.c_void_p(256)
    for dtype in (_capi.FA_F16, _capi.FA_F32, _capi.FA_F64):
        fits = _problem(dtype, 512, 512, batch=1 << 20, q=64, k=64)
        for backward in (False, True):
            assert _dispatch(fits, backward) == (1, WIDE_REASON)
        big = _problem(dtype, 512, 512, batch=1 << 29, q=64, k=64)
        for backward in (False, True):
            assert _dispatch(big, backward) == (_capi.FA_EINVAL_SHAPE, GRID_REASON)
        ws = int(_capi.lib.fa_workspace_bytes(C.byref(big), 1))
        assert _capi.lib.fa_forward(C.byref(big), one, one, one, one, one, one, None, 0, None) == _capi.FA_EINVAL_SHAPE
        assert _capi.lib.fa_backward(C.byref(big), one, one, one, one, one, one, one, one, one, one, one, ws,
                                     None) == _capi.FA_EINVAL_SHAPE
    # the forward's grid can fit where the backward's does not: dK | dV has more slices than O
    p = _problem(_capi.FA_F32, 1024, 64, batch=(1 << 31) // 4, q=32, k=32)
    assert _dispatch(p, False) == (1, WIDE_REASON)
    assert _dispatch(p, True) == (_capi.FA_EINVAL_SHAPE, GRID_REASON)


def test_channel_last_wide_heads_take_the_adapter():
    """Channel-last operands are read directly only by the fp16 tensor-core kernels; wide heads answer
    FA_EINVAL_LAYOUT, which is what sends the Python layer through the layout adapter."""
    p = _problem(_capi.FA_F16, 320, 320)
    p.layout, p.heads = _capi.FA_LAYOUT_CHANNEL_LAST, 1
    assert _dispatch(p, False)[0] == _capi.FA_EINVAL_LAYOUT
    assert _dispatch(p, True)[0] == _capi.FA_EINVAL_LAYOUT


def test_host_arenas_cover_wide_heads():
    """The host-buffer entry points size their device arena from the tensors and fa_workspace_bytes alone."""
    for dtype, e in ((_capi.FA_F16, 2), (_capi.FA_F32, 4), (_capi.FA_F64, 8)):
        b, d, v_d, q, k = 3, 320, 520, 100, 150
        p = _problem(dtype, d, v_d, batch=b, q=q, k=k)
        fwd = int(_capi.lib.fa_host_arena_bytes(C.byref(p), 0))
        bwd = int(_capi.lib.fa_host_arena_bytes(C.byref(p), 1))
        step = int(_capi.lib.fa_step_host_arena_bytes(C.byref(p)))
        tensors = e * b * (d * q + d * k + v_d * k + v_d * q) + ACC_BYTES[dtype] * b * q + e * b * q  # Q K V O l m
        assert fwd >= tensors
        assert bwd >= fwd + e * b * (v_d * q + d * q + d * k + v_d * k) + 2 * b * q * ACC_BYTES[dtype]
        assert step == bwd
