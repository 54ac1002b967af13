"""bfloat16 (dtype code 3, FA_BF16), host only: every entry point that takes a dtype accepts 3 and still refuses 4, the
host helpers and the size rules give the fp16 answers, fa_dispatch_path names the same families with the same reasons
as for fp16, and the Python dtype maps. No GPU is needed: argument checks, dispatch and sizes run on the host."""
import ctypes as C

import numpy as np
import pytest

from tests.helpers import case_id, load_pattern_golden
from tf_flash_attention_b200 import _capi
from tf_flash_attention_b200 import flash_attention as fa

F16, BF16, BAD = _capi.FA_F16, _capi.FA_BF16, 4
CASES = load_pattern_golden()


def _problem(dtype, d=128, v_d=128, batch=2, q=304, k=304, rule="causal"):
    return _capi.make_problem(dtype, 1, rule, "none_front", (batch, d, q), (batch, d, k), (batch, v_d, k))


def _golden_problem(dtype, c):
    batch = (2,)
    return _capi.make_problem(dtype, c["dims"], c["rule"], c["sync_mode"], batch + (8,) + tuple(c["q_shape"]),
                              batch + (8,) + tuple(c["k_shape"]), batch + (8,) + tuple(c["k_shape"]),
                              c["window_size"], c["log2_stride_size"], c["is_causal"])


def _dispatch(p, backward):
    buf = C.create_string_buffer(320)
    rc = _capi.lib.fa_dispatch_path(C.byref(p), int(backward), buf, len(buf))
    return rc, buf.value.decode()


def test_enum_and_error_text():
    assert BF16 == 3
    assert "bfloat16" in _capi.strerror(_capi.FA_EINVAL_DTYPE)


def test_problem_entry_points_accept_3_and_refuse_4():
    p = _problem(BF16)
    n = C.c_int64(0)
    f = C.c_float(0)
    q = np.zeros(304 * 304, dtype=np.uint8)
    qo, ko, ref = np.zeros(304, np.int32), np.zeros(304, np.int32), np.zeros(2, np.int32)
    cls = np.zeros(64, np.uint8)
    calls = {
        "fa_count_attended": lambda p: _capi.lib.fa_count_attended(C.byref(p), C.byref(n)),
        "fa_pattern_mask": lambda p: _capi.lib.fa_pattern_mask(C.byref(p), q.ctypes.data),
        "fa_pattern_mask_fast": lambda p: _capi.lib.fa_pattern_mask_fast(C.byref(p), 64, 1, q.ctypes.data),
        "fa_orders": lambda p: _capi.lib.fa_orders(C.byref(p), qo.ctypes.data, ko.ctypes.data, ref.ctypes.data),
        "fa_classify_tiles": lambda p: _capi.lib.fa_classify_tiles(C.byref(p), 128, 128, cls.ctypes.data),
        "fa_estimate_forward_flops": lambda p: _capi.lib.fa_estimate_forward_flops(C.byref(p), 0, C.byref(f)),
        "fa_dispatch_path(fwd)": lambda p: min(0, _dispatch(p, False)[0]),
        "fa_dispatch_path(bwd)": lambda p: min(0, _dispatch(p, True)[0]),
    }
    for name, call in calls.items():
        p.dtype = BF16
        assert call(p) == _capi.FA_OK, name
        p.dtype = BAD
        assert call(p) == _capi.FA_EINVAL_DTYPE, name
    # sizes answer 0 for a refused problem
    for backward in (0, 1):
        p.dtype = BF16
        assert _capi.lib.fa_workspace_bytes(C.byref(p), backward) > 0 or not backward
        assert _capi.lib.fa_host_arena_bytes(C.byref(p), backward) > 0
        p.dtype = BAD
        assert _capi.lib.fa_workspace_bytes(C.byref(p), backward) == 0
        assert _capi.lib.fa_host_arena_bytes(C.byref(p), backward) == 0
    p.dtype = BF16
    assert _capi.lib.fa_step_host_arena_bytes(C.byref(p)) > 0
    assert _capi.lib.fa_backward_accumulate_supported(C.byref(p), 0) == 1
    p.dtype = BAD
    assert _capi.lib.fa_step_host_arena_bytes(C.byref(p)) == 0
    assert _capi.lib.fa_backward_accumulate_supported(C.byref(p), 0) == 0


def test_calls_without_work_accept_3_and_refuse_4():
    """The device entry points validate the dtype before anything else; with nothing to do (batch 0, n 0) code 3
    returns FA_OK without touching a device."""
    one = C.c_void_p(256)
    p = _problem(BF16, batch=0)
    ws = int(_capi.lib.fa_workspace_bytes(C.byref(p), 1))
    for dtype, want in ((BF16, _capi.FA_OK), (BAD, _capi.FA_EINVAL_DTYPE)):
        p.dtype = dtype
        assert _capi.lib.fa_forward(C.byref(p), one, one, one, one, one, one, one, 1 << 30, None) == want
        assert _capi.lib.fa_backward(C.byref(p), *([one] * 10), one, max(ws, 1 << 30), None) == want
        assert _capi.lib.fa_backward_accumulate(C.byref(p), *([one] * 10), 0, one, 1 << 30, None) == want
        assert _capi.lib.fa_partial_merge(C.byref(p), *([one] * 6), 1, None) == want
        assert _capi.lib.fa_partial_finalize(C.byref(p), *([one] * 6), None) == want
        assert _capi.lib.fa_forward_host(C.byref(p), *([one] * 6), one, 1 << 30, None) == want
        assert _capi.lib.fa_backward_host(C.byref(p), *([one] * 10), one, 1 << 30, None) == want
        assert _capi.lib.fa_forward_backward_host(C.byref(p), *([one] * 10), one, 1 << 30, None) == want
        assert _capi.lib.fa_grad_accumulate(dtype, one, one, 0, 1, None) == want
        assert _capi.lib.fa_grad_finalize(dtype, one, one, 0, None) == want
        assert _capi.lib.fa_layout_transpose(dtype, one, one, 0, 64, 2, 64, 1, None) == want
    assert _capi.lib.fa_ring_causal_forward(None, BAD, 2, 128, 128, 64, *([one] * 7), 1 << 30,
                                            None) == _capi.FA_EINVAL_DTYPE


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_rule_helpers_give_the_fp16_answer(c):
    a, b = _golden_problem(F16, c), _golden_problem(BF16, c)
    assert _capi.count_attended(b) == _capi.count_attended(a) == int(c["mask"].sum())
    assert np.array_equal(_capi.pattern_mask(b), c["mask"])
    assert _capi.estimate_forward_flops(b) == _capi.estimate_forward_flops(a)


@pytest.mark.parametrize("d,v_d,q,k", [(128, 128, 8192, 8192), (64, 64, 1000, 88), (24, 40, 342, 343),
                                       (160, 160, 300, 300), (320, 64, 193, 277)])
def test_sizes_equal_fp16(d, v_d, q, k):
    for batch in (1, 3):
        a, b = _problem(F16, d, v_d, batch, q, k), _problem(BF16, d, v_d, batch, q, k)
        for backward in (0, 1):
            assert _capi.lib.fa_workspace_bytes(C.byref(b), backward) == _capi.lib.fa_workspace_bytes(C.byref(a),
                                                                                                    backward)
            assert _capi.lib.fa_host_arena_bytes(C.byref(b), backward) == _capi.lib.fa_host_arena_bytes(C.byref(a),
                                                                                                      backward)
        assert _capi.lib.fa_step_host_arena_bytes(C.byref(b)) == _capi.lib.fa_step_host_arena_bytes(C.byref(a))
    for world in (1, 2, 8):
        for backward in (0, 1):
            assert (_capi.lib.fa_ring_causal_arena_bytes(BF16, 4, d, v_d, 512, world, backward)
                    == _capi.lib.fa_ring_causal_arena_bytes(F16, 4, d, v_d, 512, world, backward) > 0)
    for acc in (0, 1):
        assert (_capi.lib.fa_ring_causal_slot_bytes(BF16, 4, d, v_d, 512, acc)
                == _capi.lib.fa_ring_causal_slot_bytes(F16, 4, d, v_d, 512, acc) > 0)


@pytest.mark.parametrize("d,v_d", [(8, 8), (24, 24), (64, 64), (72, 100), (128, 64), (128, 128)])
@pytest.mark.parametrize("rule", ["full", "causal", "local"])
def test_dispatch_tensor_cores_up_to_128_channels(d, v_d, rule):
    for q, k in ((8192, 8192), (1000, 88), (343, 342)):
        p = _problem(BF16, d, v_d, batch=4, q=q, k=k, rule=rule)
        for backward in (False, True):
            assert _dispatch(p, backward) == (2, "")


def test_dispatch_reasons_match_fp16():
    shapes = [dict(d=160, v_d=160), dict(d=64, v_d=200), dict(d=320, v_d=64), dict(d=1024, v_d=1024),
              dict(d=64, v_d=64, q=64, k=200000), dict(d=64, v_d=64, q=200000, k=64)]
    for kw in shapes:
        a, b = _problem(F16, **kw), _problem(BF16, **kw)
        for backward in (False, True):
            got = _dispatch(b, backward)
            assert got == _dispatch(a, backward), kw
            # the forward streams keys only: 200000 queries over 64 keys stay on the tensor cores
            assert got[0] == 1 and got[1] or (not backward and kw.get("q") == 200000 and got == (2, "")), kw
    a, b = _problem(F16), _problem(BF16)
    a.accumulate = b.accumulate = 1
    assert _dispatch(b, False) == _dispatch(a, False) == (1, "accumulate = 1 is served by the generic forward kernels")


def test_channel_last_odd_channels_is_a_layout_error():
    for d in (12, 100):
        p = _problem(BF16, d, d)
        p.layout, p.heads = _capi.FA_LAYOUT_CHANNEL_LAST, 2
        for backward in (False, True):
            assert _dispatch(p, backward)[0] == _capi.FA_EINVAL_LAYOUT
    p = _problem(BF16, 96, 96)
    p.layout, p.heads = _capi.FA_LAYOUT_CHANNEL_LAST, 2
    assert _dispatch(p, False) == (2, "") and _dispatch(p, True) == (2, "")


def test_python_dtype_maps():
    torch = pytest.importorskip("torch")
    assert fa._torch_codes()[torch.bfloat16] == BF16
    assert fa._l_dtype(torch.bfloat16) == torch.float32
    assert fa._l_dtype(torch.float16) == torch.float32
    assert fa._l_dtype(torch.float64) == torch.float64
    x = torch.zeros((2, 16, 64), dtype=torch.bfloat16)
    p = fa._problem(1, "causal", x, x, x, "none_front")
    assert p.dtype == BF16 and p.d == 16 and p.batch == 2
    with pytest.raises(_capi.InvalidArgumentError):
        fa._problem(1, "causal", x, x.float(), x, "none_front")


def test_numpy_inputs_still_raise():
    """NumPy has no bfloat16: the host path keeps refusing anything outside float16 / float32 / float64."""
    for dt in (np.int16, np.uint16, np.float128 if hasattr(np, "float128") else np.int8):
        x = np.zeros((2, 16, 64), dtype=dt)
        with pytest.raises(_capi.InvalidArgumentError) as e:
            fa.causal_1d(x, x, x, "none_front")
        assert e.value.status == _capi.FA_EINVAL_DTYPE
