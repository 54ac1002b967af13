"""Head widths above 256 channels on the GPU: the channel-sliced generic kernels against the dense oracle (float64),
at the tolerances of tests/helpers.py (fp16 2e-3 with gradients scaled by max(1, |ref|), fp32 1e-5, fp64 1e-12).
O, l, m, the sentinel rows and dQ / dK / dV are checked by test_gpu_parity._check, which also asserts that the forward
and the backward ran on the generic family (fa_last_path() == 1). fp16 gradients are checked against the backward of
the fp16 O the op receives (_check_f16_grads)."""
import ctypes as C

import numpy as np
import pytest

from oracle import dense_attention as da
from oracle import pattern
from tests.helpers import TOL, max_abs_err, scaled_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from tf_flash_attention_b200 import _capi  # noqa: E402
from tf_flash_attention_b200 import flash_attention as fa  # noqa: E402
from tests.test_gpu_parity import ATTN, SYNC, _call, _check  # noqa: E402

WIDE = [(257, 257), (320, 64), (64, 520), (512, 512), (1024, 1024)]
SHAPES = {np.float16: WIDE, np.float32: WIDE, np.float64: WIDE[:4]}
RULES = list(ATTN)


def _window(attn, dims):
    """(window_size, log2_stride_size, is_causal) of an attention class"""
    cfg = ATTN[attn]
    if cfg["rule"] != "local":
        return 1, 0, False
    if dims == 1:
        return (6, 3, cfg["is_causal"]) if cfg["strided"] else (40, 0, cfg["is_causal"])
    return (3, 1, cfg["is_causal"]) if cfg["strided"] else (4, 0, cfg["is_causal"])


def _cases():
    out, c = [], 0
    for dtype, shapes in SHAPES.items():
        for d, v_d in shapes:
            for dims in (1, 2):
                attn, sync = RULES[(c + dims) % len(RULES)], SYNC[(c + 2 * dims) % len(SYNC)]
                out.append(pytest.param(dtype, d, v_d, dims, attn, sync,
                                        id=f"{np.dtype(dtype).name}-d{d}-vd{v_d}-{dims}d-{attn}-{sync}"))
            c += 1
    return out


def _check_f16_grads(dims, rule, sync_mode, w, s, causal, batch, d, v_d, qs, ks, seed):
    """fp16 gradients against the oracle's backward of the O the op receives. The backward takes O in fp16, and
    D = rowsum(dO * O) carries O's rounding summed over v_d channels: at v_d = 520 and d = 64 that alone moves dQ by
    about 3e-3 from the gradient of the exact O, whatever the kernels do."""
    rng = np.random.default_rng(seed)
    Q, K, V, dO = da.random_inputs(rng, np.float16, batch, d, v_d, qs, ks)
    tq, tk, tv = (torch.from_numpy(x).cuda().requires_grad_(True) for x in (Q, K, V))
    O = _call(dims, rule, tq, tk, tv, sync_mode, w, s, causal)[0]
    grads = torch.autograd.grad(O, (tq, tk, tv), torch.from_numpy(dO).cuda())
    torch.cuda.synchronize()
    assert _capi.lib.fa_last_path() == 1
    Qf, Kf, Vf, _, qsh, ksh = da.flatten_inputs(Q, K, V, dims)
    mask = pattern.tests_mask(qsh, ksh, sync_mode, rule, w, s, causal)
    _, _, _, p = da.forward(Qf, Kf, Vf, mask, return_p=True)
    Kf, Qf, Vf = (x.astype(np.float64) for x in (Kf, Qf, Vf))
    Of = O.detach().cpu().numpy().astype(np.float64).reshape(Qf.shape[0], v_d, -1)
    dOf = dO.astype(np.float64).reshape(Of.shape)
    D = np.einsum("bcq,bcq->bq", dOf, Of)
    dS = p * (np.einsum("bcq,bck->bqk", dOf, Vf) - D[..., None]) / np.sqrt(np.float64(d))
    ref = {"dQ": np.einsum("bqk,bck->bcq", dS, Kf), "dK": np.einsum("bqk,bcq->bck", dS, Qf),
           "dV": np.einsum("bqk,bcq->bck", p, dOf)}
    for name, got in zip(("dQ", "dK", "dV"), grads):
        err = scaled_err(got.cpu().numpy().reshape(ref[name].shape), ref[name])
        assert err <= TOL[np.dtype(np.float16)], f"{name}: {err}"


@pytest.mark.parametrize("dtype,d,v_d,dims,attn,sync_mode", _cases())
def test_wide_heads_match_the_oracle(dtype, d, v_d, dims, attn, sync_mode):
    w, s, causal = _window(attn, dims)
    rule = ATTN[attn]["rule"]
    qs, ks = ((193,), (277,)) if dims == 1 else ((12, 17), (14, 19))   # ragged, q != k
    seed = d * 7 + v_d + dims
    f16 = dtype == np.float16
    _check(dtype, dims, rule, sync_mode, w, s, causal, (2, 2), d, v_d, qs, ks, seed, check_grad=not f16, expect_path=1)
    if f16:
        _check_f16_grads(dims, rule, sync_mode, w, s, causal, (2, 2), d, v_d, qs, ks, seed)


def _shard_forward(dtype, d, v_d, n, shards, rule="causal"):
    """Attends the key shards one after the other with accumulate = 1 and global index bases."""
    rng = np.random.default_rng(9)
    Q, K, V, _ = da.random_inputs(rng, dtype, (3,), d, v_d, (n,), (n,))
    tq = torch.from_numpy(Q).cuda()
    code = {np.float16: _capi.FA_F16, np.float32: _capi.FA_F32, np.float64: _capi.FA_F64}[dtype]
    ldt = torch.float32 if dtype == np.float16 else tq.dtype
    O = torch.empty((3, v_d, n), dtype=tq.dtype, device="cuda")
    l = torch.empty((3, n), dtype=ldt, device="cuda")
    m = torch.empty((3, n), dtype=tq.dtype, device="cuda")
    for step, (k0, k1) in enumerate(shards):
        tk = torch.from_numpy(np.ascontiguousarray(K[:, :, k0:k1])).cuda()
        tv = torch.from_numpy(np.ascontiguousarray(V[:, :, k0:k1])).cuda()
        p = _capi.make_problem(code, 1, rule, "none_front", (3, d, n), (3, d, k1 - k0), (3, v_d, k1 - k0))
        p.k_index_base, p.k_full_len, p.q_full_len, p.accumulate = k0, n, n, int(step > 0)
        need = _capi.lib.fa_workspace_bytes(C.byref(p), 0)
        assert need == 0
        _capi.check(_capi.lib.fa_forward(C.byref(p), tq.data_ptr(), tk.data_ptr(), tv.data_ptr(), O.data_ptr(),
                                         l.data_ptr(), m.data_ptr(), None, 0, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == 1
    return (Q, K, V), (O.cpu().numpy(), l.cpu().numpy().astype(np.float64), m.cpu().numpy().astype(np.float64))


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=lambda d: np.dtype(d).name)
def test_accumulate_merges_key_shards(dtype):
    """K/V-ring building block at 320 channels: two key shards attended one after the other with accumulate = 1 equal
    the whole sequence at once. Every O slice reads the incoming m and l before slice 0 replaces them."""
    (Q, K, V), (O, l, m) = _shard_forward(dtype, 320, 320, 192, ((96, 192), (0, 96)))
    ref = da.attention(Q, K, V, 1, "causal", "none_front")
    tol = TOL[np.dtype(dtype)]
    assert max_abs_err(O, ref["O"]) <= tol
    lse, lse_ref = m + np.log(l), ref["m"] + np.log(ref["l"])
    assert np.max(np.abs(lse - lse_ref)) <= max(tol * 4, 1e-12)


def test_backward_is_deterministic():
    """One writer per output element, no atomics: the backward run twice gives the same bits."""
    rng = np.random.default_rng(11)
    for dtype, d, v_d in ((np.float32, 320, 320), (np.float16, 512, 300)):
        Q, K, V, dO = da.random_inputs(rng, dtype, (2,), d, v_d, (230,), (260,))
        tq, tk, tv, tdo = (torch.from_numpy(x).cuda() for x in (Q, K, V, dO))
        O, l, m = fa.causal_1d(tq, tk, tv, "none_front", returning_l_m=True)
        runs = [fa.attention_backward(1, "causal", tq, tk, tv, O, l, m, tdo, "none_front") for _ in range(2)]
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == 1
        for a, b in zip(*runs):
            assert torch.equal(a, b)


PATTERN_CASES = [
    (1, "causal", (300,), (520,), 1, 0, False),
    (1, "local", (400,), (400,), 5, 2, False),
    (1, "local", (330,), (470,), 7, 1, True),
    (2, "causal", (18, 20), (17, 23), 1, 0, False),
    (2, "local", (19, 21), (20, 22), 3, 1, False),
]


@pytest.mark.parametrize("dims,rule,qs,ks,w,s,c", PATTERN_CASES)
def test_device_pattern_bit_exact_beyond_256_keys(dims, rule, qs, ks, w, s, c):
    """Q = K = 0 and V = identity (v_d = k > 256, so O is split into channel slices): O[j, i] > 0 exactly where
    (i, j) is attended, and l is the count of attended keys."""
    q, k = int(np.prod(qs)), int(np.prod(ks))
    Q = torch.zeros((1, 8) + qs, dtype=torch.float32, device="cuda")
    K = torch.zeros((1, 8) + ks, dtype=torch.float32, device="cuda")
    V = torch.eye(k, dtype=torch.float32, device="cuda").reshape((1, k) + ks)
    p = _capi.make_problem(_capi.FA_F32, dims, rule, "none_front", Q.shape, K.shape, V.shape, w, s, c)
    mask = _capi.pattern_mask(p)
    if rule == "causal":
        O, l, m = (fa.causal_1d if dims == 1 else fa.causal_2d)(Q, K, V, "none_front", returning_l_m=True)
    else:
        O, l, m = (fa.local_1d if dims == 1 else fa.local_2d)(Q, K, V, w, s, c, "none_front", returning_l_m=True)
    torch.cuda.synchronize()
    assert _capi.lib.fa_last_path() == 1
    got = (O.reshape(k, q).T > 0).cpu().numpy()
    assert np.array_equal(got, mask)
    assert np.array_equal(l.reshape(q).cpu().numpy(), mask.sum(axis=1).astype(np.float32))


@pytest.mark.parametrize("pipelined", [False, True])
def test_host_buffers_at_320_channels(pipelined):
    """NumPy in, NumPy out: fa.causal_1d + fa.attention_backward on host arrays, and one training step through
    fa.forward_backward_host, at d = v_d = 320."""
    rng = np.random.default_rng(13)
    Q, K, V, dO = da.random_inputs(rng, np.float32, (2, 2), 320, 320, (150,), (210,))
    ref = da.attention(Q, K, V, 1, "causal", "scale_front", dO=dO)
    O, l, m = fa.causal_1d(Q, K, V, "scale_front", returning_l_m=True)
    assert isinstance(O, np.ndarray) and max_abs_err(O, ref["O"]) <= 1e-5
    grads = fa.attention_backward(1, "causal", Q, K, V, O, l, m, dO, "scale_front")
    for name, g in zip(("dQ", "dK", "dV"), grads):
        assert scaled_err(g, ref[name]) <= 1e-5, name
    O2, l2, m2, dQ, dK, dV = fa.forward_backward_host(1, "causal", Q, K, V, dO, "scale_front", pipelined=pipelined)
    assert np.array_equal(O, O2) and np.array_equal(l, l2) and np.array_equal(m, m2)
    for g, h in zip((dQ, dK, dV), grads):
        assert np.array_equal(g, h)


def test_channel_last_320_channels_is_the_adapter_around_channel_first():
    """layout='channel_last' at 320 fp16 channels: the same bits as the channel-first call followed by
    to_channel_last, forward and gradients."""
    rng = np.random.default_rng(17)
    outer, seq, heads, ch = 2, 200, 3, 320
    Q, K, V, dO = (torch.from_numpy(rng.standard_normal((outer, seq, heads, ch)).astype(np.float16)).cuda()
                   for _ in range(4))
    tq, tk, tv = (x.clone().requires_grad_(True) for x in (Q, K, V))
    O = fa.causal_1d(tq, tk, tv, "none_front", layout="channel_last")
    grads = torch.autograd.grad(O, (tq, tk, tv), dO)
    cq, ck, cv = (fa.from_channel_last(x).requires_grad_(True) for x in (Q, K, V))
    Oc = fa.causal_1d(cq, ck, cv, "none_front")
    gc = torch.autograd.grad(Oc, (cq, ck, cv), fa.from_channel_last(dO))
    torch.cuda.synchronize()
    assert torch.equal(O, fa.to_channel_last(Oc.detach()))
    for g, h in zip(grads, gc):
        assert torch.equal(g, fa.to_channel_last(h))
