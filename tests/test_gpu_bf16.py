"""bfloat16 on the GPU: the tcgen05 16-bit kernels, the generic family, the ring pieces, the layout adapter and the
host-buffer entry points against the float64 oracle. Inputs are drawn as the other parity tests draw them and rounded
to bf16 through torch; the oracle runs on the rounded values.

Bar: 1.6e-2 * max(1, |ref|), eight times the fp16 bar of tests/helpers.py (the ratio of the unit roundoffs,
2^-8 / 2^-11). Gradient reference: the exact oracle for the precise kernels that re-derive D = rowsum(P o dP) (split
gradients with head_dim <= 64); elsewhere the oracle's backward of the bf16 O the op returned, whose
D = rowsum(dO o O) inherits O's rounding. The plain kernels (grad precision 2) are held to the bar on rows of at
least 256 keys only."""
import ctypes as C

import numpy as np
import pytest

from oracle import dense_attention as da
from oracle import pattern

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from tf_flash_attention_b200 import _capi, ring  # noqa: E402
from tf_flash_attention_b200 import flash_attention as fa  # noqa: E402
from tests.test_gpu_parity import ATTN, SYNC, _call  # noqa: E402

TOL = 1.6e-2


def _err(got, ref):
    got = np.asarray(got.detach().float().cpu().numpy() if torch.is_tensor(got) else got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64).reshape(got.shape)
    return float(np.max(np.abs(got - ref) / np.maximum(1.0, np.abs(ref)))) if ref.size else 0.0


def _inputs(seed, batch, d, v_d, qs, ks):
    """bf16 CUDA tensors and their float64 values"""
    rng = np.random.default_rng(seed)
    ts = [torch.from_numpy(x).cuda().to(torch.bfloat16) for x in da.random_inputs(rng, np.float32, batch, d, v_d, qs, ks)]
    return ts, [t.double().cpu().numpy() for t in ts]


def _window(attn, dims):
    cfg = ATTN[attn]
    if cfg["rule"] != "local":
        return 1, 0, False
    if dims == 1:
        return (6, 3, cfg["is_causal"]) if cfg["strided"] else (40, 0, cfg["is_causal"])
    return (3, 1, cfg["is_causal"]) if cfg["strided"] else (4, 0, cfg["is_causal"])


def _grad_refs(Qn, Kn, Vn, dOn, On, dims, rule, sync_mode, w, s, c):
    """(exact oracle gradients, gradients of the returned O) as dicts"""
    Qf, Kf, Vf, _, qsh, ksh = da.flatten_inputs(Qn, Kn, Vn, dims)
    mask = pattern.tests_mask(qsh, ksh, sync_mode, rule, w, s, c)
    dOf = dOn.reshape(Qf.shape[0], Vf.shape[1], Qf.shape[2])
    exact = dict(zip(("dQ", "dK", "dV"), da.backward(Qf, Kf, Vf, mask, dOf)))
    _, _, _, p = da.forward(Qf, Kf, Vf, mask, return_p=True)
    Of = On.reshape(dOf.shape)
    D = np.einsum("bcq,bcq->bq", dOf, Of)
    dS = p * (np.einsum("bcq,bck->bqk", dOf, Vf) - D[..., None]) / np.sqrt(np.float64(Qf.shape[1]))
    of_o = {"dQ": np.einsum("bqk,bck->bcq", dS, Kf), "dK": np.einsum("bqk,bcq->bck", dS, Qf),
            "dV": np.einsum("bqk,bcq->bck", p, dOf)}
    return exact, of_o, mask


def _check(dims, rule, sync_mode, w, s, c, batch, d, v_d, qs, ks, seed, mode, path=2, override=0, grads=True,
           exact=None):
    """exact: whether the gradients are held to the exact oracle (default: the precise tensor-core kernels, mode 1 at
    head_dim <= 64, which re-derive D) or to the backward of the returned O"""
    (tq, tk, tv, tdo), (Qn, Kn, Vn, dOn) = _inputs(seed, batch, d, v_d, qs, ks)
    ref = da.attention(Qn, Kn, Vn, dims, rule, sync_mode, w, s, c)
    assert _capi.lib.fa_set_grad_precision(mode) == _capi.FA_OK
    _capi.lib.fa_set_path_override(override)
    try:
        tq, tk, tv = (t.requires_grad_(grads) for t in (tq, tk, tv))
        O, l, m = _call(dims, rule, tq, tk, tv, sync_mode, w, s, c)
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == path
        assert O.dtype == torch.bfloat16 and m.dtype == torch.bfloat16 and l.dtype == torch.float32
        tag = f"{dims}d {rule} {sync_mode} w{w} s{s} c{c} d{d} vd{v_d} q{qs} k{ks} mode{mode} ov{override}"
        assert _err(O, ref["O"]) <= TOL, f"O {tag}: {_err(O, ref['O'])}"
        ln, mn = l.cpu().numpy().astype(np.float64), m.cpu()
        empty = ~np.isfinite(ref["m"])
        if empty.any():
            assert np.all(ln[empty] == 0)
            assert np.all(mn.view(torch.int16).numpy()[empty] == np.int16(-1286))   # bytes 0xFA 0xFA
            On = O.detach().float().cpu().numpy()
            assert np.all(On[np.broadcast_to(np.expand_dims(empty, -dims - 1), On.shape)] == 0)
        live = ~empty
        if live.any():
            mf = mn.double().numpy()
            lse = mf[live] + np.log(ln[live])
            assert np.max(np.abs(lse - (ref["m"][live] + np.log(ref["l"][live])))) <= TOL, f"lse {tag}"
            assert np.max(np.abs(mf[live] - ref["m"][live]) / np.maximum(1, np.abs(ref["m"][live]))) <= TOL, tag
        if not grads:
            return O, None
        g = torch.autograd.grad(O, (tq, tk, tv), tdo)
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == path
        ref_exact, of_o, mask = _grad_refs(Qn, Kn, Vn, dOn, O.detach().double().cpu().numpy(), dims, rule, sync_mode, w, s, c)
        if exact is None:
            exact = mode == 1 and d <= 64 and path == 2
        want = ref_exact if exact else of_o
        if mode == 2:
            assert mask.sum(axis=1).min() >= 256, "plain kernels are held to the bar on rows of >= 256 keys"
        for name, got in zip(("dQ", "dK", "dV"), g):
            assert got.dtype == torch.bfloat16
            e = _err(got, want[name])
            assert e <= TOL, f"{name} {tag}: {e}"
        return O, g
    finally:
        _capi.lib.fa_set_grad_precision(0)
        _capi.lib.fa_set_path_override(0)


# ---- the tensor cores -------------------------------------------------------------------------------------------
def _matrix():
    out = []
    for dims in (1, 2):
        for i, attn in enumerate(ATTN):
            for j, sync in enumerate(SYNC):
                d = (8, 12, 16, 24, 32, 20)[(i + j + dims) % 6]
                out.append(pytest.param(dims, attn, sync, d, id=f"{dims}d-{attn}-{sync}-d{d}"))
    return out


@pytest.mark.parametrize("dims,attn,sync_mode,d", _matrix())
def test_every_attention_class_on_the_tensor_cores(dims, attn, sync_mode, d):
    """Precise gradients (mode 1); ragged lengths not multiples of 8 (the pack pass runs) and q != k."""
    w, s, c = _window(attn, dims)
    qs, ks = ((301,), (262,)) if dims == 1 else ((13, 15), (14, 17))
    _check(dims, ATTN[attn]["rule"], sync_mode, w, s, c, (2,), d, d, qs, ks, 100 * dims + d, mode=1)


@pytest.mark.parametrize("d,v_d", [(64, 64), (128, 128), (128, 64), (64, 128), (48, 48), (72, 72), (100, 100),
                                   (8, 24), (32, 100)])
def test_channel_configurations(d, v_d):
    """The four kernel configurations (64 / 128 channels each side) and odd channel counts padded up to them."""
    _check(1, "causal", "none_front", 1, 0, False, (2,), d, v_d, (384,), (384,), d + v_d, mode=1)


@pytest.mark.parametrize("d,v_d", [(64, 64), (128, 128), (128, 64)])
@pytest.mark.parametrize("override", [0, 4])
def test_plain_kernels_on_long_rows(d, v_d, override):
    """Grad precision 2 on full attention over 512 keys: the fused (override 0, head_dim 128) and the two-kernel
    (override 4) plain backward."""
    _check(1, "full", "scale_front", 1, 0, False, (2, 2), d, v_d, (320,), (512,), 7 * d, mode=2, override=override)


def test_forward_override_5_and_fused_default():
    _check(1, "causal", "none_front", 1, 0, False, (2,), 64, 64, (640,), (640,), 5, mode=1, override=5)
    _check(1, "causal", "none_front", 1, 0, False, (2,), 128, 128, (1024,), (1024,), 6, mode=0)


def test_short_rows_take_the_precise_kernels_in_mode_0():
    """1000 queries over 88 keys, causal: where the fp16 plain kernels measure 4.2e-3, mode 0 picks the precise ones."""
    _check(1, "causal", "scale_end", 1, 0, False, (2,), 64, 64, (1000,), (88,), 8, mode=0, exact=True)


def test_sentinel_rows():
    _check(1, "local", "none_front", 2, 0, False, (2,), 16, 16, (200,), (40,), 21, mode=1)
    _check(2, "local", "none_front", 1, 1, True, (2,), 8, 8, (9, 12), (4, 5), 22, mode=1)


def test_c2_spot_check():
    """Two heads of C2 (causal_1d, d = 128, S = 8192) in the default mode: the fused plain backward."""
    (tq, tk, tv, tdo), (Qn, Kn, Vn, dOn) = _inputs(1234, (2,), 128, 128, (8192,), (8192,))
    tq, tk, tv = (t.requires_grad_(True) for t in (tq, tk, tv))
    O = fa.causal_1d(tq, tk, tv, "none_front")
    g = torch.autograd.grad(O, (tq, tk, tv), tdo)
    torch.cuda.synchronize()
    assert _capi.lib.fa_last_path() == 2
    for b in range(2):
        ref = da.forward_backward_chunked(Qn[b], Kn[b], Vn[b], dOn[b], (8192,), (8192,), "none_front", "causal")
        assert _err(O[b], ref["O"]) <= TOL
        for name, got in zip(("dQ", "dK", "dV"), g):
            assert _err(got[b], ref[name]) <= TOL, name


# ---- channel-last ---------------------------------------------------------------------------------------------
def test_channel_last_reads_directly():
    rng = np.random.default_rng(17)
    outer, seq, heads, ch = 2, 300, 3, 64
    Q, K, V, dO = (torch.from_numpy(rng.standard_normal((outer, seq, heads, ch)).astype(np.float32)).cuda()
                   .to(torch.bfloat16) for _ in range(4))
    _capi.lib.fa_launch_count(1)
    O = fa.causal_1d(Q, K, V, "none_front", layout="channel_last")
    torch.cuda.synchronize()
    assert _capi.lib.fa_last_path() == 2 and _capi.lib.fa_launch_count(1) == 1   # no adapter pass
    Oc = fa.causal_1d(*(fa.from_channel_last(x) for x in (Q, K, V)), "none_front")
    assert torch.equal(O, fa.to_channel_last(Oc))
    tq, tk, tv = (x.clone().requires_grad_(True) for x in (Q, K, V))
    g = torch.autograd.grad(fa.causal_1d(tq, tk, tv, "none_front", layout="channel_last"), (tq, tk, tv), dO)
    cq, ck, cv = (fa.from_channel_last(x).requires_grad_(True) for x in (Q, K, V))
    gc = torch.autograd.grad(fa.causal_1d(cq, ck, cv, "none_front"), (cq, ck, cv), fa.from_channel_last(dO))
    for a, b in zip(g, gc):
        assert _err(a, fa.to_channel_last(b).double().cpu().numpy()) <= TOL


@pytest.mark.parametrize("shape", [(2, 300, 3, 64), (1, 77, 2, 40), (3, 64, 1, 128), (2, 31, 5, 9)])
def test_layout_adapters_round_trip_bit_exactly(shape):
    x = torch.randn(shape, device="cuda").to(torch.bfloat16)
    y = fa.from_channel_last(x)
    assert torch.equal(y, x.permute(0, 2, 3, 1))
    assert torch.equal(fa.to_channel_last(y), x)


# ---- the generic family ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,v_d,override", [(160, 160, 0), (320, 64, 0), (64, 64, 1)])
def test_generic_family(d, v_d, override):
    _check(1, "causal", "scale_front", 1, 0, False, (2,), d, v_d, (193,), (277,), d + v_d, mode=0, path=1,
           override=override)


@pytest.mark.parametrize("override", [4, 1])
def test_backward_is_deterministic(override):
    (tq, tk, tv, tdo), _ = _inputs(11, (2,), 64 if override == 4 else 160, 64, (384,), (384,))
    _capi.lib.fa_set_path_override(override)
    try:
        O, l, m = fa.causal_1d(tq, tk, tv, "none_front", returning_l_m=True)
        runs = [fa.attention_backward(1, "causal", tq, tk, tv, O, l, m, tdo, "none_front") for _ in range(2)]
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == (2 if override == 4 else 1)
    finally:
        _capi.lib.fa_set_path_override(0)
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ---- ring pieces -----------------------------------------------------------------------------------------------
def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("merge", [False, True])
def test_key_shards_merge_to_one_call(merge):
    """accumulate = 1 over two key shards (generic forward), and fa_partial_merge / finalize of two tensor-core shards,
    against one call over the whole sequence."""
    n, d = 384, 64
    (tq, tk, tv, _), (Qn, Kn, Vn, _) = _inputs(9, (3,), d, d, (n,), (n,))
    ref = da.attention(Qn, Kn, Vn, 1, "causal", "none_front")
    full = fa.causal_1d(tq, tk, tv, "none_front")
    O = torch.empty((3, d, n), dtype=torch.bfloat16, device="cuda")
    l = torch.empty((3, n), dtype=torch.float32, device="cuda")
    m = torch.empty((3, n), dtype=torch.bfloat16, device="cuda")
    acc = [torch.empty(sh, dtype=torch.float32, device="cuda") for sh in ((3, d, n), (3, n), (3, n))]
    for step, (k0, k1) in enumerate(((192, 384), (0, 192))):
        sk, sv = (x[:, :, k0:k1].contiguous() for x in (tk, tv))
        p = _capi.make_problem(_capi.FA_BF16, 1, "causal", "none_front", (3, d, n), (3, d, k1 - k0), (3, d, k1 - k0))
        p.k_index_base, p.k_full_len, p.q_full_len = k0, n, n
        p.accumulate = int(step > 0 and not merge)
        if merge:
            Op, lp, mp = torch.empty_like(O), torch.empty_like(l), torch.empty_like(m)
        else:
            Op, lp, mp = O, l, m
        assert _capi.lib.fa_workspace_bytes(C.byref(p), 0) == 0
        _capi.check(_capi.lib.fa_forward(C.byref(p), tq.data_ptr(), sk.data_ptr(), sv.data_ptr(), Op.data_ptr(),
                                         lp.data_ptr(), mp.data_ptr(), None, 0, _stream()))
        torch.cuda.synchronize()
        assert _capi.lib.fa_last_path() == (1 if p.accumulate else 2)
        if merge:
            _capi.check(_capi.lib.fa_partial_merge(C.byref(p), Op.data_ptr(), lp.data_ptr(), mp.data_ptr(),
                                                   *(a.data_ptr() for a in acc), int(step == 0), _stream()))
    if merge:
        _capi.check(_capi.lib.fa_partial_finalize(C.byref(p), *(a.data_ptr() for a in acc), O.data_ptr(), l.data_ptr(),
                                                  m.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert _err(O, ref["O"]) <= TOL
    assert _err(O, full.double().cpu().numpy()) <= TOL
    lse = m.double().cpu().numpy() + np.log(l.double().cpu().numpy())
    assert np.max(np.abs(lse - (ref["m"] + np.log(ref["l"])))) <= TOL


def test_backward_accumulate_equals_backward_plus_grad_accumulate():
    B, d, nq, nk = 4, 128, 384, 512
    (tq, tk, tv, tdo), _ = _inputs(9, (B,), d, d, (nq,), (nk,))
    O, l, m = fa.full_1d(tq, tk, tv, "none_front", returning_l_m=True)
    p = _capi.make_problem(_capi.FA_BF16, 1, "full", "none_front", tq.shape, tk.shape, tv.shape)
    assert _capi.lib.fa_backward_accumulate_supported(C.byref(p), 0) == 1
    need = _capi.lib.fa_workspace_bytes(C.byref(p), 1)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    acc = torch.full((B, d, nq), 0.5, dtype=torch.float32, device="cuda")
    dk, dv = torch.empty_like(tk), torch.empty_like(tv)
    _capi.check(_capi.lib.fa_backward_accumulate(C.byref(p), tq.data_ptr(), tk.data_ptr(), tv.data_ptr(), O.data_ptr(),
                                                 l.data_ptr(), m.data_ptr(), tdo.data_ptr(), acc.data_ptr(),
                                                 dk.data_ptr(), dv.data_ptr(), 0, ws.data_ptr(), need, _stream()))
    dQ, dK, dV = fa.attention_backward(1, "full", tq, tk, tv, O, l, m, tdo, "none_front")
    acc2 = torch.full((B, d, nq), 0.5, dtype=torch.float32, device="cuda")
    _capi.check(_capi.lib.fa_grad_accumulate(_capi.FA_BF16, dQ.data_ptr(), acc2.data_ptr(), dQ.numel(), 0, _stream()))
    fin = torch.empty_like(dQ)
    _capi.check(_capi.lib.fa_grad_finalize(_capi.FA_BF16, acc2.data_ptr(), fin.data_ptr(), dQ.numel(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(fin, (dQ.float() + 0.5).to(torch.bfloat16))
    assert torch.equal(dk, dK) and torch.equal(dv, dV)
    assert _err(acc, acc2.double().cpu().numpy()) <= TOL


@pytest.mark.parametrize("driver", ["native", "python"])
def test_single_rank_ring(driver, monkeypatch):
    monkeypatch.setenv("FA_RING_DRIVER", driver)
    (tq, tk, tv, tdo), (Qn, Kn, Vn, dOn) = _inputs(3, (2, 2), 128, 128, (1024,), (1024,))
    ref = da.attention(Qn, Kn, Vn, 1, "causal", "none_front", dO=dOn)
    O, l, m = ring.ring_causal_1d(tq, tk, tv, returning_l_m=True)
    assert O.dtype == torch.bfloat16 and l.dtype == torch.float32
    assert _err(O, ref["O"]) <= TOL
    dQ, dK, dV = ring.ring_causal_1d_backward(tq, tk, tv, O, l, m, tdo)
    assert _capi.lib.fa_last_path() == 2
    _, of_o, _ = _grad_refs(Qn, Kn, Vn, dOn, O.double().cpu().numpy(), 1, "causal", "none_front", 1, 0, False)
    for name, g in (("dQ", dQ), ("dK", dK), ("dV", dV)):
        assert _err(g, of_o[name]) <= TOL, name


# ---- host buffers ------------------------------------------------------------------------------------------------
def test_host_buffers_bit_identical_to_device_calls():
    (tq, tk, tv, tdo), _ = _inputs(13, (2, 2), 64, 64, (300,), (256,))
    O, l, m = fa.causal_1d(tq, tk, tv, "scale_front", returning_l_m=True)
    dQ, dK, dV = fa.attention_backward(1, "causal", tq, tk, tv, O, l, m, tdo, "scale_front")
    p = _capi.make_problem(_capi.FA_BF16, 1, "causal", "scale_front", tq.shape, tk.shape, tv.shape)
    hq, hk, hv, hdo = (t.cpu().pin_memory() for t in (tq, tk, tv, tdo))
    ho, hl, hm = (torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in (O, l, m))
    hdq, hdk, hdv = (torch.empty(t.shape, dtype=t.dtype).pin_memory() for t in (dQ, dK, dV))
    arena = torch.empty(_capi.lib.fa_host_arena_bytes(C.byref(p), 1), dtype=torch.uint8, device="cuda")
    _capi.check(_capi.lib.fa_forward_host(C.byref(p), hq.data_ptr(), hk.data_ptr(), hv.data_ptr(), ho.data_ptr(),
                                          hl.data_ptr(), hm.data_ptr(), arena.data_ptr(), arena.numel(), _stream()))
    _capi.check(_capi.lib.fa_backward_host(C.byref(p), hq.data_ptr(), hk.data_ptr(), hv.data_ptr(), ho.data_ptr(),
                                           hl.data_ptr(), hm.data_ptr(), hdo.data_ptr(), hdq.data_ptr(), hdk.data_ptr(),
                                           hdv.data_ptr(), arena.data_ptr(), arena.numel(), _stream()))
    for h, d in ((ho, O), (hl, l), (hm, m), (hdq, dQ), (hdk, dK), (hdv, dV)):
        assert torch.equal(h, d.cpu())
