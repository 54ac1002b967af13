"""Sharded 1-D calls on the GPU: a call that sees query rows [q_index_base, q_index_base + nq) and keys
[k_index_base, k_index_base + nk) of sequences of q_full_len / k_full_len positions, on every kernel family, against the
float64 oracle of the whole sequence.

Reference: the oracle's global pattern (pattern.tests_mask on the full lengths) sliced to the block. A block's forward is
compared with da.forward on the block; merged shards and summed gradient blocks with the whole-sequence oracle. Bars are
those of the other parity tests: 2e-3 (fp16), 1.6e-2 (bf16), 1e-5 (fp32), 1e-12 (fp64) on O (max-abs; bf16 relative
to max(1, |ref|)) and on the gradients (relative to max(1, |ref|)), the lse / m bars of test_gpu_parity._check, and rows
with no attended key exactly o = 0, l = 0, m = bytes 0xFA. bf16 gradients are compared with the oracle's backward of the
bf16 O the call was given (its D = rowsum(dO o O) inherits O's rounding), as in test_gpu_bf16. Every call asserts the
kernel family it ran on (fa_last_path()), so a silent fall-back cannot pass."""
import ctypes as C

import numpy as np
import pytest

from oracle import dense_attention as da
from oracle import pattern
from tests.helpers import max_abs_err, scaled_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from tf_flash_attention_b200 import _capi, ring  # noqa: E402

lib = _capi.lib
# dtype: (C code, torch dtype, NumPy dtype the inputs are drawn in, bar, lse / m bar)
DT = {"f16": (_capi.FA_F16, torch.float16, np.float16, 2e-3, 2e-2),
      "bf16": (_capi.FA_BF16, torch.bfloat16, np.float32, 1.6e-2, 1.6e-2),
      "f32": (_capi.FA_F32, torch.float32, np.float32, 1e-5, 1e-5),
      "f64": (_capi.FA_F64, torch.float64, np.float64, 1e-12, 1e-12)}
# rule, window, log2 stride, is_causal
ATTN = {"full": ("full", 1, 0, False), "causal": ("causal", 1, 0, False), "local": ("local", 40, 0, False),
        "local_stride": ("local", 6, 2, False), "local_stride_causal": ("local", 16, 1, True),
        "narrow": ("local", 8, 0, False)}
# kernel family: dtype, d, v_d, fa_set_path_override, fa_last_path()
FAMILIES = {
    "f16-d64": ("f16", 64, 64, 0, 2),             # 64-key tiles, two CTAs per SM
    "f16-d64-ov5": ("f16", 64, 64, 5, 2),         # 128-key tiles
    "f16-d64-ov4": ("f16", 64, 64, 4, 2),         # two-slot backward
    "f16-d20": ("f16", 20, 20, 0, 2),             # channels padded to 64
    "f16-d128": ("f16", 128, 128, 0, 2),          # fused backward
    "f16-d128-ov4": ("f16", 128, 128, 4, 2),      # two-kernel backward
    "bf16-d64": ("bf16", 64, 64, 0, 2),
    "bf16-d128": ("bf16", 128, 128, 0, 2),
    "f32-64x64": ("f32", 64, 64, 0, 3),           # 3xTF32 forward, bf16x3 backward
    "f32-32x16": ("f32", 32, 16, 0, 3),
    "f64-32x48": ("f64", 32, 48, 0, 4),           # DMMA
    "f64-64x64": ("f64", 64, 64, 0, 4),
    "generic-f16": ("f16", 64, 64, 1, 1),
    "generic-bf16": ("bf16", 64, 64, 1, 1),
    "generic-f32": ("f32", 32, 16, 1, 1),
    "generic-f64": ("f64", 32, 48, 1, 1),
    "generic-f32-d320": ("f32", 320, 64, 0, 1),   # channel-sliced generic kernels
}
MAX_ERR = {}


@pytest.fixture(scope="module", autouse=True)
def _report_errors():
    yield
    print("\nlargest error per dtype (O / gradients relative to the bar's scale):",
          {k: f"{v:.3g}" for k, v in sorted(MAX_ERR.items())})


def _note(dt, err):
    MAX_ERR[dt] = max(MAX_ERR.get(dt, 0.0), err)
    return err


class _settings:
    """fa_set_path_override / fa_set_grad_precision for the duration of a block"""

    def __init__(self, override=0, grad=0):
        self.override, self.grad = override, grad

    def __enter__(self):
        lib.fa_set_path_override(self.override)
        assert lib.fa_set_grad_precision(self.grad) == _capi.FA_OK

    def __exit__(self, *exc):
        lib.fa_set_path_override(0)
        lib.fa_set_grad_precision(0)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _inputs(dt, seed, B, d, vd, qf, kf):
    """Q, K, V, dO of the whole sequence as CUDA tensors of the dtype, and their float64 values"""
    rng = np.random.default_rng(seed)
    ts = [torch.from_numpy(x).cuda().to(DT[dt][1]) for x in da.random_inputs(rng, DT[dt][2], (B,), d, vd, (qf,), (kf,))]
    return ts, [t.double().cpu().numpy() for t in ts]


def _sl(x, a, n):
    return x[..., a:a + n].contiguous()


def _mask(attn, mode, qf, kf):
    rule, w, s, c = ATTN[attn]
    return pattern.tests_mask((qf,), (kf,), mode, rule, w, s, c)


def _problem(dt, attn, mode, B, d, vd, nq, nk, qb=0, kb=0, qf=0, kf=0, accumulate=0):
    rule, w, s, c = ATTN[attn]
    p = _capi.make_problem(DT[dt][0], 1, rule, mode, (B, d, nq), (B, d, nk), (B, vd, nk), w, s, c)
    p.q_index_base, p.k_index_base, p.q_full_len, p.k_full_len, p.accumulate = qb, kb, qf, kf, accumulate
    return p


def _workspace(p, backward):
    need = lib.fa_workspace_bytes(C.byref(p), int(backward))
    return torch.empty(max(need, 256), dtype=torch.uint8, device="cuda"), need


def _new_out(p, like):
    ldt = torch.float32 if like.dtype in (torch.float16, torch.bfloat16) else like.dtype
    B, nq = p.batch, p.q_shape[0]
    return (torch.full((B, p.v_d, nq), float("nan"), dtype=like.dtype, device="cuda"),
            torch.full((B, nq), float("nan"), dtype=ldt, device="cuda"),
            torch.full((B, nq), float("nan"), dtype=like.dtype, device="cuda"))


def _forward(p, q, k, v, path, out=None):
    O, l, m = out if out is not None else _new_out(p, q)
    ws, need = _workspace(p, False)
    _capi.check(lib.fa_forward(C.byref(p), q.data_ptr(), k.data_ptr(), v.data_ptr(), O.data_ptr(), l.data_ptr(),
                               m.data_ptr(), ws.data_ptr(), need, _stream()), "fa_forward")
    torch.cuda.synchronize()
    assert lib.fa_last_path() == path, f"forward ran on family {lib.fa_last_path()}, not {path}"
    return O, l, m


def _backward(p, q, k, v, o, l, m, do, path):
    dq, dk, dv = (torch.full_like(x, float("nan")) for x in (q, k, v))
    ws, need = _workspace(p, True)
    _capi.check(lib.fa_backward(C.byref(p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), l.data_ptr(),
                                m.data_ptr(), do.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), ws.data_ptr(),
                                need, _stream()), "fa_backward")
    torch.cuda.synchronize()
    assert lib.fa_last_path() == path, f"backward ran on family {lib.fa_last_path()}, not {path}"
    return dq, dk, dv


def _check_out(dt, got, ref, tag):
    """O, l, m of a call against the oracle's (O, l, m); m = -inf marks rows with no attended key"""
    O, l, m = got
    Oref, lref, mref = ref
    tol, mtol = DT[dt][3], DT[dt][4]
    On, ln, mn = (x.double().cpu().numpy() for x in (O, l, m))
    err = scaled_err(On, Oref) if dt == "bf16" else max_abs_err(On, Oref)
    assert _note(dt, err) <= tol, f"O {tag}: {err}"
    empty = ~np.isfinite(mref)
    if empty.any():
        assert np.all(ln[empty] == 0), f"l of empty rows {tag}"
        mb = m.cpu().view(torch.uint8).numpy().reshape(m.shape + (m.element_size(),))
        assert np.all(mb[empty] == 0xFA), f"m of empty rows {tag}"
        assert np.all(On.transpose(0, 2, 1)[empty] == 0), f"O of empty rows {tag}"
    live = ~empty
    if live.any():
        lse = mn[live] + np.log(ln[live])
        assert np.max(np.abs(lse - (mref[live] + np.log(lref[live])))) <= max(mtol, tol * 4), f"lse {tag}"
        assert np.max(np.abs(mn[live] - mref[live]) / np.maximum(1, np.abs(mref[live]))) <= mtol, f"m {tag}"


def _grad_parts(Qn, Kn, Vn, dOn, mask, On=None):
    """P and dS of the whole sequence (float64); D from the exact O, or from On (the O the backward was given)"""
    O, _, _, P = da.forward(Qn, Kn, Vn, mask, return_p=True)
    D = np.einsum("bcq,bcq->bq", dOn, O if On is None else On)
    dS = P * (np.einsum("bcq,bck->bqk", dOn, Vn) - D[..., None]) / np.sqrt(np.float64(Qn.shape[1]))
    return P, dS


def _block_grads(Qn, Kn, dOn, P, dS, q0, q1, k0, k1):
    """dQ, dK, dV of the block (queries q0:q1, keys k0:k1) with the whole sequence's statistics"""
    ds, pp = dS[:, q0:q1, k0:k1], P[:, q0:q1, k0:k1]
    return (np.einsum("bqk,bck->bcq", ds, Kn[..., k0:k1]), np.einsum("bqk,bcq->bck", ds, Qn[..., q0:q1]),
            np.einsum("bqk,bcq->bck", pp, dOn[..., q0:q1]))


# ---- (a) per-block forward -----------------------------------------------------------------------------------
# attn, sync mode, q_full, k_full, (q base, rows), (k base, keys), batch. Bases 77 / 301 are not multiples of 8; the
# fp16 lengths 299, 397, 203, 333 are not either, so the pack pass runs with a base.
GEOMS = {
    "both-causal": ("causal", "none_front", 1000, 1000, (301, 299), (77, 397), 2),
    "both-stride-scale_end": ("local_stride", "scale_end", 450, 900, (77, 203), (301, 397), 2),
    "q-only-full-scale_end": ("full", "scale_end", 900, 600, (301, 333), (0, 600), 2),
    "k-only-local-scale_front": ("local", "scale_front", 400, 800, (0, 400), (77, 301), 2),
    "both-stride-causal-scale_front": ("local_stride_causal", "scale_front", 800, 400, (301, 299), (77, 203), 2),
    "all-rows-empty": ("causal", "none_front", 1000, 1000, (64, 100), (600, 200), 2),
    "some-rows-empty": ("narrow", "none_front", 1000, 1000, (301, 150), (400, 100), 2),
    "batch1-short-queries": ("local_stride_causal", "scale_end", 1000, 1000, (301, 40), (77, 900), 1),
}
FWD_FAMILIES = [f for f in FAMILIES if not f.endswith("-ov4")]


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("family", FWD_FAMILIES)
def test_block_forward(family, geom):
    dt, d, vd, override, path = FAMILIES[family]
    attn, mode, qf, kf, (qb, nq), (kb, nk), B = GEOMS[geom]
    (Q, K, V, _), (Qn, Kn, Vn, _) = _inputs(dt, 7, B, d, vd, qf, kf)
    mask = _mask(attn, mode, qf, kf)[qb:qb + nq, kb:kb + nk]
    if geom == "all-rows-empty":
        assert not mask.any()
    if geom == "some-rows-empty":
        assert mask.any() and not mask.any(axis=1).all()
    ref = da.forward(Qn[..., qb:qb + nq], Kn[..., kb:kb + nk], Vn[..., kb:kb + nk], mask)
    p = _problem(dt, attn, mode, B, d, vd, nq, nk, qb, kb, qf, kf)
    with _settings(override):
        got = _forward(p, _sl(Q, qb, nq), _sl(K, kb, nk), _sl(V, kb, nk), path)
    _check_out(dt, got, ref, f"{family} {geom}")


# ---- (b) merging key shards -----------------------------------------------------------------------------------
MERGE_FAMILIES = ["f16-d64", "f16-d128", "bf16-d64", "bf16-d128", "f32-64x64", "f32-32x16", "f64-32x48"]
MERGE_GEOMS = {"causal": ("causal", "none_front", 1000, 1000), "stride-scale_end": ("local_stride", "scale_end", 700, 1400)}


def _key_shards(kf):
    """three uneven shards, visited out of order"""
    cuts = [0, kf * 3 // 10 + 1, kf * 4 // 10 + 3, kf]
    shards = [(cuts[i], cuts[i + 1] - cuts[i]) for i in range(3)]
    return [shards[2], shards[0], shards[1]]


@pytest.mark.parametrize("how", ["partial_merge", "accumulate"])
@pytest.mark.parametrize("nq", [600, 601])
@pytest.mark.parametrize("geom", list(MERGE_GEOMS))
@pytest.mark.parametrize("family", MERGE_FAMILIES)
def test_key_shards_merge_to_the_whole_sequence(family, geom, nq, how):
    """fa_partial_merge + fa_partial_finalize over tensor-core shards (an even and an odd number of rows: the 16-bit
    pair kernels and the scalar kernels), or the accumulate = 1 chain of the generic forward, over three uneven key shards
    visited out of order, for a query shard at base 77: O, l, m equal the whole-sequence oracle."""
    dt, d, vd, override, path = FAMILIES[family]
    attn, mode, qf, kf = MERGE_GEOMS[geom]
    B, qb = 2, 77
    (Q, K, V, _), (Qn, Kn, Vn, _) = _inputs(dt, 11, B, d, vd, qf, kf)
    O, l, m = da.forward(Qn, Kn, Vn, _mask(attn, mode, qf, kf))
    ref = (O[..., qb:qb + nq], l[:, qb:qb + nq], m[:, qb:qb + nq])
    q = _sl(Q, qb, nq)
    acc_dt = torch.float64 if dt == "f64" else torch.float32
    acc = [torch.empty(sh, dtype=acc_dt, device="cuda") for sh in ((B, vd, nq), (B, nq), (B, nq))]
    out = None
    for i, (kb, nk) in enumerate(_key_shards(kf)):
        accumulate = int(how == "accumulate" and i > 0)
        p = _problem(dt, attn, mode, B, d, vd, nq, nk, qb, kb, qf, kf, accumulate)
        k, v = _sl(K, kb, nk), _sl(V, kb, nk)
        if how == "accumulate":
            out = _forward(p, q, k, v, 1 if accumulate else path, out)
            continue
        part = _forward(p, q, k, v, path)
        _capi.check(lib.fa_partial_merge(C.byref(p), *(x.data_ptr() for x in part), *(a.data_ptr() for a in acc),
                                         int(i == 0), _stream()), "fa_partial_merge")
    if how == "partial_merge":
        out = _new_out(p, q)
        _capi.check(lib.fa_partial_finalize(C.byref(p), *(a.data_ptr() for a in acc), *(x.data_ptr() for x in out),
                                            _stream()), "fa_partial_finalize")
        torch.cuda.synchronize()
    _check_out(dt, out, ref, f"{family} {geom} nq{nq} {how}")


# ---- (c) backward blocks ----------------------------------------------------------------------------------------
# attn, sync mode, q_full, k_full, query shard cuts, key shard cuts: key shards of at most 128 keys, so that grad
# precision 0 picks the precise 16-bit kernels; odd lengths at d = 20 give element counts that are not multiples of 8
BWD_GEOMS = {"causal": ("causal", "none_front", 380, 380, [0, 187, 380], [0, 125, 253, 380]),
             "stride-scale_front": ("local_stride", "scale_front", 380, 190, [0, 187, 380], [0, 61, 125, 190])}
BWD_CASES = ([(f, g) for f in ("f16-d20", "f16-d64", "f16-d64-ov4", "f16-d128", "f16-d128-ov4", "bf16-d64", "bf16-d128")
              for g in (0, 1, 2)] +
             [(f, 0) for f in ("f32-64x64", "f32-32x16", "f64-32x48", "generic-f16", "generic-bf16", "generic-f32",
                               "generic-f64", "generic-f32-d320")])


def _sum_blocks(dt, attn, mode, d, vd, path, Q, K, V, O, l, m, dO, qf, kf, qcuts, kcuts):
    """dQ, dK, dV of the whole sequence as the sums, over every (query shard, key shard) block, of fa_backward with the
    block's bases and the final O, l, m, folded with fa_grad_accumulate / fa_grad_finalize"""
    B = Q.shape[0]
    acc_dt = torch.float64 if dt == "f64" else torch.float32
    qsh = [(qcuts[i], qcuts[i + 1] - qcuts[i]) for i in range(len(qcuts) - 1)]
    ksh = [(kcuts[i], kcuts[i + 1] - kcuts[i]) for i in range(len(kcuts) - 1)]
    ksh = ksh[1:] + ksh[:1]
    dq_acc = [torch.empty((B, d, n), dtype=acc_dt, device="cuda") for _, n in qsh]
    dk_acc = [torch.empty((B, d, n), dtype=acc_dt, device="cuda") for _, n in ksh]
    dv_acc = [torch.empty((B, vd, n), dtype=acc_dt, device="cuda") for _, n in ksh]
    for i, (qb, nq) in enumerate(qsh):
        for j, (kb, nk) in enumerate(ksh):
            p = _problem(dt, attn, mode, B, d, vd, nq, nk, qb, kb, qf, kf)
            parts = _backward(p, _sl(Q, qb, nq), _sl(K, kb, nk), _sl(V, kb, nk), _sl(O, qb, nq),
                              l[:, qb:qb + nq].contiguous(), m[:, qb:qb + nq].contiguous(), _sl(dO, qb, nq), path)
            for part, acc, first in ((parts[0], dq_acc[i], j == 0), (parts[1], dk_acc[j], i == 0),
                                     (parts[2], dv_acc[j], i == 0)):
                _capi.check(lib.fa_grad_accumulate(DT[dt][0], part.data_ptr(), acc.data_ptr(), part.numel(),
                                                   int(first), _stream()), "fa_grad_accumulate")

    def fin(accs, shards):
        outs = []
        for a, _ in zip(accs, shards):
            o = torch.empty(a.shape, dtype=Q.dtype, device="cuda")
            _capi.check(lib.fa_grad_finalize(DT[dt][0], a.data_ptr(), o.data_ptr(), a.numel(), _stream()))
            outs.append(o)
        return torch.cat(outs, dim=-1)
    order = np.argsort([kb for kb, _ in ksh])
    dQ = fin(dq_acc, qsh)
    dK = fin([dk_acc[j] for j in order], ksh)
    dV = fin([dv_acc[j] for j in order], ksh)
    torch.cuda.synchronize()
    return dQ, dK, dV


@pytest.mark.parametrize("geom", list(BWD_GEOMS))
@pytest.mark.parametrize("family,grad", BWD_CASES, ids=lambda v: str(v))
def test_backward_blocks_sum_to_the_whole_sequence(family, grad, geom):
    """Two query shards x three key shards (key shards only: partial_keys on), and the two query shards over all keys
    (query-only shards: exact D / renormalisation stay on); both sums equal the whole-sequence oracle."""
    dt, d, vd, override, path = FAMILIES[family]
    attn, mode, qf, kf, qcuts, kcuts = BWD_GEOMS[geom]
    B = 3
    (Q, K, V, dO), (Qn, Kn, Vn, dOn) = _inputs(dt, 13, B, d, vd, qf, kf)
    mask = _mask(attn, mode, qf, kf)
    with _settings(override, grad):
        O, l, m = _forward(_problem(dt, attn, mode, B, d, vd, qf, kf), Q, K, V, path)
        On = O.double().cpu().numpy() if dt == "bf16" else None
        P, dS = _grad_parts(Qn, Kn, Vn, dOn, mask, On)
        want = _block_grads(Qn, Kn, dOn, P, dS, 0, qf, 0, kf)
        for cuts in (kcuts, [0, kf]):
            got = _sum_blocks(dt, attn, mode, d, vd, path, Q, K, V, O, l, m, dO, qf, kf, qcuts, cuts)
            for name, g, w in zip(("dQ", "dK", "dV"), got, want):
                err = scaled_err(g.double().cpu().numpy(), w)
                assert _note(dt, err) <= DT[dt][3], f"{name} {family} grad{grad} {geom} key cuts {cuts}: {err}"


# ---- (d) fa_backward_accumulate on sharded blocks ---------------------------------------------------------------
@pytest.mark.parametrize("dt,vd", [("f16", 128), ("f16", 64), ("bf16", 128)])
@pytest.mark.parametrize("fold", [0, 2])
def test_backward_accumulate_over_key_shards(dt, vd, fold):
    """d = 128, a query shard at base 320 and key shards at bases 320, 640 and 0 (visited in that order): dQ summed into
    the fp32 accumulator inside the launch (dq_fold = batch, or batch / 2), dK / dV of each block."""
    B, d, qf, kf, qb, nq = 4, 128, 1024, 1024, 320, 384
    (Q, K, V, dO), (Qn, Kn, Vn, dOn) = _inputs(dt, 17, B, d, vd, qf, kf)
    mask = _mask("causal", "none_front", qf, kf)
    O, l, m = _forward(_problem(dt, "causal", "none_front", B, d, vd, qf, kf), Q, K, V, 2)
    P, dS = _grad_parts(Qn, Kn, Vn, dOn, mask, O.double().cpu().numpy() if dt == "bf16" else None)
    nacc = fold or B
    acc = torch.zeros((nacc, d, nq), dtype=torch.float32, device="cuda")
    q, o, do = _sl(Q, qb, nq), _sl(O, qb, nq), _sl(dO, qb, nq)
    lq, mq = l[:, qb:qb + nq].contiguous(), m[:, qb:qb + nq].contiguous()
    tol = DT[dt][3]
    for kb, nk in ((320, 320), (640, 384), (0, 320)):
        p = _problem(dt, "causal", "none_front", B, d, vd, nq, nk, qb, kb, qf, kf)
        assert lib.fa_backward_accumulate_supported(C.byref(p), fold) == 1
        ws, need = _workspace(p, True)
        k, v = _sl(K, kb, nk), _sl(V, kb, nk)
        dk, dv = torch.full_like(k, float("nan")), torch.full_like(v, float("nan"))
        _capi.check(lib.fa_backward_accumulate(C.byref(p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                               lq.data_ptr(), mq.data_ptr(), do.data_ptr(), acc.data_ptr(), dk.data_ptr(),
                                               dv.data_ptr(), fold, ws.data_ptr(), need, _stream()),
                    "fa_backward_accumulate")
        torch.cuda.synchronize()
        assert lib.fa_last_path() == 2
        _, wk, wv = _block_grads(Qn, Kn, dOn, P, dS, qb, qb + nq, kb, kb + nk)
        for name, g, w in (("dK", dk, wk), ("dV", dv, wv)):
            err = scaled_err(g.double().cpu().numpy(), w)
            assert _note(dt, err) <= tol, f"{name} block k{kb}: {err}"
    wq = _block_grads(Qn, Kn, dOn, P, dS, qb, qb + nq, 0, kf)[0]
    wq = wq.reshape(B // nacc, nacc, d, nq).sum(axis=0)
    err = scaled_err(acc.double().cpu().numpy(), wq)
    assert _note(dt, err) <= tol, f"dQ accumulator: {err}"


# ---- (e) bit-exact invariances ----------------------------------------------------------------------------------
TC_FAMILIES = ["f16-d64", "f16-d64-ov4", "f16-d20", "f16-d128", "f16-d128-ov4", "bf16-d64", "bf16-d128", "f32-64x64",
               "f32-32x16", "f64-32x48", "generic-f16", "generic-f32"]


def _run_order(family, grad):
    """gradients whose sums are added up in a run-dependent order: dQ of the fused 16-bit head_dim-128 backward, and every
    gradient of the fp64 tensor-core backward, whose small grids split the streamed tiles and add the parts atomically"""
    dt, d, _, override, path = FAMILIES[family]
    if path == 4:
        return ("dQ", "dK", "dV")
    return ("dQ",) if dt in ("f16", "bf16") and d == 128 and override == 0 and grad != 1 else ()


def _same(a, b, dt, run_order, name):
    if name in run_order:
        assert scaled_err(a.double().cpu().numpy(), b.double().cpu().numpy()) <= DT[dt][3], name
    else:
        assert torch.equal(a, b), name


@pytest.mark.parametrize("grad", [0, 1])
@pytest.mark.parametrize("family", TC_FAMILIES)
def test_explicit_full_lengths_and_zero_bases_change_nothing(family, grad):
    """q_full_len = nq, k_full_len = nk and zero bases, set explicitly, give the bytes of a call that leaves them at 0
    (the call is not a key shard: exact D and renormalisation stay on)."""
    dt, d, vd, override, path = FAMILIES[family]
    B, nq, nk = 2, 299, 397
    (Q, K, V, dO), _ = _inputs(dt, 19, B, d, vd, nq, nk)
    runs = []
    with _settings(override, grad):
        for explicit in (False, True):
            p = _problem(dt, "causal", "scale_end", B, d, vd, nq, nk)
            if explicit:
                p.q_full_len, p.k_full_len = nq, nk
            O, l, m = _forward(p, Q, K, V, path)
            runs.append((O, l, m) + _backward(p, Q, K, V, O, l, m, dO, path))
    for name, a, b in zip(("O", "l", "m", "dQ", "dK", "dV"), *runs):
        _same(a, b, dt, _run_order(family, grad), name)


@pytest.mark.parametrize("block", ["q-only", "k-only", "both"])
@pytest.mark.parametrize("family", TC_FAMILIES)
def test_full_rule_block_equals_the_unsharded_call_on_its_slice(family, block):
    """Under the full rule the pattern does not depend on positions: a block with bases gives the bytes of an unsharded
    call on the sliced tensors - O, l, m always, and the gradients wherever the call's numerics are the same. A key
    shard (k base != 0) takes D from O and skips the fp32 backward's renormalisation, which the unsharded call does not;
    so key shards are compared bit for bit with grad precision 2 (plain 16-bit kernels, no exact D) and at the bar
    for fp32."""
    dt, d, vd, override, path = FAMILIES[family]
    B, qf, kf = 2, 700, 900
    qb, nq = (301, 299) if block != "k-only" else (0, qf)
    kb, nk = (77, 397) if block != "q-only" else (0, kf)
    grad = 2 if kb else 0
    (Q, K, V, dO), _ = _inputs(dt, 23, B, d, vd, qf, kf)
    q, k, v, do = _sl(Q, qb, nq), _sl(K, kb, nk), _sl(V, kb, nk), _sl(dO, qb, nq)
    runs = []
    with _settings(override, grad):
        for sharded in (False, True):
            p = _problem(dt, "full", "none_front", B, d, vd, nq, nk, *((qb, kb, qf, kf) if sharded else ()))
            O, l, m = _forward(p, q, k, v, path)
            runs.append((O, l, m) + _backward(p, q, k, v, O, l, m, do, path))
    for name, a, b in zip(("O", "l", "m", "dQ", "dK", "dV"), *runs):
        if kb and dt == "f32" and name in ("dQ", "dK", "dV"):
            assert scaled_err(b.double().cpu().numpy(), a.double().cpu().numpy()) <= DT[dt][3], name
        else:
            _same(a, b, dt, _run_order(family, grad), name)


# ---- (f) the per-block ring on the product backend ------------------------------------------------------------
@pytest.mark.parametrize("attn", ["full", "local", "local_stride_causal"])
@pytest.mark.parametrize("dt,d", [("f16", 64), ("f32", 32), ("f64", 16)])
def test_per_block_ring_on_the_device_backend(dt, d, attn):
    """ring.ring_forward / ring.ring_backward with ring.DeviceBackend (attend_partial, merge, finalize, grad_partial,
    grad_add, grad_finalize) on one rank: both chunks of the zig-zag layout, every block with its global bases."""
    rule, w, s, c = ATTN[attn]
    B, seq = 2, 512
    layout = ring.ZigZag(seq, 1)
    ch = layout.chunk
    (Q, K, V, dO), (Qn, Kn, Vn, dOn) = _inputs(dt, 29, B, d, d, seq, seq)
    backend = ring.DeviceBackend(DT[dt][0], rule, "none_front", w, s, c, (B,), d, d, ch, seq)
    idx = [layout.base(i) for i in layout.chunks(0)]
    qc = [_sl(Q, i, ch) for i in idx]
    kv = [_sl(K, i, ch) for i in idx] + [_sl(V, i, ch) for i in idx]
    outs = ring.ring_forward(backend, layout, 0, qc, kv, rule=rule, is_causal=c)
    torch.cuda.synchronize()
    path = {"f16": 2, "f32": 3, "f64": 4}[dt]
    assert lib.fa_last_path() == path
    mask = _mask(attn, "none_front", seq, seq)
    ref = da.forward(Qn, Kn, Vn, mask)
    for (O, l, m), i in zip(outs, idx):
        _check_out(dt, (O, l, m), (ref[0][..., i:i + ch], ref[1][:, i:i + ch], ref[2][:, i:i + ch]), f"ring {attn}")
    d_q, d_kv = ring.ring_backward(backend, layout, 0, qc, kv, [o[0] for o in outs], [o[1] for o in outs],
                                   [o[2] for o in outs], [_sl(dO, i, ch) for i in idx], rule=rule, is_causal=c)
    torch.cuda.synchronize()
    assert lib.fa_last_path() == path
    want = da.backward(Qn, Kn, Vn, mask, dOn)
    got = (torch.cat(d_q, -1), torch.cat(d_kv[:2], -1), torch.cat(d_kv[2:], -1))
    for name, g, wnt in zip(("dQ", "dK", "dV"), got, want):
        err = scaled_err(g.double().cpu().numpy(), wnt)
        assert _note(dt, err) <= DT[dt][3], f"{name} ring {attn}: {err}"
