"""Operands at unaligned addresses on the GPU: every kernel family, the ring helpers, the torch API and the host-buffer
entry points, with Q, K, V, O, l, m, dO, dQ, dK and dV placed as contiguous views at a byte offset into larger buffers.

Several launchers choose their code path from the operands' addresses, so where a tensor starts decides which code
runs. The 16-bit tensor-core calls read and write a side whose length is a multiple of 8 in place through TMA, which
needs 16-byte-aligned bases; one such operand at another address sends the call to the generic kernels, while a side of
any other length is packed into the workspace at any address. The backward's statistics pass takes pair loads only
when O and dO are 4-byte aligned and nq is even. The fp32 forward splits Q, K, V with float4 loads and stores O by TMA
only when all four are 16-byte aligned, and otherwise runs a scalar split pass and copies a padded O out. The ring
helpers vectorise per argument. Views into a fused QKV buffer, framework slices and the chunks of the host-buffer entry
points all produce such addresses.

Each call is checked four ways: against the float64 oracle at the bars of test_gpu_shards; against the same call on
aligned copies, bit for bit when both run on the same deterministic family (sums added in a run-dependent order, and
calls the address moves to another family, at the bar); for the family that FAMILIES / SIDE16 below predict; and for untouched
guard bands of 0xA5 bytes around every operand. Offsets are multiples of the element size: 2, 4 and 8 bytes for the
16-bit dtypes, 4 and 8 for fp32, 8 for fp64."""
import ctypes as C

import numpy as np
import pytest

from oracle import dense_attention as da
from oracle import pattern
from tests.helpers import scaled_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
from tests import test_gpu_shards as sh  # noqa: E402
from tf_flash_attention_b200 import _capi  # noqa: E402
from tf_flash_attention_b200 import flash_attention as fa  # noqa: E402

lib = _capi.lib
DT = sh.DT
PAD = 512                    # guard bytes on each side; the buffers torch returns are 512-byte aligned
GUARD = 0xA5
DELTAS = {"f16": (2, 4, 8), "bf16": (2, 4, 8), "f32": (4, 8), "f64": (8,)}
IS16 = ("f16", "bf16")


@pytest.fixture(scope="module", autouse=True)
def _report_errors():
    sh.MAX_ERR.clear()
    yield
    print("\nlargest error per dtype (O / gradients relative to the bar's scale):",
          {k: f"{v:.3g}" for k, v in sorted(sh.MAX_ERR.items())})
    sh.MAX_ERR.clear()


def _placed(x, delta, fill=None):
    """(raw buffer, contiguous view at byte offset PAD + delta) holding x, or `fill` for an output; the rest of the
    buffer holds the guard byte"""
    n = x.numel() * x.element_size()
    raw = torch.full((n + 2 * PAD,), GUARD, dtype=torch.uint8, device="cuda")
    view = raw[PAD + delta:PAD + delta + n].view(x.dtype).view(x.shape)
    assert view.data_ptr() % 16 == delta % 16 and view.is_contiguous()
    if fill is None:
        view.copy_(x)
    else:
        view.fill_(fill)
    return raw, view


def _off(t, delta):
    """delta, or the element size where delta is not a multiple of it (the float l of the 16-bit dtypes at +2)"""
    return delta if delta % t.element_size() == 0 else t.element_size()


def _guards_intact(placed, tag):
    torch.cuda.synchronize()
    for name, (raw, view) in placed.items():
        lo = view.data_ptr() - raw.data_ptr()
        hi = lo + view.numel() * view.element_size()
        assert bool((raw[:lo] == GUARD).all()) and bool((raw[hi:] == GUARD).all()), f"{name} {tag}: guard band written"


# ---- kernel families -------------------------------------------------------------------------------------------
# dtype, d, v_d, fa_set_path_override, fa_set_grad_precision, family on aligned tensors
FAMILIES = {
    "f16-d64": ("f16", 64, 64, 0, 0, 2),          # 64-key tiles, two CTAs per SM
    "f16-d64-ov5": ("f16", 64, 64, 5, 0, 2),      # 128-key tiles
    "f16-d64-grad1": ("f16", 64, 64, 0, 1, 2),    # precise (split-operand) backward everywhere
    "f16-d20": ("f16", 20, 20, 0, 0, 2),          # channels padded to 64 by the tensor maps
    "f16-d128": ("f16", 128, 128, 0, 0, 2),       # fused dQ/dK/dV backward
    "f16-d128-ov4": ("f16", 128, 128, 4, 0, 2),   # two-kernel backward
    "bf16-d64": ("bf16", 64, 64, 0, 0, 2),
    "bf16-d64-ov5": ("bf16", 64, 64, 5, 0, 2),
    "bf16-d20": ("bf16", 20, 20, 0, 0, 2),
    "bf16-d128": ("bf16", 128, 128, 0, 0, 2),
    "bf16-d128-ov4": ("bf16", 128, 128, 4, 0, 2),
    "f32-64x64": ("f32", 64, 64, 0, 0, 3),        # 3xTF32 forward, bf16x3 backward
    "f32-32x16": ("f32", 32, 16, 0, 0, 3),
    "f64-32x48": ("f64", 32, 48, 0, 0, 4),        # DMMA
    "generic-f16": ("f16", 64, 64, 1, 0, 1),
    "generic-bf16": ("bf16", 20, 20, 1, 0, 1),
    "generic-f32": ("f32", 32, 16, 1, 0, 1),
    "generic-f64": ("f64", 32, 48, 1, 0, 1),
    "generic-f32-d320": ("f32", 320, 64, 0, 0, 1),   # channel-sliced generic kernels
    "generic-f64-d320": ("f64", 320, 40, 0, 0, 1),
}
# Which side of a 16-bit tensor-core call each operand belongs to (sm100_f16_forward_supports / _backward_supports): on a
# side whose length is a multiple of 8 every operand listed for it must be 16-byte aligned, or the call runs on the
# generic kernels (family 1); a side of any other length is packed into the workspace and stays on family 2. None: read
# or written with element loads and stores (l and m; O in the channel-first backward, read by the statistics pass).
SIDE16 = {"fwd": {"Q": "q", "O": "q", "K": "k", "V": "k", "l": None, "m": None},
          "bwd": {"Q": "q", "dO": "q", "dQ": "q", "K": "k", "V": "k", "dK": "k", "dV": "k", "O": None, "l": None,
                  "m": None}}
# Every other family ignores operand addresses: the fp32 forward falls back to its scalar split pass and a padded O and
# the fp32 backward's split pass reads any address (family 3 throughout), the fp64 DMMA kernels and the generic kernels
# load elements.
FWD_NAMES = ("Q", "K", "V", "O", "l", "m")
BWD_NAMES = ("Q", "K", "V", "O", "l", "m", "dO", "dQ", "dK", "dV")


def expected_family(family, direction, nq, nk, offset):
    path = FAMILIES[family][5]
    if path != 2:
        return path
    packed = {"q": nq % 8 != 0, "k": nk % 8 != 0}
    sides = {SIDE16[direction][n] for n in offset} - {None}
    return 1 if any(not packed[s] for s in sides) else 2


def _run_order(family):
    """gradients added in a run-dependent order: the fused 16-bit head_dim-128 dQ and every fp64 DMMA gradient"""
    dt, d, _, override, grad, path = FAMILIES[family]
    if path == 4:
        return ("dQ", "dK", "dV")
    return ("dQ",) if dt in IS16 and d == 128 and override == 0 and grad != 1 else ()


def _lens(family):
    """(nq, nk): every combination of a length that is a multiple of 8 or not for the 16-bit tensor-core families, with
    nq even (198) and odd (197) for the statistics pass; fp32 lengths that are multiples of 4 (the exact split layout)
    or not"""
    if FAMILIES[family][5] == 2:
        return [(192, 256), (192, 213), (198, 256), (197, 213)]
    return [(192, 256), (197, 213)]


CASES = [(f, n, w) for f in FAMILIES for n in _lens(f) for w in BWD_NAMES + ("all",)]
_BASE = {}


def _base(family, nq, nk):
    """inputs, the oracle, and the forward / backward on aligned tensors (cached per family and lengths)"""
    key = (family, nq, nk)
    if key in _BASE:
        return _BASE[key]
    dt, d, vd, override, grad, path = FAMILIES[family]
    B = 2
    rng = np.random.default_rng(31)
    ts = [torch.from_numpy(x).cuda().to(DT[dt][1])
          for x in da.random_inputs(rng, DT[dt][2], (B,), d, vd, (nq,), (nk,))]
    Qn, Kn, Vn, dOn = (t.double().cpu().numpy() for t in ts)
    mask = pattern.tests_mask((nq,), (nk,), "scale_end", "causal")
    p = sh._problem(dt, "causal", "scale_end", B, d, vd, nq, nk)
    with sh._settings(override, grad):
        out = sh._forward(p, *ts[:3], path)
        grads = sh._backward(p, *ts[:3], *out, ts[3], path)
    P, dS = sh._grad_parts(Qn, Kn, Vn, dOn, mask, out[0].double().cpu().numpy() if dt == "bf16" else None)
    ref = {"fwd": da.forward(Qn, Kn, Vn, mask), "bwd": sh._block_grads(Qn, Kn, dOn, P, dS, 0, nq, 0, nk)}
    _BASE.clear()   # one entry at a time: the cases of a family and lengths are consecutive
    _BASE[key] = (p, ts, out, grads, ref)
    return _BASE[key]


def _compare(dt, names, got, want, same_family, run_order, tag):
    for name, g, w in zip(names, got, want):
        if same_family and name not in run_order:
            assert torch.equal(g, w), f"{name} {tag}: differs from the aligned call"
        else:
            err = scaled_err(g.double().cpu().numpy(), w.double().cpu().numpy())
            assert err <= DT[dt][3], f"{name} {tag}: {err} from the aligned call"


@pytest.mark.parametrize("family,lens,which", CASES,
                         ids=[f"{f}-q{n[0]}k{n[1]}-{w}" for f, n, w in CASES])
def test_operands_at_unaligned_addresses(family, lens, which):
    """One operand (or all of them) at each offset: forward and backward against the oracle, against the aligned call,
    on the expected family, with every guard band intact."""
    dt, d, vd, override, grad, path = FAMILIES[family]
    nq, nk = lens
    p, (Q, K, V, dO), (O, l, m), (dQ, dK, dV), ref = _base(family, nq, nk)
    run_order = _run_order(family)
    for delta in DELTAS[dt]:
        with sh._settings(override, grad):
            if which in FWD_NAMES or which == "all":
                offset = FWD_NAMES if which == "all" else (which,)
                placed = {}
                ins = []
                for name, t in zip(("Q", "K", "V"), (Q, K, V)):
                    if name in offset:
                        placed[name] = _placed(t, _off(t, delta))
                    ins.append(placed[name][1] if name in offset else t)
                outs = []
                for name, t in zip(("O", "l", "m"), (O, l, m)):
                    if name in offset:
                        placed[name] = _placed(t, _off(t, delta), float("nan"))
                    outs.append(placed[name][1] if name in offset else torch.full_like(t, float("nan")))
                want = expected_family(family, "fwd", nq, nk, offset)
                tag = f"{family} q{nq} k{nk} fwd {which}+{delta}"
                sh._forward(p, *ins, want, out=outs)
                _guards_intact(placed, tag)
                _compare(dt, ("O", "l", "m"), outs, (O, l, m), want == path, (), tag)
                sh._check_out(dt, outs, ref["fwd"], tag)
            if which in BWD_NAMES or which == "all":
                offset = BWD_NAMES if which == "all" else (which,)
                placed = {}
                args = []
                for name, t in zip(("Q", "K", "V", "O", "l", "m", "dO"), (Q, K, V, O, l, m, dO)):
                    if name in offset:
                        placed[name] = _placed(t, _off(t, delta))
                    args.append(placed[name][1] if name in offset else t)
                outs = []
                for name, t in zip(("dQ", "dK", "dV"), (Q, K, V)):
                    if name in offset:
                        placed[name] = _placed(t, _off(t, delta), float("nan"))
                    outs.append(placed[name][1] if name in offset else torch.full_like(t, float("nan")))
                want = expected_family(family, "bwd", nq, nk, offset)
                tag = f"{family} q{nq} k{nk} bwd {which}+{delta}"
                ws, need = sh._workspace(p, True)
                _capi.check(lib.fa_backward(C.byref(p), *(x.data_ptr() for x in args), *(x.data_ptr() for x in outs),
                                            ws.data_ptr(), need, sh._stream()), "fa_backward")
                torch.cuda.synchronize()
                assert lib.fa_last_path() == want, f"{tag}: backward ran on family {lib.fa_last_path()}, not {want}"
                _guards_intact(placed, tag)
                _compare(dt, ("dQ", "dK", "dV"), outs, (dQ, dK, dV), want == path, run_order, tag)
                for name, g, w in zip(("dQ", "dK", "dV"), outs, ref["bwd"]):
                    err = scaled_err(g.double().cpu().numpy(), w)
                    assert sh._note(dt, err) <= DT[dt][3], f"{name} {tag}: {err} from the oracle"


# ---- ring helpers ----------------------------------------------------------------------------------------------
PARTIAL_ARGS = ("o_part", "l_part", "m_part", "o_acc", "l_acc", "m_acc", "o", "l", "m")


def _partials(dt, B, vd, nq, seed, empty_rows):
    """a partial result (O, l, m) as fa_forward writes it, with the rows in empty_rows empty (o = 0, l = 0, m = 0xFA..)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    tdt = DT[dt][1]
    o = (torch.rand((B, vd, nq), generator=g, device="cuda") * 2 - 1).to(tdt)
    lp = torch.rand((B, nq), generator=g, device="cuda") * 40 + 0.5
    mp = (torch.rand((B, nq), generator=g, device="cuda") * 8 - 4).to(tdt)
    o[..., empty_rows] = 0
    lp[:, empty_rows] = 0
    mp.view(torch.int16)[:, empty_rows] = 0xFAFA - 0x10000
    empty = np.zeros((B, nq), dtype=bool)
    empty[:, empty_rows] = True
    return (o, lp, mp), (o.double().cpu().numpy(), lp.double().cpu().numpy(), mp.double().cpu().numpy(), empty)


def _merge64(parts):
    """float64 restatement of fa_partial_merge over the parts in order: o_acc, l_acc, m_acc"""
    ma, la, oa = None, None, None
    for o, lp, mp, empty in parts:
        mp = np.where(empty, -np.inf, mp)
        if ma is None:
            ma, la, oa = np.full_like(mp, -np.inf), np.zeros_like(lp), np.zeros_like(o)
        mn = np.maximum(ma, mp)
        with np.errstate(invalid="ignore"):
            wa = np.where(ma == -np.inf, 0.0, np.exp(ma - mn))
            wp = np.where(empty, 0.0, np.exp(mp - mn) * lp)
        la = la * wa + wp
        oa = oa * wa[:, None, :] + o * wp[:, None, :]
        ma = mn
    return oa, la, ma


@pytest.mark.parametrize("which", PARTIAL_ARGS + ("all",))
@pytest.mark.parametrize("dt", IS16)
def test_partial_merge_and_finalize_at_unaligned_addresses(dt, which):
    """Two key shards folded with fa_partial_merge and emitted with fa_partial_finalize, nq even: the pair kernels run on
    aligned arguments, and an argument one element off its pair alignment (2 bytes for 16-bit tensors, 4 for float ones)
    selects the scalar kernels by address alone. Same bytes as the aligned calls, and the float64 restatement of the
    online-softmax algebra (rows empty in one shard and in both included)."""
    B, vd, nq = 2, 24, 130
    p = sh._problem(dt, "full", "none_front", B, 64, vd, nq, 64)
    parts = [_partials(dt, B, vd, nq, 1, [3, 7]), _partials(dt, B, vd, nq, 2, [7, 11])]
    oa64, la64, ma64 = _merge64([x[1] for x in parts])
    live = la64 > 0
    ref = (np.where(live[:, None, :], oa64 / np.where(live, la64, 1)[:, None, :], 0.0), la64,
           np.where(live, ma64, -np.inf))

    def run(offset):
        placed = {}

        def arg(name, t, fill=None):
            if name not in offset:
                return t if fill is None else torch.full_like(t, fill)
            placed[name] = _placed(t, t.element_size(), fill)
            return placed[name][1]
        acc = [arg(n, torch.empty(sz, dtype=torch.float32, device="cuda"), float("nan"))
               for n, sz in (("o_acc", (B, vd, nq)), ("l_acc", (B, nq)), ("m_acc", (B, nq)))]
        for i, ((o, lp, mp), _) in enumerate(parts):
            pa = (arg("o_part", o), arg("l_part", lp), arg("m_part", mp))
            _capi.check(lib.fa_partial_merge(C.byref(p), *(x.data_ptr() for x in pa), *(a.data_ptr() for a in acc),
                                             int(i == 0), sh._stream()), "fa_partial_merge")
        out = [arg("o", parts[0][0][0], float("nan")), arg("l", parts[0][0][1], float("nan")),
               arg("m", parts[0][0][2], float("nan"))]
        _capi.check(lib.fa_partial_finalize(C.byref(p), *(a.data_ptr() for a in acc), *(x.data_ptr() for x in out),
                                            sh._stream()), "fa_partial_finalize")
        _guards_intact(placed, f"{dt} {which}")
        return [a.clone() for a in acc], [x.clone() for x in out]

    acc0, out0 = run(())
    acc, out = run(PARTIAL_ARGS if which == "all" else (which,))
    for name, a, b in zip(("o_acc", "l_acc", "m_acc", "o", "l", "m"), acc + out, acc0 + out0):
        assert torch.equal(a.view(torch.uint8), b.view(torch.uint8)), f"{name} {dt} {which}: differs from aligned"
    got = [a.double().cpu().numpy() for a in acc]
    assert np.array_equal(np.isfinite(got[2]), live) and np.array_equal(got[2][live], ma64[live])
    assert scaled_err(got[1], la64) <= DT["f32"][3] and scaled_err(got[0], oa64) <= DT["f32"][3]   # fp32 accumulators
    sh._check_out(dt, out, ref, f"partial {dt} {which}")


@pytest.mark.parametrize("which", ["part", "acc", "out", "all"])
@pytest.mark.parametrize("dt", IS16)
def test_grad_accumulate_and_finalize_at_unaligned_addresses(dt, which):
    """fa_grad_accumulate twice (first = 1, then 0) and fa_grad_finalize on 8 * 780 elements: the 16-byte kernels on
    aligned arguments, the scalar kernels when the 16-bit part / output is 2, 4 or 8 bytes off or the float accumulator
    4 or 8 bytes off. Same bytes as the aligned calls, and the float64 sum."""
    n = 8 * 780
    g = torch.Generator(device="cuda").manual_seed(5)
    parts = [(torch.rand(n, generator=g, device="cuda") * 4 - 2).to(DT[dt][1]) for _ in range(2)]
    want = sum(x.double() for x in parts)

    def run(delta):
        offset = ("part", "acc", "out") if which == "all" else (which,)
        placed = {}

        def arg(name, key, t, d, fill=None):
            if not delta or name not in offset:
                return t if fill is None else torch.full_like(t, fill)
            placed[key] = _placed(t, d, fill)
            return placed[key][1]
        acc = arg("acc", "acc", torch.empty(n, dtype=torch.float32, device="cuda"), max(4, delta), float("nan"))
        for i, x in enumerate(parts):
            _capi.check(lib.fa_grad_accumulate(DT[dt][0], arg("part", f"part{i}", x, delta).data_ptr(), acc.data_ptr(), n,
                                               int(i == 0), sh._stream()), "fa_grad_accumulate")
        out = arg("out", "out", parts[0], delta, float("nan"))
        _capi.check(lib.fa_grad_finalize(DT[dt][0], acc.data_ptr(), out.data_ptr(), n, sh._stream()), "fa_grad_finalize")
        _guards_intact(placed, f"{dt} {which}+{delta}")
        return acc.clone(), out.clone()

    acc0, out0 = run(0)
    assert scaled_err(acc0.double().cpu().numpy(), want.cpu().numpy()) <= 2 ** -23
    assert scaled_err(out0.double().cpu().numpy(), want.cpu().numpy()) <= DT[dt][3]
    for delta in DELTAS[dt]:
        acc, out = run(delta)
        assert torch.equal(acc, acc0) and torch.equal(out, out0), f"{dt} {which}+{delta}: differs from the aligned call"


@pytest.mark.parametrize("delta", [4, 8])
@pytest.mark.parametrize("dt", IS16)
def test_backward_accumulate_with_an_unaligned_accumulator(dt, delta):
    """fa_backward_accumulate adds dQ into its fp32 accumulator by TMA reduce-add, which needs a 16-byte-aligned
    accumulator: at +4 / +8 bytes it returns FA_EINVAL_SHAPE and launches nothing, although the pointer-free
    fa_backward_accumulate_supported() says 1. The documented fallback, fa_backward + fa_grad_accumulate into the same
    offset buffer, gives the dQ of the whole sequence over two key shards."""
    B, d, nq, nk = 2, 128, 256, 256
    (Q, K, V, dO), (Qn, Kn, Vn, dOn) = sh._inputs(dt, 37, B, d, d, nq, nk)
    mask = pattern.tests_mask((nq,), (nk,), "none_front", "causal")
    O, l, m = sh._forward(sh._problem(dt, "causal", "none_front", B, d, d, nq, nk), Q, K, V, 2)
    P, dS = sh._grad_parts(Qn, Kn, Vn, dOn, mask, O.double().cpu().numpy() if dt == "bf16" else None)
    raw, acc = _placed(torch.zeros((B, d, nq), dtype=torch.float32, device="cuda"), delta)
    for kb in (128, 0):
        p = sh._problem(dt, "causal", "none_front", B, d, d, nq, 128, 0, kb, nq, nk)
        assert lib.fa_backward_accumulate_supported(C.byref(p), 0) == 1
        k, v = sh._sl(K, kb, 128), sh._sl(V, kb, 128)
        dk, dv = torch.full_like(k, float("nan")), torch.full_like(v, float("nan"))
        ws, need = sh._workspace(p, True)
        torch.cuda.synchronize()
        lib.fa_launch_count(1)
        rc = lib.fa_backward_accumulate(C.byref(p), Q.data_ptr(), k.data_ptr(), v.data_ptr(), O.data_ptr(), l.data_ptr(),
                                        m.data_ptr(), dO.data_ptr(), acc.data_ptr(), dk.data_ptr(), dv.data_ptr(), 0,
                                        ws.data_ptr(), need, sh._stream())
        assert rc == _capi.FA_EINVAL_SHAPE and lib.fa_launch_count(0) == 0
        dq, _, _ = sh._backward(p, Q, k, v, O, l, m, dO, 2)
        _capi.check(lib.fa_grad_accumulate(DT[dt][0], dq.data_ptr(), acc.data_ptr(), dq.numel(), 0, sh._stream()))
    _guards_intact({"dq_acc": (raw, acc)}, f"{dt}+{delta}")
    want = sh._block_grads(Qn, Kn, dOn, P, dS, 0, nq, 0, nk)[0]
    err = scaled_err(acc.double().cpu().numpy(), want)
    assert sh._note(dt, err) <= DT[dt][3], f"dQ accumulator {dt}+{delta}: {err}"


# ---- torch API -------------------------------------------------------------------------------------------------
def _views(xs, delta):
    """the tensors xs as consecutive contiguous views of one buffer that starts `delta` bytes past an aligned base"""
    e = xs[0].element_size()
    buf = torch.empty(sum(x.numel() for x in xs) + 16, dtype=xs[0].dtype, device="cuda")
    out, at = [], delta // e
    for x in xs:
        v = buf[at:at + x.numel()].view(x.shape)
        v.copy_(x)
        out.append(v)
        at += x.numel()
    return out


@pytest.mark.parametrize("fn", ["causal_1d", "local_1d"])
@pytest.mark.parametrize("lens", [(256, 256), (197, 213)])
@pytest.mark.parametrize("dt", IS16)
def test_torch_api_on_views_of_a_fused_qkv_buffer(dt, lens, fn):
    """Q, K and V as views of one fused buffer 2 bytes past alignment, forward and autograd, with a dO that is itself an
    unaligned view: lengths that are multiples of 8 run on the generic kernels, other lengths are packed and stay on the
    tensor cores. Bytes of the aligned call where the family is the same, the oracle everywhere."""
    nq, nk = lens
    Bo, H, d = 2, 2, 64
    rng = np.random.default_rng(41)
    xs = [torch.from_numpy(x).cuda().to(DT[dt][1]).reshape((Bo, H) + x.shape[1:])
          for x in da.random_inputs(rng, DT[dt][2], (Bo * H,), d, d, (nq,), (nk,))]
    call = {"causal_1d": lambda q, k, v: fa.causal_1d(q, k, v, "none_front"),
            "local_1d": lambda q, k, v: fa.local_1d(q, k, v, 40, 0, False, "none_front")}[fn]
    mask = (pattern.tests_mask((nq,), (nk,), "none_front", "causal") if fn == "causal_1d"
            else pattern.tests_mask((nq,), (nk,), "none_front", "local", 40, 0, False))
    runs = []
    for unaligned in (False, True):
        if unaligned:
            q, k, v = (t.requires_grad_(True) for t in _views(xs[:3], 2))
            do = _views(xs[3:], 2)[0]
            assert all(t.data_ptr() % 16 == 2 for t in (q, k, v, do))
        else:
            q, k, v = (t.clone().requires_grad_(True) for t in xs[:3])
            do = xs[3]
        O = call(q, k, v)
        torch.cuda.synchronize()
        fwd = lib.fa_last_path()
        grads = torch.autograd.grad(O, (q, k, v), do)
        torch.cuda.synchronize()
        runs.append(((O.detach(),) + grads, fwd, lib.fa_last_path()))
    (base, _, _), (got, fwd, bwd) = runs
    want = 2 if nq % 8 and nk % 8 else 1
    assert (fwd, bwd) == (want, want) and runs[0][1:] == (2, 2)
    _compare(dt, ("O", "dQ", "dK", "dV"), got, base, want == 2, (), f"{fn} {dt} {lens}")
    flat = [t.reshape((Bo * H,) + t.shape[2:]).double().cpu().numpy() for t in xs]
    On = got[0].reshape((Bo * H, d, nq)).double().cpu().numpy()
    Oref = da.forward(*flat[:3], mask)[0]
    P, dS = sh._grad_parts(*flat, mask, On if dt == "bf16" else None)
    wants = (Oref,) + sh._block_grads(flat[0], flat[1], flat[3], P, dS, 0, nq, 0, nk)
    for name, g, w in zip(("O", "dQ", "dK", "dV"), got, wants):
        err = scaled_err(g.reshape(w.shape).double().cpu().numpy(), w)
        assert sh._note(dt, err) <= DT[dt][3], f"{name} {fn} {dt} {lens}: {err}"


@pytest.mark.parametrize("dt", IS16)
def test_channel_last_at_an_unaligned_base_takes_the_adapter(dt):
    """Channel-last tensors are read directly only at 16-byte-aligned bases; 2 bytes off, fa_forward / fa_backward say
    FA_EINVAL_LAYOUT and the torch layer runs the adapter passes around the channel-first call. The forward gives the
    bytes of the aligned channel-last call. The gradients give the bytes of the channel-first call on the transposed
    tensors; the direct channel-last backward sums D = rowsum(dO o O) in another order, so against it they agree to the
    bar (test_gpu_channel_last)."""
    b, s, h, c = 2, 200, 2, 64
    g = torch.Generator(device="cuda").manual_seed(43)
    xs = [(torch.rand((b, s, h, c), generator=g, device="cuda") * 4 - 2).to(DT[dt][1]) for _ in range(4)]

    def run(q, k, v, do, layout):
        q, k, v = (t.requires_grad_(True) for t in (q, k, v))
        O, l, m = fa.causal_1d(q, k, v, "none_front", returning_l_m=True, layout=layout)
        return (O.detach(), l, m) + torch.autograd.grad(O, (q, k, v), do)
    aligned = run(*(t.clone() for t in xs), "channel_last")
    unaligned = run(*_views(xs[:3], 2), _views(xs[3:], 2)[0], "channel_last")
    Oc, _, _, *gc = run(*(fa.from_channel_last(t) for t in xs), "channel_first")
    assert torch.equal(unaligned[0], fa.to_channel_last(Oc))
    for name, a, bb in zip(("O", "l", "m"), unaligned[:3], aligned[:3]):
        assert torch.equal(a, bb), f"{name} {dt}: differs from the aligned channel-last call"
    for name, a, bb, cc in zip(("dQ", "dK", "dV"), unaligned[3:], gc, aligned[3:]):
        assert torch.equal(a, fa.to_channel_last(bb)), f"{name} {dt}: differs from the channel-first call"
        err = scaled_err(a.double().cpu().numpy(), cc.double().cpu().numpy())
        assert err <= DT[dt][3], f"{name} {dt}: {err} from the aligned channel-last call"


# ---- host-buffer entry points ----------------------------------------------------------------------------------
def _chunk_starts(B, nch):
    """first batch element of every chunk (fa_api.cu: b0 = B * c / nch)"""
    return [B * c // nch for c in range(nch)]


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_host_entry_points_on_unaligned_batch_chunks(dt, monkeypatch):
    """fa_forward_backward_host, and fa_forward_host + fa_backward_host_resident, on a problem of more than 64 MB (so
    both pipelines cut the batch into chunks) with odd lengths and an odd channel count: the chunk starts inside the
    arena are not 16-byte aligned. Bytes of the device call on the whole batch, and the oracle on the first element of
    every chunk."""
    d = vd = 21
    nq = nk = 1023
    e = torch.empty((), dtype=DT[dt][1]).element_size()
    per = e * (2 * d * nq + 2 * d * nk)       # Q, K, V, O of one batch element
    B = -(-(64 << 20) // per) + 3
    rng = np.random.default_rng(47)
    Q, K, V, dO = da.random_inputs(rng, DT[dt][2], (B,), d, vd, (nq,), (nk,))
    p = _capi.make_problem(DT[dt][0], 1, "causal", "none_front", Q.shape, K.shape, V.shape)
    path = 2 if dt == "f16" else 3
    # chunks of the two pipelines: pick_chunks (8), and fa_forward_backward_host's default of 16, which the library reads
    # from FA_HOST_CHUNKS at each call; the variable is removed so that the library takes its default
    monkeypatch.delenv("FA_HOST_CHUNKS", raising=False)
    step_chunks = min(B, 16)
    sq, so = e * d * nq, e * vd * nq
    for nch in (min(B, 8), step_chunks):
        assert nch > 1
        assert any((b0 * sq) % 16 or (b0 * so) % 16 for b0 in _chunk_starts(B, nch)), nch

    ts = [torch.from_numpy(x).cuda() for x in (Q, K, V, dO)]
    O, l, m = sh._forward(p, *ts[:3], path)
    dev = (O, l, m) + sh._backward(p, *ts[:3], O, l, m, ts[3], path)
    dev = [t.cpu().numpy() for t in dev]

    ldt = np.float32 if dt == "f16" else DT[dt][2]
    host = [np.full(x.shape, np.nan, dtype=x.dtype) for x in dev]
    assert host[1].dtype == ldt
    arena = torch.empty(max(lib.fa_host_arena_bytes(C.byref(p), 1), lib.fa_step_host_arena_bytes(C.byref(p))),
                        dtype=torch.uint8, device="cuda")
    ptr = lambda a: a.ctypes.data   # noqa: E731
    st = sh._stream()
    _capi.check(lib.fa_forward_backward_host(C.byref(p), ptr(Q), ptr(K), ptr(V), ptr(dO), *(ptr(h) for h in host),
                                             arena.data_ptr(), arena.numel(), st), "fa_forward_backward_host")
    assert lib.fa_last_path() == path
    host2 = [np.full(x.shape, np.nan, dtype=x.dtype) for x in dev]
    _capi.check(lib.fa_forward_host(C.byref(p), ptr(Q), ptr(K), ptr(V), *(ptr(h) for h in host2[:3]), arena.data_ptr(),
                                    arena.numel(), st), "fa_forward_host")
    assert lib.fa_last_path() == path
    _capi.check(lib.fa_backward_host_resident(C.byref(p), ptr(dO), *(ptr(h) for h in host2[3:]), arena.data_ptr(),
                                              arena.numel(), st), "fa_backward_host_resident")
    assert lib.fa_last_path() == path
    names = ("O", "l", "m", "dQ", "dK", "dV")
    for tag, res in (("forward_backward_host", host), ("forward_host + backward_host_resident", host2)):
        for name, a, bb in zip(names, res, dev):
            assert np.array_equal(a.view(np.uint8), bb.view(np.uint8)), f"{name} {dt} {tag}: differs from the device call"
    sel = sorted(set(_chunk_starts(B, min(B, 8)) + _chunk_starts(B, step_chunks) + [B - 1]))
    Qs, Ks, Vs, dOs = (x[sel].astype(np.float64) for x in (Q, K, V, dO))
    mask = pattern.tests_mask((nq,), (nk,), "none_front", "causal")
    sh._check_out(dt, [torch.from_numpy(x[sel]) for x in host[:3]], da.forward(Qs, Ks, Vs, mask), f"host {dt}")
    for name, g, w in zip(names[3:], host[3:], da.backward(Qs, Ks, Vs, mask, dOs)):
        err = scaled_err(g[sel], w)
        assert sh._note(dt, err) <= DT[dt][3], f"{name} host {dt}: {err}"
