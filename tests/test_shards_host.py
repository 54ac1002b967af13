"""Sharded 1-D problems on the host: a call that sees rows [q_index_base, q_index_base + nq) and keys
[k_index_base, k_index_base + nk) of longer sequences of q_full_len / k_full_len positions evaluates the rule on global
coordinates. The host helpers (fa_pattern_mask, the tcgen05 kernels' closed-form masks, the tile classifier, the
attended count) must give the oracle's global pattern sliced to the block; the validation must refuse bases and full
lengths that do not describe a block; and fa_dispatch_path must keep such a block on the tensor cores."""
import numpy as np
import pytest

from oracle import pattern
from tf_flash_attention_b200 import _capi

CODES = {"f16": _capi.FA_F16, "f32": _capi.FA_F32, "f64": _capi.FA_F64, "bf16": _capi.FA_BF16}


def _problem(rule, mode, nq, nk, qb, kb, qf, kf, w=1, s=0, c=False, dtype=_capi.FA_F32, d=4, vd=4, batch=1):
    p = _capi.make_problem(dtype, 1, rule, mode, (batch, d, nq), (batch, d, nk), (batch, vd, nk), w, s, c)
    p.q_index_base, p.k_index_base, p.q_full_len, p.k_full_len = qb, kb, qf, kf
    return p


def _coords_mask(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk):
    """The block of the oracle's pattern from the global coordinates of pattern.tests_locations, with the mask formula
    of pattern.tests_mask: the whole (qf, kf) mask does not fit in memory at 2^21 x 2^20."""
    (qc, kc), (ql, kl) = pattern.tests_locations((qf,), (kf,), mode)
    qc, kc, ql, kl = qc[qb:qb + nq, 0], kc[kb:kb + nk, 0], ql[qb:qb + nq], kl[kb:kb + nk]
    idx_diff = ql[:, None] - kl[None, :]
    if rule == "full":
        return np.ones(idx_diff.shape, dtype=bool)
    if rule == "causal":
        return idx_diff >= 0
    diff = np.abs(qc[:, None] - kc[None, :])
    ok = (diff % (1 << s) == 0) & (diff // (1 << s) < w)
    return ok & (idx_diff >= 0) if c else ok


def _block_mask(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk):
    """The oracle's pattern of the whole (qf, kf) problem, sliced to the block."""
    if qf * kf <= 1 << 22:
        return pattern.tests_mask((qf,), (kf,), mode, rule, w, s, c)[qb:qb + nq, kb:kb + nk]
    return _coords_mask(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk)


def _check_helpers(p, want, tag):
    assert np.array_equal(_capi.pattern_mask(p), want), f"fa_pattern_mask {tag}"
    for tile, resident_is_q in ((64, 1), (128, 1), (64, 0)):
        got = _capi.pattern_mask_fast(p, tile, resident_is_q)
        assert np.array_equal(got, want), f"fa_pattern_mask_fast({tile}, {resident_is_q}) {tag}"
    for tq, tk in ((64, 64), (128, 128), (8, 16), (128, 64)):
        cls = _capi.classify_tiles(p, tq, tk)
        for a in range(cls.shape[0]):
            for b in range(cls.shape[1]):
                blk = want[a * tq:(a + 1) * tq, b * tk:(b + 1) * tk]
                assert not (cls[a, b] == 0 and blk.any()), f"tile ({a}, {b}) of {tq}x{tk} skipped but attended {tag}"
                assert not (cls[a, b] == 2 and not blk.all()), f"tile ({a}, {b}) of {tq}x{tk} full but masked {tag}"
    assert _capi.count_attended(p) == int(want.sum()), f"fa_count_attended {tag}"


def _random_cases(n, seed):
    rng = np.random.default_rng(seed)
    for _ in range(n):
        qf, kf = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        nq, nk = int(rng.integers(1, qf + 1)), int(rng.integers(1, kf + 1))
        qb, kb = int(rng.integers(0, qf - nq + 1)), int(rng.integers(0, kf - nk + 1))
        rule = pattern.RULES[int(rng.integers(0, 3))]
        mode = pattern.SYNC_MODES[int(rng.integers(0, 3))]
        w, c = int(rng.integers(1, 40)), bool(rng.integers(0, 2))
        s = int(rng.integers(0, 5)) if rule == "local" else 0
        yield rule, mode, w, s, c, qf, kf, qb, nq, kb, nk


@pytest.mark.parametrize("chunk", range(6))
def test_random_blocks_match_the_sliced_global_pattern(chunk):
    """300 seeded blocks over all rules, sync modes, strides 0-4 and independent full lengths."""
    for rule, mode, w, s, c, qf, kf, qb, nq, kb, nk in _random_cases(50, 100 + chunk):
        p = _problem(rule, mode, nq, nk, qb, kb, qf, kf, w, s, c)
        tag = f"{rule} {mode} w{w} s{s} c{c} q{qb}+{nq}/{qf} k{kb}+{nk}/{kf}"
        _check_helpers(p, _block_mask(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk), tag)


@pytest.mark.parametrize("rule,mode,w,s,c,qf,kf,qb,nq,kb,nk,empty", [
    # coordinates up to 2^21 - 1 (the reference grid's extent for these lengths); keys at stride 2 under scale_end
    ("local", "scale_end", 64, 1, True, 1 << 21, 1 << 20, 1 << 20, 96, (1 << 19) - 20, 100, False),
    ("causal", "scale_end", 1, 0, False, 1 << 21, 1 << 20, (1 << 21) - 64, 64, (1 << 20) - 50, 50, False),
    ("local", "scale_front", 5, 2, False, 1 << 20, 1 << 21, (1 << 20) - 77, 77, (1 << 21) - 200, 130, False),
    # shards of length 1
    ("causal", "none_front", 1, 0, False, 300, 300, 150, 1, 77, 100, False),
    ("local", "scale_end", 3, 1, False, 150, 300, 77, 70, 151, 1, False),
    ("full", "scale_front", 1, 0, False, 301, 77, 300, 1, 76, 1, False),
    # a causal block entirely in the future of its queries
    ("causal", "none_front", 1, 0, False, 1000, 1000, 64, 100, 600, 200, True),
    ("local", "scale_front", 40, 0, True, 500, 1000, 0, 100, 301, 300, True),
], ids=lambda v: str(v))
def test_fixed_blocks(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk, empty):
    p = _problem(rule, mode, nq, nk, qb, kb, qf, kf, w, s, c)
    want = _block_mask(rule, mode, w, s, c, qf, kf, qb, nq, kb, nk)
    assert want.any() != empty
    _check_helpers(p, want, "")


def test_coordinate_mask_is_the_sliced_tests_mask():
    for case in _random_cases(40, 7):
        rule, mode, w, s, c, qf, kf, qb, nq, kb, nk = case
        want = pattern.tests_mask((qf,), (kf,), mode, rule, w, s, c)[qb:qb + nq, kb:kb + nk]
        assert np.array_equal(_coords_mask(*case), want), case


# ---- validation ------------------------------------------------------------------------------------------------
def _status_all(p):
    """(fa_forward, fa_backward, fa_dispatch_path forward, backward) of p; null pointers are fine: validation runs first"""
    lib = _capi.lib
    import ctypes as C
    fwd = lib.fa_forward(C.byref(p), None, None, None, None, None, None, None, 0, None)
    bwd = lib.fa_backward(C.byref(p), *([None] * 11), 0, None)
    return fwd, bwd, lib.fa_dispatch_path(C.byref(p), 0, None, 0), lib.fa_dispatch_path(C.byref(p), 1, None, 0)


@pytest.mark.parametrize("dtype", list(CODES))
@pytest.mark.parametrize("qb,kb,qf,kf", [
    (-1, 0, 100, 100), (0, -3, 100, 100),            # negative base
    (1, 0, 100, 100), (0, 61, 100, 100),             # base + n > full
    (0, 0, 99, 100), (0, 0, 100, 59),                # 0 < full < n
    (0, 0, 0x7fffffff, 100),                         # a full length beyond the 2^30 reference grid
    (-0x80000000, 0, 0, 0),
])
def test_bases_and_full_lengths_outside_the_sequence_are_refused(dtype, qb, kb, qf, kf):
    p = _problem("causal", "none_front", 100, 60, 0, 0, 0, 0, dtype=CODES[dtype])
    assert _status_all(p)[2] in (1, 2, 3, 4)
    p.q_index_base, p.k_index_base, p.q_full_len, p.k_full_len = qb, kb, qf, kf
    assert _status_all(p) == (_capi.FA_EINVAL_SHAPE,) * 4


@pytest.mark.parametrize("field", ["q_index_base", "k_index_base", "q_full_len", "k_full_len"])
def test_two_dimensional_problems_take_no_base_or_full_length(field):
    p = _capi.make_problem(_capi.FA_F16, 2, "local", "none_front", (2, 16, 8, 12), (2, 16, 8, 12), (2, 16, 8, 12), 3)
    assert _status_all(p)[2] == 2
    setattr(p, field, 12 if "full" in field else 1)
    assert _status_all(p) == (_capi.FA_EINVAL_SHAPE,) * 4


# ---- dispatch ---------------------------------------------------------------------------------------------------
# the channel configurations tests/test_gpu_shards.py runs on the tensor cores
SHAPES = {"f16": [(64, 64), (128, 128), (20, 20)], "bf16": [(64, 64), (128, 128)], "f32": [(64, 64), (32, 16)],
          "f64": [(32, 48), (64, 64)]}
PATH = {"f16": 2, "f32": 3, "f64": 4, "bf16": 2}
RULES = [("causal", 1, 0, False), ("local", 40, 0, False), ("local", 6, 2, False), ("local", 16, 1, True)]


@pytest.mark.parametrize("dtype", list(CODES))
@pytest.mark.parametrize("mode", pattern.SYNC_MODES)
def test_sharded_blocks_stay_on_the_tensor_cores(dtype, mode):
    for d, vd in SHAPES[dtype]:
        for rule, w, s, c in RULES:
            for qb, nq, qf, kb, nk, kf in ((301, 299, 1000, 77, 397, 1000), (77, 203, 450, 301, 397, 900),
                                           (0, 800, 800, 77, 301, 400), (301, 333, 900, 0, 600, 600)):
                p = _problem(rule, mode, nq, nk, qb, kb, qf, kf, w, s, c, CODES[dtype], d, vd, batch=2)
                for bwd in (False, True):
                    path, why = _capi.dispatch_path(p, bwd)
                    assert path == _capi.PATH_NAMES[PATH[dtype]], (dtype, d, vd, rule, mode, qb, kb, bwd, why)
                p.accumulate = 1
                path, why = _capi.dispatch_path(p, False)
                assert path == "generic_simt" and why == "accumulate = 1 is served by the generic forward kernels"
