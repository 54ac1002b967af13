"""Workspace and host-arena alignment (CPU): fa_forward, fa_backward and fa_backward_accumulate reject a needed workspace
whose address is not a multiple of 256 bytes, and the four host-buffer entry points reject such a device arena, with
FA_EINVAL_WORKSPACE before anything touches the device. The generic kernels and the fp64 DMMA backward store double rows
straight into the workspace, and the tensor-core families carve TMA operands out of it, so a workspace a few bytes off
would reach a kernel with a misaligned address.

Every pointer here is a fake (0x1000 + offset) that must never reach a kernel, also on a machine with a GPU and also if
the check under test were missing. So each in-process call is built to fail a later host-side check when it gets past
the workspace / arena check: a channel-last layout no kernel reads, an fa_backward_accumulate shape the fused kernel
does not take, a null host tensor. A channel-first fa_forward / fa_backward that needs a workspace has no such later
check: those calls run in a child process that sees no CUDA device, where whatever gets past validation fails at its
first CUDA call."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

from tf_flash_attention_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = _capi.lib
BASE = 0x1000
BAD = (8, 16, 128)          # workspace / arena offsets from a 256-byte boundary
GOOD = (0, 256, 0x1000)
DTYPES = {"f16": _capi.FA_F16, "bf16": _capi.FA_BF16, "f32": _capi.FA_F32, "f64": _capi.FA_F64}
ONE = C.c_void_p(BASE)


def _problem(dt, d=64, vd=64, nq=203, nk=197, batch=(2, 3), layout=_capi.FA_LAYOUT_CHANNEL_FIRST):
    """Odd lengths: the 16-bit forward packs both sides into its workspace, so it needs one"""
    p = _capi.make_problem(DTYPES[dt], 1, "causal", "none_front", batch + (d, nq), batch + (d, nk), batch + (vd, nk))
    if layout == _capi.FA_LAYOUT_CHANNEL_LAST:
        p.layout, p.heads = layout, batch[-1]
    return p


def _ptr(off):
    return C.c_void_p(BASE + off)


def _forward(p, ws, nbytes):
    return lib.fa_forward(C.byref(p), ONE, ONE, ONE, ONE, ONE, ONE, ws, nbytes, None)


def _backward(p, ws, nbytes):
    return lib.fa_backward(C.byref(p), *([ONE] * 10), ws, nbytes, None)


def _backward_accumulate(p, ws, nbytes):
    return lib.fa_backward_accumulate(C.byref(p), *([ONE] * 10), 0, ws, nbytes, None)


_CHILD = r"""
import ctypes as C, json, sys
sys.path.insert(0, sys.argv[1])
import torch
assert torch.cuda.device_count() == 0, "the child must see no CUDA device"
from tests import test_alignment_host as t
out = {}
for dt in t.DTYPES:
    p = t._problem(dt)
    need_f, need_b = int(t.lib.fa_workspace_bytes(C.byref(p), 0)), int(t.lib.fa_workspace_bytes(C.byref(p), 1))
    out[dt] = {"need": [need_f, need_b],
               "fwd": {off: t._forward(p, t._ptr(off), need_f) for off in t.BAD + t.GOOD},
               "bwd": {off: t._backward(p, t._ptr(off), need_b) for off in t.BAD + t.GOOD}}
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def deviceless_calls():
    """channel-first fa_forward / fa_backward at every offset, made by a child process with no visible CUDA device"""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _CHILD, ROOT], env=env, cwd=ROOT, capture_output=True, text=True,
                         timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("dt", list(DTYPES))
def test_device_calls_reject_a_misaligned_workspace(dt, deviceless_calls):
    """A workspace at +8, +16 or +128 bytes is FA_EINVAL_WORKSPACE whenever fa_workspace_bytes() asks for one; at a
    multiple of 256 the same call passes validation and fails only for want of a device. The fp64 forward never needs a
    workspace (neither the DMMA nor the generic forward keeps anything there), so there any pointer passes."""
    res = deviceless_calls[dt]
    need_f, need_b = res["need"]
    assert need_b > 0
    assert (need_f > 0) == (dt != "f64")
    for off in BAD:
        assert res["fwd"][str(off)] == (_capi.FA_EINVAL_WORKSPACE if need_f else _capi.FA_ECUDA), off
        assert res["bwd"][str(off)] == _capi.FA_EINVAL_WORKSPACE, off
    for off in GOOD:
        assert res["fwd"][str(off)] in (_capi.FA_ECUDA, _capi.FA_ENODEVICE), off
        assert res["bwd"][str(off)] in (_capi.FA_ECUDA, _capi.FA_ENODEVICE), off
    # in process: calls whose next check after the workspace is a host-side one
    p = _problem(dt)
    cl = _problem(dt, d=5, vd=5, layout=_capi.FA_LAYOUT_CHANNEL_LAST)
    need_cl = int(lib.fa_workspace_bytes(C.byref(cl), 1))
    for off in BAD:
        assert _backward(cl, _ptr(off), need_cl) == _capi.FA_EINVAL_WORKSPACE, off
        assert _backward_accumulate(p, _ptr(off), need_b) == _capi.FA_EINVAL_WORKSPACE, off
    # a larger workspace than needed changes nothing
    assert _backward(cl, _ptr(8), need_cl + 4096) == _capi.FA_EINVAL_WORKSPACE


@pytest.mark.parametrize("dt", list(DTYPES))
def test_device_calls_accept_a_256_byte_aligned_workspace(dt):
    """Offsets that are multiples of 256 pass the workspace check and reach the next host-side check: channel-last
    tensors that no kernel reads directly (5 channels) give FA_EINVAL_LAYOUT, and fa_backward_accumulate on a shape the
    fused kernel does not take (head_dim 64, or a dtype other than fp16 / bf16) gives FA_EINVAL_SHAPE."""
    cl = _problem(dt, d=5, vd=5, layout=_capi.FA_LAYOUT_CHANNEL_LAST)
    cf = _problem(dt)
    need_cl_b = int(lib.fa_workspace_bytes(C.byref(cl), 1))
    need_cf_b = int(lib.fa_workspace_bytes(C.byref(cf), 1))
    assert need_cl_b > 0 and lib.fa_workspace_bytes(C.byref(cl), 0) == 0
    for off in GOOD:
        assert _backward(cl, _ptr(off), need_cl_b) == _capi.FA_EINVAL_LAYOUT, off
        assert _backward_accumulate(cf, _ptr(off), need_cf_b) == _capi.FA_EINVAL_SHAPE, off
    # nothing needed: a null workspace, or any pointer at all, is accepted
    for ws in (None, _ptr(8), _ptr(2)):
        assert _forward(cl, ws, 0) == _capi.FA_EINVAL_LAYOUT
    # still rejected: too small, or null while needed
    assert _backward(cl, _ptr(256), need_cl_b - 1) == _capi.FA_EINVAL_WORKSPACE
    assert _backward(cl, None, need_cl_b) == _capi.FA_EINVAL_WORKSPACE


def _arenas(p):
    return (int(lib.fa_host_arena_bytes(C.byref(p), 0)), int(lib.fa_host_arena_bytes(C.byref(p), 1)),
            int(lib.fa_step_host_arena_bytes(C.byref(p))))


def _host_calls(p, q):
    """the four host-buffer entry points with arena pointer `arena`; q is the first host pointer (None: FA_EINVAL_NULL)"""
    fwd, bwd, step = _arenas(p)
    return {
        "fa_forward_host": lambda arena: lib.fa_forward_host(C.byref(p), q, ONE, ONE, ONE, ONE, ONE, arena, fwd, None),
        "fa_backward_host": lambda arena: lib.fa_backward_host(C.byref(p), q, *([ONE] * 9), arena, bwd, None),
        "fa_backward_host_resident": lambda arena: lib.fa_backward_host_resident(C.byref(p), q, ONE, ONE, ONE, arena,
                                                                                 bwd, None),
        "fa_forward_backward_host": lambda arena: lib.fa_forward_backward_host(C.byref(p), q, *([ONE] * 9), arena, step,
                                                                               None),
    }


@pytest.mark.parametrize("dt", list(DTYPES))
def test_host_entry_points_reject_a_misaligned_arena(dt):
    """The arena holds the staged tensors and the workspace at 256-byte offsets from its base, so the base itself must be
    256-byte aligned (the ring driver's rule for its arena as well). The first host tensor is null, so with an aligned
    arena the same calls stop at the null check and never copy."""
    p = _problem(dt, d=24, vd=40)
    assert all(n > 0 for n in _arenas(p))
    for name, call in _host_calls(p, None).items():
        for off in BAD:
            assert call(_ptr(off)) == _capi.FA_EINVAL_WORKSPACE, (name, off)
        for off in GOOD:
            assert call(_ptr(off)) == _capi.FA_EINVAL_NULL, (name, off)
        assert call(None) == _capi.FA_EINVAL_WORKSPACE, name


def test_dispatch_path_still_describes_aligned_tensors():
    """fa_dispatch_path takes no pointers: its answer is the family for 256-byte-aligned tensors and workspace, and the
    workspace check does not change it."""
    for dt, fwd, bwd in (("f16", 2, 2), ("bf16", 2, 2), ("f32", 3, 3), ("f64", 4, 4)):
        p = _problem(dt, d=32, vd=32)
        assert lib.fa_dispatch_path(C.byref(p), 0, None, 0) == fwd, dt
        assert lib.fa_dispatch_path(C.byref(p), 1, None, 0) == bwd, dt
