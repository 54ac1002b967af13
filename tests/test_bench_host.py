"""Host-side checks of bench.py (no GPU): every workload describes a valid problem, the attended-pair counts the
FLOP metric is built on agree between the closed forms, the oracle and the library, the strong-scaling split keeps
whole heads together for the channel-last workload, the reference arm never loads the product library, and
--dump-outputs keeps to its size limit with a fixed sample. On a GPU: --dump-outputs writes the outputs of the timed
step, checked against the dense oracle."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from tf_flash_attention_b200 import _capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", sorted(n for n, w in bench.WORKLOADS.items() if not w.get("layout")))
def test_workload_is_a_valid_problem_with_consistent_flops(name):
    w = bench.WORKLOADS[name]
    code = {"float16": 0, "float32": 1, "float64": 2}[w["dtype"]]
    units = int(np.prod(w["batch"]))
    p = _capi.make_problem(code, w["seq_dims"], w["rule"], w["sync"], (units, w["d"]) + w["q"], (units, w["d"]) + w["k"],
                           (units, w["v_d"]) + w["k"], w["w"], w["s"], w["c"])
    nq, nk = int(np.prod(w["q"])), int(np.prod(w["k"]))
    if nq * nk <= 1 << 28:                 # the library counts by enumeration; C5 (131072^2) has its closed form below
        assert _capi.count_attended(p) == bench.attended_pairs(w)
    else:
        assert w["rule"] == "causal" and nq == nk and bench.attended_pairs(w) == nq * (nq + 1) // 2
    fwd, bwd = bench.flops_of(w, bench.attended_pairs(w))
    assert fwd == 2.0 * bench.attended_pairs(w) * (w["d"] + w["v_d"]) * units
    assert bwd == 2.0 * bench.attended_pairs(w) * (3 * w["d"] + 2 * w["v_d"]) * units
    if w.get("channel_last_heads"):
        for world in (1, 2, 4, 8):          # every rank's slice keeps whole (outer, all heads) groups
            assert (units // world) % w["channel_last_heads"] == 0
        p.layout, p.heads = _capi.FA_LAYOUT_CHANNEL_LAST, w["channel_last_heads"]
        assert _capi.dispatch_path(p) == ("tcgen05_f16", "") and _capi.dispatch_path(p, backward=True)[0] == "tcgen05_f16"
    elif not w.get("ring"):
        assert _capi.dispatch_path(p)[0] != "generic_simt", "a bench workload must not fall back to the SIMT kernels"
        assert _capi.dispatch_path(p, backward=True)[0] != "generic_simt"
    assert _capi.lib.fa_workspace_bytes(C.byref(p), 1) >= _capi.lib.fa_workspace_bytes(C.byref(p), 0) or code == 1


def test_reference_arm_runs_without_the_product_library():
    """`bench.py --impl reference` (the reference's CPU path on the host cores) prints one JSON line with the contract's
    keys and must not import tf_flash_attention_b200 (VERDICT r1 item 9a)."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'C1', '--steps', '1', "
            "'--warmup', '1', '--cpu-heads', '1']; runpy.run_path('bench.py', run_name='__main__'); "
            "assert not any(m.startswith('tf_flash_attention_b200') for m in sys.modules), 'product library imported'")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "dtype", "data", "config"):
        assert key in line


def test_dump_outputs_keeps_the_size_limit_with_a_fixed_sample(tmp_path, monkeypatch):
    """Tensors within their share of DUMP_BYTES keep their shape (fp16 widened to float32); larger ones are written as
    the same seeded, sorted sample of flat indices on every call."""
    import torch
    monkeypatch.setattr(bench, "DUMP_BYTES", 8000)
    small = torch.linspace(-2, 2, 12, dtype=torch.float16).reshape(3, 4)
    big = torch.arange(100000, dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"small": small, "big": big}, 0, 1)
    a_small, a_big = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert a_small.dtype == np.float32 and np.array_equal(a_small, small.float().numpy())
    assert a_big.dtype == np.float64 and a_big.shape == ((8000 // 2 - 1024) // 8,)
    assert np.all(np.diff(a_big) > 0) and np.all(a_big == np.round(a_big))   # distinct elements of `big`, in order
    assert np.array_equal(a_big, np.load(tmp_path / "b" / "big.npy"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 8000
    bench.dump_outputs(str(tmp_path / "r"), {"big": big}, 1, 2)
    assert os.listdir(tmp_path / "r") == ["big_rank1.npy"] and os.path.getsize(tmp_path / "r" / "big_rank1.npy") <= 4000


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_step_outputs(tmp_path):
    """`bench.py --workload C1 --dump-outputs DIR` writes O, l, m, dQ, dK, dV of its last timed step; on the bench's own
    seeded inputs they match the dense oracle."""
    import torch
    from oracle import dense_attention as da
    from tests.helpers import scaled_err
    r = subprocess.run([sys.executable, "bench.py", "--workload", "C1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                        "--no-e2e", "--no-refkernel", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("O", "l", "m", "dQ", "dK", "dV")}
    assert sorted(os.listdir(tmp_path)) == sorted(f"{n}.npy" for n in got)
    w = bench.WORKLOADS["C1"]
    g = torch.Generator(device="cuda").manual_seed(1234)       # bench.py's input recipe, rank 0

    def u(ch, seq):
        return (torch.rand(w["batch"] + (ch,) + seq, generator=g, device="cuda") * 4 - 2).cpu().numpy()
    Q, K, V, dO = u(w["d"], w["q"]), u(w["d"], w["k"]), u(w["v_d"], w["k"]), u(w["v_d"], w["q"])
    ref = da.attention(Q, K, V, 1, w["rule"], w["sync"], w["w"], w["s"], bool(w["c"]), dO=dO)
    for n in ("O", "dQ", "dK", "dV"):
        assert got[n].dtype == np.float32 and got[n].shape == ref[n].shape, n
        assert scaled_err(got[n], ref[n]) <= 1e-5, n
    lse = got["m"].astype(np.float64) + np.log(got["l"].astype(np.float64))
    assert np.max(np.abs(lse - (ref["m"] + np.log(ref["l"])))) <= 1e-4
