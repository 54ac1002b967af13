"""Times the generic kernels across the 256-channel boundary: forward and forward + backward, 16 heads, q = k = 4096,
full and causal rules, d = v_d in 256 (the whole-tile kernels) and 320 / 512 / 1024 (the channel-sliced kernels), in
fp16 / fp32 / fp64. CUDA events around back-to-back calls through the C ABI, after warm-up, over windows of at least
--window seconds. FLOPs are the unmasked ones of DESIGN.md section 4 (fwd = 2 nnz (d + v_d) B, bwd = 2 nnz (3 d + 2 v_d)
B, nnz from fa_count_attended). One more call with fa_kernel_timing on gives the per-kernel times. For context, dense
attention in torch (matmul, masked softmax, matmul) on the same shape.

    python tools/bench_wide_heads.py [--dtypes f16,f32,f64] [--widths 256,320,512,1024] [--rules full,causal]
                                     [--window 1.0] [--out results.json]

Prints one JSON object per measurement and a markdown table at the end."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tf_flash_attention_b200 import _capi  # noqa: E402

DTYPES = {"f16": (torch.float16, _capi.FA_F16), "f32": (torch.float32, _capi.FA_F32), "f64": (torch.float64, _capi.FA_F64)}
L2_BYTES = 126 << 20


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["nvidia_smi"] = q[0] if q else ""
    except (OSError, subprocess.SubprocessError) as e:
        out["nvidia_smi"] = f"unavailable: {e}"
    return out


def timed(fn, window):
    """ms per call: warm-up, then back-to-back calls between two CUDA events over at least `window` seconds"""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    n = max(3, int(window / max(time.perf_counter() - t, 1e-6)) + 1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n, n


def kernel_times(fn):
    torch.cuda.synchronize()
    _capi.kernel_timings()
    _capi.lib.fa_kernel_timing(1)
    fn()
    torch.cuda.synchronize()
    _capi.lib.fa_kernel_timing(0)
    agg = {}
    for name, ms in _capi.kernel_timings():
        agg[name] = round(agg.get(name, 0.0) + ms, 4)
    return agg


def bench_one(dt, rule, d, heads, seq, window, with_torch):
    tdt, code = DTYPES[dt]
    g = torch.Generator(device="cuda").manual_seed(d)
    mk = lambda c: torch.randn((heads, c, seq), dtype=tdt, device="cuda", generator=g)  # noqa: E731
    Q, K, V, dO = mk(d), mk(d), mk(d), mk(d)
    O, dQ, dK, dV = (torch.empty_like(x) for x in (dO, Q, K, V))
    ldt = torch.float32 if tdt == torch.float16 else tdt
    l, m = torch.empty((heads, seq), dtype=ldt, device="cuda"), torch.empty((heads, seq), dtype=tdt, device="cuda")
    p = _capi.make_problem(code, 1, rule, "none_front", Q.shape, K.shape, V.shape)
    nws = max(int(_capi.lib.fa_workspace_bytes(C.byref(p), 0)), int(_capi.lib.fa_workspace_bytes(C.byref(p), 1)), 16)
    ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def fwd():
        _capi.check(_capi.lib.fa_forward(C.byref(p), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(), l.data_ptr(),
                                         m.data_ptr(), ws.data_ptr(), nws, st), "fa_forward")

    def bwd():
        _capi.check(_capi.lib.fa_backward(C.byref(p), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(),
                                          l.data_ptr(), m.data_ptr(), dO.data_ptr(), dQ.data_ptr(), dK.data_ptr(),
                                          dV.data_ptr(), ws.data_ptr(), nws, st), "fa_backward")

    def step():
        fwd()
        bwd()

    nnz = _capi.count_attended(p)
    flops_f, flops_b = 2 * nnz * (2 * d) * heads, 2 * nnz * (5 * d) * heads
    esz = Q.element_size()
    row = {"dtype": dt, "rule": rule, "d": d, "v_d": d, "heads": heads, "q": seq, "k": seq, "nnz": nnz,
           "fwd_path": _capi.dispatch_path(p)[0], "bwd_path": _capi.dispatch_path(p, True)[0],
           "fwd_bytes": 4 * heads * d * seq * esz, "step_bytes": 8 * heads * d * seq * esz}
    row["fits_l2_fwd"] = row["fwd_bytes"] <= L2_BYTES
    row["fits_l2_step"] = row["step_bytes"] <= L2_BYTES
    row["fwd_ms"], row["fwd_calls"] = timed(fwd, window)
    row["step_ms"], row["step_calls"] = timed(step, window)
    row["fwd_tflops"] = flops_f / row["fwd_ms"] / 1e9
    row["step_tflops"] = (flops_f + flops_b) / row["step_ms"] / 1e9
    row["kernels_fwd_ms"] = kernel_times(fwd)
    row["kernels_step_ms"] = kernel_times(step)
    if with_torch:
        causal = torch.ones((seq, seq), dtype=torch.bool, device="cuda").tril() if rule == "causal" else None
        scale = d ** -0.5

        def dense():
            s = torch.matmul(Q.transpose(1, 2), K) * scale
            if causal is not None:
                s = s.masked_fill(~causal, float("-inf"))
            return torch.matmul(torch.softmax(s, dim=-1), V.transpose(1, 2))
        with torch.no_grad():
            row["torch_dense_fwd_ms"], _ = timed(dense, window)
        row["torch_dense_fwd_tflops"] = flops_f / row["torch_dense_fwd_ms"] / 1e9
    del Q, K, V, dO, O, dQ, dK, dV, ws
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--dtypes", default="f16,f32,f64")
    ap.add_argument("--widths", default="256,320,512,1024")
    ap.add_argument("--rules", default="full,causal")
    ap.add_argument("--heads", type=int, default=16)
    ap.add_argument("--seq", type=int, default=4096)
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window (at least)")
    ap.add_argument("--no-torch", action="store_true", help="skip the dense torch reference")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_wide_heads.py needs a CUDA device")
    torch.cuda.set_device(0)
    info = card()
    print(json.dumps({"card": info}), flush=True)
    rows = []
    for dt in args.dtypes.split(","):
        for rule in args.rules.split(","):
            for d in (int(w) for w in args.widths.split(",")):
                row = bench_one(dt, rule, d, args.heads, args.seq, args.window, not args.no_torch)
                rows.append(row)
                print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": info, "rows": rows}, f, indent=1)
    print("\n| dtype | rule | d = v_d | fwd ms | fwd TFLOPS | fwd+bwd ms | fwd+bwd TFLOPS | time/FLOP vs 256 (fwd, step) "
          "| torch dense fwd ms | fits L2 (fwd, step) |")
    print("|---|---|---|---|---|---|---|---|---|---|")
    base = {}
    for r in rows:
        key = (r["dtype"], r["rule"])
        if r["d"] == 256:
            base[key] = r
        b = base.get(key)
        ratio = (f"{b['fwd_tflops'] / r['fwd_tflops']:.2f}, {b['step_tflops'] / r['step_tflops']:.2f}" if b else "-")
        print(f"| {r['dtype']} | {r['rule']} | {r['d']} | {r['fwd_ms']:.3f} | {r['fwd_tflops']:.2f} | {r['step_ms']:.3f} | "
              f"{r['step_tflops']:.2f} | {ratio} | {r.get('torch_dense_fwd_ms', float('nan')):.3f} | "
              f"{'yes' if r['fits_l2_fwd'] else 'no'}, {'yes' if r['fits_l2_step'] else 'no'} |")


if __name__ == "__main__":
    main()
