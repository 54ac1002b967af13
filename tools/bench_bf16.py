"""Times bfloat16 against float16 on the tcgen05 kernels, in one process on one GPU:

  * C2 (causal_1d, 16 x 16 heads, d = 128, S = 8192) and C4's shape (full_1d, Lq = 1024, Lk = 8192, scale_end,
    16 x 16 heads, d = 64): forward, and forward + backward through the autograd function;
  * on C2, the cast workaround a bf16 model has without bf16 kernels: Q, K, V, dO cast to fp16, the fp16 kernels, and
    O, dQ, dK, dV cast back to bf16;
  * on C2, torch.nn.functional.scaled_dot_product_attention in bf16 on the same problem, its [B, H, S, d] layout
    prepared outside the timed region.

CUDA events around back-to-back calls after warm-up; every arm is timed --rounds times, the arms alternating, and the
median is reported. The working sets (>= 1 GB) are far larger than the 126 MB L2. Prints one JSON object per
measurement, the card (name, power limit, SM clock) and a markdown table.

    python tools/bench_bf16.py [--rounds 3] [--window 1.0] [--out results.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tf_flash_attention_b200 import _capi  # noqa: E402
from tf_flash_attention_b200 import flash_attention as fa  # noqa: E402

SHAPES = {
    "C2": dict(op="causal", sync="none_front", heads=(16, 16), d=128, q=8192, k=8192),
    "C4": dict(op="full", sync="scale_end", heads=(16, 16), d=64, q=1024, k=8192),
}


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        out["nvidia_smi"] = q.splitlines()[0] if q else ""
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
    return a.elapsed_time(b) / n


def attend(cfg, q, k, v):
    if cfg["op"] == "causal":
        return fa.causal_1d(q, k, v, cfg["sync"])
    return fa.full_1d(q, k, v, sync_mode=cfg["sync"])


def arms(name, cfg):
    g = torch.Generator(device="cuda").manual_seed(7)
    b, d = cfg["heads"], cfg["d"]

    def u(seq):
        return torch.rand(b + (d, seq), generator=g, device="cuda") * 4 - 2

    base = {n: u(s) for n, s in (("q", cfg["q"]), ("k", cfg["k"]), ("v", cfg["k"]), ("do", cfg["q"]))}
    out = {}
    for dt, tag in ((torch.bfloat16, "bf16"), (torch.float16, "fp16")):
        q, k, v, do = (base[n].to(dt) for n in ("q", "k", "v", "do"))
        leaf = [x.clone().requires_grad_(True) for x in (q, k, v)]

        def fwd(q=q, k=k, v=v):
            with torch.no_grad():
                attend(cfg, q, k, v)

        def step(leaf=leaf, do=do):
            o = attend(cfg, *leaf)
            torch.autograd.grad(o, leaf, do)

        out[f"{name} fwd {tag}"] = fwd
        out[f"{name} fwd+bwd {tag}"] = step
    if name == "C2":
        qb, kb, vb, dob = (base[n].to(torch.bfloat16) for n in ("q", "k", "v", "do"))

        def cast_step():
            leaf = [x.to(torch.float16).requires_grad_(True) for x in (qb, kb, vb)]
            o = attend(cfg, *leaf)
            grads = torch.autograd.grad(o, leaf, dob.to(torch.float16))
            o.detach().to(torch.bfloat16)
            [x.to(torch.bfloat16) for x in grads]

        out[f"{name} fwd+bwd bf16 via fp16 casts"] = cast_step
        # SDPA layout [B, H, S, d]: the transposes happen here, outside the timed region
        sq, sk, sv, sdo = (x.reshape((-1,) + x.shape[-2:]).transpose(-1, -2).contiguous().unsqueeze(0)
                           for x in (qb, kb, vb, dob))
        sleaf = [x.clone().requires_grad_(True) for x in (sq, sk, sv)]

        def sdpa_step():
            o = torch.nn.functional.scaled_dot_product_attention(*sleaf, is_causal=True)
            torch.autograd.grad(o, sleaf, sdo)

        out[f"{name} fwd+bwd bf16 torch SDPA"] = sdpa_step
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_bf16 needs a CUDA device")
    info = card()
    print(json.dumps({"card": info}), flush=True)
    results = []
    for name, cfg in SHAPES.items():
        fns = arms(name, cfg)
        times = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, fn in fns.items():
                times[k].append(timed(fn, args.window))
        paths = {}
        for tag, code in (("bf16", _capi.FA_BF16), ("fp16", _capi.FA_F16)):
            p = _capi.make_problem(code, 1, cfg["op"], cfg["sync"], cfg["heads"] + (cfg["d"], cfg["q"]),
                                   cfg["heads"] + (cfg["d"], cfg["k"]), cfg["heads"] + (cfg["d"], cfg["k"]))
            paths[tag] = [_capi.dispatch_path(p, bwd)[0] for bwd in (False, True)]
        for k, ts in times.items():
            r = {"measurement": k, "ms_median": statistics.median(ts), "ms_all": ts, "dispatch": paths}
            results.append(r)
            print(json.dumps(r), flush=True)
        del fns
        torch.cuda.empty_cache()
    print(f"\n{info}\n\n| measurement | ms (median of {args.rounds}) |\n|---|---|")
    for r in results:
        print(f"| {r['measurement']} | {r['ms_median']:.3f} |")
    for name in SHAPES:
        for what in ("fwd", "fwd+bwd"):
            a = next(r["ms_median"] for r in results if r["measurement"] == f"{name} {what} bf16")
            b = next(r["ms_median"] for r in results if r["measurement"] == f"{name} {what} fp16")
            print(f"{name} {what}: bf16 / fp16 = {a / b:.3f}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"card": info, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
