#!/usr/bin/env python
"""bench.py — the headline benchmark of BASELINE.json on B200.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C2|C1|C3|C4|C4f32|C4f64|C5|S1|S2|T1]
                  [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] — causal_1d fp16 forward + backward,
batch x heads = 16 x 16, head_dim 128, seq 8192 (GPT-style self-attention), inputs U(-2,2) already
resident in HBM. One "step" = one forward + one backward pass of the hot path over that batch.
With N > 1 (torchrun, one process per GPU) the batch x heads units are split contiguously over the ranks
(the unit is the reference's gridDim.y = b, flash_attention.cu:2174-2176), no communication: "strong" scaling by
default (the 256 heads of the workload are shared out, 256 / N per GPU, device-timed value AND e2e); `--scaling weak`
gives every rank the full batch instead. value = total unmasked FLOPs of all ranks / max-over-ranks time.

Metric: attention fwd/bwd TFLOPS counting only unmasked FLOPs
  fwd = 2 * nnz * (d + v_d) * batch, bwd = 2 * nnz * (3 d + 2 v_d) * batch  (BASELINE.md §3).

The product path is libfa_b200.so through its C ABI (ctypes); torch only owns device memory,
streams and the process group. oracle/ is used solely for the cpu_baseline / --impl reference legs.
"""
import argparse
import atexit
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (fn, dtype, batch_shape, d, v_d, q_shape, k_shape, rule, sync, window, log2_stride, causal)
    "C2": dict(desc="causal_1d fp16 fwd+bwd, batch*heads 16x16, head_dim 128, seq 8192", seq_dims=1,
               dtype="float16", batch=(16, 16), d=128, v_d=128, q=(8192,), k=(8192,), rule="causal",
               sync="none_front", w=1, s=0, c=0),
    # C2 with channel-last tensors [16, 8192, 16, 128] read / written directly by the kernels (SURVEY.md section 8 f3)
    "C2cl": dict(desc="causal_1d fp16 fwd+bwd, channel-last tensors [16, 8192, 16 heads, 128] read directly, seq 8192",
                 seq_dims=1, dtype="float16", batch=(16, 16), d=128, v_d=128, q=(8192,), k=(8192,), rule="causal",
                 sync="none_front", w=1, s=0, c=0, channel_last_heads=16),
    "C1": dict(desc="local_1d fp32 README example Q[8,32,1024] K[8,32,2048] V[8,16,2048] w32 s0 scale_front",
               seq_dims=1, dtype="float32", batch=(8,), d=32, v_d=16, q=(1024,), k=(2048,), rule="local",
               sync="scale_front", w=32, s=0, c=0),
    "C3": dict(desc="local_2d fp16 causal 64x64 grid, window 8, none_front, head_dim 64, 16x16 heads", seq_dims=2,
               dtype="float16", batch=(16, 16), d=64, v_d=64, q=(64, 64), k=(64, 64), rule="local",
               sync="none_front", w=8, s=0, c=1),
    "C4": dict(desc="full_1d cross-attention Lq=1024 Lk=8192 scale_end fp16 head_dim 64, 256 heads", seq_dims=1,
               dtype="float16", batch=(16, 16), d=64, v_d=64, q=(1024,), k=(8192,), rule="full",
               sync="scale_end", w=1, s=0, c=0),
    "C4f32": dict(desc="full_1d cross-attention Lq=1024 Lk=8192 scale_end fp32 (3xTF32 forward) head_dim 64, 64 heads",
                  seq_dims=1, dtype="float32", batch=(8, 8), d=64, v_d=64, q=(1024,), k=(8192,), rule="full",
                  sync="scale_end", w=1, s=0, c=0),
    "C4f64": dict(desc="full_1d cross-attention Lq=1024 Lk=8192 scale_end fp64 (DFMA) head_dim 64, 16 heads",
                  seq_dims=1, dtype="float64", batch=(4, 4), d=64, v_d=64, q=(1024,), k=(8192,), rule="full",
                  sync="scale_end", w=1, s=0, c=0),
    # bandwidth-bound short-sequence cases (north_star: "achieved HBM GB/s for the bandwidth-bound short-sequence cases")
    "S1": dict(desc="causal_1d fp16 short sequences: 16384 heads x seq 256, head_dim 64 (HBM-bound)", seq_dims=1,
               dtype="float16", batch=(64, 256), d=64, v_d=64, q=(256,), k=(256,), rule="causal",
               sync="none_front", w=1, s=0, c=0),
    "S2": dict(desc="local_1d fp16 window 32, 2048 heads x seq 4096, head_dim 64 (HBM-bound)", seq_dims=1,
               dtype="float16", batch=(8, 256), d=64, v_d=64, q=(4096,), k=(4096,), rule="local",
               sync="none_front", w=32, s=0, c=0),
    "C5": dict(desc="causal_1d fp16 single sequence 131072, head_dim 128, 16 heads, K/V ring over NCCL (fwd)",
               seq_dims=1, dtype="float16", batch=(1, 16), d=128, v_d=128, q=(131072,), k=(131072,), rule="causal",
               sync="none_front", w=1, s=0, c=0, ring=True),
    # the step either side of the op (SURVEY.md section 8 f3): channel-last activations <-> the op's channel-first layout
    "T1": dict(desc="layout adapter fp16: [16, 8192, 16, 128] channel-last -> channel-first -> channel-last (HBM-bound)",
               seq_dims=1, dtype="float16", batch=(16, 16), d=128, v_d=128, q=(8192,), k=(8192,), rule="full",
               sync="none_front", w=1, s=0, c=0, layout=True),
}


# DRAM bytes per launch measured with `ncu --set full` on the GPU (profiles/r1_*_ncu*.md); bench.py cannot
# run under a profiler, so the captured values are carried here for the workload they were taken on.
NCU_TRAFFIC = {("C2", "fwd"): 2.153e9, ("C2", "bwd"): 5.35e9,  # bwd: the fused dQ/dK/dV kernel alone
               ("T1", "layout"): 1.027e9}                     # profiles/r1_layout_ncu.md


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"tensor_burst": d.get("bf16_tflops"), "tensor_sustained": d.get("bf16_tflops_sustained"),
                "hbm": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tensor_burst": 1590.0, "tensor_sustained": 1400.0, "hbm": 6650.0,
            "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region. nvidia-smi is started
    early (before the warm-up) because its start-up can take longer than a short timed region; only the
    rows read between mark_start() and mark_end() are used."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def launch(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.terminate)     # the sampler never outlives a run that fails before stop()
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def start(self):
        if self.proc is None:
            self.launch()
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if self.t0 <= t <= self.t1 + 0.05]
        if not rows:  # timed region shorter than one sampling period: take the closest sample after it
            rows = [r for (t, r) in self.rows if t >= self.t0][:1]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def attended_pairs(w):
    """Attended (q, k) pairs per batch element, on the host, without the product library: closed form for the
    1-D causal / full rules with equal lengths (C2, C5), otherwise counted from the oracle's bit-exact rule."""
    nq, nk = int(np.prod(w["q"])), int(np.prod(w["k"]))
    if w["seq_dims"] == 1 and w["sync"] == "none_front" and nq == nk and w["rule"] == "causal":
        return nq * (nq + 1) // 2
    if w["rule"] == "full":
        return nq * nk
    from oracle import pattern
    return int(pattern.nnz(w["q"], w["k"], w["sync"], w["rule"], w["w"], w["s"], bool(w["c"])))


def flops_of(w, nnz):
    b = int(np.prod(w["batch"]))
    return 2.0 * nnz * (w["d"] + w["v_d"]) * b, 2.0 * nnz * (3 * w["d"] + 2 * w["v_d"]) * b


DUMP_BYTES = 64 * 10 ** 6   # --dump-outputs writes at most this many bytes in all, .npy headers included


def dump_outputs(out_dir, outputs, rank, world):
    """Writes each device tensor of `outputs` (name -> tensor) to out_dir/<name>.npy in float32 (float64 stays
    float64), with a _rank<r> suffix when several ranks run. A tensor whose file would exceed its equal share of
    DUMP_BYTES is written as its elements at a fixed, seeded, sorted set of flat indices (the same for every tensor of
    that size on every run), so the outputs of two builds can be compared element for element."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // (len(outputs) * world) - 1024          # 1 KB of each file's share kept for its header
    for name, t in outputs.items():
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        t = t.detach()
        n = share // (8 if dt == torch.float64 else 4)
        if t.numel() > n:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), n, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        suffix = f"_rank{rank}" if world > 1 else ""
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), t.to(dt).cpu().numpy())


def cpu_reference_leg(w, nnz, steps, warmup, heads):
    """The reference's CPU path (its tests' dense attention; oracle port) on a bounded sample."""
    import torch
    from oracle import dense_torch_cpu as cpu
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nq, nk = int(np.prod(w["q"])), int(np.prod(w["k"]))
    mask = cpu.mask_tensor(w["q"], w["k"], w["sync"], w["rule"], w["w"], w["s"], bool(w["c"]))
    sec = cpu.time_fwd_bwd(heads, w["d"], w["v_d"], nq, nk, mask, steps=steps, warmup=warmup)
    fl = 2.0 * nnz * (w["d"] + w["v_d"]) * heads + 2.0 * nnz * (3 * w["d"] + 2 * w["v_d"]) * heads
    return {"value": fl / sec / 1e12, "unit": "TFLOPS", "cores": cores, "kind": "port",
            "sample": f"{heads} of {int(np.prod(w['batch']))} heads of the same workload, full {nq}x{nk} "
                      f"logits per head, fwd + autodiff bwd in fp32 with torch CPU ops (TensorFlow absent), "
                      f"{sec:.2f} s per step", "sec_per_step": sec}


def ring_bench(args, w, nnz, config, rank, world, local_rank):
    """C5: one causal sequence of 131072 sharded zig-zag over the ranks; STRONG scaling (total work fixed).
    Forward by default; `--ring-bwd` times forward + ring backward (SURVEY.md section 8f)."""
    import torch
    import torch.distributed as dist
    from tf_flash_attention_b200 import _capi, ring
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    S = w["q"][0]
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    shard = S // world

    def u(ch):
        return (torch.rand(w["batch"] + (ch, shard), generator=g, device=dev) * 4 - 2).half()
    Q, K, V = u(w["d"]), u(w["d"]), u(w["v_d"])
    dO = u(w["v_d"])
    out = {}                                            # what the last step returned (--dump-outputs)

    def ring_step():
        if not args.ring_bwd:
            out["O"] = ring.ring_causal_1d(Q, K, V)
            return
        out["O"], out["l"], out["m"] = ring.ring_causal_1d(Q, K, V, returning_l_m=True)
        out["dQ"], out["dK"], out["dV"] = ring.ring_causal_1d_backward(Q, K, V, out["O"], out["l"], out["m"], dO)
    sampler = ClockSampler(local_rank)
    sampler.launch()
    for _ in range(max(3, args.warmup)):
        ring_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    _capi.lib.fa_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        ring_step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = int(_capi.lib.fa_launch_count(0))
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank, world)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    fwd_flops = 2.0 * nnz * (w["d"] + w["v_d"]) * int(np.prod(w["batch"]))
    if args.ring_bwd:
        fwd_flops += 2.0 * nnz * (3 * w["d"] + 2 * w["v_d"]) * int(np.prod(w["batch"]))
    value = fwd_flops / (ms * 1e-3) / 1e12
    peaks = measured_peaks()
    peak = (peaks["tensor_sustained"] or peaks["tensor_burst"]) * world
    config = dict(config, flops_per_step=fwd_flops, parallelism=f"K/V ring, zig-zag chunks, {world} rank(s), shards on the copy engines (fa_ring peer copies), "
                  f"{os.environ.get('FA_RING_DRIVER', 'native')} driver")
    config["pass"] = "fwd+bwd" if args.ring_bwd else "fwd"
    line = {"metric": f"attention {config['pass']} TFLOPS (unmasked FLOPs), single sequence K/V ring", "value": value, "unit": "TFLOPS",
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16 (fp32 accumulate)",
            "data": "synthetic U(-2,2)", "config": config, "clocks": clocks, "gpu_launches": launches,
            "roofline": {"bound": "tensor", "kernel": "fwd_f16_sm100 (per-block partials) + partial_merge" + (" + backward blocks + grad_accumulate" if args.ring_bwd else ""),
                         "achieved": value, "peak": peak, "unit": "TFLOP/s", "frac": value / peak, "traffic": None,
                         "peak_source": peaks["source"] + f", sustained bf16 GEMM x {world} GPUs"}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def layout_bench(args, w, rank, world, local_rank):
    """T1: fa_layout_transpose both ways over one activation tensor larger than L2; bytes = one read + one write per
    launch. Every rank converts its own tensor (no communication)."""
    import torch
    import torch.distributed as dist
    from tf_flash_attention_b200 import _capi
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, H, Cc, S = w["batch"][0], w["batch"][1], w["d"], w["q"][0]
    g = torch.Generator(device=dev).manual_seed(5 + rank)
    x = (torch.rand((B, S, H, Cc), generator=g, device=dev) * 4 - 2).half()
    y = torch.empty((B, H, Cc, S), dtype=x.dtype, device=dev)
    x2 = torch.empty_like(x)
    sp = torch.cuda.current_stream(dev).cuda_stream
    if args.override:
        _capi.lib.fa_set_path_override(args.override)

    def step():
        _capi.check(_capi.lib.fa_layout_transpose(0, x.data_ptr(), y.data_ptr(), B, S, H, Cc, 1, sp), "fa_layout_transpose")
        _capi.check(_capi.lib.fa_layout_transpose(0, y.data_ptr(), x2.data_ptr(), B, S, H, Cc, 0, sp), "fa_layout_transpose")
    sampler = ClockSampler(local_rank)
    sampler.launch()
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    assert torch.equal(x, x2) and torch.equal(y, x.permute(0, 2, 3, 1)), "layout adapter round trip differs"
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    _capi.lib.fa_launch_count(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = int(_capi.lib.fa_launch_count(0))
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"channel_first": y, "round_trip": x2}, rank, world)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    nbytes = x.numel() * x.element_size()
    gbs = 2 * (2 * nbytes) / (ms * 1e-3) / 1e9           # two launches per step, each one read + one write
    peaks = measured_peaks()
    line = {"metric": "layout adapter GB/s (algorithmic bytes: one read + one write per launch)", "value": gbs * world,
            "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 (byte moves)",
            "data": "synthetic U(-2,2)", "config": {"workload": f"T1: {w['desc']}", "bytes_per_launch": 2 * nbytes,
                                                    "l2": "tensor (537 MB) larger than the 126 MB L2"},
            "clocks": clocks, "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "layout_transpose", "achieved": gbs, "peak": peaks["hbm"],
                         "unit": "GB/s", "frac": gbs / peaks["hbm"], "traffic": NCU_TRAFFIC[("T1", "layout")],
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full "
                                           "(profiles/r1_layout_ncu.md)",
                         "algorithmic": f"{2 * nbytes} bytes per launch (the tensor read once and written once)",
                         "peak_source": peaks["source"]}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"{s} is not a positive integer")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-warmup", type=int, default=2)
    ap.add_argument("--cpu-heads", type=int, default=4)
    ap.add_argument("--scaling", default=None, choices=["strong", "weak"],
                    help="N > 1: strong (default) splits the workload's batch x heads over the ranks; weak replicates it")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-refkernel", action="store_true")
    ap.add_argument("--fwd-only", action="store_true")
    ap.add_argument("--override", type=int, default=0, help="fa_set_path_override value (developer A/B)")
    ap.add_argument("--grad-precision", type=int, default=0, help="fa_set_grad_precision mode (0 auto, 1 split, 2 off)")
    ap.add_argument("--graph", action="store_true", help="replay the step as one CUDA graph (launch-bound workloads)")
    ap.add_argument("--ring-bwd", action="store_true", help="C5: time forward + ring backward")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB in all: larger outputs as a fixed, seeded sample of their elements)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    scaling = args.scaling or ("weak" if (w.get("ring") or w.get("layout")) else "strong")
    if w.get("ring"):
        scaling = "strong"
    n_units = int(np.prod(w["batch"]))                 # batch x heads units of the whole workload
    if scaling == "strong" and not w.get("ring") and not w.get("layout"):
        assert n_units % world == 0, f"{n_units} batch x head units do not split over {world} ranks"
        local_units, total_units = n_units // world, n_units
    else:
        local_units, total_units = n_units, n_units * world
    nnz = attended_pairs(w)                             # oracle-free closed form or oracle.pattern (host, integer)
    fwd_flops_unit = 2.0 * nnz * (w["d"] + w["v_d"])
    bwd_flops_unit = 2.0 * nnz * (3 * w["d"] + 2 * w["v_d"])
    fwd_flops, bwd_flops = fwd_flops_unit * total_units, bwd_flops_unit * total_units   # whole job, all ranks
    step_flops = fwd_flops + (0 if args.fwd_only else bwd_flops)
    config = {"workload": f"{args.workload}: {w['desc']}", "batch_heads": total_units, "batch_heads_per_gpu": local_units,
              "head_dim": w["d"], "seq_q": int(np.prod(w["q"])), "seq_k": int(np.prod(w["k"])),
              "nnz_per_head": nnz, "flops_per_step": step_flops, "fwd_flops": fwd_flops, "bwd_flops": bwd_flops,
              "pass": "fwd" if args.fwd_only else "fwd+bwd",
              "parallelism": f"batch x head sharding ({scaling}), {world} rank(s), no communication",
              "l2": "inputs larger than the 126 MB L2 (no flush needed)"}

    # ---------------- reference arm: the reference's CPU path on the host cores ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        heads = max(1, args.cpu_heads)
        leg = cpu_reference_leg(w, nnz, max(1, args.steps), max(1, args.warmup), heads)
        line = {"impl": "reference", "metric": "attention fwd+bwd TFLOPS (unmasked FLOPs)", "value": leg["value"],
                "unit": "TFLOPS", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": leg["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "f32 (CPU; fp16 inputs computed in fp32)", "data": "synthetic U(-2,2)",
                "config": config, "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": leg["value"], "unit": "TFLOPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return

    # the product library is loaded only on our arm (the reference arm above never touches it)
    from tf_flash_attention_b200 import _capi
    if w.get("ring"):
        return ring_bench(args, w, nnz, config, rank, world, local_rank)
    if w.get("layout"):
        return layout_bench(args, w, rank, world, local_rank)
    code = {"float16": 0, "float32": 1, "float64": 2}[w["dtype"]]
    bshape = (local_units,)                             # this rank's contiguous slice of the flattened batch x heads
    prob = _capi.make_problem(code, w["seq_dims"], w["rule"], w["sync"], bshape + (w["d"],) + w["q"],
                              bshape + (w["d"],) + w["k"], bshape + (w["v_d"],) + w["k"], w["w"], w["s"], w["c"])
    assert _capi.count_attended(prob) == nnz, "attended-pair count of the library differs from the host count"
    if w.get("channel_last_heads"):
        # same element counts, the kernels address them as [outer, seq, heads, channels]; l, m stay [batch, q]
        assert local_units % w["channel_last_heads"] == 0
        prob.layout, prob.heads = _capi.FA_LAYOUT_CHANNEL_LAST, w["channel_last_heads"]
        args.no_e2e = True        # the host-buffer entry points take the reference's channel-first layout only
        args.no_refkernel = True

    # ---------------- our arm -------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    tdt = {"float16": torch.float16, "float32": torch.float32, "float64": torch.float64}[w["dtype"]]
    ldt = torch.float32 if tdt == torch.float16 else tdt
    g = torch.Generator(device=dev).manual_seed(1234 + rank)

    def u(shape):
        return (torch.rand(shape, generator=g, device=dev, dtype=torch.float32) * 4 - 2).to(tdt)

    Q, K = u(bshape + (w["d"],) + w["q"]), u(bshape + (w["d"],) + w["k"])
    V, dO = u(bshape + (w["v_d"],) + w["k"]), u(bshape + (w["v_d"],) + w["q"])
    O = torch.empty_like(dO)
    l = torch.empty(bshape + w["q"], dtype=ldt, device=dev)
    m = torch.empty(bshape + w["q"], dtype=tdt, device=dev)
    dQ, dK, dV = torch.empty_like(Q), torch.empty_like(K), torch.empty_like(V)
    if args.grad_precision:
        _capi.lib.fa_set_grad_precision(args.grad_precision)
    if args.override:
        _capi.lib.fa_set_path_override(args.override)   # before sizing the workspace: the path decides its size
    ws_bytes = max(_capi.lib.fa_workspace_bytes(C.byref(prob), 1), _capi.lib.fa_workspace_bytes(C.byref(prob), 0), 1)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream

    def fwd():
        _capi.check(_capi.lib.fa_forward(C.byref(prob), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(),
                                         l.data_ptr(), m.data_ptr(), ws.data_ptr(), ws_bytes, sp), "fa_forward")

    def bwd():
        _capi.check(_capi.lib.fa_backward(C.byref(prob), Q.data_ptr(), K.data_ptr(), V.data_ptr(), O.data_ptr(),
                                          l.data_ptr(), m.data_ptr(), dO.data_ptr(), dQ.data_ptr(), dK.data_ptr(),
                                          dV.data_ptr(), ws.data_ptr(), ws_bytes, sp), "fa_backward")

    def step():
        fwd()
        if not args.fwd_only:
            bwd()

    if args.graph:
        # capture one step (all launches are stream-ordered) and replay it; per-kernel event timing is not
        # available inside a graph, so the kernel table of this run comes from one eager step
        eager_step = step
        eager_step()
        torch.cuda.synchronize()
        cuda_graph = torch.cuda.CUDAGraph()
        _capi.lib.fa_launch_count(1)
        with torch.cuda.graph(cuda_graph):
            sp_saved = sp
            sp = torch.cuda.current_stream(dev).cuda_stream
            eager_step()
            sp = sp_saved
        graph_launches = int(_capi.lib.fa_launch_count(0))   # kernels captured per step

        def step():  # noqa: F811
            cuda_graph.replay()
    sampler = ClockSampler(local_rank)
    sampler.launch()
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    fwd_path = None
    fwd()
    fwd_path = _capi.PATH_NAMES[_capi.lib.fa_last_path()]
    bwd_path = None
    if not args.fwd_only:
        bwd()
        bwd_path = _capi.PATH_NAMES[_capi.lib.fa_last_path()]
    torch.cuda.synchronize()

    # timed region: exactly K steps, CUDA events on the launching stream, barrier + sync both sides
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    _capi.lib.fa_launch_count(1)
    # per-kernel event brackets cost two event records per launch: on for the millisecond-scale workloads (their
    # durations feed the roofline of the same timed steps), off for the launch-bound ones (--workload C1), whose
    # per-kernel table is taken from a few extra steps after the timed region
    timing_inline = w["dtype"] == "float16" or int(np.prod(w["q"])) * int(np.prod(w["k"])) * local_units >= 1 << 30
    _capi.lib.fa_kernel_timing(1 if timing_inline else 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    _capi.lib.fa_kernel_timing(0)
    launches = int(_capi.lib.fa_launch_count(0))
    if args.graph:
        launches = graph_launches * args.steps   # replayed from the captured graph, not re-issued by the library
    clocks = sampler.stop()
    if args.dump_outputs:
        outputs = {"O": O, "l": l, "m": m}
        if not args.fwd_only:
            outputs.update(dQ=dQ, dK=dK, dV=dV)
        dump_outputs(args.dump_outputs, outputs, rank, world)
    ms_total = e0.elapsed_time(e1)
    kt = _capi.kernel_timings()
    if not timing_inline and not args.graph:
        _capi.lib.fa_kernel_timing(1)
        for _ in range(min(args.steps, 20)):
            step()
        torch.cuda.synchronize()
        _capi.lib.fa_kernel_timing(0)
        kt = _capi.kernel_timings()
    if args.graph:
        # per-kernel durations of one eager step outside the timed region (events cannot be recorded into the replay)
        _capi.lib.fa_kernel_timing(1)
        eager_step()
        torch.cuda.synchronize()
        _capi.lib.fa_kernel_timing(0)
        kt = _capi.kernel_timings()
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = step_flops / (ms_per_step * 1e-3) / 1e12    # step_flops covers all ranks
    # per-launch figures of THIS rank's kernels (roofline): its own share of the units
    fwd_flops_l, bwd_flops_l = fwd_flops_unit * local_units, bwd_flops_unit * local_units

    # per-kernel durations -> roofline of the dominant kernel
    per = {}
    for name, ms in kt:
        per.setdefault(name, []).append(ms)
    share_scale = args.steps if args.graph else (1 if timing_inline else args.steps / min(args.steps, 20))
    kernels = {n: {"launches": len(v), "avg_ms": float(np.mean(v)), "share": float(np.sum(v)) * share_scale / ms_total}
               for n, v in per.items()}
    peaks = measured_peaks()
    roofline = None
    traffic = None
    if kernels:
        dom = max(kernels, key=lambda n: kernels[n]["share"])
        bwd_names = [n for n in kernels if "bwd" in n]
        if dom.startswith("fwd_") or dom == "generic_fwd":
            ach = fwd_flops_l / (kernels[dom]["avg_ms"] * 1e-3) / 1e12
            what = f"{dom}: 2*nnz*(d+v_d)*batch FLOPs per launch"
            traffic = NCU_TRAFFIC.get((args.workload, "fwd"))
        else:
            tb = sum(kernels[n]["avg_ms"] for n in bwd_names)
            if "bwd_fused_f16_sm100" in kernels:
                # every algorithmic backward FLOP runs in the fused kernel (prep / zero / convert are HBM helpers)
                dom = "bwd_fused_f16_sm100"
                ach = bwd_flops_l / (kernels[dom]["avg_ms"] * 1e-3) / 1e12
                what = f"{dom}: 2*nnz*(3d+2v_d)*batch FLOPs per launch"
            else:
                # two-kernel backward: algorithmic bwd FLOPs / sum of the backward kernels' durations
                ach = bwd_flops_l / (tb * 1e-3) / 1e12
                dom = "+".join(sorted(bwd_names))
                what = f"{dom}: 2*nnz*(3d+2v_d)*batch FLOPs per backward pass"
            traffic = NCU_TRAFFIC.get((args.workload, "bwd"))
        peak = peaks["tensor_sustained"] or peaks["tensor_burst"]
        peak_note = ", sustained bf16 GEMM"
        if w["dtype"] == "float32":
            # split precision: 3 half-rate TF32 MMAs (forward) or 6 full-rate bf16 MMAs (backward) per fp32 product
            peak = peak / 6.0
            peak_note = ", sustained bf16 GEMM / 6 (fp32 through split-precision tensor-core products)"
        elif w["dtype"] == "float64":
            # measured in this process: cuBLAS DGEMM 4096^3 (torch.matmul), best of 5 after a warm-up
            A64 = torch.rand((4096, 4096), dtype=torch.float64, device=dev)
            B64 = torch.rand((4096, 4096), dtype=torch.float64, device=dev)
            torch.matmul(A64, B64)
            best = 1e9
            for _ in range(5):
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                torch.matmul(A64, B64)
                g1.record()
                torch.cuda.synchronize()
                best = min(best, g0.elapsed_time(g1))
            peak = 2.0 * 4096 ** 3 / (best * 1e-3) / 1e12
            del A64, B64
            peak_note = f"; fp64: cuBLAS DGEMM 4096^3 measured in this run ({peak:.1f} TFLOP/s; nominal 40)"
        roofline = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": ach / peak, "traffic": traffic, "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full captures of round 2 summarised in profiles/r2_c2_ncu.md (forward 2.155 GB = the algorithmic bytes; fused backward 5.35 GB against 3.2 GB algorithmic: the fp32 dQ scratch spilling out of L2)" if traffic else None, "peak_source": peaks["source"] + peak_note,
                    "frac_of_burst": ach / (peaks["tensor_burst"] or peak), "frac_of_nominal_2250": ach / 2250.0,
                    "algorithmic": what}
        # HBM side of the roofline: algorithmic bytes of the same kernel(s) (DESIGN.md section 4) over their duration.
        # Workloads whose arithmetic intensity is below the ridge (short sequences, narrow windows) are HBM-bound
        # and report that as the primary bound.
        esz = {"float16": 2, "float32": 4, "float64": 8}[w["dtype"]]
        lsz = 4 if w["dtype"] == "float16" else esz
        nb, nq_, nk_ = local_units, int(np.prod(w["q"])), int(np.prod(w["k"]))
        fwd_bytes = esz * nb * (nq_ * w["d"] + nk_ * w["d"] + nk_ * w["v_d"] + nq_ * w["v_d"]) + nb * nq_ * (lsz + esz)
        bwd_bytes = esz * nb * (2 * nq_ * w["d"] + 2 * nk_ * w["d"] + 2 * nk_ * w["v_d"] + 2 * nq_ * w["v_d"]) + nb * nq_ * (lsz + esz)
        is_fwd = roofline["kernel"].startswith("fwd_") or roofline["kernel"] == "generic_fwd"
        k_bytes = fwd_bytes if is_fwd else bwd_bytes
        k_ms = kernels[roofline["kernel"]]["avg_ms"] if roofline["kernel"] in kernels else sum(kernels[n]["avg_ms"] for n in bwd_names)
        k_flops = fwd_flops_l if is_fwd else bwd_flops_l
        gbs = k_bytes / (k_ms * 1e-3) / 1e9
        ridge = peak * 1e12 / (peaks["hbm"] * 1e9)
        roofline["hbm"] = {"algorithmic_bytes": k_bytes, "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                           "frac": gbs / peaks["hbm"], "intensity_flop_per_byte": k_flops / k_bytes,
                           "ridge_flop_per_byte": ridge}
        if k_flops / k_bytes < ridge:
            roofline.update({"bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
                             "frac": gbs / peaks["hbm"], "tensor": {"achieved": ach, "peak": peak, "frac": ach / peak},
                             "algorithmic": what + f"; {k_bytes} algorithmic bytes (inputs and outputs once)"})
        if bwd_names:
            tb_all = sum(kernels[n]["avg_ms"] for n in bwd_names)
            roofline["backward_all_kernels"] = {"kernels": sorted(bwd_names), "ms": tb_all,
                                                "achieved": bwd_flops_l / (tb_all * 1e-3) / 1e12, "unit": "TFLOP/s",
                                                "frac": bwd_flops_l / (tb_all * 1e-3) / 1e12 / peak}
        if "fwd_f16_sm100" in kernels:
            fa_ = fwd_flops_l / (kernels["fwd_f16_sm100"]["avg_ms"] * 1e-3) / 1e12
            roofline["fwd_kernel"] = {"achieved": fa_, "frac": fa_ / peak, "frac_of_burst": fa_ / (peaks["tensor_burst"] or peak),
                                      "frac_of_nominal_2250": fa_ / 2250.0}

    line = {"metric": "attention fwd+bwd TFLOPS (unmasked FLOPs)" if not args.fwd_only else "attention fwd TFLOPS (unmasked FLOPs)",
            "value": value, "unit": "TFLOPS", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate)" if w["dtype"] == "float16" else w["dtype"], "data": "synthetic U(-2,2), seed 1234",
            "config": config, "launch": "CUDA graph replay" if args.graph else "eager launches",
            "sequences_per_s": float(total_units) / (ms_per_step * 1e-3),
            "paths": {"fwd": fwd_path, "bwd": bwd_path}, "kernels": kernels, "roofline": roofline,
            "clocks": clocks, "gpu_launches": launches, "pct_of_nominal_fp16_peak": 100.0 * value / world / 2250.0}

    # ---------------- end-to-end through the host-buffer C ABI (rank-local) ----------------
    if not args.no_e2e:
        del dQ, dK, dV, ws
        hq, hk, hv, hdo = (x.cpu().pin_memory() for x in (Q, K, V, dO))
        ho = torch.empty_like(hdo).pin_memory()
        hl = torch.empty(l.shape, dtype=ldt).pin_memory()
        hm = torch.empty(m.shape, dtype=tdt).pin_memory()
        hdq, hdk, hdv = (torch.empty_like(x).pin_memory() for x in (hq, hk, hv))
        del Q, K, V, dO, O, l, m
        torch.cuda.empty_cache()
        nb_f = _capi.lib.fa_host_arena_bytes(C.byref(prob), 0)
        nb_b = _capi.lib.fa_host_arena_bytes(C.byref(prob), 1)
        nb_s = _capi.lib.fa_step_host_arena_bytes(C.byref(prob))
        arena = torch.empty(max(nb_f, nb_b, nb_s), dtype=torch.uint8, device=dev)

        def fwd_host():
            _capi.check(_capi.lib.fa_forward_host(C.byref(prob), hq.data_ptr(), hk.data_ptr(), hv.data_ptr(),
                                                  ho.data_ptr(), hl.data_ptr(), hm.data_ptr(), arena.data_ptr(),
                                                  arena.numel(), sp), "fa_forward_host")

        def e2e_step():
            # one training step on host buffers through the C ABI: forward + gradient, chunk-pipelined in one call
            if args.fwd_only:
                return fwd_host()
            _capi.check(_capi.lib.fa_forward_backward_host(C.byref(prob), hq.data_ptr(), hk.data_ptr(), hv.data_ptr(),
                                                           hdo.data_ptr(), ho.data_ptr(), hl.data_ptr(), hm.data_ptr(),
                                                           hdq.data_ptr(), hdk.data_ptr(), hdv.data_ptr(),
                                                           arena.data_ptr(), arena.numel(), sp),
                        "fa_forward_backward_host")

        def e2e_step_two_calls():
            # the same step as the reference's host framework runs it: forward op, then its registered gradient
            # with the forward's tensors still on the device (only dO is uploaded for the backward)
            fwd_host()
            if not args.fwd_only:
                _capi.check(_capi.lib.fa_backward_host_resident(C.byref(prob), hdo.data_ptr(), hdq.data_ptr(),
                                                                hdk.data_ptr(), hdv.data_ptr(), arena.data_ptr(),
                                                                arena.numel(), sp), "fa_backward_host_resident")

        def e2e_step_stateless():
            # the same step with nothing kept on the device between the two calls (every backward input re-uploaded)
            fwd_host()
            if not args.fwd_only:
                _capi.check(_capi.lib.fa_backward_host(C.byref(prob), hq.data_ptr(), hk.data_ptr(), hv.data_ptr(),
                                                       ho.data_ptr(), hl.data_ptr(), hm.data_ptr(), hdo.data_ptr(),
                                                       hdq.data_ptr(), hdk.data_ptr(), hdv.data_ptr(),
                                                       arena.data_ptr(), arena.numel(), sp), "fa_backward_host")

        def time_e2e(fn):
            for _ in range(max(1, args.e2e_warmup)):
                fn()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                fn()
            torch.cuda.synchronize()
            sec = (time.perf_counter() - t0) / args.e2e_steps
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        nb = lambda x: x.numel() * x.element_size()  # noqa: E731
        sec = time_e2e(e2e_step)
        h2d = nb(hq) + nb(hk) + nb(hv)
        d2h = nb(ho) + nb(hl) + nb(hm)
        if not args.fwd_only:
            h2d += nb(hdo)
            d2h += nb(hdq) + nb(hdk) + nb(hdv)
        line["e2e"] = {"value": step_flops / sec / 1e12, "unit": "TFLOPS", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "bytes_are": "per rank", "ms_per_step": sec * 1e3,
                       "steps": args.e2e_steps, "warmup": max(1, args.e2e_warmup),
                       "api": "fa_forward_host (C ABI, pinned host buffers, copies inside the call)" if args.fwd_only else
                              "fa_forward_backward_host (C ABI, pinned host buffers; uploads, kernels and downloads of "
                              "successive batch chunks overlap inside the call)"}
        if not args.fwd_only:
            sec1 = time_e2e(e2e_step_two_calls)
            line["e2e_two_calls"] = {"value": step_flops / sec1 / 1e12, "unit": "TFLOPS", "h2d_bytes_per_step": h2d,
                                     "d2h_bytes_per_step": d2h, "ms_per_step": sec1 * 1e3, "steps": args.e2e_steps,
                                     "api": "fa_forward_host + fa_backward_host_resident (Q, K, V, O, l, m stay on the "
                                            "device between the forward and its gradient)"}
            sec2 = time_e2e(e2e_step_stateless)
            line["e2e_stateless"] = {"value": step_flops / sec2 / 1e12, "unit": "TFLOPS",
                                     "h2d_bytes_per_step": h2d + nb(hq) + nb(hk) + nb(hv) + nb(ho) + nb(hl) + nb(hm),
                                     "d2h_bytes_per_step": d2h, "ms_per_step": sec2 * 1e3, "steps": args.e2e_steps,
                                     "api": "fa_forward_host + fa_backward_host (every backward input re-uploaded)"}
        del arena

    # ---------------- CPU baseline (rank 0, N = 1) ------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        leg = cpu_reference_leg(w, nnz, 3, 1, max(1, args.cpu_heads))   # 1 warm-up + 3 timed steps
        line["cpu_baseline"] = {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if rank == 0 and world == 1 and not args.no_refkernel:
        try:
            from oracle import refkernel
            line["ref_kernel_baseline"] = refkernel.bench(w, nnz, heads=8, fwd_only=args.fwd_only)
        except Exception as e:  # the reference build is optional (oracle/_ref)
            line["ref_kernel_baseline"] = {"unavailable": str(e)[:200]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree and writes nothing into it
    main()
