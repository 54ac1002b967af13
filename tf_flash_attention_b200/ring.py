"""K/V ring for ONE long 1-D sequence sharded over the GPUs of a node (BASELINE.json configs[4]).

New functionality — the reference is single-GPU (SURVEY.md §5, §8e). The sequence of length S is cut
into 2G chunks; rank r owns chunks r and 2G-1-r of Q, K and V ("zig-zag", which balances the causal
triangle). In G steps every rank attends its two local query chunks to the K/V shard currently
visiting (global index bases go into fa_problem_t, so the rule is evaluated on global coordinates and
blocks that lie entirely in the future are never launched), folds the partial (O, l, m) into fp32
accumulators (fa_partial_merge) and meanwhile passes the shard on to rank r+1 with NCCL send/recv
(torch.distributed P2P, NVLink 5 / NVSwitch) into the other half of a double buffer.

The driver is written against a tiny backend interface so that the host logic (chunk ownership, step
schedule, index bases, skip rule) can be exercised on CPU with the gloo backend and the NumPy oracle
as the compute stand-in (tests/test_ring_gloo.py); the product backend is `DeviceBackend` below, which
calls the C ABI (fa_forward / fa_partial_merge / fa_partial_finalize).

Causal rings take a batched schedule instead (`ring_forward_causal` / `ring_backward_causal`): chunks are kept
chunk-major, [2, batch..., channels, c], and every ring step is ONE launch over 2 x batch problems of c x c positions
(the per-block schedule launched 2-4 blocks of `batch` problems per step, each 3.46 waves of CTAs on 148 SMs at the C5
size, plus one merge per block):
  step 0 (own shard)        causal over [Q_lo; Q_hi] x [K_lo; K_hi] pairwise (both diagonal blocks), then Q_hi x K_lo full;
  visiting shard of c < r   full over [Q_lo; Q_hi] x [K_lo(c); K_lo(c)]   (its high chunk lies in the future of both);
  visiting shard of c > r   full over [Q_hi; Q_hi] x [K_lo(c); K_hi(c)]   (Q_lo sees none of it).
No index bases are needed: every launch is a plain causal or full problem in local coordinates.

Backward (`ring_backward`): every block (local query chunk x visiting key chunk) is one fa_backward call
made with the FINAL O, l, m of the whole sequence, so block results simply add. dQ accumulates locally in
fp32; the fp32 dK / dV accumulators travel around the ring together with their K/V shard (one extra hop
at the end brings them home), K/V one step ahead of the compute, the accumulators right behind it.
"""
import ctypes as C

import numpy as np

from . import _capi


class ZigZag:
    """Chunk ownership: 2G chunks of c = S / (2G) positions; rank r owns chunks (r, 2G-1-r)."""

    def __init__(self, seq_len, world):
        if seq_len % (2 * world):
            raise _capi.InvalidArgumentError(_capi.FA_EINVAL_SHAPE,
                                             f"sequence length {seq_len} must be a multiple of 2*world = {2 * world}")
        self.seq_len, self.world, self.chunk = seq_len, world, seq_len // (2 * world)

    def chunks(self, rank):
        return (rank, 2 * self.world - 1 - rank)

    def base(self, chunk_index):
        return chunk_index * self.chunk

    def gather_index(self, rank):
        """Global positions held by `rank`, in local order (for building / checking shards)."""
        a, b = self.chunks(rank)
        return np.concatenate([np.arange(self.base(a), self.base(a) + self.chunk),
                               np.arange(self.base(b), self.base(b) + self.chunk)])


def step_plan(layout, rank, step, rule, is_causal):
    """Blocks (local q chunk slot, visiting k chunk slot, q_base, k_base) to launch at `step`, when the
    K/V shard of rank (rank - step) mod G is visiting. Causal rules drop blocks entirely in the future."""
    src = (rank - step) % layout.world
    plan = []
    causal = rule == "causal" or (rule == "local" and is_causal)
    for qa, qc in enumerate(layout.chunks(rank)):
        for kb, kc in enumerate(layout.chunks(src)):
            if causal and kc > qc:
                continue  # every key of this block is later than every query (none_front, equal lengths)
            plan.append((qa, kb, layout.base(qc), layout.base(kc)))
    return src, plan


class StepTrace:
    """Developer aid (tools/ring_trace.py): host timestamps and CUDA events at the marks of one ring pass."""

    def __init__(self, torch):
        import time
        self.torch, self.time, self.marks = torch, time, []

    def mark(self, name):
        ev = self.torch.cuda.Event(enable_timing=True)
        ev.record()
        self.marks.append((name, self.time.perf_counter(), ev))

    def report(self):
        self.torch.cuda.synchronize()
        t0, e0 = self.marks[0][1], self.marks[0][2]
        return [(n, round((t - t0) * 1e3, 3), round(e0.elapsed_time(e), 3)) for n, t, e in self.marks]


class DeviceBackend:
    """Product backend: torch CUDA tensors for memory, the C ABI for every computation."""

    def __init__(self, dtype_code, rule, sync_mode, window_size, log2_stride_size, is_causal, batch_shape, d, v_d,
                 chunk, seq_len):
        import torch
        self.torch = torch
        self.rule, self.chunk, self.seq_len = rule, chunk, seq_len
        self.batch_shape = tuple(batch_shape)
        self.p = _capi.make_problem(dtype_code, 1, rule, sync_mode, self.batch_shape + (d, chunk),
                                    self.batch_shape + (d, chunk), self.batch_shape + (v_d, chunk), window_size,
                                    log2_stride_size, is_causal)
        self.p.q_full_len = self.p.k_full_len = seq_len
        self.v_d = v_d
        self.acc_dtype = torch.float64 if dtype_code == _capi.FA_F64 else torch.float32
        self._ws = None
        self.peer_copies = True     # shards move as peer copies on the copy engines (csrc/fa_ring.cu)

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    # ---- batched schedule (causal rings): problems are derived from the tensors' own shapes ----------------
    def _problem(self, rule, q, k, v, shard=False):
        key = (rule, tuple(q.shape), tuple(k.shape), tuple(v.shape), shard)
        cache = self.__dict__.setdefault("_problems", {})
        if key not in cache:
            p = _capi.make_problem(self.p.dtype, 1, rule, "none_front", tuple(q.shape), tuple(k.shape), tuple(v.shape))
            if shard:   # the call sees a key shard of a longer sequence: no per-row renormalisation / exact row sums
                p.q_full_len = p.k_full_len = self.seq_len
            cache[key] = p
        return cache[key]

    def _workspace(self, p, backward, device):
        need = _capi.lib.fa_workspace_bytes(C.byref(p), int(backward))
        if need and (self._ws is None or self._ws.numel() < need):
            self._ws = self.torch.empty(need, dtype=self.torch.uint8, device=device)
        return (self._ws.data_ptr() if need else None), need

    def stack2(self, a, b):
        return self.torch.stack([a, b]).contiguous()

    def new_out_like(self, q, v):
        """(O, l, m) buffers for queries q [..., d, c] and values v [..., v_d, c]."""
        t = self.torch
        ldt = t.float32 if q.dtype in (t.float16, t.bfloat16) else q.dtype
        lead = tuple(q.shape[:-2])
        return (t.empty(lead + (v.shape[-2], q.shape[-1]), dtype=q.dtype, device=q.device),
                t.empty(lead + (q.shape[-1],), dtype=ldt, device=q.device),
                t.empty(lead + (q.shape[-1],), dtype=q.dtype, device=q.device))

    def new_acc_like(self, q, v):
        t = self.torch
        lead = tuple(q.shape[:-2])
        return (t.empty(lead + (v.shape[-2], q.shape[-1]), dtype=self.acc_dtype, device=q.device),
                t.empty(lead + (q.shape[-1],), dtype=self.acc_dtype, device=q.device),
                t.empty(lead + (q.shape[-1],), dtype=self.acc_dtype, device=q.device))

    def attend(self, rule, q, k, v, out):
        """One launch: `rule` ("causal" | "full", local coordinates) over all leading batch dims of q, k, v."""
        p = self._problem(rule, q, k, v)
        ws, need = self._workspace(p, False, q.device)
        o, l, m = out
        _capi.check(_capi.lib.fa_forward(C.byref(p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                         l.data_ptr(), m.data_ptr(), ws, need, self._stream()), "fa_forward")

    def merge_into(self, part, acc, first, q, k, v):
        p = self._problem("full", q, k, v)
        o, l, m = part
        oa, la, ma = acc
        _capi.check(_capi.lib.fa_partial_merge(C.byref(p), o.data_ptr(), l.data_ptr(), m.data_ptr(),
                                               oa.data_ptr(), la.data_ptr(), ma.data_ptr(), int(first),
                                               self._stream()), "fa_partial_merge")

    def finalize_into(self, acc, out, q, k, v):
        p = self._problem("full", q, k, v)
        oa, la, ma = acc
        o, l, m = out
        _capi.check(_capi.lib.fa_partial_finalize(C.byref(p), oa.data_ptr(), la.data_ptr(), ma.data_ptr(),
                                                  o.data_ptr(), l.data_ptr(), m.data_ptr(), self._stream()),
                    "fa_partial_finalize")

    def grad(self, rule, q, k, v, o, l, m, d_o, part):
        """One backward launch with the FINAL (o, l, m) of the whole sequence: block results add."""
        p = self._problem(rule, q, k, v, shard=self.seq_len != k.shape[-1])
        ws, need = self._workspace(p, True, q.device)
        dq, dk, dv = part
        _capi.check(_capi.lib.fa_backward(C.byref(p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                          l.data_ptr(), m.data_ptr(), d_o.data_ptr(), dq.data_ptr(), dk.data_ptr(),
                                          dv.data_ptr(), ws, need, self._stream()), "fa_backward")

    def new_acc(self, like_q):
        t, dev = self.torch, like_q.device
        return (t.empty(self.batch_shape + (self.v_d, self.chunk), dtype=self.acc_dtype, device=dev),
                t.empty(self.batch_shape + (self.chunk,), dtype=self.acc_dtype, device=dev),
                t.empty(self.batch_shape + (self.chunk,), dtype=self.acc_dtype, device=dev))

    def new_out(self, like_q):
        t, dev = self.torch, like_q.device
        ldt = t.float32 if like_q.dtype in (t.float16, t.bfloat16) else like_q.dtype
        return (t.empty(self.batch_shape + (self.v_d, self.chunk), dtype=like_q.dtype, device=dev),
                t.empty(self.batch_shape + (self.chunk,), dtype=ldt, device=dev),
                t.empty(self.batch_shape + (self.chunk,), dtype=like_q.dtype, device=dev))

    def attend_partial(self, q, k, v, q_base, k_base, out):
        self.p.q_index_base, self.p.k_index_base, self.p.accumulate = q_base, k_base, 0
        o, l, m = out
        need = _capi.lib.fa_workspace_bytes(C.byref(self.p), 0)
        if need and (self._ws is None or self._ws.numel() < need):
            self._ws = self.torch.empty(need, dtype=self.torch.uint8, device=q.device)
        _capi.check(_capi.lib.fa_forward(C.byref(self.p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                         l.data_ptr(), m.data_ptr(), self._ws.data_ptr() if need else None, need,
                                         self._stream()), "fa_forward")

    def merge(self, part, acc, first):
        o, l, m = part
        oa, la, ma = acc
        _capi.check(_capi.lib.fa_partial_merge(C.byref(self.p), o.data_ptr(), l.data_ptr(), m.data_ptr(),
                                               oa.data_ptr(), la.data_ptr(), ma.data_ptr(), int(first),
                                               self._stream()), "fa_partial_merge")

    def finalize(self, acc, out):
        oa, la, ma = acc
        o, l, m = out
        _capi.check(_capi.lib.fa_partial_finalize(C.byref(self.p), oa.data_ptr(), la.data_ptr(), ma.data_ptr(),
                                                  o.data_ptr(), l.data_ptr(), m.data_ptr(), self._stream()),
                    "fa_partial_finalize")

    def empty_like_kv(self, kv):
        return [self.torch.empty_like(x) for x in kv]

    # ---- backward ---------------------------------------------------------------------------
    def new_grad_acc(self, like):
        return self.torch.zeros(like.shape, dtype=self.acc_dtype, device=like.device)

    def new_grad_part(self, q, k, v):
        return (self.torch.empty_like(q), self.torch.empty_like(k), self.torch.empty_like(v))

    def grad_partial(self, q, k, v, o, l, m, d_o, q_base, k_base, part):
        self.p.q_index_base, self.p.k_index_base, self.p.accumulate = q_base, k_base, 0
        need = _capi.lib.fa_workspace_bytes(C.byref(self.p), 1)
        if need and (self._ws is None or self._ws.numel() < need):
            self._ws = self.torch.empty(need, dtype=self.torch.uint8, device=q.device)
        dq, dk, dv = part
        _capi.check(_capi.lib.fa_backward(C.byref(self.p), q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(),
                                          l.data_ptr(), m.data_ptr(), d_o.data_ptr(), dq.data_ptr(), dk.data_ptr(),
                                          dv.data_ptr(), self._ws.data_ptr() if need else None, need, self._stream()),
                    "fa_backward")

    def grad_add(self, part, acc):
        _capi.check(_capi.lib.fa_grad_accumulate(self.p.dtype, part.data_ptr(), acc.data_ptr(), part.numel(), 0,
                                                 self._stream()), "fa_grad_accumulate")

    def grad_finalize(self, acc, like):
        out = self.torch.empty_like(like)
        _capi.check(_capi.lib.fa_grad_finalize(self.p.dtype, acc.data_ptr(), out.data_ptr(), acc.numel(),
                                               self._stream()), "fa_grad_finalize")
        return out


def ring_forward(backend, layout, rank, q_chunks, kv_chunks, dist=None, group=None, rule="causal", is_causal=False):
    """q_chunks: [Q_a, Q_b] local query chunks, each [batch..., d, c] contiguous.
    kv_chunks: [K_a, K_b, V_a, V_b] local key/value chunks. Returns [(O, l, m) for the two chunks]."""
    world = layout.world
    cur = list(kv_chunks)
    nxt = backend.empty_like_kv(cur) if world > 1 else None
    acc = [backend.new_acc(q_chunks[0]), backend.new_acc(q_chunks[1])]
    part = backend.new_out(q_chunks[0])
    started = [False, False]
    for step in range(world):
        reqs = []
        if world > 1 and step + 1 < world:
            ops = []
            for t_send, t_recv in zip(cur, nxt):
                ops.append(dist.P2POp(dist.isend, t_send, (rank + 1) % world, group))
                ops.append(dist.P2POp(dist.irecv, t_recv, (rank - 1) % world, group))
            reqs = dist.batch_isend_irecv(ops)
        _, plan = step_plan(layout, rank, step, rule, is_causal)
        for qa, kb, q_base, k_base in plan:
            backend.attend_partial(q_chunks[qa], cur[kb], cur[2 + kb], q_base, k_base, part)
            backend.merge(part, acc[qa], not started[qa])
            started[qa] = True
        for r in reqs:
            r.wait()
        if world > 1 and step + 1 < world:
            cur, nxt = nxt, cur
    outs = []
    for qa in range(2):
        out = backend.new_out(q_chunks[qa])
        if not started[qa]:  # cannot happen for causal/full (the diagonal block is local), kept for local rules
            backend.attend_partial(q_chunks[qa], kv_chunks[qa], kv_chunks[2 + qa], layout.base(layout.chunks(rank)[qa]),
                                   layout.base(layout.chunks(rank)[qa]), part)
            backend.merge(part, acc[qa], True)
        backend.finalize(acc[qa], out)
        outs.append(out)
    return outs


class DistTransport:
    """Shard rotation over torch.distributed P2P (gloo in the CPU tests; NCCL send/recv when the peer-copy data plane
    is switched off with FA_RING_TRANSPORT=nccl)."""

    def __init__(self, backend, dist, group, rank, world):
        self.backend, self.dist, self.group, self.rank, self.world = backend, dist, group, rank, world
        self.nxt = self.reqs = self.acc_nxt = None

    def forward(self, step, cur):
        if self.nxt is None:
            self.nxt = self.backend.empty_like_kv(cur)
        self.reqs = _exchange(self.dist, self.group, self.rank, self.world, cur, self.nxt)

    def advance(self, step, cur, more):
        for r in self.reqs or []:
            r.wait()
        self.reqs = None
        if not more:
            return cur
        new, self.nxt = self.nxt, cur
        return new

    def hop_send(self, step, acc):
        if self.acc_nxt is None:
            self.acc_nxt = self.backend.empty_like_kv(acc)
        for r in _exchange(self.dist, self.group, self.rank, self.world, acc, self.acc_nxt):
            r.wait()
        self._arrived, self.acc_nxt = self.acc_nxt, list(acc)

    def hop_recv(self, step):
        return self._arrived


class _RawDevice:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerRing:
    """One fa_ring_t (csrc/fa_ring.cu): receive slots exported over CUDA IPC, filled by the previous rank's copy engine."""
    _cache = {}

    def __init__(self, torch, dist, group, rank, world, templates, n_slots=2):
        self.torch, self.rank, self.world, self.n_slots = torch, rank, world, n_slots
        al = lambda n: (n + 255) // 256 * 256  # noqa: E731
        self.sizes = [t.numel() * t.element_size() for t in templates]
        slot_bytes = sum(al(n) for n in self.sizes)
        blob = C.create_string_buffer(_capi.FA_RING_HANDLE_BYTES)
        self.handle = C.c_void_p()
        _capi.check(_capi.lib.fa_ring_create(rank, world, slot_bytes, n_slots, C.byref(self.handle), blob),
                    "fa_ring_create")
        mine = torch.tensor(list(blob.raw), dtype=torch.uint8, device=templates[0].device)
        blobs = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(blobs, mine, group=group)
        nb = bytes(blobs[(rank + 1) % world].cpu().tolist())
        pb = bytes(blobs[(rank - 1) % world].cpu().tolist())
        dist.barrier(group=group)          # every rank's allocation exists before anyone maps it
        _capi.check(_capi.lib.fa_ring_connect(self.handle, nb, pb), "fa_ring_connect")
        self.slots = []
        for k in range(n_slots):
            base = _capi.lib.fa_ring_slot(self.handle, k)
            views, off = [], 0
            for t, n in zip(templates, self.sizes):
                raw = torch.as_tensor(_RawDevice(base + off, n), device=t.device)
                views.append(raw.view(t.dtype).view(t.shape))
                off += al(n)
            self.slots.append(views)

    @classmethod
    def get(cls, tag, torch, dist, group, rank, world, templates):
        key = (tag, id(group), rank, world, tuple((tuple(t.shape), t.dtype) for t in templates), templates[0].device)
        if key not in cls._cache:
            cls._cache[key] = cls(torch, dist, group, rank, world, templates)
        return cls._cache[key]

    def _stream(self):
        return self.torch.cuda.current_stream().cuda_stream

    def send(self, dst_slot, tensors, forwarded_slot):
        n = len(tensors)
        src = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
        nb = (C.c_size_t * n)(*[t.numel() * t.element_size() for t in tensors])
        _capi.check(_capi.lib.fa_ring_send(self.handle, dst_slot, n, src, nb, forwarded_slot, self._stream()),
                    "fa_ring_send")

    def recv_wait(self, slot):
        _capi.check(_capi.lib.fa_ring_recv_wait(self.handle, slot, self._stream()), "fa_ring_recv_wait")

    def release(self, slot):
        _capi.check(_capi.lib.fa_ring_recv_release(self.handle, slot, self._stream()), "fa_ring_recv_release")


class PeerTransport:
    """Shard rotation on the copy engines (PeerRing): the shard of step s is pushed into slot s % 2 of the next rank
    while step s computes; arrival and slot reuse are stream-ordered flag waits."""

    def __init__(self, backend, dist, group, rank, world, kv_templates, acc_templates=None):
        t = backend.torch
        self.kv = PeerRing.get("kv", t, dist, group, rank, world, kv_templates)
        self.acc = PeerRing.get("acc", t, dist, group, rank, world, acc_templates) if acc_templates else None

    def forward(self, step, cur):
        self.kv.send(step % 2, cur, (step - 1) % 2 if step > 0 else -1)

    def advance(self, step, cur, more):
        if step > 0:
            self.kv.release((step - 1) % 2)
        if not more:
            return cur
        self.kv.recv_wait(step % 2)
        return self.kv.slots[step % 2]

    def hop_send(self, step, acc):
        self.acc.send(step % 2, acc, (step - 1) % 2 if step > 0 else -1)
        if step > 0:
            self.acc.release((step - 1) % 2)

    def hop_recv(self, step):
        self.acc.recv_wait(step % 2)
        return self.acc.slots[step % 2]


def _make_transport(backend, dist, group, rank, world, kv_templates, acc_templates=None):
    import os
    if world == 1:
        return None
    native = getattr(backend, "peer_copies", False) and os.environ.get("FA_RING_TRANSPORT", "peer") != "nccl"
    if native:
        return PeerTransport(backend, dist, group, rank, world, kv_templates, acc_templates)
    return DistTransport(backend, dist, group, rank, world)


def _exchange(dist, group, rank, world, send, recv):
    ops = []
    for t_send, t_recv in zip(send, recv):
        ops.append(dist.P2POp(dist.isend, t_send, (rank + 1) % world, group))
        ops.append(dist.P2POp(dist.irecv, t_recv, (rank - 1) % world, group))
    return dist.batch_isend_irecv(ops)


def ring_forward_causal(backend, layout, rank, q2, k2, v2, dist=None, group=None):
    """Batched causal ring (module docstring). q2, k2, v2: chunk-major local shards [2, batch..., channels, c]
    (index 0 = chunk `rank`, 1 = chunk 2G-1-rank). Returns (O, l, m) chunk-major."""
    world = layout.world
    cur = [k2, v2]
    transport = _make_transport(backend, dist, group, rank, world, cur)
    acc = backend.new_acc_like(q2, v2)
    part = backend.new_out_like(q2, v2)
    q_hh = backend.stack2(q2[1], q2[1]) if world > 1 else None
    dup = backend.empty_like_kv(cur) if world > 1 else None
    trace = getattr(backend, "trace", None)
    for step in range(world):
        if trace is not None:
            trace.mark(f"step{step}")
        more = world > 1 and step + 1 < world
        if more:
            transport.forward(step, cur)          # this step's shard travels on while it is being attended to
        if trace is not None:
            trace.mark(f"step{step}.exchange_issued")
        src = (rank - step) % world
        if step == 0:
            backend.attend("causal", q2, cur[0], cur[1], part)                    # both diagonal blocks
            backend.merge_into(part, acc, True, q2, cur[0], cur[1])
            hi = tuple(x[1] for x in part)
            backend.attend("full", q2[1], cur[0][0], cur[1][0], hi)               # Q_hi x K_lo
            backend.merge_into(hi, tuple(x[1] for x in acc), False, q2[1], cur[0][0], cur[1][0])
        elif src < rank:
            for t, x in zip(dup, cur):                                            # [K_lo(src); K_lo(src)]
                t[0].copy_(x[0])
                t[1].copy_(x[0])
            backend.attend("full", q2, dup[0], dup[1], part)
            backend.merge_into(part, acc, False, q2, dup[0], dup[1])
        else:
            backend.attend("full", q_hh, cur[0], cur[1], part)                    # Q_hi x K_lo(src), Q_hi x K_hi(src)
            acc_hi = tuple(x[1] for x in acc)
            for h in range(2):
                backend.merge_into(tuple(x[h] for x in part), acc_hi, False, q2[1], cur[0][h], cur[1][h])
        if trace is not None:
            trace.mark(f"step{step}.compute_issued")
        if world > 1:
            cur = transport.advance(step, cur, more)
    out = backend.new_out_like(q2, v2)
    backend.finalize_into(acc, out, q2, k2, v2)
    if trace is not None:
        trace.mark("end")
    return out


def ring_backward_causal(backend, layout, rank, q2, k2, v2, o2, l2, m2, do2, dist=None, group=None):
    """Gradients of ring_forward_causal with the same batched schedule: one fa_backward launch per ring step, made with
    the FINAL O, l, m. dQ accumulates locally; the dK / dV accumulators travel with their shard and come home after
    `world` hops. All arguments chunk-major; returns (dQ, dK, dV) chunk-major."""
    world = layout.world
    cur = [k2, v2]
    dq_acc = backend.new_grad_acc(q2)
    dkv_acc = [backend.new_grad_acc(x) for x in cur]          # travels with `cur`, one hop behind it
    transport = _make_transport(backend, dist, group, rank, world, cur, dkv_acc)
    part = backend.new_grad_part(q2, k2, v2)
    if world > 1:
        hh = [backend.stack2(x[1], x[1]) for x in (q2, o2, l2, m2, do2)]
        dup = backend.empty_like_kv(cur)
    for step in range(world):
        more = world > 1 and step + 1 < world
        if more:
            transport.forward(step, cur)
        src = (rank - step) % world
        # the backward launch of this step is queued BEFORE the wait for the travelling accumulators, so that their
        # transfer overlaps it
        if step == 0:
            backend.grad("causal", q2, cur[0], cur[1], o2, l2, m2, do2, part)
        elif src < rank:
            for t, x in zip(dup, cur):
                t[0].copy_(x[0])
                t[1].copy_(x[0])
            backend.grad("full", q2, dup[0], dup[1], o2, l2, m2, do2, part)
        else:
            backend.grad("full", hh[0], cur[0], cur[1], hh[1], hh[2], hh[3], hh[4], part)
        if step > 0:
            dkv_acc = transport.hop_recv(step - 1)
        if step == 0:
            backend.grad_add(part[0], dq_acc)
            backend.grad_add(part[1], dkv_acc[0])
            backend.grad_add(part[2], dkv_acc[1])
            one = tuple(x[0] for x in part)                                        # Q_hi x K_lo, full
            backend.grad("full", q2[1], cur[0][0], cur[1][0], o2[1], l2[1], m2[1], do2[1], one)
            backend.grad_add(one[0], dq_acc[1])
            backend.grad_add(one[1], dkv_acc[0][0])
            backend.grad_add(one[2], dkv_acc[1][0])
        elif src < rank:
            backend.grad_add(part[0], dq_acc)
            for h in range(2):                                                     # both halves belong to K_lo(src)
                backend.grad_add(part[1][h], dkv_acc[0][0])
                backend.grad_add(part[2][h], dkv_acc[1][0])
        else:
            for h in range(2):                                                     # both halves belong to Q_hi
                backend.grad_add(part[0][h], dq_acc[1])
            backend.grad_add(part[1], dkv_acc[0])
            backend.grad_add(part[2], dkv_acc[1])
        if world > 1:
            transport.hop_send(step, dkv_acc)     # the accumulators follow their shard (the last hop brings them home)
            cur = transport.advance(step, cur, more)
    if world > 1:
        dkv_acc = transport.hop_recv(world - 1)
    out = (backend.grad_finalize(dq_acc, q2), backend.grad_finalize(dkv_acc[0], k2),
           backend.grad_finalize(dkv_acc[1], v2))
    if world > 1 and isinstance(transport, PeerTransport):
        transport.acc.release((world - 1) % 2)    # the home-coming slot is free again once the finalize pass has read it
    return out


def ring_backward(backend, layout, rank, q_chunks, kv_chunks, o_chunks, l_chunks, m_chunks, do_chunks, dist=None,
                  group=None, rule="causal", is_causal=False):
    """Gradients of ring_forward. q/o/l/m/do_chunks: the two local query chunks (O, l, m as ring_forward
    returned them, i.e. final over the whole sequence); kv_chunks: [K_a, K_b, V_a, V_b].
    Returns ([dQ_a, dQ_b], [dK_a, dK_b, dV_a, dV_b]) for the local chunks."""
    world = layout.world
    cur = list(kv_chunks)
    nxt = backend.empty_like_kv(cur) if world > 1 else None
    dq_acc = [backend.new_grad_acc(q) for q in q_chunks]
    dkv_acc = [backend.new_grad_acc(x) for x in cur]          # travels with `cur`
    dkv_nxt = [backend.new_grad_acc(x) for x in cur] if world > 1 else None
    part = backend.new_grad_part(q_chunks[0], cur[0], cur[2])
    for step in range(world):
        reqs = []
        if world > 1 and step + 1 < world:                     # K/V shard for the next step, overlapped
            ops = []
            for t_send, t_recv in zip(cur, nxt):
                ops.append(dist.P2POp(dist.isend, t_send, (rank + 1) % world, group))
                ops.append(dist.P2POp(dist.irecv, t_recv, (rank - 1) % world, group))
            reqs = dist.batch_isend_irecv(ops)
        _, plan = step_plan(layout, rank, step, rule, is_causal)
        for qa, kb, q_base, k_base in plan:
            backend.grad_partial(q_chunks[qa], cur[kb], cur[2 + kb], o_chunks[qa], l_chunks[qa], m_chunks[qa],
                                 do_chunks[qa], q_base, k_base, part)
            backend.grad_add(part[0], dq_acc[qa])
            backend.grad_add(part[1], dkv_acc[kb])
            backend.grad_add(part[2], dkv_acc[2 + kb])
        for r in reqs:
            r.wait()
        if world > 1:
            # the accumulators follow their shard (after the last step this hop returns them to the owner)
            ops = []
            for t_send, t_recv in zip(dkv_acc, dkv_nxt):
                ops.append(dist.P2POp(dist.isend, t_send, (rank + 1) % world, group))
                ops.append(dist.P2POp(dist.irecv, t_recv, (rank - 1) % world, group))
            for r in dist.batch_isend_irecv(ops):
                r.wait()
            dkv_acc, dkv_nxt = dkv_nxt, dkv_acc
            if step + 1 < world:
                cur, nxt = nxt, cur
    d_q = [backend.grad_finalize(dq_acc[i], q_chunks[i]) for i in range(2)]
    d_kv = [backend.grad_finalize(dkv_acc[i], kv_chunks[i]) for i in range(4)]
    return d_q, d_kv


class _Template:
    """Shape / dtype / device of a tensor that travels through a PeerRing slot (no storage of its own)."""

    def __init__(self, shape, dtype, device, element_size):
        self.shape, self.dtype, self.device, self._es = tuple(shape), dtype, device, element_size

    def numel(self):
        n = 1
        for s in self.shape:
            n *= int(s)
        return n

    def element_size(self):
        return self._es


_native_arena = {}


def _native_driver(backend):
    """The native ring driver (csrc/fa_ring.cu: fa_ring_causal_forward / _backward) runs the schedule unless
    FA_RING_DRIVER=python (this module's loops, which the gloo tests pin against the oracle) or the shards are asked to
    move over NCCL (FA_RING_TRANSPORT=nccl)."""
    import os
    return (isinstance(backend, DeviceBackend) and os.environ.get("FA_RING_DRIVER", "native") == "native"
            and os.environ.get("FA_RING_TRANSPORT", "peer") != "nccl")


def _native_setup(backend, rank, world, q2, k2, v2, dist, group, backward):
    t = backend.torch
    kv = acc = None
    if world > 1:
        kv = PeerRing.get("kv", t, dist, group, rank, world, [k2, v2])
        if backward:
            es = 8 if backend.acc_dtype == t.float64 else 4
            acc = PeerRing.get("acc", t, dist, group, rank, world,
                               [_Template(k2.shape, backend.acc_dtype, k2.device, es),
                                _Template(v2.shape, backend.acc_dtype, v2.device, es)])
    batch = 1
    for n in q2.shape[1:-2]:
        batch *= int(n)
    d, v_d, c = int(q2.shape[-2]), int(v2.shape[-2]), int(q2.shape[-1])
    need = _capi.lib.fa_ring_causal_arena_bytes(backend.p.dtype, batch, d, v_d, c, world, int(backward))
    key = (q2.device, int(backward))
    arena = _native_arena.get(key)
    if arena is None or arena.numel() < need:
        arena = t.empty(max(need, 256), dtype=t.uint8, device=q2.device)
        _native_arena[key] = arena
    return kv, acc, (backend.p.dtype, batch, d, v_d, c), arena


def ring_forward_causal_native(backend, layout, rank, q2, k2, v2, dist=None, group=None):
    """ring_forward_causal as ONE C-ABI call (fa_ring_causal_forward): same arguments, same result."""
    kv, _, dims, arena = _native_setup(backend, rank, layout.world, q2, k2, v2, dist, group, False)
    o, l, m = backend.new_out_like(q2, v2)
    _capi.check(_capi.lib.fa_ring_causal_forward(kv.handle if kv else None, *dims, q2.data_ptr(), k2.data_ptr(),
                                                 v2.data_ptr(), o.data_ptr(), l.data_ptr(), m.data_ptr(),
                                                 arena.data_ptr(), arena.numel(), backend._stream()),
                "fa_ring_causal_forward")
    return o, l, m


def ring_backward_causal_native(backend, layout, rank, q2, k2, v2, o2, l2, m2, do2, dist=None, group=None):
    """ring_backward_causal as ONE C-ABI call (fa_ring_causal_backward)."""
    kv, acc, dims, arena = _native_setup(backend, rank, layout.world, q2, k2, v2, dist, group, True)
    t = backend.torch
    dq, dk, dv = t.empty_like(q2), t.empty_like(k2), t.empty_like(v2)
    _capi.check(_capi.lib.fa_ring_causal_backward(kv.handle if kv else None, acc.handle if acc else None, *dims,
                                                  q2.data_ptr(), k2.data_ptr(), v2.data_ptr(), o2.data_ptr(),
                                                  l2.data_ptr(), m2.data_ptr(), do2.data_ptr(), dq.data_ptr(),
                                                  dk.data_ptr(), dv.data_ptr(), arena.data_ptr(), arena.numel(),
                                                  backend._stream()), "fa_ring_causal_backward")
    return dq, dk, dv


def _chunk_major(x, c):
    """[..., channels, 2c] (chunk r then chunk 2G-1-r along the sequence) -> [2, ..., channels, c]."""
    import torch
    return torch.stack([x[..., :c], x[..., c:]]).contiguous()


def _shard_layout(x2):
    import torch
    return torch.cat([x2[0], x2[1]], dim=-1)


def _causal_ring_setup(Q, V, sync_mode, group):
    import torch
    import torch.distributed as dist
    if sync_mode != "none_front":
        # equal query / key lengths: the three sync modes coincide, the ring is written in plain coordinates
        if sync_mode not in _capi.SYNC_MODES:
            raise _capi.InvalidArgumentError(_capi.FA_EINVAL_SYNC_MODE, f"Unsupported sync_mode: {sync_mode}")
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    layout = ZigZag(Q.shape[-1] * world, world)
    codes = {torch.float16: _capi.FA_F16, torch.float32: _capi.FA_F32, torch.float64: _capi.FA_F64,
             torch.bfloat16: _capi.FA_BF16}
    backend = DeviceBackend(codes[Q.dtype], "causal", "none_front", 1, 0, False, Q.shape[:-2], Q.shape[-2], V.shape[-2],
                            layout.chunk, layout.seq_len)
    return dist if world > 1 else None, rank, layout, backend


def ring_causal_1d_backward(Q, K, V, O, l, m, dO, sync_mode="none_front", group=None):
    """Gradients of ring_causal_1d: all tensors are this rank's zig-zag shards (chunk r then chunk 2G-1-r);
    O, l, m as returned by ring_causal_1d(..., returning_l_m=True). Returns (dQ, dK, dV) shards."""
    dist, rank, layout, backend = _causal_ring_setup(Q, V, sync_mode, group)
    c = layout.chunk
    run = ring_backward_causal_native if _native_driver(backend) else ring_backward_causal
    d_q, d_k, d_v = run(backend, layout, rank, *(_chunk_major(x, c) for x in (Q, K, V, O, l, m, dO)), dist, group)
    return _shard_layout(d_q), _shard_layout(d_k), _shard_layout(d_v)


def ring_causal_1d(Q, K, V, sync_mode="none_front", group=None, returning_l_m=False):
    """causal_1d on a sequence sharded zig-zag over the ranks of `group` (default: world).
    Q, K, V: this rank's shard, torch CUDA tensors `batch_shape + (channel, 2*c)` holding chunk r then chunk
    2G-1-r. Returns O (and l, m) in the same sharded layout."""
    dist, rank, layout, backend = _causal_ring_setup(Q, V, sync_mode, group)
    c = layout.chunk
    run = ring_forward_causal_native if _native_driver(backend) else ring_forward_causal
    O2, l2, m2 = run(backend, layout, rank, _chunk_major(Q, c), _chunk_major(K, c), _chunk_major(V, c), dist, group)
    if not returning_l_m:
        return _shard_layout(O2)
    return _shard_layout(O2), _shard_layout(l2), _shard_layout(m2)
