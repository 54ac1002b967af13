// fa_ring.cu — the data plane of the K/V ring (BASELINE.json configs[4]) on the copy engines.
//
// New functionality (the reference is single-GPU). Round 1 rotated the shards with NCCL send/recv from Python; at 8
// GPUs the per-step trace (profiles/r2_ring.md) showed every step waiting ~1.3 ms for a 134 MB transfer behind 1.05 ms
// of attention: the NCCL kernels compete for SMs with attention CTAs that fill every SM (213 KB of shared memory
// each). Here one rank's shard goes to the next rank as plain `cudaMemcpyAsync` peer copies on a dedicated stream —
// copy engines over NVLink 5 / NVSwitch, no SM involved — into receive slots the neighbour exported with CUDA IPC:
//
//   fa_ring_create   one cudaMalloc per rank: n_slots receive slots + flag words; an IPC handle blob to hand to the
//                    neighbours (the caller moves the blobs with whatever it has: torch.distributed, MPI, a file)
//   fa_ring_connect  opens the next rank's blob (data + `ready` flags are written there) and the previous rank's (its
//                    `free` flags are written there)
//   fa_ring_send     copy stream: wait for the caller's stream (event), for the source slot's data when a received
//                    shard is being forwarded, and for the destination slot to be free; copy; raise `ready` at the receiver
//   fa_ring_recv_wait     the given stream waits (cuStreamWaitValue32, no kernel, no host sync) until the slot is filled
//   fa_ring_recv_release  once the stream's work so far and the forwarding copy are done, raise `free` at the sender
//
// Flags are 32-bit fill / drain counters per slot; a flag is raised by a 4-byte peer copy from a local table of
// integers (so signalling also stays on the copy engine and is ordered behind the payload in the same stream).
// Every rank makes the same sequence of calls, so the expected counter values are known on both sides without a
// handshake. Nothing here launches a kernel.
#include <cuda.h>
#include <cuda_runtime.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/fa_b200.h"

namespace {

constexpr int kMaxSlots = 8;
constexpr int kTable = 1 << 16;   // fill counts wrap far beyond any run; the table is replenished modulo its size

struct Blob {             // what fa_ring_create hands out (FA_RING_HANDLE_BYTES)
  cudaIpcMemHandle_t mem;
  uint64_t slot_bytes;
  int32_t n_slots, rank;
};
static_assert(sizeof(Blob) <= FA_RING_HANDLE_BYTES, "handle blob larger than the public constant");

typedef CUresult (*WaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);

}  // namespace

struct fa_ring {
  int rank = 0, world = 1, n_slots = 0;
  size_t slot_bytes = 0, flags_off = 0, total = 0;
  char* local = nullptr;        // [slots][ready flags][free flags][table]
  char* next = nullptr;         // peer mapping of the next rank's allocation (data + ready flags)
  char* prev = nullptr;         // peer mapping of the previous rank's allocation (free flags)
  cudaStream_t copy = nullptr;
  std::vector<cudaEvent_t> events;
  size_t ev_next = 0;
  uint32_t sent[kMaxSlots] = {}, expected[kMaxSlots] = {}, released[kMaxSlots] = {};
  WaitValue32Fn wait32 = nullptr;
  // layout helpers
  uint32_t* ready(char* base, int s) const { return reinterpret_cast<uint32_t*>(base + flags_off) + s; }
  uint32_t* freed(char* base, int s) const { return reinterpret_cast<uint32_t*>(base + flags_off) + kMaxSlots + s; }
  const uint32_t* table(uint32_t v) const {
    return reinterpret_cast<const uint32_t*>(local + flags_off + 2 * kMaxSlots * 4) + (v % kTable);
  }
  cudaEvent_t event() {
    if (events.size() < 64) {
      cudaEvent_t e = nullptr;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
      events.push_back(e);
      return e;
    }
    return events[ev_next++ % events.size()];
  }
};

namespace {
int cu_fail() { return FA_ECUDA; }
#define RING_CU(x)                         \
  do {                                     \
    if ((x) != cudaSuccess) return cu_fail(); \
  } while (0)
}  // namespace

extern "C" {

int fa_ring_create(int32_t rank, int32_t world, size_t slot_bytes, int32_t n_slots, fa_ring_t** out, void* handle_blob) {
  if (!out || !handle_blob) return FA_EINVAL_NULL;
  if (world < 1 || rank < 0 || rank >= world || n_slots < 1 || n_slots > kMaxSlots || slot_bytes == 0)
    return FA_EINVAL_SHAPE;
  fa_ring* r = new fa_ring();
  r->rank = rank;
  r->world = world;
  r->n_slots = n_slots;
  r->slot_bytes = (slot_bytes + 255) & ~size_t(255);
  r->flags_off = r->slot_bytes * n_slots;
  r->total = r->flags_off + 2 * kMaxSlots * 4 + size_t(kTable) * 4;
  void* f = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &f, cudaEnableDefault, &q) != cudaSuccess || !f) {
    delete r;
    return FA_ENODEVICE;
  }
  r->wait32 = reinterpret_cast<WaitValue32Fn>(f);
  if (cudaMalloc(&r->local, r->total) != cudaSuccess) {
    delete r;
    return cu_fail();
  }
  std::vector<uint32_t> init((2 * kMaxSlots) + kTable, 0u);
  for (int i = 0; i < kTable; ++i) init[2 * kMaxSlots + i] = uint32_t(i);
  Blob b{};
  if (cudaMemcpy(r->local + r->flags_off, init.data(), init.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaStreamCreateWithFlags(&r->copy, cudaStreamNonBlocking) != cudaSuccess ||
      cudaIpcGetMemHandle(&b.mem, r->local) != cudaSuccess) {
    fa_ring_destroy(r);
    return cu_fail();
  }
  b.slot_bytes = r->slot_bytes;
  b.n_slots = n_slots;
  b.rank = rank;
  memset(handle_blob, 0, FA_RING_HANDLE_BYTES);
  memcpy(handle_blob, &b, sizeof(b));
  *out = r;
  return FA_OK;
}

int fa_ring_connect(fa_ring_t* r, const void* next_blob, const void* prev_blob) {
  if (!r) return FA_EINVAL_NULL;
  if (r->world == 1) return FA_OK;
  if (!next_blob || !prev_blob) return FA_EINVAL_NULL;
  Blob nb, pb;
  memcpy(&nb, next_blob, sizeof(nb));
  memcpy(&pb, prev_blob, sizeof(pb));
  if (nb.slot_bytes != r->slot_bytes || nb.n_slots != r->n_slots || pb.slot_bytes != r->slot_bytes ||
      pb.n_slots != r->n_slots || nb.rank != (r->rank + 1) % r->world || pb.rank != (r->rank + r->world - 1) % r->world)
    return FA_EINVAL_SHAPE;
  RING_CU(cudaIpcOpenMemHandle(reinterpret_cast<void**>(&r->next), nb.mem, cudaIpcMemLazyEnablePeerAccess));
  if (r->world == 2) {
    r->prev = r->next;   // the same neighbour on both sides: one mapping
  } else {
    RING_CU(cudaIpcOpenMemHandle(reinterpret_cast<void**>(&r->prev), pb.mem, cudaIpcMemLazyEnablePeerAccess));
  }
  return FA_OK;
}

void* fa_ring_slot(fa_ring_t* r, int32_t slot) {
  if (!r || slot < 0 || slot >= r->n_slots) return nullptr;
  return r->local + size_t(slot) * r->slot_bytes;
}

int fa_ring_send(fa_ring_t* r, int32_t dst_slot, int32_t n_parts, const void* const* src, const size_t* bytes,
                 int32_t forwarded_slot, void* after_stream) {
  if (!r || !src || !bytes) return FA_EINVAL_NULL;
  if (r->world == 1) return FA_EINVAL_SHAPE;
  if (dst_slot < 0 || dst_slot >= r->n_slots || forwarded_slot >= r->n_slots || n_parts < 1) return FA_EINVAL_SHAPE;
  size_t total = 0;
  for (int i = 0; i < n_parts; ++i) total += (bytes[i] + 255) & ~size_t(255);
  if (total > r->slot_bytes) return FA_EINVAL_WORKSPACE;
  // the payload is final once the caller's stream reaches this point ...
  cudaEvent_t e = r->event();
  if (!e) return cu_fail();
  RING_CU(cudaEventRecord(e, static_cast<cudaStream_t>(after_stream)));
  RING_CU(cudaStreamWaitEvent(r->copy, e, 0));
  // ... and, when it sits in one of our receive slots, once that slot has been filled
  if (forwarded_slot >= 0 &&
      r->wait32(r->copy, reinterpret_cast<CUdeviceptr>(r->ready(r->local, forwarded_slot)), r->expected[forwarded_slot],
                CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
    return cu_fail();
  // the receiver has drained what we put into this slot before
  if (r->sent[dst_slot] > 0 &&
      r->wait32(r->copy, reinterpret_cast<CUdeviceptr>(r->freed(r->local, dst_slot)), r->sent[dst_slot],
                CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
    return cu_fail();
  char* dst = r->next + size_t(dst_slot) * r->slot_bytes;
  for (int i = 0; i < n_parts; ++i) {
    RING_CU(cudaMemcpyAsync(dst, src[i], bytes[i], cudaMemcpyDeviceToDevice, r->copy));
    dst += (bytes[i] + 255) & ~size_t(255);
  }
  r->sent[dst_slot] += 1;
  RING_CU(cudaMemcpyAsync(r->ready(r->next, dst_slot), r->table(r->sent[dst_slot]), 4, cudaMemcpyDeviceToDevice, r->copy));
  return FA_OK;
}

int fa_ring_recv_wait(fa_ring_t* r, int32_t slot, void* stream) {
  if (!r) return FA_EINVAL_NULL;
  if (slot < 0 || slot >= r->n_slots || r->world == 1) return FA_EINVAL_SHAPE;
  r->expected[slot] += 1;
  if (r->wait32(static_cast<CUstream>(stream), reinterpret_cast<CUdeviceptr>(r->ready(r->local, slot)), r->expected[slot],
                CU_STREAM_WAIT_VALUE_GEQ) != CUDA_SUCCESS)
    return cu_fail();
  return FA_OK;
}

int fa_ring_recv_release(fa_ring_t* r, int32_t slot, void* stream) {
  if (!r) return FA_EINVAL_NULL;
  if (slot < 0 || slot >= r->n_slots || r->world == 1) return FA_EINVAL_SHAPE;
  cudaEvent_t e = r->event();
  if (!e) return cu_fail();
  RING_CU(cudaEventRecord(e, static_cast<cudaStream_t>(stream)));
  RING_CU(cudaStreamWaitEvent(r->copy, e, 0));      // the copy stream also holds the forwarding copy of this slot
  r->released[slot] += 1;
  RING_CU(cudaMemcpyAsync(r->freed(r->prev, slot), r->table(r->released[slot]), 4, cudaMemcpyDeviceToDevice, r->copy));
  return FA_OK;
}

int fa_ring_destroy(fa_ring_t* r) {
  if (!r) return FA_OK;
  if (r->copy) cudaStreamSynchronize(r->copy);
  if (r->next) cudaIpcCloseMemHandle(r->next);
  if (r->prev && r->prev != r->next) cudaIpcCloseMemHandle(r->prev);
  for (auto e : r->events) cudaEventDestroy(e);
  if (r->copy) cudaStreamDestroy(r->copy);
  if (r->local) cudaFree(r->local);
  delete r;
  return FA_OK;
}


}  // extern "C"

// =====================================================================================================================
// The ring driver: causal_1d over one sequence sharded zig-zag over the ring's ranks (rank r holds chunks r and
// 2G-1-r of 2G), forward and backward, as a sequence of C-ABI calls on one stream - the batched schedule that
// ring.py's ring_forward_causal / ring_backward_causal run from Python (and that tests/test_ring_gloo.py pins against
// the oracle with a CPU backend), here in native code: one fa_forward / fa_backward launch per ring step over
// chunk-major operands [2, batch, channels, c], partial results folded with fa_partial_merge / fa_grad_accumulate, the
// K/V shards (and, in the backward, the fp32 dK / dV accumulators one hop behind them) moving on the copy engines.
// =====================================================================================================================
namespace {

size_t al256(size_t n) { return (n + 255) & ~size_t(255); }
size_t elt(int dtype) { return dtype == FA_F16 || dtype == FA_BF16 ? 2 : dtype == FA_F32 ? 4 : 8; }
size_t l_elt(int dtype) { return dtype == FA_F64 ? 8 : 4; }     // l is float for half and bf16
size_t acc_elt(int dtype) { return dtype == FA_F64 ? 8 : 4; }   // accumulators: float (double for f64)

fa_problem_t chunk_problem(int dtype, int rule, int64_t batch, int d, int v_d, int c, int64_t full_len) {
  fa_problem_t p;
  memset(&p, 0, sizeof(p));
  p.dtype = dtype;
  p.seq_dims = 1;
  p.rule = rule;
  p.window_size = 1;
  p.sync_mode = FA_SYNC_NONE_FRONT;
  p.d = d;
  p.v_d = v_d;
  p.batch = batch;
  p.q_shape[0] = p.k_shape[0] = c;
  // backward blocks see a key shard of the whole sequence: no per-row renormalisation / exact row sums there
  p.q_full_len = p.k_full_len = int32_t(full_len);
  return p;
}

struct RingArena {
  // forward
  size_t acc_o, acc_l, acc_m, part_o, part_l, part_m, q_hh, dup_k, dup_v, ws, ws_bytes;
  // backward
  size_t dq_acc, dk_acc, dv_acc, part_dq, part_dk, part_dv, o_hh, l_hh, m_hh, do_hh;
  size_t total;
};

RingArena ring_arena(int dtype, int64_t batch, int d, int v_d, int c, int world, bool backward) {
  RingArena a;
  memset(&a, 0, sizeof(a));
  size_t off = 0;
  auto take = [&off](size_t n) { size_t o = off; off += al256(n); return o; };
  const size_t es = elt(dtype), ls = l_elt(dtype), as = acc_elt(dtype);
  const size_t nq = size_t(2) * batch * d * c, nv = size_t(2) * batch * v_d * c, nr = size_t(2) * batch * c;
  if (!backward) {
    a.acc_o = take(nv * as);
    a.acc_l = take(nr * as);
    a.acc_m = take(nr * as);
    a.part_o = take(nv * es);
    a.part_l = take(nr * ls);
    a.part_m = take(nr * es);
  } else {
    a.dq_acc = take(nq * as);
    a.dk_acc = take(nq * as);
    a.dv_acc = take(nv * as);
    a.part_dq = take(nq * es);
    a.part_dk = take(nq * es);
    a.part_dv = take(nv * es);
    if (world > 1) {
      a.o_hh = take(nv * es);
      a.l_hh = take(nr * ls);
      a.m_hh = take(nr * es);
      a.do_hh = take(nv * es);
    }
  }
  if (world > 1) {
    a.q_hh = take(nq * es);
    a.dup_k = take(nq * es);
    a.dup_v = take(nv * es);
  }
  const int64_t full = int64_t(2) * c * world;
  for (int rule = FA_RULE_FULL; rule <= FA_RULE_CAUSAL; ++rule)
    for (int64_t b : {batch, 2 * batch}) {
      fa_problem_t p = chunk_problem(dtype, rule, b, d, v_d, c, backward ? full : 0);
      a.ws_bytes = std::max(a.ws_bytes, fa_workspace_bytes(&p, backward ? 1 : 0));
    }
  a.ws = take(a.ws_bytes);
  a.total = off;
  return a;
}

#define RING_OK(call)             \
  do {                            \
    int rc_ = (call);             \
    if (rc_ != FA_OK) return rc_; \
  } while (0)

int ring_args_ok(fa_ring_t* kv, int dtype, int64_t batch, int d, int v_d, int c) {
  if (dtype < FA_F16 || dtype > FA_BF16) return FA_EINVAL_DTYPE;
  if (batch < 1 || d < 1 || v_d < 1 || c < 1) return FA_EINVAL_SHAPE;
  if (kv && (kv->world < 1 || kv->n_slots < 2)) return FA_EINVAL_SHAPE;
  return FA_OK;
}

}  // namespace

extern "C" {

size_t fa_ring_causal_arena_bytes(int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk, int32_t world,
                                  int32_t backward) {
  if (dtype < FA_F16 || dtype > FA_BF16 || batch < 1 || d < 1 || v_d < 1 || chunk < 1 || world < 1) return 0;
  return ring_arena(dtype, batch, d, v_d, chunk, world, backward != 0).total;
}

size_t fa_ring_causal_slot_bytes(int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk, int32_t accumulators) {
  if (dtype < FA_F16 || dtype > FA_BF16 || batch < 1 || d < 1 || v_d < 1 || chunk < 1) return 0;
  const size_t e = accumulators ? acc_elt(dtype) : elt(dtype);
  return al256(size_t(2) * batch * d * chunk * e) + al256(size_t(2) * batch * v_d * chunk * e);
}

int fa_ring_causal_forward(fa_ring_t* kv, int32_t dtype, int64_t batch, int32_t d, int32_t v_d, int32_t chunk,
                           const void* q2, const void* k2, const void* v2, void* o2, void* l2, void* m2, void* arena,
                           size_t arena_bytes, void* stream) {
  RING_OK(ring_args_ok(kv, dtype, batch, d, v_d, chunk));
  if (!q2 || !k2 || !v2 || !o2 || !l2 || !m2 || !arena) return FA_EINVAL_NULL;
  const int world = kv ? kv->world : 1, rank = kv ? kv->rank : 0, c = chunk;
  const RingArena A = ring_arena(dtype, batch, d, v_d, c, world, false);
  if (arena_bytes < A.total || (reinterpret_cast<uintptr_t>(arena) & 255)) return FA_EINVAL_WORKSPACE;
  const size_t es = elt(dtype), ls = l_elt(dtype), as = acc_elt(dtype);
  const size_t kb = size_t(2) * batch * d * c * es, vb = size_t(2) * batch * v_d * c * es;   // one K2 / V2 shard
  if (kv && world > 1 && kv->slot_bytes < al256(kb) + al256(vb)) return FA_EINVAL_WORKSPACE;
  char* base = static_cast<char*>(arena);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char *acc_o = base + A.acc_o, *acc_l = base + A.acc_l, *acc_m = base + A.acc_m;
  char *part_o = base + A.part_o, *part_l = base + A.part_l, *part_m = base + A.part_m;
  void* ws = A.ws_bytes ? base + A.ws : nullptr;
  // element offsets of chunk 1 ("hi") inside chunk-major tensors
  const size_t hq = size_t(batch) * d * c, hv = size_t(batch) * v_d * c, hr = size_t(batch) * c;
  const char* q_hi = static_cast<const char*>(q2) + hq * es;
  const fa_problem_t causal2 = chunk_problem(dtype, FA_RULE_CAUSAL, 2 * batch, d, v_d, c, 0);
  const fa_problem_t full2 = chunk_problem(dtype, FA_RULE_FULL, 2 * batch, d, v_d, c, 0);
  const fa_problem_t full1 = chunk_problem(dtype, FA_RULE_FULL, batch, d, v_d, c, 0);
  if (world > 1) {   // [Q_hi; Q_hi]
    RING_CU(cudaMemcpyAsync(base + A.q_hh, q_hi, hq * es, cudaMemcpyDeviceToDevice, st));
    RING_CU(cudaMemcpyAsync(base + A.q_hh + hq * es, q_hi, hq * es, cudaMemcpyDeviceToDevice, st));
  }
  const char* cur_k = static_cast<const char*>(k2);
  const char* cur_v = static_cast<const char*>(v2);
  for (int step = 0; step < world; ++step) {
    const bool more = step + 1 < world;
    if (more) {   // this step's shard travels on while it is being attended to
      const void* src[2] = {cur_k, cur_v};
      const size_t nb[2] = {kb, vb};
      RING_OK(fa_ring_send(kv, step % 2, 2, src, nb, step > 0 ? (step - 1) % 2 : -1, st));
    }
    const int src_rank = ((rank - step) % world + world) % world;
    if (step == 0) {
      // both diagonal blocks, then Q_hi x K_lo
      RING_OK(fa_forward(&causal2, q2, cur_k, cur_v, part_o, part_l, part_m, ws, A.ws_bytes, st));
      RING_OK(fa_partial_merge(&causal2, part_o, part_l, part_m, acc_o, acc_l, acc_m, 1, st));
      RING_OK(fa_forward(&full1, q_hi, cur_k, cur_v, part_o + hv * es, part_l + hr * ls, part_m + hr * es, ws,
                         A.ws_bytes, st));
      RING_OK(fa_partial_merge(&full1, part_o + hv * es, part_l + hr * ls, part_m + hr * es, acc_o + hv * as,
                               acc_l + hr * as, acc_m + hr * as, 0, st));
    } else if (src_rank < rank) {
      // [K_lo(src); K_lo(src)] against both local query chunks
      char *dk = base + A.dup_k, *dv = base + A.dup_v;
      for (int h = 0; h < 2; ++h) {
        RING_CU(cudaMemcpyAsync(dk + h * hq * es, cur_k, hq * es, cudaMemcpyDeviceToDevice, st));
        RING_CU(cudaMemcpyAsync(dv + h * hv * es, cur_v, hv * es, cudaMemcpyDeviceToDevice, st));
      }
      RING_OK(fa_forward(&full2, q2, dk, dv, part_o, part_l, part_m, ws, A.ws_bytes, st));
      RING_OK(fa_partial_merge(&full2, part_o, part_l, part_m, acc_o, acc_l, acc_m, 0, st));
    } else {
      // Q_hi x K_lo(src), Q_hi x K_hi(src): both halves fold into the hi accumulators
      RING_OK(fa_forward(&full2, base + A.q_hh, cur_k, cur_v, part_o, part_l, part_m, ws, A.ws_bytes, st));
      for (int h = 0; h < 2; ++h)
        RING_OK(fa_partial_merge(&full1, part_o + h * hv * es, part_l + h * hr * ls, part_m + h * hr * es,
                                 acc_o + hv * as, acc_l + hr * as, acc_m + hr * as, 0, st));
    }
    if (world > 1) {
      if (step > 0) RING_OK(fa_ring_recv_release(kv, (step - 1) % 2, st));
      if (more) {
        RING_OK(fa_ring_recv_wait(kv, step % 2, st));
        cur_k = static_cast<const char*>(fa_ring_slot(kv, step % 2));
        cur_v = cur_k + al256(kb);
      }
    }
  }
  return fa_partial_finalize(&full2, acc_o, acc_l, acc_m, o2, l2, m2, st);
}

int fa_ring_causal_backward(fa_ring_t* kv, fa_ring_t* acc_ring, int32_t dtype, int64_t batch, int32_t d, int32_t v_d,
                            int32_t chunk, const void* q2, const void* k2, const void* v2, const void* o2,
                            const void* l2, const void* m2, const void* do2, void* dq2, void* dk2, void* dv2,
                            void* arena, size_t arena_bytes, void* stream) {
  RING_OK(ring_args_ok(kv, dtype, batch, d, v_d, chunk));
  if (!q2 || !k2 || !v2 || !o2 || !l2 || !m2 || !do2 || !dq2 || !dk2 || !dv2 || !arena) return FA_EINVAL_NULL;
  const int world = kv ? kv->world : 1, rank = kv ? kv->rank : 0, c = chunk;
  if (world > 1 && (!acc_ring || acc_ring->world != world || acc_ring->rank != rank || acc_ring->n_slots < 2))
    return FA_EINVAL_SHAPE;
  const RingArena A = ring_arena(dtype, batch, d, v_d, c, world, true);
  if (arena_bytes < A.total || (reinterpret_cast<uintptr_t>(arena) & 255)) return FA_EINVAL_WORKSPACE;
  const size_t es = elt(dtype), ls = l_elt(dtype), as = acc_elt(dtype);
  const size_t hq = size_t(batch) * d * c, hv = size_t(batch) * v_d * c, hr = size_t(batch) * c;
  const size_t kb = 2 * hq * es, vb = 2 * hv * es, kab = 2 * hq * as, vab = 2 * hv * as;
  if (world > 1 && (kv->slot_bytes < al256(kb) + al256(vb) || acc_ring->slot_bytes < al256(kab) + al256(vab)))
    return FA_EINVAL_WORKSPACE;
  char* base = static_cast<char*>(arena);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  void* ws = A.ws_bytes ? base + A.ws : nullptr;
  const int64_t full = int64_t(2) * c * world;
  const fa_problem_t causal2 = chunk_problem(dtype, FA_RULE_CAUSAL, 2 * batch, d, v_d, c, full);
  const fa_problem_t full2 = chunk_problem(dtype, FA_RULE_FULL, 2 * batch, d, v_d, c, full);
  const fa_problem_t full1 = chunk_problem(dtype, FA_RULE_FULL, batch, d, v_d, c, full);
  char *dq_acc = base + A.dq_acc, *dk_acc = base + A.dk_acc, *dv_acc = base + A.dv_acc;
  char *pdq = base + A.part_dq, *pdk = base + A.part_dk, *pdv = base + A.part_dv;
  RING_CU(cudaMemsetAsync(dq_acc, 0, 2 * hq * as, st));
  RING_CU(cudaMemsetAsync(dk_acc, 0, kab, st));
  RING_CU(cudaMemsetAsync(dv_acc, 0, vab, st));
  auto hi = [](const void* p, size_t off_bytes) { return static_cast<const char*>(p) + off_bytes; };
  if (world > 1) {   // [X_hi; X_hi] of the query-side tensors
    struct { size_t dst; const void* src; size_t half; } dup[5] = {
        {A.q_hh, hi(q2, hq * es), hq * es},  {A.o_hh, hi(o2, hv * es), hv * es}, {A.l_hh, hi(l2, hr * ls), hr * ls},
        {A.m_hh, hi(m2, hr * es), hr * es},  {A.do_hh, hi(do2, hv * es), hv * es}};
    for (auto& t : dup)
      for (int h = 0; h < 2; ++h)
        RING_CU(cudaMemcpyAsync(base + t.dst + h * t.half, t.src, t.half, cudaMemcpyDeviceToDevice, st));
  }
  auto add = [&](const void* part, void* acc, size_t n) {
    return fa_grad_accumulate(dtype, part, acc, int64_t(n), 0, st);
  };
  // dQ lands in its fp32 accumulator inside the backward launch where the fused kernel takes the shape (fp16, head_dim
  // 128): no fp16 dQ block, no fa_grad_accumulate pass for it
  const bool dq_in_kernel = fa_backward_accumulate_supported(&causal2, 2 * batch) &&
                            fa_backward_accumulate_supported(&full2, 2 * batch) &&
                            fa_backward_accumulate_supported(&full2, batch) &&
                            fa_backward_accumulate_supported(&full1, batch);
  // one block: gradients of problem p; dQ goes to dq_dst (fold = accumulator elements it spans), dK / dV to the part buffers
  auto block = [&](const fa_problem_t& p, const void* q, const void* k, const void* v, const void* o, const void* l,
                   const void* m, const void* d_o, char* dq_dst, int64_t fold) {
    if (dq_in_kernel)
      return fa_backward_accumulate(&p, q, k, v, o, l, m, d_o, dq_dst, pdk, pdv, fold, ws, A.ws_bytes, st);
    return fa_backward(&p, q, k, v, o, l, m, d_o, pdq, pdk, pdv, ws, A.ws_bytes, st);
  };
  const char* cur_k = static_cast<const char*>(k2);
  const char* cur_v = static_cast<const char*>(v2);
  for (int step = 0; step < world; ++step) {
    const bool more = step + 1 < world;
    if (more) {
      const void* src[2] = {cur_k, cur_v};
      const size_t nb[2] = {kb, vb};
      RING_OK(fa_ring_send(kv, step % 2, 2, src, nb, step > 0 ? (step - 1) % 2 : -1, st));
    }
    const int src_rank = ((rank - step) % world + world) % world;
    // this step's backward launch is queued BEFORE the wait for the travelling accumulators: their transfer overlaps it
    if (step == 0) {
      RING_OK(block(causal2, q2, cur_k, cur_v, o2, l2, m2, do2, dq_acc, 2 * batch));
    } else if (src_rank < rank) {
      char *dk = base + A.dup_k, *dv = base + A.dup_v;
      for (int h = 0; h < 2; ++h) {
        RING_CU(cudaMemcpyAsync(dk + h * hq * es, cur_k, hq * es, cudaMemcpyDeviceToDevice, st));
        RING_CU(cudaMemcpyAsync(dv + h * hv * es, cur_v, hv * es, cudaMemcpyDeviceToDevice, st));
      }
      RING_OK(block(full2, q2, dk, dv, o2, l2, m2, do2, dq_acc, 2 * batch));
    } else {
      RING_OK(block(full2, base + A.q_hh, cur_k, cur_v, base + A.o_hh, base + A.l_hh, base + A.m_hh, base + A.do_hh,
                    dq_acc + hq * as, batch));   // both halves belong to Q_hi
    }
    if (step > 0) {   // the accumulators of the shard being processed arrive one hop behind it
      RING_OK(fa_ring_recv_wait(acc_ring, (step - 1) % 2, st));
      dk_acc = static_cast<char*>(fa_ring_slot(acc_ring, (step - 1) % 2));
      dv_acc = dk_acc + al256(kab);
    }
    if (step == 0) {
      if (!dq_in_kernel) RING_OK(add(pdq, dq_acc, 2 * hq));
      RING_OK(add(pdk, dk_acc, 2 * hq));
      RING_OK(add(pdv, dv_acc, 2 * hv));
      // Q_hi x K_lo, full: results into the first halves of the part buffers
      RING_OK(block(full1, hi(q2, hq * es), cur_k, cur_v, hi(o2, hv * es), hi(l2, hr * ls), hi(m2, hr * es),
                    hi(do2, hv * es), dq_acc + hq * as, batch));
      if (!dq_in_kernel) RING_OK(add(pdq, dq_acc + hq * as, hq));
      RING_OK(add(pdk, dk_acc, hq));
      RING_OK(add(pdv, dv_acc, hv));
    } else if (src_rank < rank) {
      if (!dq_in_kernel) RING_OK(add(pdq, dq_acc, 2 * hq));
      for (int h = 0; h < 2; ++h) {   // both halves belong to K_lo(src)
        RING_OK(add(pdk + h * hq * es, dk_acc, hq));
        RING_OK(add(pdv + h * hv * es, dv_acc, hv));
      }
    } else {
      if (!dq_in_kernel)
        for (int h = 0; h < 2; ++h) RING_OK(add(pdq + h * hq * es, dq_acc + hq * as, hq));   // both belong to Q_hi
      RING_OK(add(pdk, dk_acc, 2 * hq));
      RING_OK(add(pdv, dv_acc, 2 * hv));
    }
    if (world > 1) {
      // the accumulators follow their shard (the last hop brings them home)
      const void* src[2] = {dk_acc, dv_acc};
      const size_t nb[2] = {kab, vab};
      RING_OK(fa_ring_send(acc_ring, step % 2, 2, src, nb, step > 0 ? (step - 1) % 2 : -1, st));
      if (step > 0) RING_OK(fa_ring_recv_release(acc_ring, (step - 1) % 2, st));
      if (step > 0) RING_OK(fa_ring_recv_release(kv, (step - 1) % 2, st));
      if (more) {
        RING_OK(fa_ring_recv_wait(kv, step % 2, st));
        cur_k = static_cast<const char*>(fa_ring_slot(kv, step % 2));
        cur_v = cur_k + al256(kb);
      }
    }
  }
  if (world > 1) {
    RING_OK(fa_ring_recv_wait(acc_ring, (world - 1) % 2, st));
    dk_acc = static_cast<char*>(fa_ring_slot(acc_ring, (world - 1) % 2));
    dv_acc = dk_acc + al256(kab);
  }
  RING_OK(fa_grad_finalize(dtype, dq_acc, dq2, int64_t(2 * hq), st));
  RING_OK(fa_grad_finalize(dtype, dk_acc, dk2, int64_t(2 * hq), st));
  RING_OK(fa_grad_finalize(dtype, dv_acc, dv2, int64_t(2 * hv), st));
  if (world > 1) RING_OK(fa_ring_recv_release(acc_ring, (world - 1) % 2, st));   // the home-coming slot is free again
  return FA_OK;
}

}  // extern "C"
