// p2p.cu — point-to-point send / recv (SURVEY K5; the transport under the Compiled-Graph
// GPU channel and RDT's two-sided path).
//
// Sender-push over NVLink into the receiver's inbox, chunked through per-CTA rings:
//
//   receiver's inbox[src] = kP2PRings sub-rings x kP2PSlots chunks
//   CTA b of the send kernel and CTA b of the recv kernel own sub-ring b.
//
//   send: wait until the slot was consumed (ack flag in the SENDER's signal pad),
//         store the chunk into the peer inbox, release-store "ready = seq+1" into
//         the RECEIVER's signal pad.
//   recv: acquire-wait ready == seq+1, copy the chunk from local HBM into the
//         caller's tensor, release-store "ack = seq+1" into the sender's pad.
//
// Sequence numbers persist in rank-local device memory, so messages of any size
// interleave correctly and a send completes without the receiver having been
// launched as long as the message fits the ring (eager protocol).
//
// Two copy mechanisms share this ONE protocol (each side picks its own, per launch):
//   p2p_kernel      : 512 threads x 16-byte ld/st -- small, unaligned or ragged messages
//   p2p_bulk_kernel : one thread per CTA drives the TMA bulk-copy unit (cp.async.bulk, SASS
//                     UBLKCP): user tensor -> shared ring -> peer inbox on the sender, inbox ->
//                     shared ring -> user tensor on the receiver.  A CTA keeps 192 KiB in flight,
//                     so <= 16 CTAs fill the link where the ld/st kernel needed 64; a second
//                     thread publishes the ready / ack flags so the copy thread never waits for a
//                     system-scope fence.
#include <type_traits>

#include "bulk_copy.cuh"
#include "kernel_utils.cuh"
#include "pipe.h"

namespace b200 {

struct P2PArgs {
  char *buf;
  size_t nbytes;
  size_t chunk;  // bytes per chunk of THIS message (<= slot size), same on both sides
  int peer;
};

// Chunk size is a pure function of the message size, so sender and receiver agree: big messages
// use whole ring slots; mid-size ones are cut into kP2PRings pieces so that every CTA (one per
// ring) carries one chunk and the message moves in parallel instead of through one CTA.
inline size_t p2p_chunk_bytes(size_t nbytes, size_t slot_bytes) {
  size_t c = (nbytes + kP2PRings - 1) / kP2PRings;
  c = (c + 4095) & ~size_t(4095);
  if (c < (size_t(16) << 10)) c = size_t(16) << 10;
  return c < slot_bytes ? c : slot_bytes;
}

__device__ __forceinline__ bool cta_wait_flag(const DevComm &c, const uint32_t *flag, uint32_t target) {
  __shared__ int ok;
  if (threadIdx.x == 0) ok = wait_flag_ge(c, flag, target) ? 1 : 0;
  __syncthreads();
  return ok != 0;
}

template <bool SEND>
__global__ void __launch_bounds__(kThreads, 1) p2p_kernel(DevComm c, P2PArgs a) {
  const int me = c.rank, peer = a.peer;
  const int b = blockIdx.x, G = gridDim.x;
  const size_t ring_bytes = c.inbox_bytes / kP2PRings;
  const size_t slot_bytes = ring_bytes / kP2PSlots;
  const size_t chunk = a.chunk;
  const size_t nchunks = (a.nbytes + chunk - 1) / chunk;
  const bool al = is_aligned16(a.buf);

  uint32_t *seq_word = SEND ? &c.st->send_seq[peer][b] : &c.st->recv_seq[peer][b];
  uint32_t seq = *seq_word;

  // sender: data lands in the peer's inbox[me]; receiver: reads its own inbox[peer]
  char *ring = (SEND ? c.inbox[peer] + size_t(me) * c.inbox_bytes : c.inbox[me] + size_t(peer) * c.inbox_bytes) +
               size_t(b) * ring_bytes;
  // ready flags live in the receiver's pad, ack flags in the sender's pad
  uint32_t *ready = (SEND ? c.sig[peer] + kSigP2PReady + (size_t(me) * kP2PRings + b) * kP2PSlots
                          : c.sig[me] + kSigP2PReady + (size_t(peer) * kP2PRings + b) * kP2PSlots);
  uint32_t *ack = (SEND ? c.sig[me] + kSigP2PAck + size_t(peer) * kP2PRings + b
                        : c.sig[peer] + kSigP2PAck + size_t(me) * kP2PRings + b);

  for (size_t j = b; j < nchunks; j += G) {
    const size_t lo = j * chunk;
    const size_t len = (a.nbytes - lo) < chunk ? (a.nbytes - lo) : chunk;
    const Units un = make_units(len);
    const size_t U = un.total();
    const uint32_t slot = seq % kP2PSlots;
    char *slot_ptr = ring + size_t(slot) * slot_bytes;
    char *user = a.buf + lo;
    if (SEND) {
      // slot free once the receiver consumed chunk (seq - kP2PSlots)
      if (!cta_wait_flag(c, ack, seq + 1u - kP2PSlots)) break;
      // 8 x 16 B per thread in flight (one CTA sustains ~20 GB/s this way; large aligned messages
      // take p2p_bulk_kernel instead)
      for (size_t u0 = threadIdx.x; u0 < U; u0 += size_t(kThreads) * 8) {
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const size_t u = u0 + size_t(k) * kThreads;
          if (u < U) v[k] = load_user_unit(user, u, un, al);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const size_t u = u0 + size_t(k) * kThreads;
          if (u < U) st_vec(slot_ptr + (u << 4), v[k]);
        }
      }
      __syncthreads();
      if (threadIdx.x == 0) st_release_sys(ready + slot, seq + 1u);
    } else {
      if (!cta_wait_flag(c, ready + slot, seq + 1u)) break;
      for (size_t u0 = threadIdx.x; u0 < U; u0 += size_t(kThreads) * 8) {
        uint4 v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const size_t u = u0 + size_t(k) * kThreads;
          if (u < U) v[k] = ld_peer(slot_ptr + (u << 4));
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const size_t u = u0 + size_t(k) * kThreads;
          if (u < U) store_user_unit(user, u, un, al, v[k]);
        }
      }
      __syncthreads();
      if (threadIdx.x == 0) st_release_sys(ack, seq + 1u);
    }
    ++seq;
  }
  __syncthreads();
  if (threadIdx.x == 0) *seq_word = seq;
}

// ---------------------------------------------------------------------------
// bulk-copy variant: same rings, same flags, same sequence numbers
// ---------------------------------------------------------------------------
template <bool SEND>
__global__ void __launch_bounds__(kThreads, 1) p2p_bulk_kernel(DevComm c, P2PArgs a) {
  extern __shared__ __align__(128) char dyn_smem[];
  __shared__ volatile uint32_t mailbox;  // chunks of this CTA whose bytes have all been moved
  __shared__ volatile int stop;
  const int me = c.rank, peer = a.peer;
  const int b = blockIdx.x, G = gridDim.x;
  const size_t ring_bytes = c.inbox_bytes / kP2PRings;
  const size_t slot_bytes = ring_bytes / kP2PSlots;
  const size_t chunk = a.chunk;
  const size_t nchunks = (a.nbytes + chunk - 1) / chunk;
  const size_t nq = nchunks > size_t(b) ? (nchunks - 1 - size_t(b)) / size_t(G) + 1 : 0;  // chunks of this CTA

  uint32_t *seq_word = SEND ? &c.st->send_seq[peer][b] : &c.st->recv_seq[peer][b];
  const uint32_t seq0 = *seq_word;
  char *ring = (SEND ? c.inbox[peer] + size_t(me) * c.inbox_bytes : c.inbox[me] + size_t(peer) * c.inbox_bytes) +
               size_t(b) * ring_bytes;
  uint32_t *ready = (SEND ? c.sig[peer] + kSigP2PReady + (size_t(me) * kP2PRings + b) * kP2PSlots
                          : c.sig[me] + kSigP2PReady + (size_t(peer) * kP2PRings + b) * kP2PSlots);
  uint32_t *ack = (SEND ? c.sig[me] + kSigP2PAck + size_t(peer) * kP2PRings + b
                        : c.sig[peer] + kSigP2PAck + size_t(me) * kP2PRings + b);
  if (threadIdx.x == 0) {
    mailbox = 0;
    stop = 0;
  }
  const BulkRing br = bulk_ring_init(dyn_smem);  // contains the __syncthreads

  const uint32_t nq32 = uint32_t(nq);
  if (threadIdx.x == 0 && nq > 0) {
    // ---- copy thread: one segment per chunk ---------------------------------------------------
    auto seg = [&](uint32_t q) {
      const size_t lo = (size_t(b) + size_t(q) * size_t(G)) * chunk;
      const uint32_t len = uint32_t((a.nbytes - lo) < chunk ? (a.nbytes - lo) : chunk);
      char *slot = ring + size_t((seq0 + q) % kP2PSlots) * slot_bytes;
      return SEND ? BulkSeg{a.buf + lo, slot, len} : BulkSeg{slot, a.buf + lo, len};
    };
    auto gate = [&](uint32_t q, bool block) {
      const uint32_t seq = seq0 + q;
      // sender: the slot was consumed (ack in MY pad); receiver: the chunk landed (ready in MY pad)
      const uint32_t *flag = SEND ? ack : ready + seq % kP2PSlots;
      const uint32_t target = SEND ? seq + 1u - kP2PSlots : seq + 1u;
      if (block) {
        if (!wait_flag_ge(c, flag, target)) return -1;
      } else if (int32_t(ld_acquire_sys(flag) - target) < 0) {
        return 0;
      }
      if (!SEND) fence_proxy_async();  // the peer's stores before our bulk reads
      return 1;
    };
    auto done = [&](uint32_t q) {
      __threadfence_block();
      mailbox = q + 1;
    };
    // the sender's stores cross NVLink, the receiver's stay in local HBM
    const bool ok = SEND ? bulk_copy_segments<BulkRemote>(br, nq32, seg, gate, done)
                         : bulk_copy_segments<BulkLocal>(br, nq32, seg, gate, done);
    if (!ok) stop = 1;
  } else if (threadIdx.x == 32 && nq > 0) {
    // ---- flag thread: publishes "ready" (sender) / "ack" (receiver) for completed chunks ------
    uint32_t published = 0;
    while (published < nq) {
      const uint32_t avail = mailbox;
      if (avail == published) {
        if (stop) break;
        __nanosleep(64);
        continue;
      }
      __threadfence_block();
      fence_proxy_async();
      __threadfence_system();
      for (; published < avail; ++published) {
        const uint32_t seq = seq0 + published;
        if (SEND) st_relaxed_sys(ready + seq % kP2PSlots, seq + 1u);
        else st_relaxed_sys(ack, seq + 1u);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *seq_word = seq0 + uint32_t(stop ? mailbox : nq);
}

// ---------------------------------------------------------------------------
// one-sided get: the receiver pulls [src_off, src_off + nbytes) of a PEER's symmetric heap into a
// local tensor.  No kernel runs on the owner of the data (RDT's one-sided contract,
// experimental/rdt/cuda_ipc_transport.py:57-186); ordering against the owner's writes is the
// caller's event.  Aligned transfers use bulk loads over NVLink + bulk stores (segment engine).
// ---------------------------------------------------------------------------
struct GetArgs {
  const char *src;  // peer mapping of the owner's heap + offset
  char *dst;
  size_t nbytes;
  size_t seg_bytes;
};

__global__ void __launch_bounds__(kThreads, 1) get_bulk_kernel(GetArgs a) {
  extern __shared__ __align__(128) char dyn_smem[];
  const BulkRing br = bulk_ring_init(dyn_smem);
  if (threadIdx.x != 0) return;
  const size_t nseg = (a.nbytes + a.seg_bytes - 1) / a.seg_bytes;
  const uint32_t b = blockIdx.x, G = gridDim.x;
  const uint32_t mine = nseg > b ? uint32_t((nseg - 1 - b) / G + 1) : 0;
  bulk_copy_segments<BulkPull>(
      br, mine,
      [&](uint32_t i) {
        const size_t lo = (size_t(b) + size_t(i) * G) * a.seg_bytes;
        const uint32_t len = uint32_t((a.nbytes - lo) < a.seg_bytes ? (a.nbytes - lo) : a.seg_bytes);
        return BulkSeg{a.src + lo, a.dst + lo, len};
      },
      [&](uint32_t, bool) { return 1; }, [&](uint32_t) {});
}

__global__ void __launch_bounds__(kThreads) get_ldst_kernel(GetArgs a) {
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const bool sal = is_aligned16(a.src), dal = is_aligned16(a.dst);
  for (size_t u = size_t(blockIdx.x) * kThreads + threadIdx.x; u < U; u += size_t(gridDim.x) * kThreads) {
    uint4 v;
    if (sal && u < un.full) v = ld_peer(a.src + (u << 4));
    else v = load_user_unit(a.src, u, un, false);
    store_user_unit(a.dst, u, un, dal, v);
  }
}

static int p2p_common(b200_comm *c, void *buf, size_t nbytes, int peer, cudaStream_t stream, bool send) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (peer < 0 || peer >= c->world) {
    set_error("peer rank %d out of range for world size %d", peer, c->world);
    return B200_ERR_INVALID;
  }
  if (peer == c->rank) {
    set_error("peer rank %d is this rank", peer);
    return B200_ERR_INVALID;
  }
  if (nbytes == 0) return B200_OK;
  if (!buf) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t chunk = p2p_chunk_bytes(nbytes, c->inbox_bytes / kP2PRings / kP2PSlots);
  const size_t nchunks = (nbytes + chunk - 1) / chunk;
  // Grid is a pure function of the message size so both sides pair CTA b with CTA b.
  int g = int(nchunks < size_t(kP2PRings) ? nchunks : size_t(kP2PRings));
  P2PArgs a{static_cast<char *>(buf), nbytes, chunk, peer};
  // The protocol (rings, slots, chunking) is a function of the message size alone; HOW this side
  // moves its bytes is a local choice: the bulk-copy unit when the tensor is 16-byte aligned, a
  // whole number of 16-byte units and the chunks are big enough to be worth a TMA pipeline.
  const long long pb = c->params[B200_PARAM_P2P_BULK_MIN_CHUNK];
  const size_t bulk_min_chunk = pb >= 0 ? size_t(pb) : (size_t(32) << 10);
  const bool bulk = is_aligned16(buf) && (nbytes & 15) == 0 && chunk >= bulk_min_chunk && pb != 0;
  if (bulk) {
    auto k = send ? p2p_bulk_kernel<true> : p2p_bulk_kernel<false>;
    if (int rc2 = set_dyn_smem(c->device, reinterpret_cast<const void *>(k))) return rc2;
    k<<<g, kThreads, kBulkSmemBytes, stream>>>(c->dev(), a);
  } else if (send) {
    p2p_kernel<true><<<g, kThreads, 0, stream>>>(c->dev(), a);
  } else {
    p2p_kernel<false><<<g, kThreads, 0, stream>>>(c->dev(), a);
  }
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

const void *p2p_module_kernel() { return reinterpret_cast<const void *>(get_ldst_kernel); }

}  // namespace b200

using namespace b200;

extern "C" int b200_send(b200_comm_t c, const void *buf, size_t nbytes, int peer, void *stream) {
  return p2p_common(c, const_cast<void *>(buf), nbytes, peer, static_cast<cudaStream_t>(stream), true);
}

extern "C" int b200_recv(b200_comm_t c, void *buf, size_t nbytes, int peer, void *stream) {
  return p2p_common(c, buf, nbytes, peer, static_cast<cudaStream_t>(stream), false);
}

extern "C" int b200_symm_base(b200_comm_t c, void **base, size_t *bytes) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (base) *base = reinterpret_cast<char *>(c->data.va[c->rank]) + 2 * c->staging_bytes;
  if (bytes) *bytes = c->heap_bytes;
  return B200_OK;
}

extern "C" int b200_get(b200_comm_t c, void *dst, int src_rank, size_t src_heap_offset, size_t nbytes, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (src_rank < 0 || src_rank >= c->world) {
    set_error("source rank %d out of range for world size %d", src_rank, c->world);
    return B200_ERR_INVALID;
  }
  if (src_heap_offset + nbytes > c->heap_bytes) {
    set_error("[%zu, %zu) is outside the %zu-byte symmetric heap", src_heap_offset, src_heap_offset + nbytes,
              c->heap_bytes);
    return B200_ERR_INVALID;
  }
  if (nbytes == 0) return B200_OK;
  if (!dst) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  GetArgs a{reinterpret_cast<const char *>(c->data.va[src_rank]) + 2 * c->staging_bytes + src_heap_offset,
            static_cast<char *>(dst), nbytes, size_t(256) << 10};
  if (is_aligned16(a.src) && is_aligned16(a.dst) && (nbytes & 15) == 0 && nbytes >= (size_t(256) << 10)) {
    const size_t nseg = (nbytes + a.seg_bytes - 1) / a.seg_bytes;
    const int g = int(nseg < 16 ? nseg : 16);
    if (int rc2 = set_dyn_smem(c->device, reinterpret_cast<const void *>(get_bulk_kernel))) return rc2;
    get_bulk_kernel<<<g, kThreads, kBulkSmemBytes, stream>>>(a);
  } else {
    const size_t U = make_units(nbytes).total();
    const int g = int((U + kThreads - 1) / kThreads < 32 ? (U + kThreads - 1) / kThreads : 32);
    get_ldst_kernel<<<g, kThreads, 0, stream>>>(a);
  }
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}
