// allreduce_pipe.cu — chunk-pipelined all-reduce for large messages on ORDINARY tensors
// (operands that do not live in the symmetric heap).
//
// The phase-by-phase kernels in allreduce.cu run stage-in, the NVLink phase and stage-out one
// after the other on the whole grid: two full HBM passes that are never overlapped with the link
// (round-1 verdict: 0.45-0.63 of the link at 64 MiB).  Here the message is cut into chunks of
// C bytes and the CTAs of ONE launch take fixed roles that work on different chunks at the same
// time, synchronised by per-chunk flags in the signal pad (never by a grid-wide or host barrier):
//
//   allreduce_pipe_kernel (n >= 3; NVLS when the multicast mapping exists, peer ld/st otherwise)
//     copy-in  CTAs : user tensor -> own symmetric slot, TMA bulk copies      -> flag0[k][rank]
//     reduce   CTAs : wait flag0[k][*]; reduce the stripe of chunk k this rank owns
//                     (multimem.ld_reduce + multimem.st, or n peer loads + n peer stores)
//                                                                              -> flag1[k][rank]
//     copy-out CTAs : wait flag1[k][*]; own slot -> user tensor, TMA bulk copies
//
// A copy role is one thread driving the bulk-copy unit (bulk_copy.cuh), so it costs a few CTAs;
// the reduce roles are ordinary 512-thread CTAs with 16-byte accesses.
//
// Flags carry the launch epoch (launch counter * 4 + phase), which only grows, so nothing is ever
// reset; per-chunk arrival counters live in rank-local memory and are re-zeroed by the last
// arriver.  Slot rotation and its safety argument are unchanged (DESIGN.md, "slot rotation"):
// every rank's completion of a launch depends on every peer having started that launch.
#include "allreduce_core.cuh"
#include "bulk_copy.cuh"
#include "pipe.h"

#include <algorithm>
#include <utility>
#include <vector>

namespace b200 {

struct PipeArgs {
  const char *in;
  char *out;
  size_t nbytes;         // multiple of 16; in/out 16-byte aligned
  size_t staging_bytes;
  size_t chunk_bytes;    // C: multiple of copy_ctas * kBulkTile
  int copy_ctas;         // CTAs per copy role (power of two)
  uint32_t ring_chunks;  // 0: chunk k lives at slot offset k*C (message fits the slot);
                         // R > 0: chunk k lives at (k % R)*C -- the slot is a ring of R chunks
};

struct PipeGeom {
  size_t S, C;
  uint32_t K;      // chunks
  uint32_t G;      // copy CTAs per role
  uint32_t share;  // bytes of a full chunk each copy CTA moves: C / G (a multiple of kBulkTile)
  uint32_t R;      // ring length in chunks (0 = no ring)
};
__host__ __device__ __forceinline__ PipeGeom make_geom(const PipeArgs &a) {
  PipeGeom g;
  g.S = a.nbytes;
  g.C = a.chunk_bytes;
  g.K = uint32_t((g.S + g.C - 1) / g.C);
  g.G = uint32_t(a.copy_ctas);
  g.share = uint32_t(g.C / g.G);
  g.R = a.ring_chunks;
  return g;
}
__host__ __device__ __forceinline__ size_t chunk_len(const PipeGeom &g, uint32_t k) {
  const size_t lo = size_t(k) * g.C;
  return (g.S - lo) < g.C ? (g.S - lo) : g.C;
}
// Copy CTA j moves bytes [j*share, (j+1)*share) of every chunk (clipped by the message end).
__host__ __device__ __forceinline__ size_t share_off(const PipeGeom &g, uint32_t j, uint32_t k) {
  return size_t(k) * g.C + size_t(j) * g.share;
}
// Where chunk k sits in the staging slot.  With a ring the slot holds R chunks and chunk k reuses
// the place of chunk k - R, so ONE launch handles a message of any size with R*C bytes of staging:
// the copy-in of chunk k (share j) waits until the copy-out of chunk k - R (share j) is done, which
// in turn implies every rank's reducers are done with chunk k - R (they published it).
__host__ __device__ __forceinline__ size_t slot_chunk_off(const PipeGeom &g, uint32_t k) {
  return size_t(g.R ? k % g.R : k) * g.C;
}
__host__ __device__ __forceinline__ uint32_t share_len(const PipeGeom &g, uint32_t j, uint32_t k) {
  const size_t len = chunk_len(g, k), lo = size_t(j) * g.share;
  if (lo >= len) return 0;
  return uint32_t((len - lo) < size_t(g.share) ? (len - lo) : size_t(g.share));
}
// chunks in which copy CTA j has bytes: all full chunks, plus the ragged last one if it reaches j's share
__host__ __device__ __forceinline__ uint32_t chunks_of_cta(const PipeGeom &g, uint32_t j) {
  if (g.K == 0) return 0;
  return share_len(g, j, g.K - 1) ? g.K : g.K - 1;
}
// copy CTAs that own bytes of chunk k (= arrivals expected on its counter)
__host__ __device__ __forceinline__ uint32_t copy_arrivals(const PipeGeom &g, uint32_t k) {
  const size_t pieces = (chunk_len(g, k) + g.share - 1) / g.share;
  return uint32_t(pieces < size_t(g.G) ? pieces : size_t(g.G));
}

// Copy CTAs split the work between two threads: thread 0 drives the bulk-copy unit and only
// bumps a shared-memory mailbox when its last tile of a chunk has completed; thread 32 turns
// mailbox increments into chunk arrivals and flags, so the system-scope fences that publishing
// needs never stall the copy pipeline.  A copy CTA owns tiles in chunks 0 .. nchunks-1 (in order).
struct CopyMailbox {
  volatile uint32_t chunks_done;
  volatile int stop;
};
__device__ __forceinline__ void mailbox_post(CopyMailbox *mb, uint32_t chunks_done) {
  __threadfence_block();
  mb->chunks_done = chunks_done;
}

// One thread: count this CTA's arrival on a chunk; the last arriver re-zeroes the counter and
// returns true.  The caller has executed __threadfence_system() after the writes the arrival
// stands for (one fence may cover a batch of arrivals: with bulk stores to a peer in flight a
// system-scope fence costs ~4 us -- measured, profiles/r02/trace_push_v1.log), so by the time any
// CTA observes the final count every contribution has been performed system-wide, and the flag
// stores that follow the observation are issued after it.
__device__ __forceinline__ bool chunk_arrive_fenced(uint32_t *cnt, uint32_t expected) {
  const uint32_t old = atomicAdd(cnt, 1u);
  if (old + 1u == expected) {
    *cnt = 0;
    return true;
  }
  return false;
}
__device__ __forceinline__ void signal_all(const DevComm &c, size_t flag_word, uint32_t value) {
  for (int i = 0; i < c.world; ++i) {
    int p = c.rank + i;  // own pad first (local consumers), then walk the peers
    if (p >= c.world) p -= c.world;
    st_relaxed_sys(c.sig[p] + flag_word + c.rank, value);
  }
}

// Scout thread: the consumers of a chunk flag (copy-out, pull) must not pay for the flag wait in
// their issue loop -- an ld.acquire.sys poll of n flags plus fence.proxy.async measured ~2 us per
// chunk (profiles/r02/trace_pull_v1.log), more than the chunk's copy time.  A spare thread walks
// the chunks in order, does the acquiring waits and the proxy fence, and publishes its progress in
// shared memory; the consumer's gate is then one shared-memory load.
struct ChunkScout {
  volatile uint32_t ready;  // chunks [0, ready) are flagged by every rank
  volatile int stop;
};
__device__ __forceinline__ void scout_thread(const DevComm &c, size_t flag_base, uint32_t value, uint32_t nchunks,
                                             ChunkScout *sc) {
  for (uint32_t k = 0; k < nchunks; ++k) {
    const uint32_t *f = c.sig[c.rank] + flag_base + size_t(k) * kMaxRanks;
    for (int p = 0; p < c.world; ++p) {
      if (!wait_flag_ge(c, f + p, value)) {
        sc->stop = 1;
        return;
      }
    }
    fence_proxy_async();  // the flagged stores (generic proxy) before the consumer's bulk reads
    __threadfence_block();
    sc->ready = k + 1;
  }
}
__device__ __forceinline__ int scout_gate(ChunkScout *sc, uint32_t k, bool block) {
  if (sc->ready > k) return 1;
  if (!block) return 0;
  while (sc->ready <= k) {
    if (sc->stop) return -1;
  }
  return 1;
}

// Flag thread of a copy-in CTA: publish flag0 of every chunk this CTA finished.
__device__ __forceinline__ void copy_flag_thread(const DevComm &c, const PipeGeom &g, CopyMailbox *mb,
                                                 uint32_t nchunks, uint32_t value) {
  uint32_t published = 0;
  while (published < nchunks) {
    const uint32_t avail = mb->chunks_done;
    if (avail == published) {
      if (mb->stop) break;
      __nanosleep(100);
      continue;
    }
    __threadfence_block();
    trace_event(c, 9, avail);
    fence_proxy_async();
    trace_event(c, 10, avail);
    __threadfence_system();  // ONE fence for every chunk completed so far
    trace_event(c, 13, avail);
    for (; published < avail; ++published) {
      if (chunk_arrive_fenced(&c.st->pipe_cnt[0][published], copy_arrivals(g, published))) {
        signal_all(c, kSigPipe0 + size_t(published) * kMaxRanks, value);
        trace_event(c, 12, published);
      }
      trace_event(c, 11, published);
    }
  }
}

// The copy-in role shared by the pipelined kernels: CTA j of g.G copies its tiles of the caller's
// tensor into this rank's slot with the bulk-copy unit and publishes flag0[k][rank] per chunk.
__device__ __forceinline__ void role_copy_in(const DevComm &c, const PipeArgs &a, const PipeGeom &g, size_t off,
                                             uint32_t ep, char *dyn_smem, uint32_t j) {
  __shared__ CopyMailbox mb;
  if (threadIdx.x == 0) {
    mb.chunks_done = 0;
    mb.stop = 0;
  }
  const BulkRing ring = bulk_ring_init(dyn_smem);
  const uint32_t my_chunks = chunks_of_cta(g, j);
  if (threadIdx.x == 0) {
    char *slot = c.data[c.rank] + off;
    const uint32_t tag = (ep >> 2) << 10;  // launch << 10
    const bool ok = bulk_copy_segments<BulkLocal>(
        ring, my_chunks,
        [&](uint32_t k) {
          return BulkSeg{a.in + share_off(g, j, k), slot + slot_chunk_off(g, k) + size_t(j) * g.share, share_len(g, j, k)};
        },
        [&](uint32_t k, bool block) {
          if (g.R == 0 || k < g.R) return 1;
          const uint32_t *prog = &c.st->pipe_out_progress[j];
          const uint32_t need = tag + (k - g.R + 1);
          if (block) return wait_flag_ge(c, prog, need) ? 1 : -1;
          return int32_t(ld_acquire_sys(prog) - need) >= 0 ? 1 : 0;
        },
        [&](uint32_t k) { mailbox_post(&mb, k + 1); });
    if (!ok) mb.stop = 1;
  } else if (threadIdx.x == 32) {
    copy_flag_thread(c, g, &mb, my_chunks, ep + 1);
  }
}

constexpr int kItemUnroll = 4;
constexpr size_t kItemUnits = size_t(kThreads) * kItemUnroll;  // 16-byte units per reduce work item

// The reduce work of one rank: chunk k's stripe [lo, hi) (16-byte units) is cut into items of
// kItemUnits units; items are dealt round-robin, chunk-major, to the Gr reduce CTAs.  Workers and
// the arrival thread of a CTA walk the same sequence.
struct ItemIter {
  const PipeGeom &g;
  uint32_t rank, world, me, Gr;
  uint32_t k = 0;        // next chunk to look at
  size_t item_base = 0;  // global index of chunk k's first item
  // the item most recently returned by next():
  size_t lo = 0, hi = 0, it = 0;
  uint32_t nitems = 0, cur_k = 0;
  bool in_chunk = false;
  __host__ __device__ ItemIter(const PipeGeom &g_, int r, int n, uint32_t me_, uint32_t Gr_)
      : g(g_), rank(uint32_t(r)), world(uint32_t(n)), me(me_), Gr(Gr_) {}
  __host__ __device__ bool next(uint32_t &k_out) {
    if (in_chunk) {
      it += Gr;
      if (it < nitems) {
        k_out = cur_k;
        return true;
      }
      in_chunk = false;
    }
    for (; k < g.K; ++k) {
      const size_t cu = chunk_len(g, k) >> 4;
      lo = cu * size_t(rank) / size_t(world);
      hi = cu * size_t(rank + 1) / size_t(world);
      const size_t items = (hi - lo + kItemUnits - 1) / kItemUnits;
      nitems = uint32_t(items ? items : 1);  // an empty stripe still publishes
      it = (size_t(me) + size_t(Gr) - item_base % size_t(Gr)) % size_t(Gr);
      item_base += nitems;
      if (it < nitems) {
        cur_k = k_out = k;
        ++k;
        in_chunk = true;
        return true;
      }
    }
    return false;
  }
};

// ---------------------------------------------------------------------------
// n >= 3: copy-in | reduce (NVLS or peer ld/st) | copy-out
// ---------------------------------------------------------------------------
template <typename T, int OP, bool NVLS>
__global__ void __launch_bounds__(kThreads + 32, 1) allreduce_pipe_kernel(DevComm c, PipeArgs a) {
  extern __shared__ __align__(128) char dyn_smem[];
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const PipeGeom g = make_geom(a);
  const int n = c.world, r = c.rank;
  const int G = int(g.G), Gr = int(gridDim.x) - 2 * G;
  const int b = blockIdx.x;

  if (b < G) {
    role_copy_in(c, a, g, off, ep, dyn_smem, uint32_t(b));
  } else if (b < G + Gr) {
    // ---- reduce ------------------------------------------------------------------------------
    // 512 workers + one service warp (the kernel runs kThreads + 32 threads).  The workers only
    // load, reduce and store; waiting for chunk flags (scout, service lane 0) and publishing
    // arrivals behind a system-scope fence (service lane 1) happen beside them, so a worker never
    // executes a fence or an acquiring poll.
    __shared__ ChunkScout sc;
    __shared__ CopyMailbox mb;  // chunks_done counts this CTA's finished work items here
    if (threadIdx.x == 0) {
      sc.ready = 0;
      sc.stop = 0;
      mb.chunks_done = 0;
      mb.stop = 0;
    }
    __syncthreads();
    ItemIter iter(g, r, n, uint32_t(b - G), uint32_t(Gr));
    if (threadIdx.x >= kThreads) {
      if (threadIdx.x == kThreads) {
        scout_thread(c, kSigPipe0, ep + 1, g.K, &sc);
      } else if (threadIdx.x == kThreads + 1) {
        uint32_t published = 0, k = 0;
        bool have = iter.next(k);
        while (have) {
          const uint32_t avail = mb.chunks_done;
          if (avail == published) {
            if (mb.stop) break;
            __nanosleep(100);
            continue;
          }
          __threadfence_block();
          __threadfence_system();  // one fence for every item finished so far
          for (; published < avail && have; ++published) {
            if (chunk_arrive_fenced(&c.st->pipe_cnt[1][k], iter.nitems))
              signal_all(c, kSigPipe1 + size_t(k) * kMaxRanks, ep + 2);
            have = iter.next(k);
          }
        }
      }
    } else {
      uint32_t k = 0, done_items = 0;
      while (iter.next(k)) {
        // chunk k staged on every rank?
        if (sc.ready <= k) {
          bool alive = true;
          while (sc.ready <= k) {
            if (sc.stop) {
              alive = false;
              break;
            }
          }
          if (!alive) break;
        }
        const size_t cbase = off + slot_chunk_off(g, k);
        const size_t hi = iter.hi;
        const size_t u0 = iter.lo + iter.it * kItemUnits + threadIdx.x;
        if (NVLS) {
          char *mc = c.mc_data + cbase;
          uint4 v[kItemUnroll];
#pragma unroll
          for (int q = 0; q < kItemUnroll; ++q) {
            const size_t u = u0 + size_t(q) * kThreads;
            if (u < hi) v[q] = Multimem<T>::ld_reduce_sum(mc + (u << 4));
          }
#pragma unroll
          for (int q = 0; q < kItemUnroll; ++q) {
            const size_t u = u0 + size_t(q) * kThreads;
            if (u < hi) {
              if (OP == B200_AVG) {
                typename Tr::Acc acc = Tr::unpack(v[q]);
                Tr::average(acc, n);
                v[q] = Tr::pack(acc);
              }
              multimem_st(mc + (u << 4), v[q]);
            }
          }
        } else {
#pragma unroll 1
          for (int q0 = 0; q0 < kItemUnroll; q0 += 2) {
            uint4 v[2][kMaxRanks];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const size_t u = u0 + size_t(q0 + q) * kThreads;
              if (u < hi) {
#pragma unroll
                for (int p = 0; p < kMaxRanks; ++p)
                  if (p < n) v[q][p] = ld_peer(c.data[p] + cbase + (u << 4));
              }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const size_t u = u0 + size_t(q0 + q) * kThreads;
              if (u < hi) {
                typename Tr::Acc acc = Tr::unpack(v[q][0]);
#pragma unroll
                for (int p = 1; p < kMaxRanks; ++p)
                  if (p < n) Tr::template reduce<OP>(acc, Tr::unpack(v[q][p]));  // rank-ascending
                if (OP == B200_AVG) Tr::average(acc, n);
                const uint4 res = Tr::pack(acc);
#pragma unroll
                for (int i = 0; i < kMaxRanks; ++i) {
                  if (i < n) {
                    int p = r + i;
                    if (p >= n) p -= n;
                    st_vec(c.data[p] + cbase + (u << 4), res);
                  }
                }
              }
            }
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");  // workers only
        if (threadIdx.x == 0) mailbox_post(&mb, ++done_items);
      }
      if (threadIdx.x == 0 && sc.stop) mb.stop = 1;
    }
  } else {
    // ---- copy-out ------------------------------------------------------------------------
    __shared__ ChunkScout sc;
    if (threadIdx.x == 0) {
      sc.ready = 0;
      sc.stop = 0;
    }
    const BulkRing ring = bulk_ring_init(dyn_smem);
    const uint32_t j = uint32_t(b - G - Gr);
    const uint32_t my_chunks = chunks_of_cta(g, j);
    if (threadIdx.x == 0) {
      const char *slot = c.data[r] + off;
      const uint32_t tag = launch << 10;
      bulk_copy_segments<BulkLocal>(
          ring, my_chunks,
          [&](uint32_t k) {
            return BulkSeg{slot + slot_chunk_off(g, k) + size_t(j) * g.share, a.out + share_off(g, j, k), share_len(g, j, k)};
          },
          [&](uint32_t k, bool block) { return scout_gate(&sc, k, block); },
          [&](uint32_t k) {
            // chunk k has left the slot (its bulk loads landed long ago, its stores completed):
            // the copy-in CTA with the same share may reuse the ring position
            if (g.R) *reinterpret_cast<volatile uint32_t *>(&c.st->pipe_out_progress[j]) = tag + k + 1;
          });
    } else if (threadIdx.x == 32) {
      scout_thread(c, kSigPipe1, ep + 2, my_chunks, &sc);
    }
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// n == 2, pull: copy-in | pull-reduce
//
// Measured on B200 (profiles/r02/bulk_bench*.log): bulk LOADS from a peer reach 770 GB/s with 16
// CTAs and complete on an mbarrier the moment the bytes are in shared memory, while bulk STORES
// to a peer top out at 705 GB/s and are only known to be complete ~10 us later (wait_group) --
// a lag the consumer of a push design has to sit out.  So each rank stages its tensor in its OWN
// slot (local copy, cheap completion) and the PEER pulls it:
//
//   copy-in CTAs : user tensor -> own slot (bulk copies)                        -> flag0[k][rank]
//   pull CTAs    : one thread keeps kPullLookahead bulk loads of the peer's slot in flight into a
//                  shared-memory ring (plus a bulk load of the matching piece of the caller's
//                  tensor); all 512 threads wait on the tile's mbarrier and write
//                  out = rank0 (op) rank1 straight into the caller's tensor, then release the
//                  stage on an "empty" mbarrier.
// ---------------------------------------------------------------------------
constexpr int kPullLookahead = 4;  // + the tile being consumed = 5 of the 6 ring stages in flight
constexpr int kPullTile = kBulkTile / 2;  // payload bytes per tile (a stage holds both operands)

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

template <typename T, int OP>
__global__ void __launch_bounds__(kThreads + 32, 1) allreduce_pull_kernel(DevComm c, PipeArgs a) {
  extern __shared__ __align__(128) char dyn_smem[];
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const PipeGeom g = make_geom(a);
  const int r = c.rank, peer = 1 - c.rank;
  const int G = int(g.G), Gr = int(gridDim.x) - G;
  const int b = blockIdx.x;

  if (b < G) {
    role_copy_in(c, a, g, off, ep, dyn_smem, uint32_t(b));
  } else {
    __shared__ int bail;
    __shared__ ChunkScout sc;
    const uint32_t tiles_smem = smem_u32(dyn_smem);
    const uint32_t full = tiles_smem + kBulkStages * kBulkTile;  // mbarriers: tile landed
    const uint32_t empty = full + 8 * kBulkStages;               // mbarriers: tile consumed
    if (threadIdx.x == 0) {
      bail = 0;
      sc.ready = 0;
      sc.stop = 0;
      for (int s = 0; s < kBulkStages; ++s) {
        mbar_init(full + 8 * s, 1);
        mbar_init(empty + 8 * s, kThreads);
      }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // A ring stage holds BOTH operands of one tile: [peer's kPullTile bytes | own kPullTile bytes],
    // each fetched by its own bulk load (remote slot / local caller tensor) onto the same mbarrier,
    // so the 512 consumer threads never wait on a global-memory load of their own.
    const uint32_t me = uint32_t(b - G);
    const uint32_t total_tiles = uint32_t((g.S + kPullTile - 1) / kPullTile);
    const uint32_t nt = total_tiles > me ? (total_tiles - 1 - me) / uint32_t(Gr) + 1 : 0;  // tiles me, me+Gr, ...
    const uint32_t tiles_per_chunk = uint32_t(g.C / kPullTile);
    const char *peer_slot = c.data[peer] + off;
    if (threadIdx.x >= kThreads) {
      // service warp (the kernel runs kThreads + 32 threads): its first lane is the scout.  A chunk
      // is usable once BOTH ranks flagged it: the peer's slot is readable, and the local copy-in
      // CTAs are done reading the caller's tensor, so it may be overwritten in place.
      if (threadIdx.x == kThreads && nt > 0) scout_thread(c, kSigPipe0, ep + 1, g.K, &sc);
      finish_launch(c);
      return;
    }
    uint32_t next_load = 0;
    for (uint32_t it = 0; it < nt; ++it) {
      if (threadIdx.x == 0) {
        // keep the ring full: tiles it .. it + kPullLookahead
        while (next_load < nt && next_load <= it + uint32_t(kPullLookahead)) {
          const uint32_t t = me + next_load * uint32_t(Gr);
          const int st = scout_gate(&sc, t / tiles_per_chunk, next_load == it);
          if (st < 0) bail = 1;
          if (st <= 0) break;
          const uint32_t s = next_load % kBulkStages;
          if (next_load >= uint32_t(kBulkStages)) {  // stage consumed by everyone?
            const uint32_t par = (next_load / kBulkStages - 1) & 1u;
            while (!mbar_try_wait(empty + 8 * s, par)) {
            }
          }
          const size_t o = size_t(t) * kPullTile;
          const uint32_t bytes = uint32_t((g.S - o) < size_t(kPullTile) ? (g.S - o) : size_t(kPullTile));
          mbar_expect_tx(full + 8 * s, 2 * bytes);
          bulk_g2s(tiles_smem + s * kBulkTile, peer_slot + o, bytes, full + 8 * s);
          bulk_g2s(tiles_smem + s * kBulkTile + kPullTile, a.in + o, bytes, full + 8 * s);
          trace_event(c, 30, next_load);
          ++next_load;
        }
      }
      const uint32_t s = it % kBulkStages;
      const uint32_t par = (it / kBulkStages) & 1u;
      unsigned spins = 0;
      bool alive = true;
      while (!mbar_try_wait(full + 8 * s, par)) {
        if ((++spins & 0xff) == 0 && *reinterpret_cast<volatile int *>(&bail)) {
          alive = false;
          break;
        }
      }
      if (!alive) break;
      if (threadIdx.x == 0) trace_event(c, 33, it);
      const uint32_t t = me + it * uint32_t(Gr);
      const size_t o = size_t(t) * kPullTile;
      const uint32_t units = uint32_t(((g.S - o) < size_t(kPullTile) ? (g.S - o) : size_t(kPullTile)) >> 4);
      constexpr int kPerThread = kPullTile / 16 / kThreads;
      uint4 mine[kPerThread], theirs[kPerThread];
#pragma unroll
      for (int q = 0; q < kPerThread; ++q) {
        const uint32_t u = threadIdx.x + uint32_t(q) * kThreads;
        if (u < units) {
          theirs[q] = lds_v4(tiles_smem + s * kBulkTile + (u << 4));
          mine[q] = lds_v4(tiles_smem + s * kBulkTile + kPullTile + (u << 4));
        }
      }
      mbar_arrive(empty + 8 * s);  // this thread is done with the stage
#pragma unroll
      for (int q = 0; q < kPerThread; ++q) {
        const uint32_t u = threadIdx.x + uint32_t(q) * kThreads;
        if (u < units) {
          typename Tr::Acc acc = Tr::unpack(r == 0 ? mine[q] : theirs[q]);
          Tr::template reduce<OP>(acc, Tr::unpack(r == 0 ? theirs[q] : mine[q]));  // rank-ascending
          if (OP == B200_AVG) Tr::average(acc, 2);
          st_vec(a.out + o + (size_t(u) << 4), Tr::pack(acc));
        }
      }
    }
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// all-gather, pull: copy-in | pull-copy
//
//   copy-in CTAs : own tensor -> own slot (bulk copies)                         -> flag0[k][rank]
//   pull CTAs    : for every peer p and chunk k (chunk-major): bulk-load p's slot over NVLink into
//                  the shared ring, bulk-store into the caller's output tensor for p.  The rank's
//                  own tensor goes straight from the input to its output.  A scout thread per
//                  pull CTA follows the peers' chunk flags.
// NVLink carries only loads (775 GB/s measured, completion known exactly); nothing is staged twice.
// ---------------------------------------------------------------------------
struct GatherOuts {
  char *p[kMaxRanks];
};

__global__ void __launch_bounds__(kThreads, 1) allgather_pull_kernel(DevComm c, PipeArgs a, GatherOuts outs) {
  extern __shared__ __align__(128) char dyn_smem[];
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const PipeGeom g = make_geom(a);
  const int n = c.world, r = c.rank;
  const int G = int(g.G), Gp = int(gridDim.x) - G;
  const int b = blockIdx.x;
  if (b < G) {
    role_copy_in(c, a, g, off, ep, dyn_smem, uint32_t(b));
  } else {
    __shared__ volatile uint32_t ready[kMaxRanks];  // ready[p]: chunks of peer p that are staged
    __shared__ volatile int stop;
    if (threadIdx.x < kMaxRanks) ready[threadIdx.x] = 0;
    if (threadIdx.x == 0) stop = 0;
    const BulkRing ring = bulk_ring_init(dyn_smem);
    const uint32_t me = uint32_t(b - G);
    const uint32_t total = g.K * uint32_t(n);                       // segments (k, q), chunk-major
    const uint32_t mine = total > me ? (total - 1 - me) / uint32_t(Gp) + 1 : 0;
    auto decode = [&](uint32_t i, uint32_t &k, int &p) {
      const uint32_t sidx = me + i * uint32_t(Gp);
      k = sidx / uint32_t(n);
      p = r + int(sidx - k * uint32_t(n));  // q = 0 is this rank itself, then the peers in ring order
      if (p >= n) p -= n;
    };
    if (threadIdx.x == 0) {
      const bool ok = bulk_copy_segments<BulkPull>(
          ring, mine,
          [&](uint32_t i) {
            uint32_t k;
            int p;
            decode(i, k, p);
            const size_t o = size_t(k) * g.C;
            const uint32_t len = uint32_t(chunk_len(g, k));
            return BulkSeg{p == r ? a.in + o : c.data[p] + off + o, outs.p[p] + o, len};
          },
          [&](uint32_t i, bool block) {
            uint32_t k;
            int p;
            decode(i, k, p);
            if (p == r || ready[p] > k) return 1;
            if (!block) return 0;
            while (ready[p] <= k) {
              if (stop) return -1;
            }
            return 1;
          },
          [&](uint32_t) {});
      (void)ok;
    } else if (threadIdx.x == 32 && mine > 0) {
      // scout: chunk-major walk over the peers' flags (a flag is written by its rank only)
      for (uint32_t k = 0; k < g.K && !stop; ++k) {
        for (int q = 1; q < n; ++q) {
          int p = r + q;
          if (p >= n) p -= n;
          if (!wait_flag_ge(c, c.sig[r] + kSigPipe0 + size_t(k) * kMaxRanks + p, ep + 1)) {
            stop = 1;
            break;
          }
          fence_proxy_async();
          __threadfence_block();
          ready[p] = k + 1;
        }
      }
    }
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int pow2_floor(int x) {
  int p = 1;
  while (p * 2 <= x) p *= 2;
  return p;
}

// Opt the kernel into kBulkSmemBytes of dynamic shared memory, once per (device, kernel): the
// attribute call is kept out of the steady-state launch path (and out of stream capture).
int set_dyn_smem(int device, const void *fn) {
  static std::mutex mu;
  static std::vector<std::pair<int, const void *>> seen;
  std::lock_guard<std::mutex> lk(mu);
  for (auto &e : seen)
    if (e.first == device && e.second == fn) return B200_OK;
  B200_CHECK_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kBulkSmemBytes)));
  seen.emplace_back(device, fn);
  return B200_OK;
}

// Defaults measured on 2 / 4 / 8 B200s (profiles/r02/tune_n2.log, tune_n4.log, tune_n8.log):
//   2 ranks (pull)      : 1 MiB chunks, 32 copy-in + 32 pull CTAs
//   3-4 ranks (NVLS)    : 4 MiB chunks, 16 + 16 copy CTAs, 64 reduce CTAs
//   5-8 ranks (NVLS)    : 8 MiB chunks, 16 + 16 copy CTAs, 32 reduce CTAs (more CTAs on the
//                         switch reduction measured slower, as in round 1)
size_t pipe_chunk_bytes(const b200_comm *c) {
  const long long v = c->params[B200_PARAM_PIPE_CHUNK_BYTES];
  size_t C = v > 0 ? size_t(v) : (c->world == 2 ? (size_t(1) << 20) : (c->world <= 4 ? (size_t(4) << 20) : (size_t(8) << 20)));
  const size_t quantum = size_t(32) * kBulkTile;  // C / G is a whole number of tiles for any power-of-two G <= 32
  C = round_up(C, quantum);
  const size_t fit = c->staging_bytes / quantum * quantum;  // a chunk must fit the staging slot
  return C < fit ? C : fit;                                 // 0: slot too small for the pipeline
}

// chunk ring of the n >= 3 pipeline, used whenever the slot holds at least 4 chunks: one launch
// beat splitting the message into launches in every measured case (profiles/r02/ring_check.log)
static bool pipe_ring_enabled(const b200_comm *c, int variant) {
  if (variant != PIPE_NVLS && variant != PIPE_PEER) return false;  // pull kernels: the READER is a peer
  const size_t C = pipe_chunk_bytes(c);
  return C && c->staging_bytes / C >= 4;
}

size_t pipe_max_bytes(const b200_comm *c, int variant) {
  const size_t C = pipe_chunk_bytes(c);
  if (C == 0) return 0;
  size_t cap = pipe_ring_enabled(c, variant) ? ~size_t(0) : c->staging_bytes;
  const size_t by_chunks = size_t(kMaxPipeChunks) * C;
  cap = cap < by_chunks ? cap : by_chunks;
  return cap / C * C;  // whole chunks, so a split message continues on a chunk boundary
}

template <typename T, int OP>
int launch_allreduce_pipe(b200_comm *c, const char *in, char *out, size_t nbytes, int variant,
                          cudaStream_t stream) {
  PipeArgs a{in, out, nbytes, c->staging_bytes, pipe_chunk_bytes(c), 0, 0};
  if (pipe_ring_enabled(c, variant) && nbytes > c->staging_bytes / a.chunk_bytes * a.chunk_bytes)
    a.ring_chunks = uint32_t(c->staging_bytes / a.chunk_bytes);
  const long long pc = c->params[B200_PARAM_PIPE_COPY_CTAS];
  const long long pr = c->params[B200_PARAM_PIPE_RED_CTAS];
  int G = pc > 0 ? int(pc) : (variant == PIPE_PULL ? 32 : 16);
  int Gr = pr > 0 ? int(pr) : (variant == PIPE_PULL ? 32 : (c->world <= 4 ? 64 : 32));
  const int roles = variant == PIPE_PULL ? 1 : 2;
  int cap = c->forced_blocks > 0 ? c->forced_blocks : c->sm_count;
  if (roles * G + Gr > cap) {  // shared-GPU harness / small parts: shrink, keep at least one reducer
    while (G > 1 && roles * G + 1 > cap / 2) G /= 2;
    Gr = cap - roles * G;
    if (Gr < 1) {
      set_error("pipelined all-reduce needs at least %d CTAs (have %d)", roles + 1, cap);
      return B200_ERR_UNSUPPORTED;
    }
  }
  G = pow2_floor(G > 32 ? 32 : G);
  a.copy_ctas = G;
  const int grid = roles * G + Gr;
  DevComm dc = c->dev();
  int rc = B200_OK;
  if (variant == PIPE_PULL) {
    if (c->world != 2) {
      set_error("the pull all-reduce is a 2-rank kernel");
      return B200_ERR_UNSUPPORTED;
    }
    auto k = allreduce_pull_kernel<T, OP>;
    if ((rc = set_dyn_smem(c->device, reinterpret_cast<const void *>(k)))) return rc;
    k<<<grid, kThreads + 32, kBulkSmemBytes, stream>>>(dc, a);  // + one service warp (scout)
  } else if (variant == PIPE_NVLS) {
    if constexpr (Multimem<T>::kSum && (OP == B200_SUM || OP == B200_AVG)) {
      auto k = allreduce_pipe_kernel<T, OP, true>;
      if ((rc = set_dyn_smem(c->device, reinterpret_cast<const void *>(k)))) return rc;
      k<<<grid, kThreads + 32, kBulkSmemBytes, stream>>>(dc, a);  // + one service warp
    } else {
      set_error("NVLS all-reduce supports SUM/AVG on f32/f16/bf16 only");
      return B200_ERR_UNSUPPORTED;
    }
  } else {
    auto k = allreduce_pipe_kernel<T, OP, false>;
    if ((rc = set_dyn_smem(c->device, reinterpret_cast<const void *>(k)))) return rc;
    k<<<grid, kThreads + 32, kBulkSmemBytes, stream>>>(dc, a);  // + one service warp
  }
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

int launch_allreduce_pipe_dyn(b200_comm *c, const char *in, char *out, size_t nbytes, int dtype, int op,
                              int variant, cudaStream_t stream) {
  int rc = B200_OK;
  B200_DISPATCH_DTYPE(dtype, T, B200_DISPATCH_OP(op, OP, {
                        rc = launch_allreduce_pipe<T, OP>(c, in, out, nbytes, variant, stream);
                      }));
  return rc;
}

// in / outs[p] 16-byte aligned, nbytes a multiple of 16 and <= pipe_max_bytes()
int launch_allgather_pull(b200_comm *c, const char *in, char *const *outs, size_t nbytes, cudaStream_t stream) {
  PipeArgs a{in, nullptr, nbytes, c->staging_bytes, pipe_chunk_bytes(c), 0, 0};
  if (c->params[B200_PARAM_PIPE_CHUNK_BYTES] <= 0) a.chunk_bytes = round_up(size_t(1) << 20, size_t(32) * kBulkTile);
  const long long pc = c->params[B200_PARAM_PIPE_COPY_CTAS];
  const long long pr = c->params[B200_PARAM_PIPE_RED_CTAS];
  int G = pc > 0 ? int(pc) : 16;
  // pull CTAs also move the rank's own tensor (in -> out): half of all bytes at 2 ranks, 1/8 at 8
  int Gp = pr > 0 ? int(pr) : (c->world == 2 ? 64 : (c->world <= 4 ? 48 : 32));
  int cap = c->forced_blocks > 0 ? c->forced_blocks : c->sm_count;
  if (G + Gp > cap) {
    while (G > 1 && G + 1 > cap / 2) G /= 2;
    Gp = cap - G;
    if (Gp < 1) {
      set_error("pull all-gather needs at least 2 CTAs (have %d)", cap);
      return B200_ERR_UNSUPPORTED;
    }
  }
  G = pow2_floor(G > 32 ? 32 : G);
  a.copy_ctas = G;
  if (a.chunk_bytes > c->staging_bytes) a.chunk_bytes = c->staging_bytes / (size_t(32) * kBulkTile) * (size_t(32) * kBulkTile);
  GatherOuts o{};
  for (int p = 0; p < c->world; ++p) o.p[p] = outs[p];
  int rc = set_dyn_smem(c->device, reinterpret_cast<const void *>(allgather_pull_kernel));
  if (rc) return rc;
  allgather_pull_kernel<<<G + Gp, kThreads, kBulkSmemBytes, stream>>>(c->dev(), a, o);
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

// ---------------------------------------------------------------------------
// Host-side self-test of the work decomposition (the SAME inline functions the kernels use):
// every byte of the message is copied in / out by exactly one copy CTA, the arrival counts the
// flag threads expect are the numbers of CTAs that really own bytes of a chunk, every 16-byte unit
// of every chunk is reduced by exactly one (rank, reduce CTA, work item), and ring positions of
// chunks that can be in flight together never overlap.  Runs without a GPU (tests/test_pipe_geometry_cpu.py).
// ---------------------------------------------------------------------------
int selftest_pipe_geometry(size_t nbytes, size_t chunk_bytes, int copy_ctas, int world, int red_ctas,
                           unsigned ring_chunks) {
  if (nbytes == 0 || (nbytes & 15) || chunk_bytes == 0 || chunk_bytes % (size_t(copy_ctas) * kBulkTile) || copy_ctas < 1 ||
      world < 2 || world > kMaxRanks || red_ctas < 1) {
    set_error("invalid self-test arguments");
    return B200_ERR_INVALID;
  }
  PipeArgs a{nullptr, nullptr, nbytes, 0, chunk_bytes, copy_ctas, ring_chunks};
  const PipeGeom g = make_geom(a);
  // ---- copy roles --------------------------------------------------------------------------
  std::vector<std::pair<size_t, size_t>> iv;  // [begin, end)
  std::vector<uint32_t> owners(g.K, 0);
  for (uint32_t j = 0; j < g.G; ++j) {
    const uint32_t nc = chunks_of_cta(g, j);
    for (uint32_t k = 0; k < g.K; ++k) {
      const uint32_t len = share_len(g, j, k);
      if ((k < nc) != (len > 0)) {
        set_error("copy CTA %u: chunks_of_cta=%u disagrees with share_len of chunk %u", j, nc, k);
        return B200_ERR_INVALID;
      }
      if (!len) continue;
      if (len & 15) {
        set_error("share of CTA %u in chunk %u is not a multiple of 16 bytes", j, k);
        return B200_ERR_INVALID;
      }
      ++owners[k];
      iv.emplace_back(share_off(g, j, k), share_off(g, j, k) + len);
      if (g.R) {  // the share must stay inside the ring position of its chunk
        const size_t pos = slot_chunk_off(g, k) + size_t(j) * g.share;
        if (pos + len > size_t(g.R) * g.C || pos / g.C != k % g.R) {
          set_error("ring placement of chunk %u share %u leaves its position", k, j);
          return B200_ERR_INVALID;
        }
      }
    }
  }
  std::sort(iv.begin(), iv.end());
  size_t at = 0;
  for (auto &e : iv) {
    if (e.first != at) {
      set_error("copy shares do not tile the message at byte %zu (next share starts at %zu)", at, e.first);
      return B200_ERR_INVALID;
    }
    at = e.second;
  }
  if (at != nbytes) {
    set_error("copy shares end at %zu, message has %zu bytes", at, nbytes);
    return B200_ERR_INVALID;
  }
  for (uint32_t k = 0; k < g.K; ++k)
    if (owners[k] != copy_arrivals(g, k)) {
      set_error("chunk %u: %u copy CTAs own bytes, flag thread expects %u arrivals", k, owners[k], copy_arrivals(g, k));
      return B200_ERR_INVALID;
    }
  // ---- reduce role ---------------------------------------------------------------------------
  std::vector<std::pair<size_t, size_t>> units;  // global 16-byte unit ranges
  for (int r = 0; r < world; ++r) {
    std::vector<uint32_t> items(g.K, 0), expect(g.K, 0);
    for (int me = 0; me < red_ctas; ++me) {
      ItemIter iter(g, r, world, uint32_t(me), uint32_t(red_ctas));
      uint32_t k = 0;
      while (iter.next(k)) {
        ++items[k];
        expect[k] = iter.nitems;
        const size_t base = (size_t(k) * g.C) >> 4;
        const size_t lo = iter.lo + iter.it * kItemUnits;
        const size_t hi = lo + kItemUnits < iter.hi ? lo + kItemUnits : iter.hi;
        if (lo < hi) units.emplace_back(base + lo, base + hi);
      }
    }
    for (uint32_t k = 0; k < g.K; ++k)
      if (items[k] != expect[k] || items[k] == 0) {
        set_error("rank %d chunk %u: %u work items dealt, arrival thread expects %u", r, k, items[k], expect[k]);
        return B200_ERR_INVALID;
      }
  }
  std::sort(units.begin(), units.end());
  at = 0;
  for (auto &e : units) {
    if (e.first != at) {
      set_error("reduce items do not tile the message at unit %zu (next item starts at %zu)", at, e.first);
      return B200_ERR_INVALID;
    }
    at = e.second;
  }
  if (at != (nbytes >> 4)) {
    set_error("reduce items end at unit %zu, message has %zu units", at, nbytes >> 4);
    return B200_ERR_INVALID;
  }
  return B200_OK;
}

const void *allreduce_pipe_module_kernel() { return reinterpret_cast<const void *>(allgather_pull_kernel); }

}  // namespace b200

extern "C" int b200_selftest_pipe_geometry(size_t nbytes, size_t chunk_bytes, int copy_ctas, int world, int red_ctas,
                                           unsigned ring_chunks) {
  return b200::selftest_pipe_geometry(nbytes, chunk_bytes, copy_ctas, world, red_ctas, ring_chunks);
}
