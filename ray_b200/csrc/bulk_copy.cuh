// bulk_copy.cuh — TMA bulk-copy engine (cp.async.bulk, SASS UBLKCP) driven by ONE thread of a CTA.
//
// The copy phases of the collectives (user tensor -> symmetric slot, slot -> user tensor, user
// tensor -> a peer's slot or inbox over NVLink) are pure byte movement.  Done with ld/st they need
// tens of CTAs x 512 threads to keep enough bytes in flight; done with the bulk-copy unit a single
// thread keeps NST x TILE bytes in flight per CTA:
//
//     global --cp.async.bulk + mbarrier complete_tx--> shared ring --cp.async.bulk.bulk_group--> global
//
// so a copy role costs a handful of CTAs (one busy thread each) instead of the whole GPU, and the
// SMs stay available to the kernels the collective overlaps with (DDP backward).
//
// Requirements: source, destination and length of every tile are multiples of 16 bytes.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b200 {

constexpr int kBulkTile = 32 << 10;  // bytes per tile
constexpr int kBulkStages = 6;       // ring depth (6 x 32 KiB = 192 KiB of shared memory)
// loads issued ahead of the store cursor -- measured with scripts/bulk_bench.cu (profiles/r02/
// bulk_bench*.log): 3 is as good as anything for local HBM -> local HBM (49.6 GB/s per CTA) and
// for local -> peer over NVLink (16 CTAs: 711 GB/s); waiting for completion with a lag of 2+
// tiles costs nothing
constexpr int kBulkLookaheadLocal = 3;
constexpr int kBulkLookaheadRemote = 3;
// A ring buffer is free again as soon as its store has READ it (wait_group.read); the store's
// global writes may still be in flight then.  Measured on B200 (profiles/r02): a bulk store to a
// peer over NVLink takes ~6 us to COMPLETE, so bounding the stores in flight by the ring depth
// (12 x 16 KiB in the first version) capped a CTA at 18 GB/s.  Completion is therefore tracked
// separately and lazily: done(i) is reported once tile i + D has been issued (wait_group D).
constexpr int kBulkLagRemote = 4;  // completion lag D for stores that cross NVLink
constexpr int kBulkLagLocal = 2;   // ... and for stores into local HBM
// the two flavours of the engine
struct BulkLocal {
  static constexpr int kLookahead = kBulkLookaheadLocal, kLag = kBulkLagLocal;
};
struct BulkRemote {
  static constexpr int kLookahead = kBulkLookaheadRemote, kLag = kBulkLagRemote;
};
// source on a peer (bulk loads over NVLink), destination local: 5 loads in flight measured 703 GB/s
// with 16 CTAs against 530 with 3 (profiles/r02/bulk_bench_pull.log)
struct BulkPull {
  static constexpr int kLookahead = 5, kLag = kBulkLagLocal;
};
constexpr size_t kBulkSmemBytes = size_t(kBulkStages) * kBulkTile + 16 * kBulkStages;

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// shared -> global (local HBM or a peer's memory over NVLink), tracked by bulk async-groups
__device__ __forceinline__ void bulk_s2g(void *dst, uint32_t src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait() {  // all but the N most recent groups have COMPLETED (writes done)
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_read() {  // all but the N most recent groups have read their source
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// orders async-proxy accesses (bulk copies) against generic-proxy accesses (ld/st, flags)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// Shared-memory carve-up of a copy CTA (dynamic shared memory, kBulkSmemBytes).
struct BulkRing {
  uint32_t tiles;  // shared address of tile 0
  uint32_t bars;   // shared address of mbarrier 0
};

// Every thread of the CTA calls this once before the copy role starts.
__device__ __forceinline__ BulkRing bulk_ring_init(char *dyn_smem) {
  BulkRing r;
  r.tiles = smem_u32(dyn_smem);
  r.bars = r.tiles + kBulkStages * kBulkTile;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kBulkStages; ++s) mbar_init(r.bars + 8 * s, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  return r;
}

// ---------------------------------------------------------------------------
// Segment engine.  One thread issues every tile, and a single thread retires a dependent
// instruction every ~5 cycles, so the per-tile instruction count IS the throughput limit
// (measured: a first, index-based engine with two divisions and three lambda calls per tile
// reached 30-36 GB/s per CTA where the bulk-copy unit does 50).  Here the work is a list of
// SEGMENTS -- contiguous byte ranges [src, src+bytes) -> [dst, dst+bytes) -- and the tiles of a
// segment are walked with pointer increments; the callbacks run once per segment, not per tile:
//   seg(i)         -> BulkSeg of segment i (bytes > 0)
//   gate(i, block) -> before the first load of segment i: 1 = source valid / destination free,
//                     0 = not yet (only when !block), -1 = abandon (abort / watchdog).  The
//                     engine first asks without blocking; when nothing else can make progress it
//                     drains its pending stores (every done() it owes has then been delivered -- a
//                     peer may be waiting for exactly that) and asks again with block = true
//   done(i)        -> once every store of segment i has completed, in order (lazily, Cfg::kLag tiles)
// ---------------------------------------------------------------------------
struct BulkSeg {
  const char *src;
  char *dst;
  uint32_t bytes;  // multiple of 16
};

template <typename Cfg, typename SegFn, typename GateFn, typename DoneFn>
__device__ __forceinline__ bool bulk_copy_segments(const BulkRing &ring, uint32_t nsegs, SegFn seg, GateFn gate,
                                                   DoneFn done) {
  constexpr int LAG = Cfg::kLag;
  constexpr uint32_t LA = Cfg::kLookahead;
  constexpr int kReadPending = kBulkStages - Cfg::kLookahead - 1;
  // load cursor
  uint32_t l_seg = 0, l_left = 0, l_stage = 0;
  const char *l_src = nullptr;
  bool l_open = false;  // segment l_seg passed its gate and l_src / l_left are valid
  // store cursor
  uint32_t s_seg = 0, s_left = 0, s_stage = 0, s_parity = 0;
  char *s_dst = nullptr;
  bool s_open = false;
  // completion cursor
  uint32_t c_seg = 0, c_tiles_left = 0;
  bool c_open = false;
  uint32_t loads = 0, stores = 0, completed = 0;  // tile counters
  (void)s_seg;
  bool ok = true;

  auto retire = [&](uint32_t upto) {  // tiles [completed, upto) have completed
    while (completed < upto) {
      if (!c_open) {
        c_tiles_left = (seg(c_seg).bytes + kBulkTile - 1) / kBulkTile;
        c_open = true;
      }
      ++completed;
      if (--c_tiles_left == 0) {
        done(c_seg);
        ++c_seg;
        c_open = false;
      }
    }
  };

  while (true) {
    // ---- issue loads while the lookahead window has room --------------------------------
    while (loads - stores < LA) {
      if (!l_open) {
        if (l_seg >= nsegs) break;
        const int g = gate(l_seg, false);
        if (g < 0) ok = false;
        if (g <= 0) break;
        const BulkSeg d = seg(l_seg);
        l_src = d.src;
        l_left = d.bytes;
        l_open = true;
      }
      if (l_left == 0) {
        ++l_seg;
        l_open = false;
        continue;
      }
      const uint32_t bytes = l_left < uint32_t(kBulkTile) ? l_left : uint32_t(kBulkTile);
      mbar_expect_tx(ring.bars + 8 * l_stage, bytes);
      bulk_g2s(ring.tiles + l_stage * kBulkTile, l_src, bytes, ring.bars + 8 * l_stage);
      l_src += bytes;
      l_left -= bytes;
      l_stage = l_stage + 1 == uint32_t(kBulkStages) ? 0 : l_stage + 1;
      ++loads;
    }
    // ---- store the oldest landed tile -----------------------------------------------------
    if (stores < loads) {
      if (!s_open) {
        const BulkSeg d = seg(s_seg);
        s_dst = d.dst;
        s_left = d.bytes;
        s_open = true;
      }
      while (!mbar_try_wait(ring.bars + 8 * s_stage, s_parity)) {
      }
      const uint32_t bytes = s_left < uint32_t(kBulkTile) ? s_left : uint32_t(kBulkTile);
      bulk_s2g(s_dst, ring.tiles + s_stage * kBulkTile, bytes);
      bulk_commit();
      s_dst += bytes;
      s_left -= bytes;
      if (s_left == 0) {
        ++s_seg;
        s_open = false;
      }
      if (++s_stage == uint32_t(kBulkStages)) {
        s_stage = 0;
        s_parity ^= 1u;
      }
      ++stores;
      bulk_wait_read<kReadPending>();
      if (stores > uint32_t(LAG)) {
        bulk_wait<LAG>();
        retire(stores - uint32_t(LAG));
      }
      continue;
    }
    // ---- nothing in flight ------------------------------------------------------------------
    bulk_wait<0>();
    retire(stores);
    if (!ok || (l_seg >= nsegs && !l_open)) break;
    if (!l_open) {
      // every remaining step needs segment l_seg's gate: everything owed has been reported, block
      if (gate(l_seg, true) < 0) {
        ok = false;
        break;
      }
      const BulkSeg d = seg(l_seg);
      l_src = d.src;
      l_left = d.bytes;
      l_open = true;
    }
  }
  bulk_wait<0>();
  retire(stores);
  return ok;
}

}  // namespace b200
