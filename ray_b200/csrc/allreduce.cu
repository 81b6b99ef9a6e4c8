// allreduce.cu — all-reduce kernels (SURVEY K1) and their dispatcher.
//
// Three algorithms, all in ONE launch each (stage-in, cross-GPU barrier, reduce,
// barrier, stage-out are phases of the same persistent grid):
//
//   one-shot : every rank stages its input in its own symmetric slot, then reads
//              all n staged inputs over NVLink and reduces rank-ascending.  One
//              barrier; latency path for small messages.
//   two-shot : the message is cut into rows of n*512 16-byte units; rank r owns
//              units [r*512,(r+1)*512) of every row.  The owner loads its units
//              from all n peers' HBM (rank-ascending reduction), and pushes the
//              result back into all n peers' slots.  Every element is read and
//              written by exactly one thread system-wide, so the reduce-scatter
//              and all-gather halves fuse without a barrier between them.
//   NVLS     : same ownership, but the n loads are one multimem.ld_reduce and the
//              n stores one multimem.st on the NVSwitch multicast alias.
//
// CTA b of every rank works on the same rows in every phase, so a barrier between
// CTA b's of all ranks (flags in the signal pad) is the only synchronisation needed:
// no grid-wide sync, no host involvement.
#include "allreduce_core.cuh"
#include "pipe.h"

namespace b200 {

struct ARArgs {
  const char *in;
  char *out;
  size_t nbytes;
  size_t staging_bytes;
  long long sym_off;  // >= 0: operand lives in the symmetric data region at this offset
                      //       (zero-copy, in place); < 0: stage through the rotating slot
  int red_ctas;       // CTAs that run the reduce phase (0 or >= grid: all of them)
};

// ---------------------------------------------------------------------------
// one-shot
// ---------------------------------------------------------------------------
template <typename T, int OP>
__global__ void __launch_bounds__(kThreads, 1) allreduce_oneshot_kernel(DevComm c, ARArgs a) {
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const int n = c.world, r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const bool in_al = is_aligned16(a.in), out_al = is_aligned16(a.out);
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const size_t stride = size_t(gridDim.x) * kThreads;
  const size_t first = size_t(blockIdx.x) * kThreads + threadIdx.x;

  char *mine = c.data[r] + off;
  for (size_t u = first; u < U; u += stride) st_vec(mine + (u << 4), load_user_unit(a.in, u, un, in_al));

  if (!cta_barrier_all(c, ep + 1)) {
    finish_launch(c);
    return;
  }

  for (size_t u = first; u < U; u += stride) {
    uint4 v[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p)
      if (p < n) v[p] = ld_peer(c.data[p] + off + (u << 4));
    typename Tr::Acc acc = Tr::unpack(v[0]);
#pragma unroll
    for (int p = 1; p < kMaxRanks; ++p)
      if (p < n) Tr::template reduce<OP>(acc, Tr::unpack(v[p]));
    if (OP == B200_AVG) Tr::average(acc, n);
    store_user_unit(a.out, u, un, out_al, Tr::pack(acc));
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// low-latency (LL) one-shot: every rank pushes its message straight into each peer's LL slot as
// (word, flag) pairs -- 16-byte stores carrying two pairs, each 8-byte pair lands atomically --
// and then polls its own slots until the flags of this launch appear.  No barrier, no staging
// pass: one NVLink traversal end to end.  At most one 16-byte unit per thread.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void ll_store(void *p, uint32_t a, uint32_t b, uint32_t flag) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(a), "r"(flag), "r"(b), "r"(flag)
               : "memory");
}
__device__ __forceinline__ uint4 ll_load(const void *p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p)
               : "memory");
  return v;
}

template <typename T, int OP>
__global__ void __launch_bounds__(kThreads, 1) allreduce_ll_kernel(DevComm c, ARArgs a) {
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t flag = launch + 1u;  // never 0, never equal to what the slot held two launches ago
  const int n = c.world, r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const size_t u = size_t(blockIdx.x) * kThreads + threadIdx.x;
  const size_t par_off = (launch & 1u) ? size_t(kMaxRanks) * kLLSlotBytes : 0;
  if (u < U) {
    const uint4 mine = load_user_unit(a.in, u, un, is_aligned16(a.in));
    // push (start with the next rank so the eight peers are not hit in lock step)
#pragma unroll
    for (int i = 1; i < kMaxRanks; ++i) {
      if (i < n) {
        int p = r + i;
        if (p >= n) p -= n;
        char *dst = c.ll[p] + par_off + size_t(r) * kLLSlotBytes + (u << 5);
        ll_store(dst, mine.x, mine.y, flag);
        ll_store(dst + 16, mine.z, mine.w, flag);
      }
    }
    // collect, rank-ascending
    const char *base = c.ll[r] + par_off + (u << 5);
    typename Tr::Acc acc;
    bool alive = true;
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p) {
      if (p < n) {
        uint4 v = mine;
        if (p != r) {
          const char *src = base + size_t(p) * kLLSlotBytes;
          uint4 lo, hi;
          unsigned spins = 0;
          unsigned long long t0 = 0;
          while (alive) {
            lo = ll_load(src);
            hi = ll_load(src + 16);
            if (lo.y == flag && lo.w == flag && hi.y == flag && hi.w == flag) break;
            if ((++spins & 0x3ff) == 0) {
              if (*c.abort != 0) {
                give_up(c, B200_ERR_ABORTED);
                alive = false;
              }
              const unsigned long long now = globaltimer_ns();
              if (t0 == 0) t0 = now;
              else if (now - t0 > c.timeout_ns) {
                give_up(c, B200_ERR_TIMEOUT);
                alive = false;
              }
            }
          }
          v = make_uint4(lo.x, lo.z, hi.x, hi.z);
        }
        if (p == 0) acc = Tr::unpack(v);
        else Tr::template reduce<OP>(acc, Tr::unpack(v));
      }
    }
    if (alive) {
      if (OP == B200_AVG) Tr::average(acc, n);
      store_user_unit(a.out, u, un, is_aligned16(a.out), Tr::pack(acc));
    }
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// two-shot / NVLS
// ---------------------------------------------------------------------------
template <typename T, int OP, bool NVLS>
__global__ void __launch_bounds__(kThreads, 1) allreduce_twoshot_kernel(DevComm c, ARArgs a) {
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const Units un = make_units(a.nbytes);
  const RowGeom g = make_rows(un.total(), c.world);
  const bool staged = a.sym_off < 0;
  const size_t off = staged ? staging_slot_offset(launch, a.staging_bytes) : size_t(a.sym_off);

  // phase 0: stage this CTA's rows into the local symmetric slot
  if (staged) {
    const bool in_al = is_aligned16(a.in);
    stage_in_rows(c, off, g, [&](size_t u) { return load_user_unit(a.in, u, un, in_al); });
  }
  // phase 1: reduce the units this rank owns, publish to every peer
  if (!reduce_phase<T, OP, NVLS>(c, ep, off, g, a.red_ctas)) {
    finish_launch(c);
    return;
  }
  // phase 2: copy this CTA's rows out of the local slot
  if (staged) {
    const bool out_al = is_aligned16(a.out);
    stage_out_rows(c, off, g, [&](size_t u, uint4 v) { store_user_unit(a.out, u, un, out_al, v); });
  }
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// multi-tensor (SURVEY K9): the same three phases, but stage-in gathers from / stage-out
// scatters to a table of tensors, so a list of tensors is reduced as ONE message in ONE
// launch with no host-side flatten (dag/collective_node.py:220-232 uses parameters_to_vector).
// ---------------------------------------------------------------------------
template <typename T, int OP, bool NVLS>
__global__ void __launch_bounds__(kThreads, 1)
allreduce_multi_kernel(DevComm c, const __grid_constant__ TensorTable tb, size_t staging_bytes, int red_ctas) {
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const RowGeom g = make_rows(tb.ustart[tb.count], c.world);
  const size_t off = staging_slot_offset(launch, staging_bytes);

  stage_in_rows(c, off, g, [&](size_t u) {
    const int i = table_find(tb, u);
    return load_user_unit(tb.ptr[i], u - tb.ustart[i], make_units(tb.nbytes[i]), is_aligned16(tb.ptr[i]));
  });
  if (!reduce_phase<T, OP, NVLS>(c, ep, off, g, red_ctas)) {
    finish_launch(c);
    return;
  }
  stage_out_rows(c, off, g, [&](size_t u, uint4 v) {
    const int i = table_find(tb, u);
    store_user_unit(tb.ptr[i], u - tb.ustart[i], make_units(tb.nbytes[i]), is_aligned16(tb.ptr[i]), v);
  });
  finish_launch(c);
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int nvls_ctas(const b200_comm *c);
static size_t ll_limit(const b200_comm *c);
template <typename T, int OP>
static int launch_allreduce(b200_comm *c, const char *in, char *out, size_t nbytes, int algo,
                            long long sym_off, cudaStream_t stream) {
  DevComm dc = c->dev();
  ARArgs a{in, out, nbytes, c->staging_bytes, sym_off, 0};
  const size_t U = make_units(nbytes).total();
  if (algo == B200_ALGO_LL) {
    a.sym_off = -1;
    allreduce_ll_kernel<T, OP><<<int((U + kThreads - 1) / kThreads), kThreads, 0, stream>>>(dc, a);
  } else if (algo == B200_ALGO_ONESHOT) {
    a.sym_off = -1;
    int g = pick_blocks(c, (U + kThreads - 1) / kThreads, 32);
    allreduce_oneshot_kernel<T, OP><<<g, kThreads, 0, stream>>>(dc, a);
  } else {
    const size_t rows = (U + size_t(c->world) * kThreads - 1) / (size_t(c->world) * kThreads);
    int g = pick_blocks(c, rows, c->sm_count);
    if (algo == B200_ALGO_NVLS) {
      a.red_ctas = nvls_ctas(c);
      if (sym_off >= 0) {  // nothing to stage: the whole launch is the reduce phase, which
        const int cap = a.red_ctas > 0 ? a.red_ctas : 64;  // saturates the switch with ~64 CTAs
        if (g > cap && c->forced_blocks == 0) g = cap;
        a.red_ctas = 0;
      }
      if constexpr (Multimem<T>::kSum && (OP == B200_SUM || OP == B200_AVG)) {
        allreduce_twoshot_kernel<T, OP, true><<<g, kThreads, 0, stream>>>(dc, a);
      } else {
        set_error("NVLS all-reduce supports SUM/AVG on f32/f16/bf16 only");
        return B200_ERR_UNSUPPORTED;
      }
    } else {
      allreduce_twoshot_kernel<T, OP, false><<<g, kThreads, 0, stream>>>(dc, a);
    }
  }
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

static bool nvls_capable(int dtype, int op) {
  return (dtype == B200_F32 || dtype == B200_F16 || dtype == B200_BF16) &&
         (op == B200_SUM || op == B200_AVG);
}

// Measured on 2/4/8 B200s (profiles/r01): with two ranks the switch reduction saves no
// traffic and the peer-load kernel is faster; from five ranks on NVLS wins at every size.
static bool nvls_pays_off(const b200_comm *c, size_t nbytes) {
  const long long min_world = c->params[B200_PARAM_NVLS_MIN_WORLD];
  if (min_world >= 0) return c->world >= min_world;
  if (c->world <= 2) return false;
  if (c->world <= 4) return nbytes >= (size_t(128) << 20);
  return true;
}

// Zero-copy operands: the NVSwitch reduction saturates with far fewer CTAs than the GPU has SMs
// (8 B200s, profiles/r01/tune_w8_v2_graph.log: 64 CTAs beat 100 and 148), so those launches are
// capped at 64 CTAs.  Staged operands keep CTA-to-CTA barriers over the whole grid by default:
// running their reduce phase on fewer CTAs (this parameter > 0) needs grid-wide waits, which
// serialise the phases and measured slower (profiles/r01/sweep_w4_nvls_ctas.log).
static int nvls_ctas(const b200_comm *c) {
  const long long v = c->params[B200_PARAM_NVLS_CTAS];
  return v > 0 ? int(v) : 0;
}

// LL pays n-1 flag-doubled pushes per rank: measured break-even against the one-shot kernel is
// ~32 KiB with 2 ranks and ~4 KiB with 8 (profiles/r01/final_w8_graph_sweeps.log).
static size_t ll_limit(const b200_comm *c) {
  const long long v = c->params[B200_PARAM_LL_MAX_BYTES];
  const size_t lim = v >= 0 ? size_t(v) : (size_t(64) << 10) / size_t(c->world) / (c->world > 4 ? 2 : 1);
  return lim < kLLMaxPayload ? lim : kLLMaxPayload;
}

// Measured break-even of the pipelined kernels against the phase-by-phase ones (profiles/r02).
static size_t pipe_min_bytes(const b200_comm *c) {
  const long long v = c->params[B200_PARAM_PIPE_MIN_BYTES];
  if (v >= 0) return size_t(v);
  // 2 ranks: the pull kernel wins from 16 MiB (350 vs 330 GB/s; 64 MiB 519 vs 440, 1 GiB 619 vs 411);
  // NVLS roles: from 128 MiB (8 ranks: 586 vs 559, 256 MiB 673 vs 611, 1 GiB 694 vs 627 GB/s)
  return c->world == 2 ? (size_t(16) << 20) : (size_t(128) << 20);
}

static size_t oneshot_limit(const b200_comm *c) {
  if (c->params[B200_PARAM_ONESHOT_MAX_BYTES] >= 0) return size_t(c->params[B200_PARAM_ONESHOT_MAX_BYTES]);
  // each rank reads world * nbytes in the one-shot scheme.  Break-even against the two-shot kernel
  // (profiles/r01 sweeps: 2 ranks ~1 MiB, 8 ranks ~256 KiB; profiles/r02/bench_n4: 256 KiB one-shot
  // 16 us, 1 MiB two-shot 24 us); the 0.5 MB PPO gradient vector of BASELINE configs[3] falls on
  // the one-shot side at 2 and 4 ranks.
  return (size_t(5) << 19) / size_t(c->world);  // 2.5 MiB / n
}

const void *allreduce_module_kernel() {
  return reinterpret_cast<const void *>(allreduce_ll_kernel<float, B200_SUM>);
}

}  // namespace b200

using namespace b200;

extern "C" int b200_allreduce(b200_comm_t c, const void *in, void *out, size_t count, int dtype,
                              int op, int algo, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  const size_t es = b200_dtype_size(dtype);
  if (es == 0) {
    set_error("unsupported dtype %d", dtype);
    return B200_ERR_UNSUPPORTED;
  }
  if (op < 0 || op >= B200_OP_COUNT) {
    set_error("unsupported reduce op %d", op);
    return B200_ERR_UNSUPPORTED;
  }
  if (count == 0) return B200_OK;
  if (!in || !out) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t total = count * es;
  if (c->world == 1) {
    if (in != out) B200_CHECK_CUDA(cudaMemcpyAsync(out, in, total, cudaMemcpyDeviceToDevice, stream));
    return B200_OK;
  }
  if (algo == B200_ALGO_NVLS && !c->mc_active) {
    set_error("NVLS requested but the multicast mapping is not active");
    return B200_ERR_UNSUPPORTED;
  }

  // zero-copy when the operand sits in the symmetric heap (and is updated in place)
  // The reduce phase works on whole 16-byte units straight in the heap, so a tensor whose size is
  // not a multiple of 16 bytes would have the bytes that follow it reduced as well: such operands
  // take the staged path (which zero-pads the tail unit in the slot instead).  Every rank must pass
  // the tensor at the same heap offset (b200_symm_alloc / the pool hand out identical offsets when
  // ranks allocate in the same order, which both interfaces require).
  long long sym_off = -1;
  if (in == out && (total & 15) == 0 && b200_symm_contains(c, in, total) && is_aligned16(in))
    sym_off = static_cast<const char *>(in) - reinterpret_cast<const char *>(c->data.va[c->rank]);

  const char *src = static_cast<const char *>(in);
  char *dst = static_cast<char *>(out);

  // Ordinary (staged) operands from pipe_min_bytes() on: the chunk-pipelined kernels, which overlap
  // the two staging passes with the NVLink phase (allreduce_pipe.cu).  They move whole 16-byte
  // units with the bulk-copy engine, so they need aligned operands.
  int pipe_variant = -1;
  if (sym_off < 0 && is_aligned16(in) && is_aligned16(out) && (total & 15) == 0 && pipe_chunk_bytes(c) > 0 &&
      (algo == B200_ALGO_PIPE || (algo == B200_ALGO_AUTO && total >= pipe_min_bytes(c)))) {
    if (c->world == 2) pipe_variant = PIPE_PULL;
    else if (c->mc_active && nvls_capable(dtype, op)) pipe_variant = PIPE_NVLS;
    else if (algo == B200_ALGO_PIPE) pipe_variant = PIPE_PEER;  // AUTO without NVLS keeps the two-shot kernel
    if (algo == B200_ALGO_PIPE && c->params[B200_PARAM_PIPE_VARIANT] >= 0)
      pipe_variant = int(c->params[B200_PARAM_PIPE_VARIANT]);
    if (pipe_variant == PIPE_NVLS && !(c->mc_active && nvls_capable(dtype, op))) pipe_variant = PIPE_PEER;
  } else if (algo == B200_ALGO_PIPE) {
    set_error("the pipelined all-reduce needs 16-byte aligned operands outside the symmetric heap "
              "and a size that is a multiple of 16 bytes");
    return B200_ERR_UNSUPPORTED;
  }

  // Messages larger than one staging slot are processed slot by slot.
  const size_t chunk_max = sym_off >= 0 ? total : (pipe_variant >= 0 ? pipe_max_bytes(c, pipe_variant) : c->staging_bytes);
  for (size_t done = 0; done < total;) {
    const size_t nbytes = (total - done) < chunk_max ? (total - done) : chunk_max;
    if (pipe_variant >= 0 && (algo == B200_ALGO_PIPE || nbytes >= pipe_min_bytes(c) || nbytes > c->staging_bytes)) {
      rc = launch_allreduce_pipe_dyn(c, src + done, dst + done, nbytes, dtype, op, pipe_variant, stream);
      if (rc) return rc;
      done += nbytes;
      continue;
    }
    int a = algo;
    if (a == B200_ALGO_AUTO || a == B200_ALGO_PIPE) {
      if (nbytes <= ll_limit(c)) a = B200_ALGO_LL;
      else if (sym_off < 0 && nbytes <= oneshot_limit(c)) a = B200_ALGO_ONESHOT;
      else if (c->mc_active && nvls_capable(dtype, op) && nvls_pays_off(c, nbytes)) a = B200_ALGO_NVLS;
      else a = B200_ALGO_TWOSHOT;
    }
    if (a == B200_ALGO_LL && nbytes > kLLMaxPayload) a = B200_ALGO_ONESHOT;
    if (a == B200_ALGO_ONESHOT && nbytes > c->staging_bytes) a = B200_ALGO_TWOSHOT;
    const long long so = sym_off >= 0 ? sym_off + (long long)done : -1;
    B200_DISPATCH_DTYPE(dtype, T, B200_DISPATCH_OP(op, OP, {
                          rc = launch_allreduce<T, OP>(c, src + done, dst + done, nbytes, a, so, stream);
                        }));
    if (rc) return rc;
    done += nbytes;
  }
  return B200_OK;
}


// ---- multi-tensor entry ------------------------------------------------------------
namespace b200 {
template <typename T, int OP>
static int launch_multi(b200_comm *c, const TensorTable &tb, cudaStream_t stream) {
  const size_t U = tb.ustart[tb.count];
  const size_t rows = (U + size_t(c->world) * kThreads - 1) / (size_t(c->world) * kThreads);
  int g = pick_blocks(c, rows, c->sm_count);
  if constexpr (Multimem<T>::kSum && (OP == B200_SUM || OP == B200_AVG)) {
    if (c->mc_active) {
      allreduce_multi_kernel<T, OP, true><<<g, kThreads, 0, stream>>>(c->dev(), tb, c->staging_bytes, nvls_ctas(c));
      B200_LAUNCH_CHECK(c);
      return B200_OK;
    }
  }
  allreduce_multi_kernel<T, OP, false><<<g, kThreads, 0, stream>>>(c->dev(), tb, c->staging_bytes, 0);
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}
}  // namespace b200

// Reduces `ntensors` same-dtype tensors as one message: tensors are packed (each starting on
// a 16-byte unit) into launches of up to kMaxTableTensors tensors / one staging slot.  The
// single-launch kernel exists for the floating-point types (gradients, activations); other
// dtypes take one fused launch per tensor.
extern "C" int b200_allreduce_multi(b200_comm_t c, void *const *ptrs, const size_t *counts,
                                    int ntensors, int dtype, int op, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  const size_t es = b200_dtype_size(dtype);
  if (es == 0) {
    set_error("unsupported dtype %d", dtype);
    return B200_ERR_UNSUPPORTED;
  }
  if (op < 0 || op >= B200_OP_COUNT) {
    set_error("unsupported reduce op %d", op);
    return B200_ERR_UNSUPPORTED;
  }
  if (ntensors < 0 || (ntensors > 0 && (!ptrs || !counts))) {
    set_error("invalid tensor list");
    return B200_ERR_INVALID;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool table_ok = (dtype == B200_F32 || dtype == B200_F16 || dtype == B200_BF16 || dtype == B200_F64) &&
                        c->world > 1;
  int i = 0;
  while (i < ntensors) {
    if (counts[i] == 0) {
      ++i;
      continue;
    }
    if (!ptrs[i]) {
      set_error("tensor %d is null", i);
      return B200_ERR_INVALID;
    }
    const size_t bytes_i = counts[i] * es;
    if (!table_ok || bytes_i > c->staging_bytes / 2) {
      // large tensors (or dtypes without a table kernel) go through the single-tensor path
      rc = b200_allreduce(c, ptrs[i], ptrs[i], counts[i], dtype, op, B200_ALGO_AUTO, stream_);
      if (rc) return rc;
      ++i;
      continue;
    }
    B200_CHECK_CUDA(cudaSetDevice(c->device));
    TensorTable tb{};
    size_t units = 0;
    while (i < ntensors && tb.count < kMaxTableTensors) {
      if (counts[i] == 0) {
        ++i;
        continue;
      }
      const size_t b = counts[i] * es;
      const size_t u = (b + 15) >> 4;
      if (!ptrs[i] || b > c->staging_bytes / 2 || ((units + u) << 4) > c->staging_bytes) break;
      tb.ptr[tb.count] = static_cast<char *>(ptrs[i]);
      tb.nbytes[tb.count] = b;
      tb.ustart[tb.count] = static_cast<unsigned int>(units);
      units += u;
      ++tb.count;
      ++i;
    }
    tb.ustart[tb.count] = static_cast<unsigned int>(units);
    if (tb.count == 0) continue;
    switch (dtype) {
      case B200_F32: B200_DISPATCH_OP(op, OP, { rc = launch_multi<float, OP>(c, tb, stream); }); break;
      case B200_F64: B200_DISPATCH_OP(op, OP, { rc = launch_multi<double, OP>(c, tb, stream); }); break;
      case B200_F16: B200_DISPATCH_OP(op, OP, { rc = launch_multi<__half, OP>(c, tb, stream); }); break;
      default: B200_DISPATCH_OP(op, OP, { rc = launch_multi<__nv_bfloat16, OP>(c, tb, stream); }); break;
    }
    if (rc) return rc;
  }
  return B200_OK;
}
