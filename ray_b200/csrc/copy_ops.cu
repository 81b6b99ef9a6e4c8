// copy_ops.cu — all-gather (SURVEY K2 with the K6 un-flatten copies fused away),
// broadcast (K4) and the flag-only barrier (K7).  These kernels move bytes; they do
// not depend on the element type.
#include "kernel_utils.cuh"
#include "pipe.h"

namespace b200 {

struct AGArgs {
  const char *in;
  char *outs[kMaxRanks];
  size_t nbytes;  // per rank
  size_t staging_bytes;
};

// Every rank stages its tensor in its own slot, then pulls each peer's slot over
// NVLink straight into the caller's output tensor for that peer.
__global__ void __launch_bounds__(kThreads, 1) allgather_kernel(DevComm c, AGArgs a) {
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const int n = c.world, r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const bool in_al = is_aligned16(a.in);
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
    for (int i = 0; i < kMaxRanks; ++i) {
      if (i < n) {
        int p = r + i;
        if (p >= n) p -= n;
        v[i] = ld_peer(c.data[p] + off + (u << 4));
      }
    }
#pragma unroll
    for (int i = 0; i < kMaxRanks; ++i) {
      if (i < n) {
        int p = r + i;
        if (p >= n) p -= n;
        store_user_unit(a.outs[p], u, un, is_aligned16(a.outs[p]), v[i]);
      }
    }
  }
  finish_launch(c);
}

struct BcastArgs {
  char *buf;
  size_t nbytes;
  size_t staging_bytes;
  int root;
};

// NVLS = false: root stages, every other rank pulls root's slot.
// NVLS = true : root writes its tensor once to the multicast alias (the switch
//               replicates it into every rank's slot), the others copy out locally.
template <bool NVLS>
__global__ void __launch_bounds__(kThreads, 1) broadcast_kernel(DevComm c, BcastArgs a) {
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const int r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const bool al = is_aligned16(a.buf);
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const size_t stride = size_t(gridDim.x) * kThreads;
  const size_t first = size_t(blockIdx.x) * kThreads + threadIdx.x;

  if (r == a.root) {
    char *dst = (NVLS ? c.mc_data : c.data[r]) + off;
    for (size_t u = first; u < U; u += stride) {
      const uint4 v = load_user_unit(a.buf, u, un, al);
      if (NVLS) multimem_st(dst + (u << 4), v);
      else st_vec(dst + (u << 4), v);
    }
  }

  if (!cta_barrier_all(c, ep + 1)) {
    finish_launch(c);
    return;
  }

  if (r != a.root) {
    const char *src = (NVLS ? c.data[r] : c.data[a.root]) + off;
    for (size_t u = first; u < U; u += stride) store_user_unit(a.buf, u, un, al, ld_peer(src + (u << 4)));
  }
  finish_launch(c);
}

__global__ void barrier_kernel(DevComm c) {
  const uint32_t ep = c.st->launch_ctr * 4u;
  cta_barrier_all(c, ep + 1);
  finish_launch(c);
}

const void *copy_ops_module_kernel() { return reinterpret_cast<const void *>(barrier_kernel); }

}  // namespace b200

using namespace b200;

extern "C" int b200_allgather(b200_comm_t c, const void *in, void *const *outs, size_t count,
                              int dtype, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  const size_t es = b200_dtype_size(dtype);
  if (es == 0) {
    set_error("unsupported dtype %d", dtype);
    return B200_ERR_UNSUPPORTED;
  }
  if (count == 0) return B200_OK;
  if (!in || !outs) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  for (int p = 0; p < c->world; ++p)
    if (!outs[p]) {
      set_error("output tensor %d is null", p);
      return B200_ERR_INVALID;
    }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t total = count * es;
  if (c->world == 1) {
    if (outs[0] != in) B200_CHECK_CUDA(cudaMemcpyAsync(outs[0], in, total, cudaMemcpyDeviceToDevice, stream));
    return B200_OK;
  }
  // Large aligned operands: the pull kernel (TMA copy-in + bulk loads of the peers' slots straight
  // into the caller's output tensors, allreduce_pipe.cu).  B200_PARAM_AG_PULL_MIN_BYTES = per-rank
  // size from which it is used (default 4 MiB; 0 = never).
  {
    const long long pm = c->params[B200_PARAM_AG_PULL_MIN_BYTES];
    const size_t pull_min = pm >= 0 ? size_t(pm) : (size_t(4) << 20);  // 4 ranks: 1 MiB/rank 49 us pulled vs 28 us staged
    bool aligned = is_aligned16(in) && (total & 15) == 0 && pm != 0 && pipe_chunk_bytes(c) > 0;
    for (int p = 0; p < c->world; ++p) aligned = aligned && is_aligned16(outs[p]);
    if (aligned && total >= pull_min) {
      const size_t cap = pipe_max_bytes(c, PIPE_PULL) / (size_t(1) << 20) * (size_t(1) << 20);
      const size_t step = cap ? cap : c->staging_bytes;
      for (size_t done = 0; done < total;) {
        const size_t nbytes = (total - done) < step ? (total - done) : step;
        char *o[kMaxRanks] = {};
        for (int p = 0; p < c->world; ++p) o[p] = static_cast<char *>(outs[p]) + done;
        rc = launch_allgather_pull(c, static_cast<const char *>(in) + done, o, nbytes, stream);
        if (rc) return rc;
        done += nbytes;
      }
      return B200_OK;
    }
  }
  for (size_t done = 0; done < total;) {
    const size_t nbytes = (total - done) < c->staging_bytes ? (total - done) : c->staging_bytes;
    AGArgs a{};
    a.in = static_cast<const char *>(in) + done;
    for (int p = 0; p < c->world; ++p) a.outs[p] = static_cast<char *>(outs[p]) + done;
    a.nbytes = nbytes;
    a.staging_bytes = c->staging_bytes;
    const size_t U = make_units(nbytes).total();
    int g = pick_blocks(c, (U + kThreads - 1) / kThreads, c->sm_count);
    allgather_kernel<<<g, kThreads, 0, stream>>>(c->dev(), a);
    B200_LAUNCH_CHECK(c);
    done += nbytes;
  }
  return B200_OK;
}

extern "C" int b200_broadcast(b200_comm_t c, void *buf, size_t count, int dtype, int root,
                              void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  const size_t es = b200_dtype_size(dtype);
  if (es == 0) {
    set_error("unsupported dtype %d", dtype);
    return B200_ERR_UNSUPPORTED;
  }
  if (root < 0 || root >= c->world) {
    set_error("root rank %d out of range for world size %d", root, c->world);
    return B200_ERR_INVALID;
  }
  if (count == 0 || c->world == 1) return B200_OK;
  if (!buf) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t total = count * es;
  for (size_t done = 0; done < total;) {
    const size_t nbytes = (total - done) < c->staging_bytes ? (total - done) : c->staging_bytes;
    BcastArgs a{static_cast<char *>(buf) + done, nbytes, c->staging_bytes, root};
    const size_t U = make_units(nbytes).total();
    int g = pick_blocks(c, (U + kThreads - 1) / kThreads, c->sm_count);
    // The multicast store pays off once more than one peer would pull from the root.
    const bool nvls = c->mc_active && c->world > 2 && nbytes >= (size_t(64) << 10);
    if (nvls) broadcast_kernel<true><<<g, kThreads, 0, stream>>>(c->dev(), a);
    else broadcast_kernel<false><<<g, kThreads, 0, stream>>>(c->dev(), a);
    B200_LAUNCH_CHECK(c);
    done += nbytes;
  }
  return B200_OK;
}

extern "C" int b200_barrier(b200_comm_t c, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (c->world == 1) return B200_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  barrier_kernel<<<1, 32, 0, stream>>>(c->dev());
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}
