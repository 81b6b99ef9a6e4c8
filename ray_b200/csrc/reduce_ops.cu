// reduce_ops.cu — reduce-scatter (SURVEY K3, fusing away the K6 flatten copies) and
// reduce-to-root (a6).
//
// reduce-scatter is push based: rank r reads its n input tensors straight from the
// caller's list and writes tensor q into sub-slot r of rank q's staging slot over
// NVLink (the local copy-in and the transfer are the same instruction stream).  After
// one barrier every rank reduces its n sub-slots from local HBM, rank-ascending, into
// the caller's output tensor.
#include "kernel_utils.cuh"

namespace b200 {

struct RSArgs {
  const char *ins[kMaxRanks];
  char *out;
  size_t nbytes;  // per tensor
  size_t staging_bytes;
};

template <typename T, int OP>
__global__ void __launch_bounds__(kThreads, 1) reducescatter_kernel(DevComm c, RSArgs a) {
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const int n = c.world, r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const size_t sub = U << 4;  // bytes per sub-slot
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const size_t stride = size_t(gridDim.x) * kThreads;
  const size_t first = size_t(blockIdx.x) * kThreads + threadIdx.x;

  // push: tensor (r+i)%n goes to rank (r+i)%n, sub-slot r
  for (size_t u = first; u < U; u += stride) {
    uint4 v[kMaxRanks];
#pragma unroll
    for (int i = 0; i < kMaxRanks; ++i) {
      if (i < n) {
        int q = r + i;
        if (q >= n) q -= n;
        v[i] = load_user_unit(a.ins[q], u, un, is_aligned16(a.ins[q]));
      }
    }
#pragma unroll
    for (int i = 0; i < kMaxRanks; ++i) {
      if (i < n) {
        int q = r + i;
        if (q >= n) q -= n;
        st_vec(c.data[q] + off + size_t(r) * sub + (u << 4), v[i]);
      }
    }
  }

  if (!cta_barrier_all(c, ep + 1)) {
    finish_launch(c);
    return;
  }

  const bool out_al = is_aligned16(a.out);
  const char *mine = c.data[r] + off;
  for (size_t u = first; u < U; u += stride) {
    uint4 v[kMaxRanks];
#pragma unroll
    for (int p = 0; p < kMaxRanks; ++p)
      if (p < n) v[p] = ld_peer(mine + size_t(p) * sub + (u << 4));
    typename Tr::Acc acc = Tr::unpack(v[0]);
#pragma unroll
    for (int p = 1; p < kMaxRanks; ++p)
      if (p < n) Tr::template reduce<OP>(acc, Tr::unpack(v[p]));
    if (OP == B200_AVG) Tr::average(acc, n);
    store_user_unit(a.out, u, un, out_al, Tr::pack(acc));
  }
  finish_launch(c);
}

struct ReduceArgs {
  char *buf;
  size_t nbytes;
  size_t staging_bytes;
  int root;
};

// Every rank stages its tensor; the root pulls all n copies and reduces in place.
template <typename T, int OP>
__global__ void __launch_bounds__(kThreads, 1) reduce_kernel(DevComm c, ReduceArgs a) {
  using Tr = Traits<T>;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const int n = c.world, r = c.rank;
  const Units un = make_units(a.nbytes);
  const size_t U = un.total();
  const bool al = is_aligned16(a.buf);
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const size_t stride = size_t(gridDim.x) * kThreads;
  const size_t first = size_t(blockIdx.x) * kThreads + threadIdx.x;

  char *mine = c.data[r] + off;
  for (size_t u = first; u < U; u += stride) st_vec(mine + (u << 4), load_user_unit(a.buf, u, un, al));

  if (!cta_barrier_all(c, ep + 1)) {
    finish_launch(c);
    return;
  }

  if (r == a.root) {
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
      store_user_unit(a.buf, u, un, al, Tr::pack(acc));
    }
  }
  finish_launch(c);
}

template <typename T, int OP>
static int launch_rs(b200_comm *c, const RSArgs &a, cudaStream_t stream) {
  const size_t U = make_units(a.nbytes).total();
  int g = pick_blocks(c, (U + kThreads - 1) / kThreads, c->sm_count);
  reducescatter_kernel<T, OP><<<g, kThreads, 0, stream>>>(c->dev(), a);
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

template <typename T, int OP>
static int launch_reduce(b200_comm *c, const ReduceArgs &a, cudaStream_t stream) {
  const size_t U = make_units(a.nbytes).total();
  int g = pick_blocks(c, (U + kThreads - 1) / kThreads, c->sm_count);
  reduce_kernel<T, OP><<<g, kThreads, 0, stream>>>(c->dev(), a);
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

const void *reduce_ops_module_kernel() {
  return reinterpret_cast<const void *>(reducescatter_kernel<float, B200_SUM>);
}

}  // namespace b200

using namespace b200;

extern "C" int b200_reducescatter(b200_comm_t c, const void *const *ins, void *out, size_t count,
                                  int dtype, int op, void *stream_) {
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
  if (!ins || !out) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  for (int p = 0; p < c->world; ++p)
    if (!ins[p]) {
      set_error("input tensor %d is null", p);
      return B200_ERR_INVALID;
    }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t total = count * es;
  if (c->world == 1) {
    if (ins[0] != out) B200_CHECK_CUDA(cudaMemcpyAsync(out, ins[0], total, cudaMemcpyDeviceToDevice, stream));
    return B200_OK;
  }
  // n sub-slots of the chunk must fit one staging slot; keep chunks 16-byte multiples
  size_t chunk_max = (c->staging_bytes / size_t(c->world)) & ~size_t(15);
  for (size_t done = 0; done < total;) {
    const size_t nbytes = (total - done) < chunk_max ? (total - done) : chunk_max;
    RSArgs a{};
    for (int p = 0; p < c->world; ++p) a.ins[p] = static_cast<const char *>(ins[p]) + done;
    a.out = static_cast<char *>(out) + done;
    a.nbytes = nbytes;
    a.staging_bytes = c->staging_bytes;
    B200_DISPATCH_DTYPE(dtype, T, B200_DISPATCH_OP(op, OP, { rc = launch_rs<T, OP>(c, a, stream); }));
    if (rc) return rc;
    done += nbytes;
  }
  return B200_OK;
}

extern "C" int b200_reduce(b200_comm_t c, void *buf, size_t count, int dtype, int op, int root,
                           void *stream_) {
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
  if (root < 0 || root >= c->world) {
    set_error("root rank %d out of range for world size %d", root, c->world);
    return B200_ERR_INVALID;
  }
  if (count == 0) return B200_OK;
  if (!buf) {
    set_error("null tensor pointer");
    return B200_ERR_INVALID;
  }
  if (c->world == 1) return B200_OK;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t total = count * es;
  for (size_t done = 0; done < total;) {
    const size_t nbytes = (total - done) < c->staging_bytes ? (total - done) : c->staging_bytes;
    ReduceArgs a{static_cast<char *>(buf) + done, nbytes, c->staging_bytes, root};
    B200_DISPATCH_DTYPE(dtype, T, B200_DISPATCH_OP(op, OP, { rc = launch_reduce<T, OP>(c, a, stream); }));
    if (rc) return rc;
    done += nbytes;
  }
  return B200_OK;
}
