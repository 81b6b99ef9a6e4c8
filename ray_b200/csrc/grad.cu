// grad.cu — fused data-parallel gradient synchronisation (SURVEY K8).
//
// One launch per DDP bucket does what the reference path does in four to six kernels
// (c10d reducer div_ / bf16_compress_hook casts + ncclAllReduce + cast back, reached
// from train/torch/config.py:144 and train/torch/train_loop_utils.py:456-480):
//
//   stage-in : read the fp32 bucket, multiply by `scale` (1/world for DDP's mean),
//              cast to the wire dtype, write to the symmetric slot
//   reduce   : two-shot over peer HBM, or NVLS multimem.ld_reduce(.acc::f32)+multimem.st
//   stage-out: read the reduced wire values, cast back to fp32, write the bucket
//
// With wire = bf16 the NVLink traffic and the staging traffic are halved.
#include <type_traits>

#include "allreduce_core.cuh"

namespace b200 {

struct GradArgs {
  float *grad;
  size_t count;
  float scale;
  size_t staging_bytes;
  int red_ctas;  // CTAs of the NVLS reduce phase (0 = all)
};

template <typename W>
struct Wire;
template <>
struct Wire<float> {
  static constexpr int kElems = 4;
  static __device__ __forceinline__ uint4 pack(const float *f) {
    return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
  }
  static __device__ __forceinline__ void unpack(uint4 v, float *f) {
    f[0] = __uint_as_float(v.x);
    f[1] = __uint_as_float(v.y);
    f[2] = __uint_as_float(v.z);
    f[3] = __uint_as_float(v.w);
  }
};
template <>
struct Wire<__nv_bfloat16> {
  static constexpr int kElems = 8;
  static __device__ __forceinline__ uint4 pack(const float *f) {
    uint4 v;
    __nv_bfloat162 *p = reinterpret_cast<__nv_bfloat162 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
    return v;
  }
  static __device__ __forceinline__ void unpack(uint4 v, float *f) {
    const __nv_bfloat162 *p = reinterpret_cast<const __nv_bfloat162 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 t = __bfloat1622float2(p[i]);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
};
template <>
struct Wire<__half> {
  static constexpr int kElems = 8;
  static __device__ __forceinline__ uint4 pack(const float *f) {
    uint4 v;
    __half2 *p = reinterpret_cast<__half2 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
    return v;
  }
  static __device__ __forceinline__ void unpack(uint4 v, float *f) {
    const __half2 *p = reinterpret_cast<const __half2 *>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float2 t = __half22float2(p[i]);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
};

// wire unit u covers gradient elements [u*E, u*E+E)
template <typename W>
__device__ __forceinline__ uint4 load_grad_unit(const float *g, size_t u, size_t count, float scale, bool aligned) {
  constexpr int E = Wire<W>::kElems;
  float f[E];
  const size_t e0 = u * E;
  if (aligned && e0 + E <= count) {
#pragma unroll
    for (int k = 0; k < E / 4; ++k) {
      const uint4 v = ld_stream(g + e0 + 4 * k);
      f[4 * k + 0] = __uint_as_float(v.x);
      f[4 * k + 1] = __uint_as_float(v.y);
      f[4 * k + 2] = __uint_as_float(v.z);
      f[4 * k + 3] = __uint_as_float(v.w);
    }
  } else {
#pragma unroll
    for (int i = 0; i < E; ++i) f[i] = (e0 + i < count) ? g[e0 + i] : 0.f;
  }
#pragma unroll
  for (int i = 0; i < E; ++i) f[i] *= scale;
  return Wire<W>::pack(f);
}

template <typename W>
__device__ __forceinline__ void store_grad_unit(float *g, size_t u, size_t count, bool aligned, uint4 w) {
  constexpr int E = Wire<W>::kElems;
  float f[E];
  Wire<W>::unpack(w, f);
  const size_t e0 = u * E;
  if (aligned && e0 + E <= count) {
#pragma unroll
    for (int k = 0; k < E / 4; ++k)
      st_vec(g + e0 + 4 * k, make_uint4(__float_as_uint(f[4 * k]), __float_as_uint(f[4 * k + 1]),
                                       __float_as_uint(f[4 * k + 2]), __float_as_uint(f[4 * k + 3])));
  } else {
#pragma unroll
    for (int i = 0; i < E; ++i)
      if (e0 + i < count) g[e0 + i] = f[i];
  }
}

template <typename W, bool NVLS>
__global__ void __launch_bounds__(kThreads, 1) grad_allreduce_kernel(DevComm c, GradArgs a) {
  constexpr int E = Wire<W>::kElems;
  const uint32_t launch = c.st->launch_ctr;
  const uint32_t ep = launch * 4u;
  const RowGeom g = make_rows((a.count + E - 1) / E, c.world);
  const size_t off = staging_slot_offset(launch, a.staging_bytes);
  const bool al = is_aligned16(a.grad);

  stage_in_rows(c, off, g, [&](size_t u) { return load_grad_unit<W>(a.grad, u, a.count, a.scale, al); });
  if (!reduce_phase<W, B200_SUM, NVLS>(c, ep, off, g, a.red_ctas)) {
    finish_launch(c);
    return;
  }
  stage_out_rows(c, off, g, [&](size_t u, uint4 v) { store_grad_unit<W>(a.grad, u, a.count, al, v); });
  finish_launch(c);
}

// world == 1: the same arithmetic without any peer (scale, round-trip through the wire type).
// Pure HBM streaming (8 B per element).  One-shot grid: every thread owns one 16-byte unit and the
// hardware CTA scheduler does the load balancing -- no flag rows are involved, so the grid is NOT
// clamped to kMaxBlocks (round-1 ran this kernel at 43 % occupancy because of that clamp).  One
// unit per thread was best or tied against 2, 4 and 8 at every bucket size and wire type
// (profiles/r02/grad_local_sweep_events.txt, grad_local_sweep_ncu.txt).
constexpr int kLocalThreads = 256;
// One thread = 16 bytes of the fp32 bucket (4 elements), whatever the wire type: nothing is
// stored in wire format here, so the 8-element wire units of the multi-rank kernels would only
// halve the thread count (ncu, 60 MB bucket: 20.0 us with 8-element units, 15.1 us with 4).
template <typename W>
__device__ __forceinline__ uint4 wire_round_trip(uint4 v, float scale) {
  float f[4] = {__uint_as_float(v.x) * scale, __uint_as_float(v.y) * scale, __uint_as_float(v.z) * scale,
                __uint_as_float(v.w) * scale};
  if constexpr (std::is_same<W, __nv_bfloat16>::value) {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = __bfloat162float(__float2bfloat16_rn(f[i]));
  } else if constexpr (std::is_same<W, __half>::value) {
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = __half2float(__float2half_rn(f[i]));
  }
  return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
}

template <typename W>
__global__ void __launch_bounds__(kLocalThreads) grad_local_kernel(GradArgs a) {
  const size_t U = a.count >> 2;  // whole 16-byte units; the host sends the ragged tail separately
  const size_t u = size_t(blockIdx.x) * kLocalThreads + threadIdx.x;
  uint4 *g = reinterpret_cast<uint4 *>(a.grad);
  if (u < U) st_vec(g + u, wire_round_trip<W>(ld_stream(g + u), a.scale));
}

// unaligned buckets / the last count % 4 elements
template <typename W>
__global__ void grad_local_scalar_kernel(GradArgs a) {
  for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < a.count; i += size_t(gridDim.x) * blockDim.x) {
    float f = a.grad[i] * a.scale;
    if constexpr (std::is_same<W, __nv_bfloat16>::value) f = __bfloat162float(__float2bfloat16_rn(f));
    else if constexpr (std::is_same<W, __half>::value) f = __half2float(__float2half_rn(f));
    a.grad[i] = f;
  }
}

template <typename W>
static void launch_grad_local(const GradArgs &a, cudaStream_t stream) {
  if (!is_aligned16(a.grad)) {
    grad_local_scalar_kernel<W><<<1184, 256, 0, stream>>>(a);
    return;
  }
  const size_t U = a.count >> 2;
  if (U) grad_local_kernel<W><<<unsigned((U + kLocalThreads - 1) / kLocalThreads), kLocalThreads, 0, stream>>>(a);
  if (a.count & 3) {
    GradArgs tail = a;
    tail.grad = a.grad + (U << 2);
    tail.count = a.count & 3;
    grad_local_scalar_kernel<W><<<1, 32, 0, stream>>>(tail);
  }
}

template <typename W>
static int launch_grad(b200_comm *c, GradArgs a, cudaStream_t stream) {
  constexpr int E = Wire<W>::kElems;
  const size_t U = (a.count + E - 1) / E;
  if (c->world == 1) {
    launch_grad_local<W>(a, stream);
    B200_LAUNCH_CHECK(c);
    return B200_OK;
  }
  const size_t rows = (U + size_t(c->world) * kThreads - 1) / (size_t(c->world) * kThreads);
  int g = pick_blocks(c, rows, c->sm_count);
  const long long min_world = c->params[B200_PARAM_NVLS_MIN_WORLD] >= 0 ? c->params[B200_PARAM_NVLS_MIN_WORLD] : 3;
  const bool nvls = c->mc_active && c->world >= min_world;
  if (!nvls) a.red_ctas = 0;  // peer-load reducers want the whole grid
  if (nvls) grad_allreduce_kernel<W, true><<<g, kThreads, 0, stream>>>(c->dev(), a);
  else grad_allreduce_kernel<W, false><<<g, kThreads, 0, stream>>>(c->dev(), a);
  B200_LAUNCH_CHECK(c);
  return B200_OK;
}

const void *grad_module_kernel() { return reinterpret_cast<const void *>(grad_local_scalar_kernel<float>); }

}  // namespace b200

using namespace b200;

extern "C" int b200_grad_allreduce(b200_comm_t c, float *grad, size_t count, float scale,
                                   int wire_dtype, void *stream_) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (wire_dtype != B200_F32 && wire_dtype != B200_BF16 && wire_dtype != B200_F16) {
    set_error("wire dtype must be f32, bf16 or f16 (got %d)", wire_dtype);
    return B200_ERR_UNSUPPORTED;
  }
  if (count == 0) return B200_OK;
  if (!grad) {
    set_error("null gradient pointer");
    return B200_ERR_INVALID;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  const size_t wire_es = b200_dtype_size(wire_dtype);
  // elements per launch so the wire image fits one staging slot (multiple of 8 elements)
  const size_t chunk_elems = (c->staging_bytes / wire_es) & ~size_t(7);
  for (size_t done = 0; done < count;) {
    const size_t n = (count - done) < chunk_elems ? (count - done) : chunk_elems;
    const long long rc_param = c->params[B200_PARAM_NVLS_CTAS];
    GradArgs a{grad + done, n, scale, c->staging_bytes, rc_param > 0 ? int(rc_param) : 0};
    if (wire_dtype == B200_F32) rc = launch_grad<float>(c, a, stream);
    else if (wire_dtype == B200_BF16) rc = launch_grad<__nv_bfloat16>(c, a, stream);
    else rc = launch_grad<__half>(c, a, stream);
    if (rc) return rc;
    done += n;
  }
  return B200_OK;
}
