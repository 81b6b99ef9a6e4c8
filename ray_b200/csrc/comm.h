// comm.h — host-side communicator object shared by the translation units of
// libb200_collective.so.  Not part of the public ABI (see include/b200_collective.h).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

namespace b200 {

void set_error(const char *fmt, ...);

#define B200_CHECK_CUDA(expr)                                                              \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      b200::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,    \
                      __LINE__);                                                           \
      return B200_ERR_CUDA;                                                                \
    }                                                                                      \
  } while (0)

struct Region {
  size_t bytes = 0;                                   // mapped size (granularity multiple)
  CUmemGenericAllocationHandle own = 0;               // this rank's physical allocation
  int own_fd = -1;                                    // exported POSIX fd of `own`
  CUmemGenericAllocationHandle imported[kMaxRanks] = {};  // peers' allocations
  CUdeviceptr va[kMaxRanks] = {};                     // where each peer's copy is mapped here
};

}  // namespace b200

struct b200_comm {
  int world = 0;
  int rank = 0;
  int device = 0;
  b200_config_t cfg{};
  size_t staging_bytes = 0;  // per slot
  size_t heap_bytes = 0;
  size_t inbox_bytes = 0;    // per source
  size_t heap_used = 0;

  b200::Region data, sig, inbox, ll;

  // NVLS
  bool mc_supported = false;  // this device + config allow multicast
  bool mc_active = false;
  CUmemGenericAllocationHandle mc_handle = 0;
  int mc_fd = -1;
  CUdeviceptr mc_va = 0;
  size_t mc_bytes = 0;

  b200::LocalState *d_state = nullptr;
  int *h_abort = nullptr;  // cudaHostAlloc'd, mapped
  int *d_abort = nullptr;  // device alias of h_abort
  unsigned long long *d_trace = nullptr;  // optional kernel event trace
  unsigned int trace_cap = 0;

  // bootstrap endpoint (abstract unix socket served by `server`)
  std::string sock_name;
  int listen_fd = -1;
  std::thread server;
  std::atomic<bool> server_stop{false};
  std::vector<std::string> peer_socks;
  unsigned char token[16] = {};                          // secret of this rank's endpoint
  std::vector<std::array<unsigned char, 16>> peer_tokens;  // ... and of the peers', from their handles
  bool connected = false;
  uint32_t host_barrier_seq = 0;

  std::atomic<uint64_t> launches{0};
  int forced_blocks = 0;
  long long params[B200_PARAM_COUNT];  // b200_comm_set_param values; -1 = default
  int sm_count = 148;
  std::atomic<bool> aborted{false};
  std::mutex mu;

  b200_comm() { std::fill(std::begin(params), std::end(params), -1ll); }
  b200::DevComm dev() const;
};

namespace b200 {
// implemented in bootstrap.cu
int check_usable(b200_comm *c);
inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// One kernel of every translation unit that defines kernels (each is a module of its own in the
// shared object): b200_comm_create loads every function of these modules up front.
const void *allreduce_module_kernel();
const void *allreduce_pipe_module_kernel();
const void *copy_ops_module_kernel();
const void *grad_module_kernel();
const void *p2p_module_kernel();
const void *reduce_ops_module_kernel();
}  // namespace b200
