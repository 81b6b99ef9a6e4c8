// bootstrap.cu — communicator lifecycle: symmetric memory through the CUDA virtual
// memory management API, peer mapping by POSIX-fd passing, NVLS multicast binding.
//
// What travels through Ray's store is ONE opaque blob per rank (b200_comm_export_handle);
// it names an abstract unix socket on which that rank serves the file descriptors of its
// allocations (SCM_RIGHTS) and, on rank 0, a tiny agreement barrier used while the
// multicast object is assembled.  This replaces the ncclUniqueId rendezvous of the
// reference (util/collective/collective_group/nccl_collective_group.py:36-125,414-468;
// experimental/channel/torch_tensor_accelerator_channel.py:738-844).
//
// The driver API is reached through cudaGetDriverEntryPoint so the library has no
// link-time dependency on libcuda.so (it must load on a GPU-less build host).
#include <errno.h>
#include <poll.h>
#include <sys/socket.h>
#include <sys/un.h>
#include <unistd.h>

#include <array>

#include <chrono>
#include <cstring>
#include <map>
#include <set>

#include "comm.h"
#include "pipe.h"

namespace b200 {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------------------
// driver entry points
// ---------------------------------------------------------------------------
struct Driver {
  CUresult (*GetErrorString)(CUresult, const char **) = nullptr;
  CUresult (*DeviceGet)(CUdevice *, int) = nullptr;
  CUresult (*DeviceGetAttribute)(int *, CUdevice_attribute, CUdevice) = nullptr;
  CUresult (*MemGetAllocationGranularity)(size_t *, const CUmemAllocationProp *,
                                          CUmemAllocationGranularity_flags) = nullptr;
  CUresult (*MemCreate)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *,
                        unsigned long long) = nullptr;
  CUresult (*MemRelease)(CUmemGenericAllocationHandle) = nullptr;
  CUresult (*MemAddressReserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr,
                                unsigned long long) = nullptr;
  CUresult (*MemAddressFree)(CUdeviceptr, size_t) = nullptr;
  CUresult (*MemMap)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle,
                     unsigned long long) = nullptr;
  CUresult (*MemUnmap)(CUdeviceptr, size_t) = nullptr;
  CUresult (*MemSetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t) = nullptr;
  CUresult (*MemExportToShareableHandle)(void *, CUmemGenericAllocationHandle,
                                         CUmemAllocationHandleType, unsigned long long) = nullptr;
  CUresult (*MemImportFromShareableHandle)(CUmemGenericAllocationHandle *, void *,
                                           CUmemAllocationHandleType) = nullptr;
  CUresult (*MulticastCreate)(CUmemGenericAllocationHandle *, const CUmulticastObjectProp *) = nullptr;
  CUresult (*MulticastAddDevice)(CUmemGenericAllocationHandle, CUdevice) = nullptr;
  CUresult (*MulticastBindMem)(CUmemGenericAllocationHandle, size_t, CUmemGenericAllocationHandle,
                               size_t, size_t, unsigned long long) = nullptr;
  CUresult (*MulticastUnbind)(CUmemGenericAllocationHandle, CUdevice, size_t, size_t) = nullptr;
  CUresult (*MulticastGetGranularity)(size_t *, const CUmulticastObjectProp *,
                                      CUmulticastGranularity_flags) = nullptr;
  CUresult (*FuncGetModule)(CUmodule *, CUfunction) = nullptr;
  CUresult (*ModuleGetFunctionCount)(unsigned int *, CUmodule) = nullptr;
  CUresult (*ModuleEnumerateFunctions)(CUfunction *, unsigned int, CUmodule) = nullptr;
  CUresult (*FuncLoad)(CUfunction) = nullptr;
  bool ok = false;
  bool has_multicast = false;
  bool has_func_load = false;
};

template <typename F>
static bool load_sym(const char *name, F *out) {
  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qr;
  cudaError_t e = cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &qr);
  if (e != cudaSuccess || qr != cudaDriverEntryPointSuccess || fn == nullptr) {
    (void)cudaGetLastError();
    *out = nullptr;
    return false;
  }
  *out = reinterpret_cast<F>(fn);
  return true;
}

static Driver &driver() {
  static Driver d;
  static std::once_flag once;
  std::call_once(once, [] {
    bool ok = true;
    ok &= load_sym("cuGetErrorString", &d.GetErrorString);
    ok &= load_sym("cuDeviceGet", &d.DeviceGet);
    ok &= load_sym("cuDeviceGetAttribute", &d.DeviceGetAttribute);
    ok &= load_sym("cuMemGetAllocationGranularity", &d.MemGetAllocationGranularity);
    ok &= load_sym("cuMemCreate", &d.MemCreate);
    ok &= load_sym("cuMemRelease", &d.MemRelease);
    ok &= load_sym("cuMemAddressReserve", &d.MemAddressReserve);
    ok &= load_sym("cuMemAddressFree", &d.MemAddressFree);
    ok &= load_sym("cuMemMap", &d.MemMap);
    ok &= load_sym("cuMemUnmap", &d.MemUnmap);
    ok &= load_sym("cuMemSetAccess", &d.MemSetAccess);
    ok &= load_sym("cuMemExportToShareableHandle", &d.MemExportToShareableHandle);
    ok &= load_sym("cuMemImportFromShareableHandle", &d.MemImportFromShareableHandle);
    d.ok = ok;
    bool mc = true;
    mc &= load_sym("cuMulticastCreate", &d.MulticastCreate);
    mc &= load_sym("cuMulticastAddDevice", &d.MulticastAddDevice);
    mc &= load_sym("cuMulticastBindMem", &d.MulticastBindMem);
    mc &= load_sym("cuMulticastUnbind", &d.MulticastUnbind);
    mc &= load_sym("cuMulticastGetGranularity", &d.MulticastGetGranularity);
    d.has_multicast = mc;
    bool fl = true;
    fl &= load_sym("cuFuncGetModule", &d.FuncGetModule);
    fl &= load_sym("cuModuleGetFunctionCount", &d.ModuleGetFunctionCount);
    fl &= load_sym("cuModuleEnumerateFunctions", &d.ModuleEnumerateFunctions);
    fl &= load_sym("cuFuncLoad", &d.FuncLoad);
    d.has_func_load = fl;
  });
  return d;
}

#define B200_CHECK_CU(expr)                                                            \
  do {                                                                                 \
    CUresult _r = (expr);                                                              \
    if (_r != CUDA_SUCCESS) {                                                          \
      const char *_s = nullptr;                                                        \
      if (b200::driver().GetErrorString) b200::driver().GetErrorString(_r, &_s);       \
      b200::set_error("%s failed: %s (%d) (%s:%d)", #expr, _s ? _s : "?", int(_r),     \
                      __FILE__, __LINE__);                                             \
      return B200_ERR_CUDA;                                                            \
    }                                                                                  \
  } while (0)

// ---------------------------------------------------------------------------
// bootstrap blob
// ---------------------------------------------------------------------------
struct Blob {
  uint32_t magic;
  uint32_t version;
  int32_t pid;
  int32_t rank;
  int32_t world;
  int32_t device;
  int32_t mc_supported;
  int32_t reserved;
  unsigned char uuid[16];
  uint64_t data_bytes;
  uint64_t sig_bytes;
  uint64_t inbox_region_bytes;
  uint64_t staging_bytes;
  uint64_t heap_bytes;
  uint64_t inbox_bytes;
  char sock[96];
  unsigned char token[16];  // per-communicator secret: every request to this rank's endpoint must carry it
  char host[32];            // the group must live on one host (one NVSwitch domain)
};
static_assert(sizeof(Blob) <= B200_HANDLE_BYTES, "blob too large");
constexpr uint32_t kMagic = 0xB200C011u;
constexpr uint32_t kVersion = 2;

// ---------------------------------------------------------------------------
// unix-socket helpers
// ---------------------------------------------------------------------------
enum : uint32_t { OP_GET_FD = 1, OP_AGREE = 2 };
enum : uint32_t { FD_DATA = 0, FD_SIG = 1, FD_INBOX = 2, FD_MC = 3, FD_LL = 4 };
struct Req {
  uint32_t magic;
  uint32_t op;
  uint32_t arg;    // GET_FD: kind; AGREE: sequence number
  int32_t value;   // AGREE: this rank's vote (AND-reduced)
  unsigned char token[16];  // the secret from the SERVING rank's handle blob
};

// The endpoint lives in the abstract unix namespace (no file permissions) under a guessable name,
// and what it hands out are read-write fds of GPU memory.  Two checks before serving anything:
// the peer runs under our uid (SO_PEERCRED), and it knows the 128-bit token that only travelled
// inside the handle blob through the rendezvous store.
static bool peer_is_trusted(int conn, const Req &rq, const unsigned char *token) {
  ucred cred{};
  socklen_t len = sizeof(cred);
  if (getsockopt(conn, SOL_SOCKET, SO_PEERCRED, &cred, &len) != 0 || cred.uid != geteuid()) return false;
  unsigned char diff = 0;
  for (int i = 0; i < 16; ++i) diff |= rq.token[i] ^ token[i];  // constant time
  return diff == 0;
}

static void make_addr(const std::string &name, sockaddr_un *addr, socklen_t *len) {
  memset(addr, 0, sizeof(*addr));
  addr->sun_family = AF_UNIX;
  // abstract namespace: leading NUL, no filesystem entry, vanishes with the process
  size_t n = name.size() < sizeof(addr->sun_path) - 2 ? name.size() : sizeof(addr->sun_path) - 2;
  memcpy(addr->sun_path + 1, name.data(), n);
  *len = socklen_t(offsetof(sockaddr_un, sun_path) + 1 + n);
}

static bool read_full(int fd, void *buf, size_t n, int timeout_ms) {
  char *p = static_cast<char *>(buf);
  while (n) {
    pollfd pf{fd, POLLIN, 0};
    int pr = poll(&pf, 1, timeout_ms);
    if (pr <= 0) return false;
    ssize_t r = read(fd, p, n);
    if (r <= 0) {
      if (r < 0 && (errno == EINTR || errno == EAGAIN)) continue;
      return false;
    }
    p += r;
    n -= size_t(r);
  }
  return true;
}

static bool write_full(int fd, const void *buf, size_t n) {
  const char *p = static_cast<const char *>(buf);
  while (n) {
    ssize_t r = send(fd, p, n, MSG_NOSIGNAL);
    if (r <= 0) {
      if (r < 0 && (errno == EINTR || errno == EAGAIN)) continue;
      return false;
    }
    p += r;
    n -= size_t(r);
  }
  return true;
}

static bool send_fd(int sock, int fd, int32_t status) {
  msghdr msg{};
  iovec iov{&status, sizeof(status)};
  msg.msg_iov = &iov;
  msg.msg_iovlen = 1;
  alignas(cmsghdr) char ctrl[CMSG_SPACE(sizeof(int))];
  if (fd >= 0) {
    memset(ctrl, 0, sizeof(ctrl));
    msg.msg_control = ctrl;
    msg.msg_controllen = sizeof(ctrl);
    cmsghdr *cm = CMSG_FIRSTHDR(&msg);
    cm->cmsg_level = SOL_SOCKET;
    cm->cmsg_type = SCM_RIGHTS;
    cm->cmsg_len = CMSG_LEN(sizeof(int));
    memcpy(CMSG_DATA(cm), &fd, sizeof(int));
  }
  return sendmsg(sock, &msg, MSG_NOSIGNAL) == ssize_t(sizeof(status));
}

static int recv_fd(int sock, int32_t *status, int timeout_ms) {
  pollfd pf{sock, POLLIN, 0};
  if (poll(&pf, 1, timeout_ms) <= 0) return -1;
  msghdr msg{};
  iovec iov{status, sizeof(*status)};
  msg.msg_iov = &iov;
  msg.msg_iovlen = 1;
  alignas(cmsghdr) char ctrl[CMSG_SPACE(sizeof(int))];
  msg.msg_control = ctrl;
  msg.msg_controllen = sizeof(ctrl);
  ssize_t r = recvmsg(sock, &msg, MSG_CMSG_CLOEXEC);
  if (r != ssize_t(sizeof(*status))) return -1;
  for (cmsghdr *cm = CMSG_FIRSTHDR(&msg); cm; cm = CMSG_NXTHDR(&msg, cm)) {
    if (cm->cmsg_level == SOL_SOCKET && cm->cmsg_type == SCM_RIGHTS) {
      int fd;
      memcpy(&fd, CMSG_DATA(cm), sizeof(int));
      return fd;
    }
  }
  return -1;
}

static int connect_to(const std::string &name, int timeout_ms) {
  auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(timeout_ms);
  while (true) {
    int s = socket(AF_UNIX, SOCK_STREAM | SOCK_CLOEXEC, 0);
    if (s < 0) return -1;
    sockaddr_un addr;
    socklen_t len;
    make_addr(name, &addr, &len);
    if (connect(s, reinterpret_cast<sockaddr *>(&addr), len) == 0) return s;
    close(s);
    if (std::chrono::steady_clock::now() > deadline) return -1;
    std::this_thread::sleep_for(std::chrono::milliseconds(20));
  }
}

// Serves fds of this rank's allocations; on rank 0 also the agreement barrier.
static void server_loop(b200_comm *c) {
  std::map<uint32_t, std::vector<std::pair<int, int32_t>>> pending;  // seq -> (conn, vote)
  while (!c->server_stop.load()) {
    pollfd pf{c->listen_fd, POLLIN, 0};
    int pr = poll(&pf, 1, 100);
    if (pr <= 0) continue;
    int conn = accept4(c->listen_fd, nullptr, nullptr, SOCK_CLOEXEC);
    if (conn < 0) continue;
    Req rq{};
    // 500 ms: a client that connects and stays silent must not stall the (single-threaded) loop
    if (!read_full(conn, &rq, sizeof(rq), 500) || rq.magic != kMagic || !peer_is_trusted(conn, rq, c->token)) {
      close(conn);
      continue;
    }
    if (rq.op == OP_GET_FD) {
      int fd = -1;
      {
        std::lock_guard<std::mutex> lk(c->mu);
        switch (rq.arg) {
          case FD_DATA: fd = c->data.own_fd; break;
          case FD_SIG: fd = c->sig.own_fd; break;
          case FD_INBOX: fd = c->inbox.own_fd; break;
          case FD_MC: fd = c->mc_fd; break;
          case FD_LL: fd = c->ll.own_fd; break;
          default: break;
        }
      }
      send_fd(conn, fd, fd >= 0 ? 0 : -1);
      close(conn);
    } else if (rq.op == OP_AGREE) {
      auto &v = pending[rq.arg];
      v.emplace_back(conn, rq.value);
      if (int(v.size()) == c->world) {
        int32_t all = 1;
        for (auto &pr2 : v) all = all && pr2.second;
        for (auto &pr2 : v) {
          write_full(pr2.first, &all, sizeof(all));
          close(pr2.first);
        }
        pending.erase(rq.arg);
      }
    } else {
      close(conn);
    }
  }
  for (auto &kv : pending)
    for (auto &pr2 : kv.second) close(pr2.first);
  // nothing is served any more: stop accepting, so a late (or rogue) connect is refused outright
  std::lock_guard<std::mutex> lk(c->mu);
  if (c->listen_fd >= 0) {
    close(c->listen_fd);
    c->listen_fd = -1;
  }
}

static int fetch_fd(b200_comm *c, int peer, uint32_t kind) {
  int s = connect_to(c->peer_socks[peer], 30000);
  if (s < 0) {
    set_error("cannot reach bootstrap socket of rank %d (%s)", peer, strerror(errno));
    return -1;
  }
  Req rq{kMagic, OP_GET_FD, kind, 0, {}};
  memcpy(rq.token, c->peer_tokens[peer].data(), 16);
  int fd = -1;
  int32_t status = -1;
  if (write_full(s, &rq, sizeof(rq))) fd = recv_fd(s, &status, 30000);
  close(s);
  if (fd < 0) set_error("rank %d did not hand out fd kind %u", peer, kind);
  return fd;
}

// AND-agreement across all ranks through rank 0's endpoint.  Returns the agreed
// value (0/1) or -1 on failure.
static int host_agree(b200_comm *c, int vote) {
  if (c->world == 1) return vote ? 1 : 0;
  uint32_t seq = c->host_barrier_seq++;
  int s = connect_to(c->peer_socks[0], 30000);
  if (s < 0) {
    set_error("cannot reach rank 0 for host barrier %u", seq);
    return -1;
  }
  Req rq{kMagic, OP_AGREE, seq, vote ? 1 : 0, {}};
  memcpy(rq.token, c->peer_tokens[0].data(), 16);
  int32_t all = 0;
  int timeout_ms = 300000;
  bool ok = write_full(s, &rq, sizeof(rq)) && read_full(s, &all, sizeof(all), timeout_ms);
  close(s);
  if (!ok) {
    set_error("host barrier %u failed (a peer did not arrive)", seq);
    return -1;
  }
  return all ? 1 : 0;
}

// ---------------------------------------------------------------------------
// VMM helpers
// ---------------------------------------------------------------------------
static CUmemAllocationProp alloc_prop(int device) {
  CUmemAllocationProp prop{};
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = device;
  prop.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
  return prop;
}

static int map_handle(int device, CUmemGenericAllocationHandle h, size_t bytes, size_t align,
                      CUdeviceptr *va) {
  Driver &d = driver();
  B200_CHECK_CU(d.MemAddressReserve(va, bytes, align, 0, 0));
  B200_CHECK_CU(d.MemMap(*va, bytes, 0, h, 0));
  CUmemAccessDesc acc{};
  acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  acc.location.id = device;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  B200_CHECK_CU(d.MemSetAccess(*va, bytes, &acc, 1));
  return B200_OK;
}

static int region_create(b200_comm *c, Region *r, size_t bytes, size_t gran) {
  Driver &d = driver();
  r->bytes = round_up(bytes, gran);
  CUmemAllocationProp prop = alloc_prop(c->device);
  B200_CHECK_CU(d.MemCreate(&r->own, r->bytes, &prop, 0));
  int fd = -1;
  B200_CHECK_CU(d.MemExportToShareableHandle(&fd, r->own, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0));
  r->own_fd = fd;
  int rc = map_handle(c->device, r->own, r->bytes, gran, &r->va[c->rank]);
  if (rc) return rc;
  B200_CHECK_CUDA(cudaMemset(reinterpret_cast<void *>(r->va[c->rank]), 0, r->bytes));
  return B200_OK;
}

static int region_import(b200_comm *c, Region *r, int peer, uint32_t kind, size_t gran) {
  Driver &d = driver();
  int fd = fetch_fd(c, peer, kind);
  if (fd < 0) return B200_ERR_SYSTEM;
  CUresult res = d.MemImportFromShareableHandle(&r->imported[peer], reinterpret_cast<void *>(intptr_t(fd)),
                                                CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
  close(fd);
  B200_CHECK_CU(res);
  return map_handle(c->device, r->imported[peer], r->bytes, gran, &r->va[peer]);
}

static void region_destroy(b200_comm *c, Region *r) {
  Driver &d = driver();
  for (int p = 0; p < kMaxRanks; ++p) {
    if (r->va[p]) {
      d.MemUnmap(r->va[p], r->bytes);
      d.MemAddressFree(r->va[p], r->bytes);
      r->va[p] = 0;
    }
    if (r->imported[p]) {
      d.MemRelease(r->imported[p]);
      r->imported[p] = 0;
    }
  }
  if (r->own) {
    d.MemRelease(r->own);
    r->own = 0;
  }
  if (r->own_fd >= 0) {
    close(r->own_fd);
    r->own_fd = -1;
  }
  (void)c;
}

int check_usable(b200_comm *c) {
  if (!c) {
    set_error("null communicator");
    return B200_ERR_INVALID;
  }
  if (c->aborted.load()) {
    set_error("communicator was aborted");
    return B200_ERR_ABORTED;
  }
  if (!c->connected) {
    set_error("communicator is not connected (call b200_comm_connect first)");
    return B200_ERR_INVALID;
  }
  // A kernel that gave up (watchdog / abort) leaves the flag protocol in an undefined state: the
  // launch counter still advanced, peers may be mid-collective.  Treat it as fatal for the
  // communicator -- later launches are refused instead of running against stale flags.
  if (c->h_abort) {
    const int st = __atomic_load_n(&c->h_abort[1], __ATOMIC_ACQUIRE);
    if (st != 0) {
      set_error(st == B200_ERR_TIMEOUT ? "a previous collective timed out waiting for a peer (device watchdog); "
                                         "the communicator is unusable"
                                       : "a previous collective was aborted; the communicator is unusable");
      return st;
    }
  }
  return B200_OK;
}

// CUDA loads kernels lazily by default, and loading a kernel at its first launch may synchronise the
// context.  The collective kernels spin until their peers' kernels run, so where ranks share a context
// (several ranks on one GPU, thread actors of one process) a first launch can wait for a kernel that
// is itself waiting for that launch, until the device watchdog gives up.  Every kernel of the library
// is therefore loaded on a device before the first communicator there can launch anything.
static int preload_kernels(int device) {
  static std::mutex mu;
  static std::set<int> done;
  std::lock_guard<std::mutex> lk(mu);
  if (done.count(device)) return B200_OK;
  Driver &d = driver();
  if (!d.has_func_load) {
    set_error("CUDA driver lacks cuModuleEnumerateFunctions / cuFuncLoad (needs CUDA 12.4 or newer)");
    return B200_ERR_UNSUPPORTED;
  }
  for (const void *k : {allreduce_module_kernel(), allreduce_pipe_module_kernel(), copy_ops_module_kernel(),
                        grad_module_kernel(), p2p_module_kernel(), reduce_ops_module_kernel()}) {
    cudaFunction_t f = nullptr;
    B200_CHECK_CUDA(cudaGetFuncBySymbol(&f, k));
    CUmodule mod = nullptr;
    B200_CHECK_CU(d.FuncGetModule(&mod, f));
    unsigned int n = 0;
    B200_CHECK_CU(d.ModuleGetFunctionCount(&n, mod));
    std::vector<CUfunction> fns(n);
    B200_CHECK_CU(d.ModuleEnumerateFunctions(fns.data(), n, mod));
    for (CUfunction fn : fns) B200_CHECK_CU(d.FuncLoad(fn));
  }
  done.insert(device);
  return B200_OK;
}

}  // namespace b200

using namespace b200;

b200::DevComm b200_comm::dev() const {
  DevComm d{};
  d.rank = rank;
  d.world = world;
  for (int p = 0; p < kMaxRanks; ++p) {
    d.data[p] = reinterpret_cast<char *>(data.va[p]);
    d.sig[p] = reinterpret_cast<uint32_t *>(sig.va[p]);
    d.inbox[p] = reinterpret_cast<char *>(inbox.va[p]);
    d.ll[p] = reinterpret_cast<char *>(ll.va[p]);
  }
  d.mc_data = mc_active ? reinterpret_cast<char *>(mc_va) : nullptr;
  d.st = d_state;
  d.abort = d_abort;
  d.host_status = d_abort + 1;
  d.timeout_ns = (unsigned long long)(cfg.timeout_ms) * 1000000ull;
  d.inbox_bytes = inbox_bytes;
  d.trace = d_trace;
  d.trace_cap = trace_cap;
  return d;
}

static std::atomic<uint32_t> g_comm_serial{0};
static std::mutex g_pool_mu;
static b200_comm *g_pool_comm = nullptr;
static std::map<size_t, std::vector<void *>> g_pool_free;  // rounded size -> recycled blocks

extern "C" {

int b200_comm_create(int world_size, int rank, int device, const b200_config_t *cfg,
                     b200_comm_t *out) {
  if (!out) {
    set_error("out is null");
    return B200_ERR_INVALID;
  }
  *out = nullptr;
  if (world_size < 1 || world_size > kMaxRanks || rank < 0 || rank >= world_size) {
    set_error("invalid world_size/rank %d/%d (max %d ranks)", world_size, rank, kMaxRanks);
    return B200_ERR_INVALID;
  }
  int ndev = 0;
  B200_CHECK_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) {
    set_error("device %d not visible (%d devices)", device, ndev);
    return B200_ERR_INVALID;
  }
  B200_CHECK_CUDA(cudaSetDevice(device));
  B200_CHECK_CUDA(cudaFree(nullptr));
  Driver &d = driver();
  if (!d.ok) {
    set_error("CUDA driver lacks the virtual memory management API");
    return B200_ERR_UNSUPPORTED;
  }
  const int pre = preload_kernels(device);
  if (pre) return pre;

  b200_comm *c = new b200_comm();
  c->world = world_size;
  c->rank = rank;
  c->device = device;
  if (cfg) c->cfg = *cfg;
  else c->cfg.enable_multicast = 1;
  if (c->cfg.staging_bytes == 0) c->cfg.staging_bytes = size_t(256) << 20;
  if (c->cfg.inbox_bytes == 0) c->cfg.inbox_bytes = size_t(32) << 20;
  // device watchdog: minutes, not seconds -- a rank may legitimately be late by a checkpoint, an
  // evaluation pass or a first-step compile (c10d's default collective timeout is 10-30 minutes)
  if (c->cfg.timeout_ms <= 0) c->cfg.timeout_ms = 600000;

  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    set_error("cudaGetDeviceProperties failed");
    delete c;
    return B200_ERR_CUDA;
  }
  c->sm_count = prop.multiProcessorCount;

  CUmemAllocationProp aprop = alloc_prop(device);
  size_t gran = 0;
  CUresult gr = d.MemGetAllocationGranularity(&gran, &aprop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED);
  if (gr != CUDA_SUCCESS || gran == 0) {
    set_error("cuMemGetAllocationGranularity failed (%d)", int(gr));
    delete c;
    return B200_ERR_CUDA;
  }

  // Multicast capability of this device.
  int mc_attr = 0;
  CUdevice cudev;
  if (d.has_multicast && c->cfg.enable_multicast && world_size > 1 &&
      d.DeviceGet(&cudev, device) == CUDA_SUCCESS &&
      d.DeviceGetAttribute(&mc_attr, CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED, cudev) == CUDA_SUCCESS &&
      mc_attr) {
    c->mc_supported = true;
    CUmulticastObjectProp mp{};
    mp.numDevices = unsigned(world_size);
    mp.size = gran;
    mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    size_t mgran = 0;
    if (d.MulticastGetGranularity(&mgran, &mp, CU_MULTICAST_GRANULARITY_RECOMMENDED) == CUDA_SUCCESS &&
        mgran > gran)
      gran = mgran;
  }

  // staging slots are multiples of 2 MiB so slot 1 and the heap start aligned
  c->staging_bytes = round_up(c->cfg.staging_bytes, size_t(2) << 20);
  c->heap_bytes = round_up(c->cfg.heap_bytes, size_t(2) << 20);
  c->inbox_bytes = round_up(c->cfg.inbox_bytes, size_t(kP2PRings) * kP2PSlots * 4096);

  int rc = region_create(c, &c->data, 2 * c->staging_bytes + c->heap_bytes, gran);
  if (!rc) rc = region_create(c, &c->sig, kSigWords * sizeof(uint32_t), gran);
  if (!rc) rc = region_create(c, &c->inbox, size_t(kMaxRanks) * c->inbox_bytes, gran);
  if (!rc) rc = region_create(c, &c->ll, kLLRegionBytes, gran);
  if (!rc) {
    cudaError_t e = cudaMalloc(&c->d_state, sizeof(LocalState));
    if (e == cudaSuccess) e = cudaMemset(c->d_state, 0, sizeof(LocalState));
    if (e == cudaSuccess) e = cudaHostAlloc(&c->h_abort, 2 * sizeof(int), cudaHostAllocMapped);
    if (e == cudaSuccess) {
      c->h_abort[0] = 0;  // abort request (host -> device)
      c->h_abort[1] = 0;  // status mirror (device -> host)
      e = cudaHostGetDevicePointer(&c->d_abort, c->h_abort, 0);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
      set_error("local state allocation failed: %s", cudaGetErrorString(e));
      rc = B200_ERR_CUDA;
    }
  }
  if (rc) {
    b200_comm_destroy(c);
    return rc;
  }

  // bootstrap endpoint + its secret
  {
    FILE *ur = fopen("/dev/urandom", "rb");
    if (!ur || fread(c->token, 1, 16, ur) != 16) {
      if (ur) fclose(ur);
      set_error("cannot read /dev/urandom for the bootstrap token");
      b200_comm_destroy(c);
      return B200_ERR_SYSTEM;
    }
    fclose(ur);
  }
  char name[96];
  snprintf(name, sizeof(name), "b200coll-%d-%u-r%d", int(getpid()), g_comm_serial.fetch_add(1), rank);
  c->sock_name = name;
  c->listen_fd = socket(AF_UNIX, SOCK_STREAM | SOCK_CLOEXEC, 0);
  sockaddr_un addr;
  socklen_t len;
  make_addr(c->sock_name, &addr, &len);
  if (c->listen_fd < 0 || bind(c->listen_fd, reinterpret_cast<sockaddr *>(&addr), len) != 0 ||
      listen(c->listen_fd, 64) != 0) {
    set_error("cannot create bootstrap socket: %s", strerror(errno));
    b200_comm_destroy(c);
    return B200_ERR_SYSTEM;
  }
  c->server = std::thread(server_loop, c);
  *out = c;
  return B200_OK;
}

int b200_comm_export_handle(b200_comm_t c, void *blob) {
  if (!c || !blob) {
    set_error("null argument");
    return B200_ERR_INVALID;
  }
  Blob b{};
  b.magic = kMagic;
  b.version = kVersion;
  b.pid = int32_t(getpid());
  b.rank = c->rank;
  b.world = c->world;
  b.device = c->device;
  b.mc_supported = c->mc_supported ? 1 : 0;
  cudaDeviceProp prop;
  B200_CHECK_CUDA(cudaGetDeviceProperties(&prop, c->device));
  memcpy(b.uuid, &prop.uuid, 16);
  b.data_bytes = c->data.bytes;
  b.sig_bytes = c->sig.bytes;
  b.inbox_region_bytes = c->inbox.bytes;
  b.staging_bytes = c->staging_bytes;
  b.heap_bytes = c->heap_bytes;
  b.inbox_bytes = c->inbox_bytes;
  snprintf(b.sock, sizeof(b.sock), "%s", c->sock_name.c_str());
  memcpy(b.token, c->token, 16);
  gethostname(b.host, sizeof(b.host) - 1);
  memset(blob, 0, B200_HANDLE_BYTES);
  memcpy(blob, &b, sizeof(b));
  return B200_OK;
}

int b200_comm_connect(b200_comm_t c, const void *blobs) {
  if (!c || !blobs) {
    set_error("null argument");
    return B200_ERR_INVALID;
  }
  if (c->connected) {
    set_error("already connected");
    return B200_ERR_INVALID;
  }
  Driver &d = driver();
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  std::vector<Blob> bs(c->world);
  bool all_mc = c->mc_supported;
  bool distinct = true;
  for (int p = 0; p < c->world; ++p) {
    memcpy(&bs[p], static_cast<const char *>(blobs) + size_t(p) * B200_HANDLE_BYTES, sizeof(Blob));
    const Blob &b = bs[p];
    if (b.magic != kMagic || b.version != kVersion || b.rank != p || b.world != c->world) {
      set_error("handle %d is not a valid rank-%d handle of a %d-rank group", p, p, c->world);
      return B200_ERR_INVALID;
    }
    if (b.data_bytes != c->data.bytes || b.sig_bytes != c->sig.bytes ||
        b.inbox_region_bytes != c->inbox.bytes || b.staging_bytes != c->staging_bytes ||
        b.heap_bytes != c->heap_bytes || b.inbox_bytes != c->inbox_bytes) {
      set_error("rank %d was created with a different memory configuration", p);
      return B200_ERR_INVALID;
    }
    {
      char mine[sizeof(b.host)] = {};
      gethostname(mine, sizeof(mine) - 1);
      if (strncmp(b.host, mine, sizeof(mine)) != 0) {
        set_error("rank %d runs on host '%s', this rank on '%s': a b200 group spans ONE host (<= %d GPUs of one "
                  "NVSwitch domain); use the nccl backend across hosts", p, b.host, mine, kMaxRanks);
        return B200_ERR_UNSUPPORTED;
      }
    }
    all_mc = all_mc && b.mc_supported;
    for (int q = 0; q < p; ++q)
      if (memcmp(bs[q].uuid, b.uuid, 16) == 0) distinct = false;
  }
  c->peer_socks.resize(c->world);
  c->peer_tokens.resize(c->world);
  for (int p = 0; p < c->world; ++p) {
    c->peer_socks[p] = bs[p].sock;
    memcpy(c->peer_tokens[p].data(), bs[p].token, 16);
  }

  // Map every peer's regions.  Ranks that share a physical GPU (several actors on
  // one device, or the single-GPU test harness) map each other the same way.
  for (int off = 1; off < c->world; ++off) {
    int p = (c->rank + off) % c->world;
    if (memcmp(bs[p].uuid, bs[c->rank].uuid, 16) != 0) {
      // locate the peer's device ordinal in this process to verify P2P capability
      int ndev = 0, peer_dev = -1;
      cudaGetDeviceCount(&ndev);
      for (int i = 0; i < ndev; ++i) {
        cudaDeviceProp pr;
        if (cudaGetDeviceProperties(&pr, i) == cudaSuccess && memcmp(&pr.uuid, bs[p].uuid, 16) == 0)
          peer_dev = i;
      }
      if (peer_dev >= 0) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, c->device, peer_dev);
        if (!can) {
          set_error("device %d cannot access peer device %d (rank %d)", c->device, peer_dev, p);
          return B200_ERR_UNSUPPORTED;
        }
      }
    }
    size_t gran = size_t(2) << 20;
    int rc = region_import(c, &c->data, p, FD_DATA, gran);
    if (!rc) rc = region_import(c, &c->sig, p, FD_SIG, gran);
    if (!rc) rc = region_import(c, &c->inbox, p, FD_INBOX, gran);
    if (!rc) rc = region_import(c, &c->ll, p, FD_LL, gran);
    if (rc) return rc;
  }

  // NVLS multicast object over the data region.
  bool want_mc = all_mc && distinct && c->world > 1;
  if (want_mc) {
    bool ok = true;
    c->mc_bytes = c->data.bytes;
    if (c->rank == 0) {
      CUmulticastObjectProp mp{};
      mp.numDevices = unsigned(c->world);
      mp.size = c->mc_bytes;
      mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
      CUresult r = d.MulticastCreate(&c->mc_handle, &mp);
      if (r == CUDA_SUCCESS) {
        int fd = -1;
        r = d.MemExportToShareableHandle(&fd, c->mc_handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0);
        if (r == CUDA_SUCCESS) {
          std::lock_guard<std::mutex> lk(c->mu);
          c->mc_fd = fd;
        }
      }
      ok = (r == CUDA_SUCCESS);
    }
    int agreed = host_agree(c, ok);
    if (agreed < 0) return B200_ERR_SYSTEM;
    if (agreed) {
      CUdevice cudev;
      ok = d.DeviceGet(&cudev, c->device) == CUDA_SUCCESS;
      if (ok && c->rank != 0) {
        int fd = fetch_fd(c, 0, FD_MC);
        ok = fd >= 0 &&
             d.MemImportFromShareableHandle(&c->mc_handle, reinterpret_cast<void *>(intptr_t(fd)),
                                            CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR) == CUDA_SUCCESS;
        if (fd >= 0) close(fd);
      }
      if (ok) ok = d.MulticastAddDevice(c->mc_handle, cudev) == CUDA_SUCCESS;
      agreed = host_agree(c, ok);  // every device must be added before any bind
      if (agreed < 0) return B200_ERR_SYSTEM;
      if (agreed) {
        ok = d.MulticastBindMem(c->mc_handle, 0, c->data.own, 0, c->mc_bytes, 0) == CUDA_SUCCESS;
        if (ok) ok = map_handle(c->device, c->mc_handle, c->mc_bytes, size_t(2) << 20, &c->mc_va) == B200_OK;
        agreed = host_agree(c, ok);
        if (agreed < 0) return B200_ERR_SYSTEM;
        c->mc_active = agreed == 1;
      }
    }
  }

  // Nobody may touch peer memory before every rank finished mapping.
  if (host_agree(c, 1) < 0) return B200_ERR_SYSTEM;
  // Every rank has imported what it needs: stop serving (the fds of the GPU regions are no longer
  // reachable through the socket for the rest of the communicator's life) and drop our own
  // exported descriptors.  The server thread leaves its loop after finishing the iteration that
  // answered the final agreement.
  c->server_stop.store(true);
  {
    std::lock_guard<std::mutex> lk(c->mu);
    for (Region *r : {&c->data, &c->sig, &c->inbox, &c->ll}) {
      if (r->own_fd >= 0) {
        close(r->own_fd);
        r->own_fd = -1;
      }
    }
    if (c->mc_fd >= 0) {
      close(c->mc_fd);
      c->mc_fd = -1;
    }
  }
  c->connected = true;
  return B200_OK;
}

int b200_comm_abort(b200_comm_t c) {
  if (!c) return B200_ERR_INVALID;
  c->aborted.store(true);
  if (c->h_abort) {
    __atomic_store_n(c->h_abort, 1, __ATOMIC_RELEASE);
  }
  return B200_OK;
}

int b200_comm_status(b200_comm_t c) {
  if (!c) return B200_ERR_INVALID;
  if (c->aborted.load()) return B200_ERR_ABORTED;
  if (!c->h_abort) return B200_ERR_INVALID;
  // host-mapped mirror written by the kernel that gave up: no CUDA call on this path
  return __atomic_load_n(&c->h_abort[1], __ATOMIC_ACQUIRE);
}

int b200_comm_destroy(b200_comm_t c) {
  if (!c) return B200_OK;
  Driver &d = driver();
  b200_comm_abort(c);
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();  // kernels leave their waits once the abort word is set
  c->server_stop.store(true);
  if (c->server.joinable()) c->server.join();
  if (c->listen_fd >= 0) {
    close(c->listen_fd);
    c->listen_fd = -1;
  }
  if (c->mc_va) {
    d.MemUnmap(c->mc_va, c->mc_bytes);
    d.MemAddressFree(c->mc_va, c->mc_bytes);
  }
  if (c->mc_handle) {
    if (c->mc_active) {
      CUdevice cudev;
      if (d.DeviceGet(&cudev, c->device) == CUDA_SUCCESS)
        d.MulticastUnbind(c->mc_handle, cudev, 0, c->mc_bytes);
    }
    d.MemRelease(c->mc_handle);
  }
  if (c->mc_fd >= 0) close(c->mc_fd);
  region_destroy(c, &c->data);
  region_destroy(c, &c->sig);
  region_destroy(c, &c->inbox);
  region_destroy(c, &c->ll);
  if (c->d_state) cudaFree(c->d_state);
  if (c->h_abort) cudaFreeHost(c->h_abort);
  if (c->d_trace) cudaFree(c->d_trace);
  (void)cudaGetLastError();
  {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    if (g_pool_comm == c) {
      g_pool_comm = nullptr;
      g_pool_free.clear();
    }
  }
  delete c;
  return B200_OK;
}

int b200_comm_rank(b200_comm_t c) { return c ? c->rank : B200_ERR_INVALID; }
int b200_comm_world_size(b200_comm_t c) { return c ? c->world : B200_ERR_INVALID; }
int b200_comm_has_multicast(b200_comm_t c) { return c && c->mc_active ? 1 : 0; }

int b200_symm_alloc(b200_comm_t c, size_t nbytes, void **out) {
  int rc = check_usable(c);
  if (rc) return rc;
  if (!out) {
    set_error("out is null");
    return B200_ERR_INVALID;
  }
  size_t need = round_up(nbytes ? nbytes : 1, 256);
  if (c->heap_used + need > c->heap_bytes) {
    set_error("symmetric heap exhausted: %zu used + %zu requested > %zu", c->heap_used, need,
              c->heap_bytes);
    return B200_ERR_TOO_LARGE;
  }
  *out = reinterpret_cast<char *>(c->data.va[c->rank]) + 2 * c->staging_bytes + c->heap_used;
  c->heap_used += need;
  return B200_OK;
}

int b200_symm_reset(b200_comm_t c) {
  int rc = check_usable(c);
  if (rc) return rc;
  c->heap_used = 0;
  return B200_OK;
}

int b200_symm_contains(b200_comm_t c, const void *ptr, size_t nbytes) {
  if (!c || !c->heap_bytes) return 0;
  const char *base = reinterpret_cast<const char *>(c->data.va[c->rank]) + 2 * c->staging_bytes;
  const char *p = static_cast<const char *>(ptr);
  return p >= base && p + nbytes <= base + c->heap_bytes;
}

// ---- torch pluggable-allocator bridge ---------------------------------------------------

int b200_pool_bind(b200_comm_t c) {
  std::lock_guard<std::mutex> lk(g_pool_mu);
  if (c) {
    int rc = check_usable(c);
    if (rc) return rc;
    if (c->heap_bytes == 0) {
      set_error("communicator was created without a symmetric heap (heap_bytes = 0)");
      return B200_ERR_INVALID;
    }
  }
  g_pool_comm = c;
  g_pool_free.clear();
  return B200_OK;
}

void *b200_pool_alloc(size_t size, int device, void *stream) {
  (void)stream;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  b200_comm *c = g_pool_comm;
  if (!c || c->device != device) return nullptr;
  const size_t need = round_up(size ? size : 1, 512);
  auto it = g_pool_free.find(need);
  if (it != g_pool_free.end() && !it->second.empty()) {
    void *p = it->second.back();
    it->second.pop_back();
    return p;
  }
  void *out = nullptr;
  if (b200_symm_alloc(c, need, &out) != B200_OK) return nullptr;
  return out;
}

void b200_pool_free(void *ptr, size_t size, int device, void *stream) {
  (void)device;
  (void)stream;
  std::lock_guard<std::mutex> lk(g_pool_mu);
  if (!g_pool_comm || !ptr) return;
  g_pool_free[round_up(size ? size : 1, 512)].push_back(ptr);
}

const char *b200_last_error(void) { return g_err; }
const char *b200_version(void) { return "b200_collective 0.3 (sm_100a)"; }

size_t b200_dtype_size(int dtype) {
  switch (dtype) {
    case B200_U8:
    case B200_I8: return 1;
    case B200_F16:
    case B200_BF16: return 2;
    case B200_I32:
    case B200_U32:
    case B200_F32: return 4;
    case B200_I64:
    case B200_U64:
    case B200_F64: return 8;
    default: return 0;
  }
}

uint64_t b200_comm_launch_count(b200_comm_t c) { return c ? c->launches.load() : 0; }

int b200_comm_set_blocks(b200_comm_t c, int nblocks) {
  if (!c || nblocks < 0 || nblocks > kMaxBlocks) {
    set_error("nblocks must be in [0, %d]", kMaxBlocks);
    return B200_ERR_INVALID;
  }
  c->forced_blocks = nblocks;
  return B200_OK;
}

int b200_comm_trace_enable(b200_comm_t c, unsigned int capacity) {
  if (!c) return B200_ERR_INVALID;
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  if (c->d_trace) {
    B200_CHECK_CUDA(cudaDeviceSynchronize());
    B200_CHECK_CUDA(cudaFree(c->d_trace));
    c->d_trace = nullptr;
    c->trace_cap = 0;
  }
  if (capacity == 0) return B200_OK;
  const size_t bytes = (2 + 2 * size_t(capacity)) * sizeof(unsigned long long);
  B200_CHECK_CUDA(cudaMalloc(&c->d_trace, bytes));
  B200_CHECK_CUDA(cudaMemset(c->d_trace, 0, bytes));
  c->trace_cap = capacity;
  return B200_OK;
}

int b200_comm_trace_read(b200_comm_t c, unsigned long long *out, unsigned int max_events, int reset) {
  if (!c || !out) return B200_ERR_INVALID;
  if (!c->d_trace) return 0;
  B200_CHECK_CUDA(cudaSetDevice(c->device));
  B200_CHECK_CUDA(cudaDeviceSynchronize());
  unsigned long long n = 0;
  B200_CHECK_CUDA(cudaMemcpy(&n, c->d_trace, sizeof(n), cudaMemcpyDeviceToHost));
  if (n > c->trace_cap) n = c->trace_cap;
  if (n > max_events) n = max_events;
  if (n) B200_CHECK_CUDA(cudaMemcpy(out, c->d_trace + 2, n * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (reset) B200_CHECK_CUDA(cudaMemset(c->d_trace, 0, 2 * sizeof(unsigned long long)));
  return int(n);
}

int b200_comm_set_param(b200_comm_t c, int param, long long value) {
  if (!c || param < 0 || param >= B200_PARAM_COUNT) {
    set_error("unknown parameter %d", param);
    return B200_ERR_INVALID;
  }
  if (param == B200_PARAM_PIPE_VARIANT && value != -1 && value != PIPE_NVLS && value != PIPE_PEER && value != PIPE_PULL) {
    set_error("B200_PARAM_PIPE_VARIANT must be -1, %d (NVLS), %d (peer) or %d (pull), got %lld", PIPE_NVLS, PIPE_PEER,
              PIPE_PULL, value);
    return B200_ERR_INVALID;
  }
  c->params[param] = value;
  return B200_OK;
}

}  // extern "C"
