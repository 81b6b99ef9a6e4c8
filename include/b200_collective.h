/*
 * b200_collective.h — C ABI of libb200_collective.so
 *
 * Blackwell-native (sm_100a) replacement for the device-side work that Ray's
 * GPU collective / tensor-transport hot path delegates to libnccl.  Every entry
 * point takes plain pointers, sizes and a raw cudaStream_t: no torch, cupy or
 * Ray types cross this boundary.  All functions return 0 on success or a
 * negative b200_status_t; b200_last_error() returns a per-thread message.
 *
 * Each function cites the reference call site it replaces
 * (paths relative to the reference tree, python/ray/...).
 *
 * Threading: a communicator may be used from any host thread, one call at a
 * time (the reference guards only its group map, util/collective/collective.py:136-138).
 * b200_comm_abort() and b200_comm_status() are safe from any thread at any time.
 *
 * Stream semantics: every collective is enqueued on the caller's stream and
 * returns without host synchronisation (util/collective/collective_group/
 * nccl_collective_group.py:591-639 enqueues and returns as well).  Collectives of
 * one communicator must be stream-ordered with respect to each other.
 */
#ifndef B200_COLLECTIVE_H_
#define B200_COLLECTIVE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_MAX_RANKS 8      /* one NVSwitch domain of a single HGX B200 host */
#define B200_HANDLE_BYTES 256 /* size of the opaque bootstrap blob */

typedef struct b200_comm *b200_comm_t;

typedef enum {
  B200_OK = 0,
  B200_ERR_INVALID = -1,      /* bad argument (maps to ValueError / RuntimeError in Python) */
  B200_ERR_CUDA = -2,         /* a CUDA runtime / driver call failed */
  B200_ERR_SYSTEM = -3,       /* socket / fd passing failure during bootstrap */
  B200_ERR_UNSUPPORTED = -4,  /* dtype/op combination or feature not available */
  B200_ERR_ABORTED = -5,      /* b200_comm_abort() was called (maps to RayChannelError) */
  B200_ERR_TIMEOUT = -6,      /* a device-side wait exceeded the watchdog */
  B200_ERR_TOO_LARGE = -7     /* message does not fit the staging / inbox configuration */
} b200_status_t;

/* Element types.  Mirrors the dtypes the reference maps onto ncclDataType_t
 * (util/collective/collective_group/nccl_util.py:30-71; torch.bool travels as int8). */
typedef enum {
  B200_U8 = 0,
  B200_I8 = 1,
  B200_I32 = 2,
  B200_U32 = 3,
  B200_I64 = 4,
  B200_U64 = 5,
  B200_F16 = 6,
  B200_BF16 = 7,
  B200_F32 = 8,
  B200_F64 = 9,
  B200_DTYPE_COUNT = 10
} b200_dtype_t;

/* Reduction operators.  Numbering follows ray.util.collective.types.ReduceOp
 * (util/collective/types.py:55-59: SUM0 PRODUCT1 MIN2 MAX3); AVG is the extra
 * value the Compiled-Graph enum carries (experimental/util/types.py:11-17).  The
 * Python layer translates the cgraph numbering (MAX2 MIN3 AVG4) to this one. */
typedef enum {
  B200_SUM = 0,
  B200_PROD = 1,
  B200_MIN = 2,
  B200_MAX = 3,
  B200_AVG = 4,
  B200_OP_COUNT = 5
} b200_op_t;

/* Algorithm selector for b200_allreduce (B200_ALGO_AUTO picks by size / dtype / op). */
typedef enum {
  B200_ALGO_AUTO = 0,
  B200_ALGO_ONESHOT = 1,  /* every rank reads all peers' staged inputs (latency path) */
  B200_ALGO_TWOSHOT = 2,  /* owner reduces its stripe from peer HBM, pushes result to all peers */
  B200_ALGO_NVLS = 3,     /* multimem.ld_reduce + multimem.st through the NVSwitch */
  B200_ALGO_LL = 4,       /* flag-in-data push, no barrier (<= 64 KiB) */
  B200_ALGO_PIPE = 5      /* chunk-pipelined: TMA copy-in | reduce | TMA copy-out roles in one launch
                             (n == 2: TMA copy-in | bulk-load the peer's slot and reduce into the output) */
} b200_algo_t;

typedef struct {
  size_t staging_bytes; /* per-slot staging size; two slots are allocated (0 -> default 256 MiB) */
  size_t heap_bytes;    /* symmetric user heap for zero-copy operands (0 -> none) */
  size_t inbox_bytes;   /* per-peer point-to-point inbox (0 -> default 32 MiB) */
  int enable_multicast; /* 1: try to create the NVLS multicast mapping, 0: never */
  int timeout_ms;       /* device-side watchdog for peer waits (0 -> default 600000 = 10 min) */
} b200_config_t;

/* ---- lifecycle / bootstrap ------------------------------------------------
 * Replaces NCCLGroup._get_nccl_collective_communicator + Rendezvous
 * (util/collective/collective_group/nccl_collective_group.py:36-125,414-468) and
 * _NcclGroup.__init__ (experimental/channel/nccl_group.py:29-114): instead of an
 * ncclUniqueId, every rank publishes one opaque B200_HANDLE_BYTES blob through
 * Ray's store (named actor / GCS KV / __ray_call__), then maps its peers.  */

/* Allocate this rank's symmetric memory on `device`, start the fd-passing
 * endpoint.  `cfg` may be NULL for defaults. */
int b200_comm_create(int world_size, int rank, int device, const b200_config_t *cfg,
                     b200_comm_t *out);

/* Fill `blob` (B200_HANDLE_BYTES) with this rank's bootstrap handle. */
int b200_comm_export_handle(b200_comm_t comm, void *blob);

/* `blobs` = world_size consecutive handles in rank order.  Maps every peer's
 * buffers, sets up the multicast mapping when available.  Collective: blocks
 * until all ranks called it. */
int b200_comm_connect(b200_comm_t comm, const void *blobs);

/* Replaces _NcclGroup.destroy (nccl_group.py:347-365) / NCCLGroup.destroy_group
 * (nccl_collective_group.py:161-185).  Implies abort. */
int b200_comm_destroy(b200_comm_t comm);

/* Unblocks every device-side wait of this communicator (ncclCommAbort stand-in,
 * nccl_group.py:360-364).  Sticky: later calls fail with B200_ERR_ABORTED. */
int b200_comm_abort(b200_comm_t comm);

/* 0 while healthy; B200_ERR_ABORTED / B200_ERR_TIMEOUT once a kernel gave up.
 * Reading it is only meaningful after the stream was synchronised. */
int b200_comm_status(b200_comm_t comm);

int b200_comm_rank(b200_comm_t comm);
int b200_comm_world_size(b200_comm_t comm);
/* 1 when the NVLS multicast mapping is active. */
int b200_comm_has_multicast(b200_comm_t comm);

/* Symmetric user heap: collective bump allocation (all ranks must issue the
 * same sequence).  Tensors placed here are reduced in place with no staging
 * copies.  `*out` is a device pointer valid on this rank. */
int b200_symm_alloc(b200_comm_t comm, size_t nbytes, void **out);
/* Resets the bump pointer (collective). */
int b200_symm_reset(b200_comm_t comm);
/* 1 if [ptr, ptr+nbytes) lies inside this rank's symmetric heap. */
int b200_symm_contains(b200_comm_t comm, const void *ptr, size_t nbytes);

/* torch.cuda.memory.CUDAPluggableAllocator entry points: after b200_pool_bind(comm) every
 * allocation torch routes through them comes from comm's symmetric heap, so ordinary
 * torch tensors created under `torch.cuda.use_mem_pool(...)` are zero-copy operands
 * (the counterpart of ncclMemAlloc + buffer registration).  All ranks must allocate the
 * same sequence of sizes.  Blocks are recycled through size-keyed free lists. */
int b200_pool_bind(b200_comm_t comm);
void *b200_pool_alloc(size_t size, int device, void *stream);
void b200_pool_free(void *ptr, size_t size, int device, void *stream);

/* ---- collectives ------------------------------------------------------------ */

/* out[i] = op over ranks of in[i]; in == out allowed (in place).
 * Replaces ncclAllReduce at nccl_collective_group.py:200-207 and nccl_group.py:293-312. */
int b200_allreduce(b200_comm_t comm, const void *in, void *out, size_t count,
                   int dtype, int op, int algo, void *stream);

/* outs[p] (p < world_size) receives rank p's `in` (count elements each).
 * Writes straight into the caller's n output tensors: replaces ncclAllGather plus
 * the flat scratch buffer and n device copies at nccl_collective_group.py:283-319,
 * 685-726; with outs[p] = base + p*count*elsize it is nccl_group.py:274-291. */
int b200_allgather(b200_comm_t comm, const void *in, void *const *outs, size_t count,
                   int dtype, void *stream);

/* out = op over ranks q of (rank q's ins[this rank]).  Reads the caller's n input
 * tensors directly: replaces the n device copies + ncclReduceScatter at
 * nccl_collective_group.py:321-360 and nccl_group.py:314-333. */
int b200_reducescatter(b200_comm_t comm, const void *const *ins, void *out, size_t count,
                       int dtype, int op, void *stream);

/* In-place copy of root's buffer to every rank.  Replaces ncclBroadcast at
 * nccl_collective_group.py:257-281. */
int b200_broadcast(b200_comm_t comm, void *buf, size_t count, int dtype, int root,
                   void *stream);

/* Only root's buffer is modified.  Replaces ncclReduce at nccl_collective_group.py:231-255. */
int b200_reduce(b200_comm_t comm, void *buf, size_t count, int dtype, int op, int root,
                void *stream);

/* Flag-only device barrier (the reference all-reduces a 1-element array,
 * nccl_collective_group.py:211-229). */
int b200_barrier(b200_comm_t comm, void *stream);

/* Point-to-point.  Replaces ncclSend / ncclRecv at nccl_collective_group.py:362-412,
 * 641-682 and nccl_group.py:149-241.  Eager up to the inbox size. */
int b200_send(b200_comm_t comm, const void *buf, size_t nbytes, int peer, void *stream);
int b200_recv(b200_comm_t comm, void *buf, size_t nbytes, int peer, void *stream);

/* One-sided get (RDT's one-sided transport, experimental/rdt/cuda_ipc_transport.py:57-186, without
 * its same-GPU restriction): copies [src_heap_offset, +nbytes) of rank `src_rank`'s symmetric heap
 * into `dst` with a kernel that runs on THIS rank only.  The caller orders it after the owner's
 * writes (an interprocess event in the RDT transport).  b200_symm_base returns this rank's heap
 * base and size, so that an address inside it can be turned into the offset a peer passes here. */
int b200_symm_base(b200_comm_t comm, void **base, size_t *bytes);
int b200_get(b200_comm_t comm, void *dst, int src_rank, size_t src_heap_offset, size_t nbytes, void *stream);

/* Fused data-parallel gradient synchronisation (SURVEY K8): for a flat fp32
 * bucket computes grad[i] = sum_r wire(grad_r[i] * scale) in one launch, where
 * wire() is a cast to `wire_dtype` (B200_BF16 / B200_F16 compress the NVLink
 * traffic; B200_F32 keeps DDP's exact arithmetic).  Replaces the c10d reducer's
 * div + ncclAllReduce (+ bf16_compress_hook casts) reached from
 * train/torch/config.py:144 and train/torch/train_loop_utils.py:456-480. */
int b200_grad_allreduce(b200_comm_t comm, float *grad, size_t count, float scale,
                        int wire_dtype, void *stream);

/* Multi-tensor all-reduce (SURVEY K9): reduces `ntensors` same-dtype tensors as one
 * message without a host-side flatten (replaces parameters_to_vector + views at
 * dag/collective_node.py:220-232).  ptrs/counts are host arrays. */
int b200_allreduce_multi(b200_comm_t comm, void *const *ptrs, const size_t *counts,
                         int ntensors, int dtype, int op, void *stream);

/* ---- introspection ---------------------------------------------------------- */
const char *b200_last_error(void);
const char *b200_version(void);
size_t b200_dtype_size(int dtype);
/* Number of device kernels this library launched on behalf of `comm` so far. */
uint64_t b200_comm_launch_count(b200_comm_t comm);
/* Tuning knob: force the CTA count used by collectives (0 = automatic). */
int b200_comm_set_blocks(b200_comm_t comm, int nblocks);

/* In-kernel event trace (profiling aid, off by default): allocates room for `capacity` events
 * (0 frees it); instrumented kernels then record (globaltimer ns, CTA, event id, argument).
 * b200_comm_trace_read synchronises the device, copies up to max_events events (2 x u64 each:
 * ns, blockIdx << 40 | event << 32 | argument) and returns how many; `reset` != 0 clears it. */
int b200_comm_trace_enable(b200_comm_t comm, unsigned int capacity);
int b200_comm_trace_read(b200_comm_t comm, unsigned long long *out, unsigned int max_events, int reset);

/* Host-side self-test (no GPU needed) of the work decomposition of the pipelined kernels: runs the
 * very inline functions the kernels use and checks that copy shares tile the message, that the
 * expected arrival counts match, that reduce work items tile every chunk exactly once and that
 * ring positions are respected.  0 = consistent; otherwise b200_last_error() says what broke. */
int b200_selftest_pipe_geometry(size_t nbytes, size_t chunk_bytes, int copy_ctas, int world, int red_ctas,
                                unsigned ring_chunks);

/* Tuning parameters (must be set identically on every rank; -1 restores the default). */
typedef enum {
  B200_PARAM_ONESHOT_MAX_BYTES = 0, /* all-reduce messages up to this size use the one-shot kernel */
  B200_PARAM_NVLS_MIN_WORLD = 1,    /* AUTO uses the NVLS kernels from this world size on (default 3) */
  B200_PARAM_NVLS_CTAS = 2,         /* CTAs of the NVSwitch reduce phase: zero-copy default 64, staged default all */
  B200_PARAM_LL_MAX_BYTES = 3,      /* all-reduce messages up to this size use the LL kernel (default 32 KiB / 2 ranks ... 4 KiB / 8 ranks) */
  B200_PARAM_PIPE_MIN_BYTES = 4,    /* AUTO uses the pipelined kernels from this size on (ordinary, 16-byte aligned tensors) */
  B200_PARAM_PIPE_CHUNK_BYTES = 5,  /* pipeline chunk size, rounded up to 1 MiB multiples (all-reduce default 1 MiB at 2 ranks, 4 MiB at <= 4, 8 MiB above; pull all-gather 1 MiB) */
  B200_PARAM_PIPE_COPY_CTAS = 6,    /* CTAs per TMA copy role (power of two; default 32 for the 2-rank pull all-reduce, 16 otherwise) */
  B200_PARAM_PIPE_RED_CTAS = 7,     /* CTAs of the reduce / pull role (all-reduce default 32 for the 2-rank pull kernel, 64 at <= 4 ranks, 32 above; pull all-gather 64 at 2 ranks, 48 at <= 4, 32 above) */
  B200_PARAM_PIPE_VARIANT = 8,      /* B200_ALGO_PIPE only: force 1 = NVLS roles, 2 = peer ld/st roles, 3 = pull (2 ranks); other values are rejected */
  B200_PARAM_P2P_BULK_MIN_CHUNK = 9, /* send/recv: chunks from this size on move with the TMA bulk-copy kernel (0 = never; default 32 KiB) */
  B200_PARAM_AG_PULL_MIN_BYTES = 10, /* all-gather: per-rank size from which the pull kernel is used (0 = never; default 4 MiB) */
  B200_PARAM_COUNT = 11
} b200_param_t;
int b200_comm_set_param(b200_comm_t comm, int param, long long value);

#ifdef __cplusplus
}
#endif
#endif /* B200_COLLECTIVE_H_ */
