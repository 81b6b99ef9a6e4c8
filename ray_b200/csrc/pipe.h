// pipe.h — host-side interface of the chunk-pipelined all-reduce kernels (allreduce_pipe.cu).
#pragma once
#include "kernel_utils.cuh"

namespace b200 {

// values of B200_PARAM_PIPE_VARIANT
enum PipeVariant {
  PIPE_NVLS = 1,  // copy-in | multimem.ld_reduce + multimem.st | copy-out
  PIPE_PEER = 2,  // copy-in | peer loads + peer stores         | copy-out
  PIPE_PULL = 3   // n == 2: copy-in | bulk-load the peer's slot + reduce into the caller's tensor
};

// chunk size C of the pipeline (B200_PARAM_PIPE_CHUNK_BYTES; default 1 MiB at 2 ranks, 4 MiB at
// <= 4, 8 MiB above); 0 when the staging slot is too small for the pipeline
size_t pipe_chunk_bytes(const b200_comm *c);
// largest message one launch can take (a multiple of C)
size_t pipe_max_bytes(const b200_comm *c, int variant);
// `in`/`out` 16-byte aligned, nbytes a multiple of 16 and <= pipe_max_bytes()
int launch_allreduce_pipe_dyn(b200_comm *c, const char *in, char *out, size_t nbytes, int dtype, int op,
                              int variant, cudaStream_t stream);

// pull all-gather (copy-in | bulk-pull from every peer's slot); same operand requirements
int launch_allgather_pull(b200_comm *c, const char *in, char *const *outs, size_t nbytes, cudaStream_t stream);
// cudaFuncAttributeMaxDynamicSharedMemorySize = bulk-copy ring, once per (device, kernel)
int set_dyn_smem(int device, const void *fn);

}  // namespace b200
