// mpi4jax_b200 -- host-side runtime objects and the C ABI.
//
// B2Seg   : one symmetric-memory segment (same size on every rank), backed by
//           the CUDA VMM API (cuMemCreate + POSIX fd export) or, as a fallback,
//           by cudaMalloc + cudaIpc handles.  Peers' segments are mapped into
//           this process' address space; file descriptors / IPC handles are
//           exchanged by the Python control plane (unix sockets / gloo).
// B2Mc    : an NVLS multicast object bound to a segment on every rank
//           (multimem.ld_reduce / multimem.st address space).
// B2Comm  : a communicator: rank/size, control segment (flags, p2p rings, LL
//           buffers, halo buffers), growable staging segment, local counters.
//
// This is the B200-native counterpart of the reference's native bridge layer
// (mpi4jax/_src/xla_bridge/mpi_xla_bridge_cuda.cpp + mpi_ops_common.h); the
// reference hands device pointers to a CUDA-aware MPI, we own the transport.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include "b2_common.h"

struct B2Seg {
  int mode;                 // 0 = VMM, 1 = cudaIpc
  int device;
  int nranks;
  int rank;
  size_t bytes;             // rounded-up size
  CUmemGenericAllocationHandle handle;      // local physical allocation (VMM)
  CUmemGenericAllocationHandle peer_handle[B2_MAX_RANKS];
  void* ptr[B2_MAX_RANKS];  // mapped address of every rank's segment (ptr[rank] = local)
  int export_fd;
};

struct B2Mc {
  CUmemGenericAllocationHandle handle;
  size_t bytes;
  int device;
  void* ptr;                // mapped multicast VA
  int export_fd;
  int bound;
};

struct B2Comm {
  B2DevComm dev;
  int device;
  int sm_count;
  B2Seg* ctl;
  B2Seg* stage;
  B2Mc* stage_mc;
  // algorithm thresholds (bytes); tunable from Python (measured table)
  size_t ll_max;
  size_t oneshot_max;
  size_t nvls_min;
  size_t bcast_mc_min;          // bcast: root multimem.st from this size on
  int nvls_pipeline;            // software-pipelined NVLS allreduce (default on)
  unsigned long long* trace;    // device buffer for the phase timeline of CTA 0 (scripts/allreduce_phases.py)
  int trace_cap;
  int max_blocks;
  B2ErrorRecord* err_host;      // host pointer of the mapped error record
  int launches;                 // kernels launched through this communicator
};

#ifdef __cplusplus
extern "C" {
#endif

// --- library / logging -------------------------------------------------------
const char* b2_version(void);
const char* b2_last_error(void);
void b2_set_logging(int enable);
int b2_get_logging(void);
typedef void (*b2_print_fn)(const char*);
void b2_set_print_callback(b2_print_fn fn);
int b2_launch_count(void);

// --- device / driver ---------------------------------------------------------
int b2_init(int device);
int b2_multicast_supported(int device);
int b2_vmm_supported(int device);
size_t b2_granularity(int device, int for_multicast);

// --- segments ----------------------------------------------------------------
B2Seg* b2_seg_create(int device, int rank, int nranks, size_t bytes, int mode);
int b2_seg_export_fd(B2Seg* s);                       // VMM: fd to send to peers
int b2_seg_import_fd(B2Seg* s, int peer, int fd);     // VMM: map a peer's allocation
int b2_seg_ipc_handle(B2Seg* s, void* out64);         // IPC: 64-byte handle
int b2_seg_import_ipc(B2Seg* s, int peer, const void* handle64);
void* b2_seg_ptr(B2Seg* s, int peer);
size_t b2_seg_bytes(B2Seg* s);
int b2_seg_destroy(B2Seg* s);

// --- multicast ---------------------------------------------------------------
B2Mc* b2_mc_create(int device, int nranks, size_t bytes);      // rank 0
int b2_mc_export_fd(B2Mc* m);
B2Mc* b2_mc_import(int device, int fd, size_t bytes);           // other ranks
int b2_mc_add_device(B2Mc* m);
int b2_mc_bind(B2Mc* m, B2Seg* s);
void* b2_mc_ptr(B2Mc* m);
int b2_mc_destroy(B2Mc* m);

// --- communicator ------------------------------------------------------------
size_t b2_layout_bytes(int nranks, size_t slot_bytes, size_t ll_cap, size_t halo_cap);
B2Comm* b2_comm_create(int device, int rank, int nranks, B2Seg* ctl, size_t slot_bytes,
                       size_t ll_cap, size_t halo_cap, double timeout_s);
int b2_comm_set_stage(B2Comm* c, B2Seg* stage, B2Mc* mc);
size_t b2_comm_stage_half(B2Comm* c);
int b2_comm_set_tuning(B2Comm* c, long long ll_max, long long oneshot_max, long long nvls_min,
                       int max_blocks);
int b2_comm_set_option(B2Comm* c, const char* key, long long value);
long long b2_comm_get_option(B2Comm* c, const char* key);   // "bcast_mc_min", "nvls_pipeline"
int b2_comm_check_error(B2Comm* c, char* buf, int buflen);     // 0 = ok
int b2_comm_destroy(B2Comm* c);
size_t b2_stage_need(int opcode, int nranks, size_t blk_bytes); // staging half needed by an op

// Layout of a non-contiguous input (elements, innermost dimension last); nd == 0: contiguous.
// Dimension 0 of an alltoall / scatter input (the per-peer blocks) is described separately.
struct B2Strided {
  int nd;
  int esize;                 // element size in bytes: 1, 2, 4, 8 or 16
  long long shape[4];
  long long stride[4];       // in elements
  long long blk_stride;      // elements between consecutive blocks
};

// --- collectives (all enqueue on `stream`, never synchronise the host) --------
int b2_barrier(B2Comm* c, cudaStream_t stream);
int b2_allreduce(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op, int algo,
                 cudaStream_t stream);
int b2_allreduce_sym(B2Comm* c, void* mc, size_t count, int dtype, cudaStream_t stream);
int b2_reduce(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op, int root,
              cudaStream_t stream);
int b2_scan(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
            cudaStream_t stream);
// MPI_Reduce_scatter_block: `in` holds size blocks of `count` elements, rank r receives the reduction of
// block r over all ranks in `out` (`count` elements)
int b2_reduce_scatter(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op, int algo,
                      cudaStream_t stream);
// `lay` (may be null = contiguous) describes a strided input; the pack is fused into the staging copy
int b2_allgather(B2Comm* c, const void* in, void* out, size_t blk_bytes, const B2Strided* lay,
                 cudaStream_t stream);
int b2_alltoall(B2Comm* c, const void* in, void* out, size_t blk_bytes, const B2Strided* lay,
                cudaStream_t stream);
int b2_bcast(B2Comm* c, const void* in, void* out, size_t nbytes, int root, const B2Strided* lay,
             cudaStream_t stream);
int b2_gather(B2Comm* c, const void* in, void* out, size_t blk_bytes, int root, const B2Strided* lay,
              cudaStream_t stream);
int b2_scatter(B2Comm* c, const void* in, void* out, size_t blk_bytes, int root, const B2Strided* lay,
               cudaStream_t stream);

// --- point to point ----------------------------------------------------------
// source/tag may be -1 (ANY).  `status` is a host-mapped B2StatusRecord or null.
B2StatusRecord* b2_status_alloc(void);
void b2_status_free(B2StatusRecord* s);
int b2_send(B2Comm* c, const void* buf, size_t nbytes, int dest, int tag, cudaStream_t stream);
int b2_recv(B2Comm* c, void* buf, size_t nbytes, int source, int tag, B2StatusRecord* status,
            cudaStream_t stream);
int b2_sendrecv(B2Comm* c, const void* sendbuf, size_t send_bytes, int dest, int sendtag,
                void* recvbuf, size_t recv_bytes, int source, int recvtag, B2StatusRecord* status,
                cudaStream_t stream);

// --- tensor-parallel linear: tcgen05 GEMM + in-switch allreduce in one kernel (b2_gemm.cu) ---
int b2_gemm_allreduce(B2Comm* c, const void* A, const void* B, void* out, int M, int N, int K,
                      cudaStream_t stream);

// --- fused halo exchange + shallow-water stencils (see b2_halo.cu, b2_swe.cu) --
struct B2HaloDesc {
  int nfields;
  float* field[B2_HALO_MAX_FIELDS];   // (ny, nx) row-major fp32 arrays with a 1-cell halo
  int kind[B2_HALO_MAX_FIELDS];       // 0 = "h", 1 = "u", 2 = "v"  (wall conditions)
  int ny, nx;
  int pitch;                          // row pitch in floats (>= nx)
  int west, east, south, north;       // neighbour ranks, -1 = wall
  int sw, se, nw, ne;                 // diagonal neighbours (-1 where south/north is a wall)
  int periodic_x;
  int at_east_wall;                   // last column of processes (u wall, non-periodic only)
  int at_north_wall;                  // last row of processes (v wall)
};
int b2_halo_exchange(B2Comm* c, const B2HaloDesc* d, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
