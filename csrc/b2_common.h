// mpi4jax_b200 native core -- shared host/device definitions.
//
// The native core is frontend-agnostic: every entry point takes raw device
// pointers, element counts, a dtype/op code, a communicator handle and a
// cudaStream_t.  The PyTorch frontend binds it through ctypes
// (mpi4jax_b200/_src/native/__init__.py); an XLA-FFI shim could bind the same
// C ABI.
//
// Role in the parity map: this header plus b2_runtime.cpp / b2_logging.cpp
// replace the reference's shared bridge header
// (mpi4jax/_src/xla_bridge/mpi_ops_common.h:1-457): error/abort path, logging
// switch, debug timer, handle plumbing.  Nothing here is derived from that
// file's code; the transport is peer-mapped HBM over NVLink instead of MPI.
#pragma once

#include <cstddef>
#include <cstdint>

#define B2_ABI_VERSION 11   // bump whenever a struct shared with Python or a C signature changes
#define B2_MAX_RANKS 16          // ranks per NVLink domain we support (8 on HGX B200)
#define B2_MAX_BLOCKS 1024       // max CTAs per collective launch (flag rows)
#define B2_P2P_NSLOT 8           // ring slots per directed pair
#define B2_P2P_MAX_LANES 64      // CTAs cooperating on one p2p message
#define B2_P2P_LL_MAX 8192       // payload bytes up to which a p2p message travels flag-in-data
#define B2_HALO_MAX_FIELDS 8

// ---- dtype / op codes (must match mpi4jax_b200/_src/native/codes.py) -------
enum B2DType : int {
  B2_F32 = 0, B2_F64 = 1, B2_F16 = 2, B2_BF16 = 3,
  B2_I8 = 4, B2_I16 = 5, B2_I32 = 6, B2_I64 = 7,
  B2_U8 = 8, B2_U16 = 9, B2_U32 = 10, B2_U64 = 11,
  B2_BOOL = 12, B2_C64 = 13, B2_C128 = 14,
  B2_DTYPE_COUNT = 15
};

enum B2Op : int {
  B2_SUM = 0, B2_PROD = 1, B2_MIN = 2, B2_MAX = 3,
  B2_LAND = 4, B2_LOR = 5, B2_LXOR = 6,
  B2_BAND = 7, B2_BOR = 8, B2_BXOR = 9,
  B2_OP_COUNT = 10
};

// allreduce algorithm selector (B2_ALGO_AUTO = measured size table)
enum B2Algo : int {
  B2_ALGO_AUTO = 0,
  B2_ALGO_LL = 1,        // flag-in-data push, no barrier            (latency path)
  B2_ALGO_ONESHOT = 2,   // stage -> barrier -> pull all peers       (small / P=2)
  B2_ALGO_TWOSHOT = 3,   // stage -> RS by pull -> AG by push        (mid / large)
  B2_ALGO_NVLS = 4       // stage -> multimem.ld_reduce + multimem.st (large, in-switch)
};

// error codes written by kernels into the host-mapped error record
enum B2Err : int {
  B2_OK = 0,
  B2_ERR_TIMEOUT = 1,        // device-side spin wait exceeded the watchdog
  B2_ERR_TAG_MISMATCH = 2,   // p2p: next message in the pair FIFO has another tag
  B2_ERR_TRUNCATE = 3,       // p2p: message size differs from the receive buffer
  B2_ERR_BAD_ARG = 4
};

// Written by the device (host-mapped pinned memory) right before __trap().
struct B2ErrorRecord {
  volatile int code;
  volatile int rank;
  volatile int opcode;      // B2OpCode of the kernel that failed
  volatile int peer;
  volatile unsigned expected;
  volatile unsigned observed;
  volatile int block;
  volatile int aux;
};

// p2p receive status, one record per Status object (host-mapped pinned memory)
struct B2StatusRecord {
  volatile int source;
  volatile int tag;
  volatile long long count_bytes;
  volatile int error;
  volatile int ready;       // written last; host checks after stream sync
};

// identifies the kernel family for diagnostics / debug log lines
enum B2OpCode : int {
  B2_OPC_BARRIER = 0, B2_OPC_ALLREDUCE, B2_OPC_REDUCE, B2_OPC_SCAN, B2_OPC_ALLGATHER,
  B2_OPC_ALLTOALL, B2_OPC_BCAST, B2_OPC_GATHER, B2_OPC_SCATTER, B2_OPC_SEND, B2_OPC_RECV,
  B2_OPC_SENDRECV, B2_OPC_HALO, B2_OPC_REDUCE_SCATTER, B2_OPC_COUNT
};

static inline size_t b2_dtype_size(int dt) {
  switch (dt) {
    case B2_F32: case B2_I32: case B2_U32: return 4;
    case B2_F64: case B2_I64: case B2_U64: case B2_C64: return 8;
    case B2_F16: case B2_BF16: case B2_I16: case B2_U16: return 2;
    case B2_I8: case B2_U8: case B2_BOOL: return 1;
    case B2_C128: return 16;
    default: return 0;
  }
}

// ---------------------------------------------------------------------------
// Symmetric-heap layout (identical offsets on every rank).
//
//   [flags]      B2_MAX_BLOCKS x B2_MAX_RANKS u32   block-paired barrier flags
//   [p2p hdr]    P x NSLOT x LANES x 16 B           inbox headers (written by the sender)
//   [p2p ack]    P x NSLOT x LANES x 4 B            slot credits  (written by the receiver)
//   [ll]         2 parities x P x ll_cap            flag-in-data allreduce buffers
//   [p2p slots]  P x NSLOT x slot_bytes             eager/streaming payload ring
//   [p2p LL]     P x NSLOT x 16 KiB                 small messages, 8-byte {word, seq} stores
//   [halo LL]    2 parities x 8 sides x halo_ll_cap flag-in-data halo buffers
//   -- separate, growable segment --
//   [staging]    2 parities x stage_half            collective staging
// ---------------------------------------------------------------------------
struct B2Layout {
  size_t flags_off;
  size_t p2p_hdr_off;
  size_t p2p_ack_off;
  size_t ll_off;
  size_t ll_cap;          // bytes per (parity, source) LL buffer (wire bytes = 2x payload)
  size_t p2p_slot_off;
  size_t p2p_slot_bytes;
  size_t p2p_ll_off;      // P x NSLOT x (2 * B2_P2P_LL_MAX): flag-in-data copies of small messages
  size_t halo_cap;        // halo payload limit: nfields x max(ny, nx) x 4 B per exchange
  size_t halo_ll_off;     // flag-in-data halo buffers (b2_halo_ll.cuh)
  size_t halo_ll_cap;     // bytes per (parity, side): 8 B per element
  size_t total;
};

// Device-visible communicator state; passed to kernels BY VALUE (pointers are
// stable for the lifetime of the communicator, so CUDA graphs can bake them).
struct B2DevComm {
  int rank;
  int size;
  unsigned long long timeout_ns;        // device watchdog for spin waits
  char* heap[B2_MAX_RANKS];             // control+p2p segment of every rank, as mapped here
  char* stage[B2_MAX_RANKS];            // staging segment of every rank, as mapped here
  char* stage_mc;                       // multicast alias of the staging segment (or null)
  size_t stage_half;                    // bytes per parity
  B2Layout lay;
  // local (non-symmetric) device memory
  unsigned* epoch;                      // [B2_MAX_BLOCKS] per-CTA barrier epochs
  unsigned* ticket;                     // [0] collective ticket [1] finish ctr [6] halo finish ctr
                                        // [32..39] halo msgs received per side [40..47] sent per side
  unsigned* p2p_send_seq;               // [P] fragments sent to each destination
  unsigned* p2p_recv_seq;               // [P] fragments consumed from each source
  unsigned* p2p_ctl;                    // [8] arrive counters / any-source election word
  B2ErrorRecord* err;                   // host-mapped
};
