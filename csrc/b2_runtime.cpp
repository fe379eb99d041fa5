// mpi4jax_b200 -- symmetric heap, NVLS multicast objects and communicator state.
//
// The CUDA driver entry points are resolved at run time through
// cudaGetDriverEntryPoint so that the shared library has no link-time
// dependency on libcuda.so (it must import on GPU-less build hosts).
//
// Parity: this file is the B200 counterpart of what the reference delegates to
// the MPI library + mpi4py handles (mpi4jax/_src/utils.py:60-97) and to
// mpi_xla_bridge_cuda.cpp's cudaMemcpy staging (:55-67, :185-206): here the
// "communicator" is a set of peer-mapped HBM segments, flags and counters.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <unistd.h>

#include "b2_runtime.h"

extern "C" void b2_set_error(const char* fmt, ...);

// ---------------------------------------------------------------------------
// driver API loader
// ---------------------------------------------------------------------------
#define B2_DRV_FUNCS(X)                \
  X(cuMemCreate)                       \
  X(cuMemRelease)                      \
  X(cuMemAddressReserve)               \
  X(cuMemAddressFree)                  \
  X(cuMemMap)                          \
  X(cuMemUnmap)                        \
  X(cuMemSetAccess)                    \
  X(cuMemExportToShareableHandle)      \
  X(cuMemImportFromShareableHandle)    \
  X(cuMemGetAllocationGranularity)     \
  X(cuMulticastCreate)                 \
  X(cuMulticastAddDevice)              \
  X(cuMulticastBindMem)                \
  X(cuMulticastGetGranularity)         \
  X(cuDeviceGetAttribute)              \
  X(cuTensorMapEncodeTiled)            \
  X(cuGetErrorString)

#define B2_DECL(name) static decltype(&name) p_##name = nullptr;
B2_DRV_FUNCS(B2_DECL)
#undef B2_DECL

static bool g_drv_ok = false;

static bool load_driver() {
  if (g_drv_ok) return true;
#define B2_LOAD(name)                                                                      \
  {                                                                                        \
    void* fn = nullptr;                                                                    \
    cudaDriverEntryPointQueryResult qr;                                                    \
    cudaError_t e = cudaGetDriverEntryPoint(#name, &fn, cudaEnableDefault, &qr);           \
    if (e != cudaSuccess || fn == nullptr) {                                               \
      b2_set_error("driver entry point %s not available: %s", #name, cudaGetErrorString(e)); \
      return false;                                                                        \
    }                                                                                      \
    p_##name = reinterpret_cast<decltype(&name)>(fn);                                      \
  }
  B2_DRV_FUNCS(B2_LOAD)
#undef B2_LOAD
  g_drv_ok = true;
  return true;
}

static const char* drv_err(CUresult r) {
  const char* s = nullptr;
  if (p_cuGetErrorString && p_cuGetErrorString(r, &s) == CUDA_SUCCESS && s) return s;
  return "unknown driver error";
}

#define DRV_CHECK(call, ret)                                                  \
  do {                                                                        \
    CUresult _r = (call);                                                     \
    if (_r != CUDA_SUCCESS) {                                                 \
      b2_set_error("%s failed: %s (%d)", #call, drv_err(_r), (int)_r);        \
      return ret;                                                             \
    }                                                                         \
  } while (0)

#define RT_CHECK(call, ret)                                                   \
  do {                                                                        \
    cudaError_t _e = (call);                                                  \
    if (_e != cudaSuccess) {                                                  \
      b2_set_error("%s failed: %s", #call, cudaGetErrorString(_e));           \
      return ret;                                                             \
    }                                                                         \
  } while (0)

static size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

extern "C" int b2_init(int device) {
  RT_CHECK(cudaSetDevice(device), 1);
  RT_CHECK(cudaFree(0), 1);
  if (!load_driver()) return 2;
  return 0;
}

extern "C" int b2_vmm_supported(int device) {
  if (!load_driver()) return 0;
  int v = 0;
  if (p_cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR_SUPPORTED,
                             device) != CUDA_SUCCESS)
    return 0;
  return v;
}

extern "C" int b2_multicast_supported(int device) {
  if (!load_driver()) return 0;
  int v = 0;
  if (p_cuDeviceGetAttribute(&v, CU_DEVICE_ATTRIBUTE_MULTICAST_SUPPORTED, device) != CUDA_SUCCESS)
    return 0;
  return v;
}

static CUmemAllocationProp alloc_prop(int device) {
  CUmemAllocationProp prop;
  memset(&prop, 0, sizeof prop);
  prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
  prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  prop.location.id = device;
  prop.requestedHandleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
  return prop;
}

extern "C" size_t b2_granularity(int device, int for_multicast) {
  if (!load_driver()) return 0;
  size_t g = 0;
  CUmemAllocationProp prop = alloc_prop(device);
  if (p_cuMemGetAllocationGranularity(&g, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) !=
      CUDA_SUCCESS)
    g = 2u << 20;
  if (for_multicast) {
    CUmulticastObjectProp mp;
    memset(&mp, 0, sizeof mp);
    mp.numDevices = 2;
    mp.size = g;
    mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
    size_t mg = 0;
    if (p_cuMulticastGetGranularity(&mg, &mp, CU_MULTICAST_GRANULARITY_RECOMMENDED) ==
            CUDA_SUCCESS && mg > g)
      g = mg;
  }
  return g;
}

// ---------------------------------------------------------------------------
// segments
// ---------------------------------------------------------------------------
static int map_handle(int device, CUmemGenericAllocationHandle h, size_t bytes, void** out) {
  CUdeviceptr va = 0;
  DRV_CHECK(p_cuMemAddressReserve(&va, bytes, 0, 0, 0), 1);
  DRV_CHECK(p_cuMemMap(va, bytes, 0, h, 0), 1);
  CUmemAccessDesc acc;
  memset(&acc, 0, sizeof acc);
  acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
  acc.location.id = device;
  acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
  DRV_CHECK(p_cuMemSetAccess(va, bytes, &acc, 1), 1);
  *out = reinterpret_cast<void*>(va);
  return 0;
}

extern "C" B2Seg* b2_seg_create(int device, int rank, int nranks, size_t bytes, int mode) {
  if (nranks < 1 || nranks > B2_MAX_RANKS || rank < 0 || rank >= nranks) {
    b2_set_error("b2_seg_create: bad rank/nranks %d/%d", rank, nranks);
    return nullptr;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    b2_set_error("cudaSetDevice(%d) failed", device);
    return nullptr;
  }
  B2Seg* s = new B2Seg();
  memset(s, 0, sizeof *s);
  s->mode = mode;
  s->device = device;
  s->rank = rank;
  s->nranks = nranks;
  s->export_fd = -1;
  if (mode == 0) {
    if (!load_driver()) { delete s; return nullptr; }
    const size_t gran = b2_granularity(device, 1);
    s->bytes = round_up(bytes, gran ? gran : (2u << 20));
    CUmemAllocationProp prop = alloc_prop(device);
    CUresult r = p_cuMemCreate(&s->handle, s->bytes, &prop, 0);
    if (r != CUDA_SUCCESS) {
      b2_set_error("cuMemCreate(%zu bytes) failed: %s", s->bytes, drv_err(r));
      delete s;
      return nullptr;
    }
    if (map_handle(device, s->handle, s->bytes, &s->ptr[rank]) != 0) {
      p_cuMemRelease(s->handle);
      delete s;
      return nullptr;
    }
  } else {
    s->bytes = round_up(bytes, 2u << 20);
    if (cudaMalloc(&s->ptr[rank], s->bytes) != cudaSuccess) {
      b2_set_error("cudaMalloc(%zu) failed", s->bytes);
      delete s;
      return nullptr;
    }
  }
  if (cudaMemset(s->ptr[rank], 0, s->bytes) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    b2_set_error("zero-filling the segment failed");
    delete s;
    return nullptr;
  }
  return s;
}

extern "C" int b2_seg_export_fd(B2Seg* s) {
  if (s->mode != 0) { b2_set_error("segment is not VMM-backed"); return -1; }
  if (s->export_fd >= 0) return s->export_fd;
  int fd = -1;
  DRV_CHECK(p_cuMemExportToShareableHandle(&fd, s->handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0),
            -1);
  s->export_fd = fd;
  return fd;
}

extern "C" int b2_seg_import_fd(B2Seg* s, int peer, int fd) {
  if (peer < 0 || peer >= s->nranks || peer == s->rank) { b2_set_error("bad peer %d", peer); return 1; }
  DRV_CHECK(p_cuMemImportFromShareableHandle(&s->peer_handle[peer], (void*)(uintptr_t)fd,
                                             CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR), 1);
  return map_handle(s->device, s->peer_handle[peer], s->bytes, &s->ptr[peer]);
}

extern "C" int b2_seg_ipc_handle(B2Seg* s, void* out64) {
  if (s->mode != 1) { b2_set_error("segment is not IPC-backed"); return 1; }
  cudaIpcMemHandle_t h;
  RT_CHECK(cudaIpcGetMemHandle(&h, s->ptr[s->rank]), 1);
  memcpy(out64, &h, sizeof h);
  return 0;
}

extern "C" int b2_seg_import_ipc(B2Seg* s, int peer, const void* handle64) {
  if (peer < 0 || peer >= s->nranks || peer == s->rank) { b2_set_error("bad peer %d", peer); return 1; }
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof h);
  RT_CHECK(cudaIpcOpenMemHandle(&s->ptr[peer], h, cudaIpcMemLazyEnablePeerAccess), 1);
  return 0;
}

extern "C" void* b2_seg_ptr(B2Seg* s, int peer) { return s->ptr[peer]; }
extern "C" size_t b2_seg_bytes(B2Seg* s) { return s->bytes; }

extern "C" int b2_seg_destroy(B2Seg* s) {
  if (!s) return 0;
  cudaDeviceSynchronize();
  for (int p = 0; p < s->nranks; ++p) {
    if (!s->ptr[p]) continue;
    if (s->mode == 0) {
      p_cuMemUnmap((CUdeviceptr)s->ptr[p], s->bytes);
      p_cuMemAddressFree((CUdeviceptr)s->ptr[p], s->bytes);
      if (p != s->rank && s->peer_handle[p]) p_cuMemRelease(s->peer_handle[p]);
    } else if (p != s->rank) {
      cudaIpcCloseMemHandle(s->ptr[p]);
    }
  }
  if (s->mode == 0) {
    if (s->handle) p_cuMemRelease(s->handle);
    if (s->export_fd >= 0) close(s->export_fd);
  } else if (s->ptr[s->rank]) {
    cudaFree(s->ptr[s->rank]);
  }
  delete s;
  return 0;
}

// ---------------------------------------------------------------------------
// multicast (NVLS)
// ---------------------------------------------------------------------------
extern "C" B2Mc* b2_mc_create(int device, int nranks, size_t bytes) {
  if (!load_driver()) return nullptr;
  CUmulticastObjectProp mp;
  memset(&mp, 0, sizeof mp);
  mp.numDevices = (unsigned)nranks;
  mp.size = bytes;
  mp.handleTypes = CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR;
  B2Mc* m = new B2Mc();
  memset(m, 0, sizeof *m);
  m->bytes = bytes;
  m->device = device;
  m->export_fd = -1;
  CUresult r = p_cuMulticastCreate(&m->handle, &mp);
  if (r != CUDA_SUCCESS) {
    b2_set_error("cuMulticastCreate(%zu bytes, %d devices) failed: %s", bytes, nranks, drv_err(r));
    delete m;
    return nullptr;
  }
  return m;
}

extern "C" int b2_mc_export_fd(B2Mc* m) {
  if (m->export_fd >= 0) return m->export_fd;
  int fd = -1;
  DRV_CHECK(p_cuMemExportToShareableHandle(&fd, m->handle, CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR, 0),
            -1);
  m->export_fd = fd;
  return fd;
}

extern "C" B2Mc* b2_mc_import(int device, int fd, size_t bytes) {
  if (!load_driver()) return nullptr;
  B2Mc* m = new B2Mc();
  memset(m, 0, sizeof *m);
  m->bytes = bytes;
  m->device = device;
  m->export_fd = -1;
  CUresult r = p_cuMemImportFromShareableHandle(&m->handle, (void*)(uintptr_t)fd,
                                                CU_MEM_HANDLE_TYPE_POSIX_FILE_DESCRIPTOR);
  if (r != CUDA_SUCCESS) {
    b2_set_error("importing the multicast handle failed: %s", drv_err(r));
    delete m;
    return nullptr;
  }
  return m;
}

extern "C" int b2_mc_add_device(B2Mc* m) {
  DRV_CHECK(p_cuMulticastAddDevice(m->handle, m->device), 1);
  return 0;
}

extern "C" int b2_mc_bind(B2Mc* m, B2Seg* s) {
  if (s->mode != 0) { b2_set_error("multicast needs a VMM-backed segment"); return 1; }
  if (s->bytes != m->bytes) { b2_set_error("multicast/segment size mismatch"); return 1; }
  DRV_CHECK(p_cuMulticastBindMem(m->handle, 0, s->handle, 0, s->bytes, 0), 1);
  m->bound = 1;
  return map_handle(m->device, m->handle, m->bytes, &m->ptr);
}

extern "C" void* b2_mc_ptr(B2Mc* m) { return m ? m->ptr : nullptr; }

extern "C" int b2_mc_destroy(B2Mc* m) {
  if (!m) return 0;
  cudaDeviceSynchronize();
  if (m->ptr) {
    p_cuMemUnmap((CUdeviceptr)m->ptr, m->bytes);
    p_cuMemAddressFree((CUdeviceptr)m->ptr, m->bytes);
  }
  if (m->handle) p_cuMemRelease(m->handle);
  if (m->export_fd >= 0) close(m->export_fd);
  delete m;
  return 0;
}

// ---------------------------------------------------------------------------
// communicator
// ---------------------------------------------------------------------------
static B2Layout make_layout(int nranks, size_t slot_bytes, size_t ll_cap, size_t halo_cap) {
  B2Layout L;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = round_up(off + bytes, 4096); return o; };
  L.flags_off = take((size_t)B2_MAX_BLOCKS * B2_MAX_RANKS * 4);
  L.p2p_hdr_off = take((size_t)nranks * B2_P2P_NSLOT * B2_P2P_MAX_LANES * 16);
  L.p2p_ack_off = take((size_t)nranks * B2_P2P_NSLOT * 4);
  L.ll_cap = round_up(ll_cap, 4096);
  L.ll_off = take(2 * (size_t)nranks * L.ll_cap);
  L.p2p_slot_bytes = round_up(slot_bytes, 4096);
  L.p2p_slot_off = take((size_t)nranks * B2_P2P_NSLOT * L.p2p_slot_bytes);
  L.p2p_ll_off = take((size_t)nranks * B2_P2P_NSLOT * 2 * B2_P2P_LL_MAX);
  L.halo_cap = round_up(halo_cap, 4096);
  // 8 B per element; the extra 4 KiB covers padding each field to a multiple of 4 elements, so every
  // halo that fits halo_cap as 4-byte floats fits here
  L.halo_ll_cap = 2 * L.halo_cap + 4096;
  L.halo_ll_off = take(2 * 8 * L.halo_ll_cap);
  L.total = off;
  return L;
}

extern "C" size_t b2_layout_bytes(int nranks, size_t slot_bytes, size_t ll_cap, size_t halo_cap) {
  return make_layout(nranks, slot_bytes, ll_cap, halo_cap).total;
}

extern "C" B2Comm* b2_comm_create(int device, int rank, int nranks, B2Seg* ctl, size_t slot_bytes,
                                  size_t ll_cap, size_t halo_cap, double timeout_s) {
  if (cudaSetDevice(device) != cudaSuccess) { b2_set_error("cudaSetDevice failed"); return nullptr; }
  B2Layout L = make_layout(nranks, slot_bytes, ll_cap, halo_cap);
  if (ctl->bytes < L.total) {
    b2_set_error("control segment too small: %zu < %zu", ctl->bytes, L.total);
    return nullptr;
  }
  B2Comm* c = new B2Comm();
  memset(c, 0, sizeof *c);
  c->device = device;
  c->ctl = ctl;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return nullptr; }
  c->sm_count = prop.multiProcessorCount;
  B2DevComm& d = c->dev;
  d.rank = rank;
  d.size = nranks;
  d.timeout_ns = (unsigned long long)(timeout_s * 1e9);
  d.lay = L;
  for (int p = 0; p < nranks; ++p) d.heap[p] = (char*)ctl->ptr[p];
  // local counters: epoch[B2_MAX_BLOCKS] | ticket[8] | send_seq[16] | recv_seq[16] | p2p_ctl[32]
  const size_t nwords = B2_MAX_BLOCKS + 64 + B2_MAX_RANKS + B2_MAX_RANKS + 32;
  unsigned* local = nullptr;
  if (cudaMalloc(&local, nwords * 4) != cudaSuccess || cudaMemset(local, 0, nwords * 4) != cudaSuccess) {
    b2_set_error("allocating local counters failed");
    delete c;
    return nullptr;
  }
  d.epoch = local;
  d.ticket = local + B2_MAX_BLOCKS;
  d.p2p_send_seq = d.ticket + 64;
  d.p2p_recv_seq = d.p2p_send_seq + B2_MAX_RANKS;
  d.p2p_ctl = d.p2p_recv_seq + B2_MAX_RANKS;
  // any-source election generation starts at 1 (0 would match the zero-filled word)
  unsigned one = 1;
  cudaMemcpy(d.p2p_ctl + 3, &one, 4, cudaMemcpyHostToDevice);
  // host-mapped error record
  B2ErrorRecord* eh = nullptr;
  if (cudaHostAlloc((void**)&eh, sizeof(B2ErrorRecord), cudaHostAllocMapped) != cudaSuccess) {
    b2_set_error("cudaHostAlloc(error record) failed");
    delete c;
    return nullptr;
  }
  memset((void*)eh, 0, sizeof *eh);
  c->err_host = eh;
  void* edev = nullptr;
  cudaHostGetDevicePointer(&edev, (void*)eh, 0);
  d.err = (B2ErrorRecord*)edev;
  // measured on 8 x B200 (profiles/r1_collectives_sweep_8gpu_v1.json): LL wins up to its 64 KiB
  // buffer limit (7-12 us vs 13+), in-switch reduction wins from there on, one-shot beats
  // two-shot up to ~512 KiB when multicast is unavailable
  c->ll_max = 64 * 1024;
  c->oneshot_max = 512 * 1024;
  c->nvls_min = 64 * 1024 + 1;
  c->bcast_mc_min = 256 * 1024;
  c->nvls_pipeline = 1;
  c->trace = nullptr;
  c->trace_cap = 0;
  // one 512-thread CTA of the collective kernels (<= 128 registers per thread) fits per SM: grids are
  // capped at the co-resident count (see pick_chunks in b2_collectives.cu)
  c->max_blocks = 2 * c->sm_count;       // upper bound; every launch is further capped at its kernel's co-resident count
  if (c->max_blocks > B2_MAX_BLOCKS) c->max_blocks = B2_MAX_BLOCKS;
  cudaDeviceSynchronize();
  return c;
}

extern "C" int b2_comm_set_stage(B2Comm* c, B2Seg* stage, B2Mc* mc) {
  c->stage = stage;
  c->stage_mc = mc;
  for (int p = 0; p < c->dev.size; ++p) c->dev.stage[p] = stage ? (char*)stage->ptr[p] : nullptr;
  c->dev.stage_mc = (mc && mc->ptr) ? (char*)mc->ptr : nullptr;
  // two parities; keep halves 4 KiB aligned
  c->dev.stage_half = stage ? (stage->bytes / 2) / 4096 * 4096 : 0;
  return 0;
}

extern "C" size_t b2_comm_stage_half(B2Comm* c) { return c->dev.stage_half; }

extern "C" int b2_comm_set_tuning(B2Comm* c, long long ll_max, long long oneshot_max,
                                  long long nvls_min, int max_blocks) {
  if (ll_max >= 0) c->ll_max = (size_t)ll_max;
  if (oneshot_max >= 0) c->oneshot_max = (size_t)oneshot_max;
  if (nvls_min >= 0) c->nvls_min = (size_t)nvls_min;
  if (max_blocks > 0) c->max_blocks = max_blocks > B2_MAX_BLOCKS ? B2_MAX_BLOCKS : max_blocks;
  return 0;
}

extern "C" int b2_comm_set_option(B2Comm* c, const char* key, long long value) {
  if (strcmp(key, "bcast_mc_min") == 0) c->bcast_mc_min = (size_t)value;
  else if (strcmp(key, "nvls_pipeline") == 0) c->nvls_pipeline = value != 0;
  else if (strcmp(key, "trace_ptr") == 0) c->trace = (unsigned long long*)(uintptr_t)value;
  else if (strcmp(key, "trace_cap") == 0) c->trace_cap = (int)value;
  else { b2_set_error("unknown communicator option '%s'", key); return B2_ERR_BAD_ARG; }
  return 0;
}

// read back what the launches use (tests/test_coresidency.py checks the grid cap against the SM count)
extern "C" long long b2_comm_get_option(B2Comm* c, const char* key) {
  if (strcmp(key, "max_blocks") == 0) return c->max_blocks;
  if (strcmp(key, "sm_count") == 0) return c->sm_count;
  if (strcmp(key, "bcast_mc_min") == 0) return (long long)c->bcast_mc_min;
  if (strcmp(key, "nvls_pipeline") == 0) return c->nvls_pipeline ? 1 : 0;
  b2_set_error("unknown communicator option '%s'", key);
  return -1;
}

static const char* opcode_name(int opc) {
  static const char* names[] = {"Barrier", "Allreduce", "Reduce", "Scan", "Allgather", "Alltoall",
                                "Bcast", "Gather", "Scatter", "Send", "Recv", "Sendrecv", "Halo",
                                "Reduce_scatter_block"};
  if (opc < 0 || opc >= B2_OPC_COUNT) return "Unknown";
  return names[opc];
}

// Formats the device-side error record the same way the reference's abort path does
// ("r<rank> | MPI_<Op> returned error code <n>: <msg> - aborting", mpi_ops_common.h:60-78).
extern "C" int b2_comm_check_error(B2Comm* c, char* buf, int buflen) {
  B2ErrorRecord* e = c->err_host;
  if (!e || e->code == 0) return 0;
  const char* what = "unknown";
  switch (e->code) {
    case B2_ERR_TIMEOUT: what = "timed out waiting for a peer (deadlock or dead rank)"; break;
    case B2_ERR_TAG_MISMATCH: what = "next message from this source carries a different tag"; break;
    case B2_ERR_TRUNCATE: what = "message size does not match the receive buffer"; break;
    case B2_ERR_BAD_ARG: what = "invalid argument"; break;
  }
  snprintf(buf, buflen,
           "r%d | MPI_%s returned error code %d: %s (peer %d, expected %u, observed %u, block %d) - aborting",
           e->rank, opcode_name(e->opcode), e->code, what, e->peer, e->expected, e->observed, e->block);
  return e->code;
}

extern "C" int b2_comm_destroy(B2Comm* c) {
  if (!c) return 0;
  cudaDeviceSynchronize();
  if (c->dev.epoch) cudaFree(c->dev.epoch);
  if (c->err_host) cudaFreeHost((void*)c->err_host);
  delete c;
  return 0;
}

// ---------------------------------------------------------------------------
// TMA descriptor for a row-major (rows x cols) bf16 matrix, box = box_rows x box_cols,
// 128-byte swizzle (what the tcgen05 K-major SWIZZLE_128B shared-memory descriptor expects)
// ---------------------------------------------------------------------------
extern "C" int b2_tensor_map_2d_bf16(CUtensorMap* out, const void* ptr, unsigned long long rows,
                                     unsigned long long cols, unsigned box_rows, unsigned box_cols) {
  if (!load_driver()) return 1;
  if (((uintptr_t)ptr & 15) != 0 || (cols * 2) % 16 != 0 || box_cols * 2 != 128) {
    b2_set_error("tensor map: need a 16-byte aligned base, a row pitch that is a multiple of 16 bytes "
                 "and a 128-byte box row");
    return 1;
  }
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = p_cuTensorMapEncodeTiled(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr),
                                        dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    b2_set_error("cuTensorMapEncodeTiled failed: %s", drv_err(r));
    return 1;
  }
  return 0;
}

// ---------------------------------------------------------------------------
// p2p status records (host-mapped, written by the receive kernel)
// ---------------------------------------------------------------------------
extern "C" B2StatusRecord* b2_status_alloc(void) {
  B2StatusRecord* s = nullptr;
  if (cudaHostAlloc((void**)&s, sizeof(B2StatusRecord), cudaHostAllocMapped) != cudaSuccess) {
    b2_set_error("cudaHostAlloc(status) failed");
    return nullptr;
  }
  memset((void*)s, 0, sizeof *s);
  s->source = -1;
  s->tag = -1;
  return s;
}
extern "C" void b2_status_free(B2StatusRecord* s) {
  if (s) cudaFreeHost((void*)s);
}
