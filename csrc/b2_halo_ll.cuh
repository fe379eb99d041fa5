// mpi4jax_b200 -- flag-in-data ("LL") halo transport shared by the stand-alone exchange kernel
// (b2_halo.cu) and the deep exchange of the communication-avoiding shallow-water step (b2_swe_ca.cu).
//
// A halo element travels as ONE 8-byte store {value, flag}; 8-byte stores are atomic, so a reader
// that sees the flag sees the value: no fence, no separate signal, one NVLink one-way latency.
// flag = (messages sent on this side so far) + 1, buffer parity = that count & 1; both ends of
// a channel count the same messages in device memory (c.ticket[32..47]), so kernels using this
// transport can be mixed freely and replayed from CUDA graphs.
#pragma once

#include "b2_device.cuh"

enum { FS_W = 0, FS_E, FS_S, FS_N, FS_SW, FS_SE, FS_NW, FS_NE, FS_NSIDES };

// ticket words (local device memory)
#define TK_FIN 6       // finish counter
#define TK_RX 32       // [8] messages received per side
#define TK_TX 40       // [8] messages sent per side

__device__ __forceinline__ uint2* fz_buf(const B2DevComm& c, int rank, unsigned parity, int side) {
  return (uint2*)(c.heap[rank] + c.lay.halo_ll_off +
                  ((size_t)parity * FS_NSIDES + side) * c.lay.halo_ll_cap);
}
__device__ __forceinline__ void fz_put(uint2* p, float v, unsigned flag) {
  // no "memory" clobber: the value comes from registers and nothing in the kernel reads the
  // (remote) target, so the compiler stays free to overlap other loads with the push
  asm volatile("st.relaxed.sys.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)),
               "r"(flag));
}
__device__ __forceinline__ void fz_put2(uint2* p, float v0, float v1, unsigned flag) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p),
               "r"(__float_as_uint(v0)), "r"(flag), "r"(__float_as_uint(v1)), "r"(flag));
}
__device__ __forceinline__ float fz_get(const B2DevComm& c, const uint2* p, unsigned flag, int side) {
  unsigned v, f;
  unsigned long long t0 = 0;
  unsigned spins = 0;
  while (true) {
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(f) : "l"(p) : "memory");
    if (f == flag) break;
    if ((++spins & 0xfffu) == 0) {
      unsigned long long now = b2_gtime();
      if (t0 == 0) t0 = now;
      else if (now - t0 > c.timeout_ns) b2_fatal(c, B2_ERR_TIMEOUT, B2_OPC_HALO, side, flag, f, 5);
    }
  }
  return __uint_as_float(v);
}
