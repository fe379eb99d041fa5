// mpi4jax_b200 -- collective entry points and the data-movement kernels.
//
// Data-movement collectives (allgather, alltoall, bcast, gather, scatter) share
// ONE kernel: every rank stages the blocks its peers will need into its own
// symmetric staging buffer, a block-paired barrier publishes them, then every
// rank PULLS what it needs from the peers' staging straight into the final
// layout of its (ordinary, non-symmetric) output tensor.  The "unpack" the
// reference leaves to XLA concat/dynamic-update-slice ops after MPI_Allgather /
// MPI_Alltoall / MPI_Gather / MPI_Scatter / MPI_Bcast
// (mpi_ops_common.h:222-306; mpi_xla_bridge_cuda.cpp:99-148, 227-503) is fused
// into the NVLink pull; there is no host sync and no host staging.
//
// Reduction collectives live in b2_reduce.cuh; this file adds the kernels that go through the
// NVSwitch multicast object -- the NVLS allreduce of staged data (b2_k_allreduce_nvls), the
// in-place allreduce of symmetric tensors (b2_k_allreduce_sym), the multicast bcast
// (b2_k_bcast_mc), the reduce-to-root (b2_k_reduce_root_nvls), the in-switch reduce-scatter
// (b2_k_reduce_scatter_nvls) --, the size-based algorithm selection and the grid cap that keeps every
// launch co-resident (coresident_blocks).
#include <cstdio>
#include <cstring>

#include "b2_reduce.cuh"
#include "b2_runtime.h"

b2_reduce_launch_fn b2_reduce_table[B2_DTYPE_COUNT][B2_OP_COUNT];
b2_ll_launch_fn b2_ll_table[B2_DTYPE_COUNT][B2_OP_COUNT];
b2_rs_launch_fn b2_rs_table[B2_DTYPE_COUNT][B2_OP_COUNT];
b2_rs_launch_fn b2_rs_ll_table[B2_DTYPE_COUNT][B2_OP_COUNT];
void b2_register_reduce_group_0();
void b2_register_reduce_group_1();
void b2_register_reduce_group_2();
void b2_register_reduce_group_3();

extern "C" void b2_set_error(const char* fmt, ...);
extern "C" void b2_count_launch(B2Comm* c);
struct B2DebugScope;
extern "C" B2DebugScope* b2_debug_begin(B2Comm* c, const char* opname, const char* details,
                                         cudaStream_t stream);
extern "C" void b2_debug_end(B2DebugScope* s, int code);

static void b2_ensure_tables() {
  static bool done = false;
  if (done) return;
  b2_register_reduce_group_0();
  b2_register_reduce_group_1();
  b2_register_reduce_group_2();
  b2_register_reduce_group_3();
  done = true;
}

// ---------------------------------------------------------------------------
// barrier
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(32) b2_k_barrier(const B2DevComm c) {
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  b2_barrier_all(c, ++e, B2_OPC_BARRIER);
  if (threadIdx.x == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
}

// ---------------------------------------------------------------------------
// stage -> barrier -> pull
// ---------------------------------------------------------------------------
struct B2MoveArgs {
  const void* in;
  void* out;
  size_t blk_bytes;     // bytes of one per-rank block (chunks index into it)
  size_t blk_stride;    // staging stride between blocks (blk_bytes rounded up to 16)
  size_t chunk;
  int nin;              // blocks staged by this rank (0, 1 or size)
  int nsrc;             // blocks pulled by this rank
  int src_rank[B2_MAX_RANKS];
  int src_blk[B2_MAX_RANKS];
  int dst_blk[B2_MAX_RANKS];
  int opcode;
  int vec_ok;           // out and every block offset are 16-byte aligned -> batched vector pulls
  // strided input ("fused pack"): when lay.nd > 0 the blocks are gathered element by element from a
  // non-contiguous tensor while they are staged -- what the reference leaves to an XLA transpose /
  // copy kernel in front of MPI_Alltoall (tests/collective_ops/test_alltoall.py:43-65)
  B2Strided lay;
  long long in_blk_stride;   // bytes between consecutive input blocks (strided input only)
};

// stage `len` bytes of a block, starting at byte `off` of its row-major order, from strided memory
__device__ __forceinline__ void b2_gather_bytes(char* __restrict__ dst, const char* __restrict__ base,
                                                const B2Strided& L, size_t off, size_t len) {
  const size_t es = (size_t)L.esize;
  const size_t e0 = off / es, n = len / es;          // chunks are multiples of 16 bytes >= esize
  for (size_t k = threadIdx.x; k < n; k += blockDim.x) {
    size_t lin = e0 + k;
    long long src = 0;
#pragma unroll
    for (int d = 3; d >= 0; --d)
      if (d < L.nd) {
        const size_t q = lin / (size_t)L.shape[d];
        src += (long long)(lin - q * (size_t)L.shape[d]) * L.stride[d];
        lin = q;
      }
    const char* sp = base + src * (long long)es;
    char* dp = dst + k * es;
    switch (L.esize) {
      case 1: *dp = *sp; break;
      case 2: *(unsigned short*)dp = *(const unsigned short*)sp; break;
      case 4: *(unsigned*)dp = *(const unsigned*)sp; break;
      case 8: *(unsigned long long*)dp = *(const unsigned long long*)sp; break;
      default: *(ulonglong2*)dp = *(const ulonglong2*)sp; break;
    }
  }
}

// stage one chunk of every input block (plain local copy, or the fused gather of a strided input)
__device__ __forceinline__ void move_stage(const B2MoveArgs& a, char* mine, const char* in, size_t off, size_t len) {
  for (int j = 0; j < a.nin; ++j) {
    if (a.lay.nd > 0)
      b2_gather_bytes(mine + (size_t)j * a.blk_stride + off, in + (long long)j * a.in_blk_stride, a.lay, off, len);
    else
      b2_copy_bytes<false>(mine + (size_t)j * a.blk_stride + off, in + (size_t)j * a.blk_bytes + off, len);
  }
}

// Pull chunk [off, off + len) from the peers' staging into the output AND stage chunk [noff, noff + nlen)
// of this rank's input, in ONE loop: the NVLink loads (~3 us round trip) and the local HBM loads of a
// thread are in flight together, U vectors each -- a CTA is one per SM (co-residency, pick_chunks), so
// what it cannot overlap inside a thread it cannot overlap at all.  Measured before (2 GPUs, 256 MiB,
// profiles/r2_bw_probe_n2.log): 460 GB/s for every collective, proportional to the CTA count, next to
// 625 GB/s for the p2p ring on 64 CTAs -- latency-bound phases in a row, not the link.
template <int NS, int NI, int U, bool SPLIT>
__device__ __noinline__ void move_pull_and_stage(const B2DevComm& c, const B2MoveArgs& a, const size_t par,
                                                 char* mine, const char* in, char* out, const size_t off,
                                                 const size_t len, const size_t noff, const size_t nlen) {
  // (a real call per chunk: every instantiation gets its own register allocation; everything the loop
  // needs is read from the argument structs ONCE -- the stores below go through char pointers, which
  // may alias anything as far as the compiler knows)
  const int t = threadIdx.x, nt = blockDim.x;
  const int nsrc = a.nsrc, nin = a.nin;
  const size_t nvp = len >> 4, nvi = nlen >> 4;
  const size_t nvmax = nvp > nvi ? nvp : nvi;
  const char* psrc[NS];
  char* pdst[NS];
  const char* ssrc[NI];
  char* sdst[NI];
#pragma unroll
  for (int s2 = 0; s2 < NS; ++s2) {
    const int k = s2 < nsrc ? (s2 + c.rank) % nsrc : 0;      // stagger peers across ranks
    psrc[s2] = c.stage[a.src_rank[k]] + par + (size_t)a.src_blk[k] * a.blk_stride + off;
    pdst[s2] = out + (size_t)a.dst_blk[k] * a.blk_bytes + off;
  }
#pragma unroll
  for (int j = 0; j < NI; ++j) {
    ssrc[j] = in + (size_t)j * a.blk_bytes + noff;
    sdst[j] = mine + (size_t)j * a.blk_stride + noff;
  }
  (void)nvmax;
  // main part: whole tiles of U x blockDim vectors on BOTH sides, no per-vector conditions (arrays that
  // are defined under a condition end up in local memory)
  const size_t tile = (size_t)U * nt;
  const size_t nvmin = nvp < nvi ? nvp : nvi;
  const size_t full = nvmin / tile * tile;
  for (size_t base = 0; base < full; base += tile) {
    uint4 pv[U][NS], sv[U][NI];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t i = base + (size_t)u * nt + t;
#pragma unroll
      for (int s2 = 0; s2 < NS; ++s2) {
        pv[u][s2] = make_uint4(0, 0, 0, 0);
        if (s2 < nsrc) pv[u][s2] = b2_ld_peer16(psrc[s2] + (i << 4));
      }
      if (!SPLIT) {
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          sv[u][j] = make_uint4(0, 0, 0, 0);
          if (j < nin) sv[u][j] = b2_ld_stream16(ssrc[j] + (i << 4));
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t i = base + (size_t)u * nt + t;
#pragma unroll
      for (int s2 = 0; s2 < NS; ++s2)
        if (s2 < nsrc) b2_st16(pdst[s2] + (i << 4), pv[u][s2]);
      if (SPLIT) {        // (2 x 8 vectors live at once do not fit the register file: one side after the other)
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          sv[u][j] = make_uint4(0, 0, 0, 0);
          if (j < nin) sv[u][j] = b2_ld_stream16(ssrc[j] + (i << 4));
        }
      }
#pragma unroll
      for (int j = 0; j < NI; ++j)
        if (j < nin) b2_st16(sdst[j] + (i << 4), sv[u][j]);
    }
  }
  // remainders (the last tile of a chunk, a shorter or missing next chunk): one side after the other
  for (size_t i = full + t; i < nvp; i += nt) {
    uint4 pv[NS];
#pragma unroll
    for (int s2 = 0; s2 < NS; ++s2) {
      pv[s2] = make_uint4(0, 0, 0, 0);
      if (s2 < nsrc) pv[s2] = b2_ld_peer16(psrc[s2] + (i << 4));
    }
#pragma unroll
    for (int s2 = 0; s2 < NS; ++s2)
      if (s2 < nsrc) b2_st16(pdst[s2] + (i << 4), pv[s2]);
  }
  for (size_t i = full + t; i < nvi; i += nt) {
#pragma unroll
    for (int j = 0; j < NI; ++j)
      if (j < nin) b2_st16(sdst[j] + (i << 4), b2_ld_stream16(ssrc[j] + (i << 4)));
  }
  // the last < 16 bytes of either chunk
  const size_t ptail = len & 15, stail = nlen & 15;
  if (ptail && (size_t)t < ptail) {
#pragma unroll
    for (int s2 = 0; s2 < NS; ++s2)
      if (s2 < nsrc) pdst[s2][(nvp << 4) + t] = ((const volatile char*)psrc[s2])[(nvp << 4) + t];
  }
  if (stail && (size_t)t < stail) {
#pragma unroll
    for (int j = 0; j < NI; ++j)
      if (j < nin) sdst[j][(nvi << 4) + t] = ssrc[j][(nvi << 4) + t];
  }
}

__global__ void __launch_bounds__(B2_THREADS, 1)
b2_k_move(const __grid_constant__ B2DevComm c, const __grid_constant__ B2MoveArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  const size_t nchunks = (a.blk_bytes + a.chunk - 1) / a.chunk;
  // the fused loop moves whole 16-byte vectors on both sides
  const bool fuse = a.vec_ok && a.lay.nd == 0 && ((((uintptr_t)in) & 15) == 0) && (a.nin <= 1 || (a.blk_bytes & 15) == 0);
#define CH_OFF(ch) ((ch) * a.chunk)
#define CH_LEN(ch) ((a.blk_bytes - CH_OFF(ch) < a.chunk) ? (a.blk_bytes - CH_OFF(ch)) : a.chunk)
  size_t ch = blockIdx.x;
  unsigned e_cur = e;
  if (ch < nchunks) {
    move_stage(a, mine, in, CH_OFF(ch), CH_LEN(ch));
    b2_barrier_arrive(c, ++e);
    e_cur = e;
  }
  for (; ch < nchunks; ch += gridDim.x) {
    const size_t nxt = ch + gridDim.x;
    const bool more = nxt < nchunks;
    const size_t off = CH_OFF(ch), len = CH_LEN(ch);
    const size_t noff = more ? CH_OFF(nxt) : 0, nlen = more ? CH_LEN(nxt) : 0;
    b2_barrier_wait(c, e_cur, a.opcode);            // every rank staged this chunk
    if (fuse && a.nin <= 1 && a.nsrc <= 8) {
      if (a.nsrc <= 1) move_pull_and_stage<1, 1, 4, false>(c, a, par, mine, in, out, off, len, noff, nlen);
      else if (a.nsrc <= 3) move_pull_and_stage<3, 1, 2, false>(c, a, par, mine, in, out, off, len, noff, nlen);
      else move_pull_and_stage<8, 1, 1, false>(c, a, par, mine, in, out, off, len, noff, nlen);
    } else if (fuse && a.nsrc <= 8 && a.nin <= 8) {       // alltoall, the root of a scatter
      if (a.nsrc <= 2 && a.nin <= 2) move_pull_and_stage<2, 2, 2, false>(c, a, par, mine, in, out, off, len, noff, nlen);
      else if (a.nsrc <= 4 && a.nin <= 4) move_pull_and_stage<4, 4, 1, false>(c, a, par, mine, in, out, off, len, noff, nlen);
      else move_pull_and_stage<8, 8, 1, true>(c, a, par, mine, in, out, off, len, noff, nlen);
    } else {
      for (int s2 = 0; s2 < a.nsrc; ++s2) {
        const int k = (s2 + c.rank) % a.nsrc;
        b2_copy_bytes<true>(out + (size_t)a.dst_blk[k] * a.blk_bytes + off,
                            c.stage[a.src_rank[k]] + par + (size_t)a.src_blk[k] * a.blk_stride + off, len);
      }
      if (more) move_stage(a, mine, in, noff, nlen);
    }
    if (more) {
      b2_barrier_arrive(c, ++e);
      e_cur = e;
    }
  }
#undef CH_OFF
#undef CH_LEN
  __syncthreads();
  if (threadIdx.x == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// NVLS allreduce (SUM; f32 / bf16 / f16 with fp32 accumulation in the switch)
// ---------------------------------------------------------------------------
template <int DT>
__device__ __forceinline__ uint4 b2_mc_ld_reduce(const void* mc) {
  uint4 v;
  if (DT == B2_F32) {
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
  } else if (DT == B2_BF16) {
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
  } else {
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.f16x2 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
  }
  return v;
}
__device__ __forceinline__ void b2_mc_st(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// in-switch reduction of this rank's sub-slice of a chunk, broadcast back through the switch
template <int DT>
__device__ __forceinline__ void b2_nvls_slice(const B2DevComm& c, char* mc, size_t off, size_t len) {
  const int t = threadIdx.x, nt = blockDim.x;
  const size_t nv = (len + 15) >> 4;
  const size_t per = (nv + c.size - 1) / c.size;
  size_t v0 = per * (size_t)c.rank;
  if (v0 > nv) v0 = nv;
  size_t v1 = v0 + per;
  if (v1 > nv) v1 = nv;
  size_t i = v0 + t;
  for (; i + 3 * (size_t)nt < v1; i += 4 * (size_t)nt) {
    uint4 r0 = b2_mc_ld_reduce<DT>(mc + off + (i << 4));
    uint4 r1 = b2_mc_ld_reduce<DT>(mc + off + ((i + nt) << 4));
    uint4 r2 = b2_mc_ld_reduce<DT>(mc + off + ((i + 2 * (size_t)nt) << 4));
    uint4 r3 = b2_mc_ld_reduce<DT>(mc + off + ((i + 3 * (size_t)nt) << 4));
    b2_mc_st(mc + off + (i << 4), r0);
    b2_mc_st(mc + off + ((i + nt) << 4), r1);
    b2_mc_st(mc + off + ((i + 2 * (size_t)nt) << 4), r2);
    b2_mc_st(mc + off + ((i + 3 * (size_t)nt) << 4), r3);
  }
  for (; i < v1; i += nt) b2_mc_st(mc + off + (i << 4), b2_mc_ld_reduce<DT>(mc + off + (i << 4)));
}

// Software-pipelined over the chunks of a CTA (all CTAs co-resident, chunk k of CTA b is chunk
// b + k * grid on every rank):
//
//   stage(0) A1(0) | stage(1) W1(0) nvls(0) A2(0) A1(1) | stage(2) W2(0) out(0) W1(1) nvls(1) A2(1) A1(2) | ...
//
// A = arrive (flags to the peers), W = wait.  The local HBM copies (stage the next chunk, copy
// the previous result out) sit between an arrive and its wait, so they hide the flag round trip,
// and CTAs drift to different phases, so HBM copies overlap other CTAs' NVLink phases.
template <int DT>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_allreduce_nvls(const B2DevComm c, const B2ReduceArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  char* mc = c.stage_mc + par;
  const size_t nchunks = (a.nbytes + a.chunk - 1) / a.chunk;
  const int t = threadIdx.x;
#define CH_OFF(ch) ((ch) * a.chunk)
#define CH_LEN(ch) ((a.nbytes - CH_OFF(ch) < a.chunk) ? (a.nbytes - CH_OFF(ch)) : a.chunk)
  const bool pipe = a.pipeline != 0;
  unsigned e_a1 = e;
  bool staged = false;
  // phase timeline of CTA 0 (debug option "trace_ptr"): %globaltimer after every phase
  int tr_n = 0;
#define TRACE() do { if (a.trace != nullptr && blockIdx.x == 0) { __syncthreads(); \
    if (t == 0 && tr_n < a.trace_cap) a.trace[tr_n] = b2_gtime(); ++tr_n; } } while (0)
  TRACE();
  for (size_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const size_t nxt = ch + gridDim.x;
    const bool more = pipe && nxt < nchunks;
    if (!staged) {
      b2_copy_bytes<false>(mine + CH_OFF(ch), in + CH_OFF(ch), CH_LEN(ch));
      b2_barrier_arrive(c, ++e);                                 // A1
      e_a1 = e;
    }
    TRACE();                                                     // 1: staged (or nothing)
    if (more) b2_copy_bytes<false>(mine + CH_OFF(nxt), in + CH_OFF(nxt), CH_LEN(nxt));
    TRACE();                                                     // 2: next chunk staged
    b2_barrier_wait(c, e_a1, a.opcode);                          // W1: every rank staged this chunk
    TRACE();                                                     // 3: W1
    b2_nvls_slice<DT>(c, mc, CH_OFF(ch), CH_LEN(ch));
    TRACE();                                                     // 4: in-switch reduction + broadcast issued
    b2_barrier_arrive(c, ++e);                                   // A2
    const unsigned e_a2 = e;
    staged = more;
    if (more) {                                                  // A1 of the next chunk (staged above)
      b2_barrier_arrive(c, ++e);
      e_a1 = e;
    }
    b2_barrier_wait(c, e_a2, a.opcode);                          // W2: every sub-slice has landed here
    TRACE();                                                     // 5: W2
    b2_copy_bytes<true>(out + CH_OFF(ch), mine + CH_OFF(ch), CH_LEN(ch));
    TRACE();                                                     // 6: copied out
  }
#undef TRACE
#undef CH_OFF
#undef CH_LEN
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// allreduce of a SYMMETRIC tensor, in place (mpi4jax_b200.symmetric_empty / allreduce_): the buffer
// lives in a multicast-bound segment at the same offset on every rank, so there is nothing to stage
// and nothing to copy out -- barrier, every rank reduces its 1/P of the vectors inside the switch
// (multimem.ld_reduce) and broadcasts them back through it (multimem.st), barrier.  No chunks: the
// two barriers are the only synchronisation, the links are busy in between.
// ---------------------------------------------------------------------------
struct B2SymArgs {
  char* mc;          // multicast address of the buffer
  size_t nbytes;     // multiple of 16
  int opcode;
};
template <int DT>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_allreduce_sym(const B2DevComm c, const B2SymArgs a) {
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  b2_barrier_all(c, ++e, a.opcode);                  // every rank's kernels that wrote the buffer are done
  const int t = threadIdx.x, nt = blockDim.x;
  const size_t nv = a.nbytes >> 4;
  const size_t per = (nv + c.size - 1) / c.size;     // this rank's slice of the vectors
  size_t v0 = per * (size_t)c.rank;
  if (v0 > nv) v0 = nv;
  size_t v1 = v0 + per;
  if (v1 > nv) v1 = nv;
  // tiles of 4 x blockDim vectors, round-robin over the CTAs: four in-switch reductions in flight per thread
  const size_t tile = 4 * (size_t)nt;
  for (size_t base = v0 + (size_t)blockIdx.x * tile; base < v1; base += (size_t)gridDim.x * tile) {
    const size_t i0 = base + t, i1 = i0 + nt, i2 = i1 + nt, i3 = i2 + nt;
    uint4 r0 = make_uint4(0, 0, 0, 0), r1 = r0, r2 = r0, r3 = r0;
    if (i0 < v1) r0 = b2_mc_ld_reduce<DT>(a.mc + (i0 << 4));
    if (i1 < v1) r1 = b2_mc_ld_reduce<DT>(a.mc + (i1 << 4));
    if (i2 < v1) r2 = b2_mc_ld_reduce<DT>(a.mc + (i2 << 4));
    if (i3 < v1) r3 = b2_mc_ld_reduce<DT>(a.mc + (i3 << 4));
    if (i0 < v1) b2_mc_st(a.mc + (i0 << 4), r0);
    if (i1 < v1) b2_mc_st(a.mc + (i1 << 4), r1);
    if (i2 < v1) b2_mc_st(a.mc + (i2 << 4), r2);
    if (i3 < v1) b2_mc_st(a.mc + (i3 << 4), r3);
  }
  b2_barrier_all(c, ++e, a.opcode);                  // every slice has landed everywhere
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
}

// ---------------------------------------------------------------------------
// bcast: the root writes its data ONCE with multimem.st -- the NVSwitch replicates it into every
// rank's staging -- instead of P-1 peers pulling P-1 copies over the root's links
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(B2_THREADS)
b2_k_bcast_mc(const B2DevComm c, const B2MoveArgs a, const int root) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  char* mc = c.stage_mc + par;
  const size_t nchunks = (a.blk_bytes + a.chunk - 1) / a.chunk;
  const int t = threadIdx.x, nt = blockDim.x;
  for (size_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const size_t off = ch * a.chunk;
    const size_t len = (a.blk_bytes - off < a.chunk) ? (a.blk_bytes - off) : a.chunk;
    if (c.rank == root) {
      const size_t nv = len >> 4, tail = len & 15;
      size_t i = t;
      for (; i + 3 * (size_t)nt < nv; i += 4 * (size_t)nt) {       // four HBM loads in flight per thread
        const uint4 v0 = b2_ld_stream16(in + off + (i << 4));
        const uint4 v1 = b2_ld_stream16(in + off + ((i + nt) << 4));
        const uint4 v2 = b2_ld_stream16(in + off + ((i + 2 * (size_t)nt) << 4));
        const uint4 v3 = b2_ld_stream16(in + off + ((i + 3 * (size_t)nt) << 4));
        b2_mc_st(mc + off + (i << 4), v0);
        b2_mc_st(mc + off + ((i + nt) << 4), v1);
        b2_mc_st(mc + off + ((i + 2 * (size_t)nt) << 4), v2);
        b2_mc_st(mc + off + ((i + 3 * (size_t)nt) << 4), v3);
      }
      for (; i < nv; i += nt) b2_mc_st(mc + off + (i << 4), b2_ld_stream16(in + off + (i << 4)));
      if (tail && t == 0) {
        alignas(16) unsigned char tmp[16] = {0};
        for (size_t k = 0; k < tail; ++k) tmp[k] = ((const unsigned char*)in)[off + (nv << 4) + k];
        b2_mc_st(mc + off + (nv << 4), *reinterpret_cast<const uint4*>(tmp));
      }
    }
    b2_barrier_all(c, ++e, a.opcode);
    if (c.rank != root) b2_copy_bytes<true>(out + off, mine + off, len);
  }
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// reduce (SUM, f32 / bf16 / f16): the root reads the in-switch sum of all ranks' staging with
// multimem.ld_reduce -- one stream of S bytes into the root instead of P-1
template <int DT>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_reduce_root_nvls(const B2DevComm c, const B2ReduceArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  const char* mc = c.stage_mc + par;
  const size_t nchunks = (a.nbytes + a.chunk - 1) / a.chunk;
  const int t = threadIdx.x, nt = blockDim.x;
#define CH_OFF(ch) ((ch) * a.chunk)
#define CH_LEN(ch) ((a.nbytes - CH_OFF(ch) < a.chunk) ? (a.nbytes - CH_OFF(ch)) : a.chunk)
  // software pipeline: the next chunk is staged while this one is reduced -- on the root in the SAME
  // loop as the multimem.ld_reduce, so the switch round trips and the HBM loads overlap
  size_t ch = blockIdx.x;
  unsigned e_cur = e;
  if (ch < nchunks) {
    b2_copy_bytes<false>(mine + CH_OFF(ch), in + CH_OFF(ch), CH_LEN(ch));
    b2_barrier_arrive(c, ++e);
    e_cur = e;
  }
  const bool vec_in = ((((uintptr_t)in) | ((uintptr_t)out)) & 15) == 0;
  for (; ch < nchunks; ch += gridDim.x) {
    const size_t nxt = ch + gridDim.x;
    const bool more = nxt < nchunks;
    const size_t off = CH_OFF(ch), len = CH_LEN(ch);
    const size_t noff = more ? CH_OFF(nxt) : 0, nlen = more ? CH_LEN(nxt) : 0;
    b2_barrier_wait(c, e_cur, a.opcode);              // every rank staged this chunk
    size_t staged = 0;                                // vectors of the next chunk staged by the fused loop
    if (a.has_out) {
      const size_t nv = (len + 15) >> 4;
      const size_t nfull = len >> 4;                  // whole output vectors
      const size_t nvi = vec_in ? (nlen >> 4) : 0;
      const size_t both = (nfull < nvi ? nfull : nvi) / (2 * (size_t)nt) * (2 * (size_t)nt);
      for (size_t base = 0; base < both; base += 2 * (size_t)nt) {
        const size_t i0 = base + t, i1 = i0 + nt;
        const uint4 r0 = b2_mc_ld_reduce<DT>(mc + off + (i0 << 4));
        const uint4 r1 = b2_mc_ld_reduce<DT>(mc + off + (i1 << 4));
        const uint4 s0 = b2_ld_stream16(in + noff + (i0 << 4));
        const uint4 s1 = b2_ld_stream16(in + noff + (i1 << 4));
        b2_st16(out + off + (i0 << 4), r0);
        b2_st16(out + off + (i1 << 4), r1);
        b2_st16(mine + noff + (i0 << 4), s0);
        b2_st16(mine + noff + (i1 << 4), s1);
      }
      staged = both;
      size_t i = both + t;
      for (; i + 3 * (size_t)nt < nfull; i += 4 * (size_t)nt) {
        const uint4 r0 = b2_mc_ld_reduce<DT>(mc + off + (i << 4));
        const uint4 r1 = b2_mc_ld_reduce<DT>(mc + off + ((i + nt) << 4));
        const uint4 r2 = b2_mc_ld_reduce<DT>(mc + off + ((i + 2 * (size_t)nt) << 4));
        const uint4 r3 = b2_mc_ld_reduce<DT>(mc + off + ((i + 3 * (size_t)nt) << 4));
        b2_st16(out + off + (i << 4), r0);
        b2_st16(out + off + ((i + nt) << 4), r1);
        b2_st16(out + off + ((i + 2 * (size_t)nt) << 4), r2);
        b2_st16(out + off + ((i + 3 * (size_t)nt) << 4), r3);
      }
      for (; i < nv; i += nt) {
        const uint4 r = b2_mc_ld_reduce<DT>(mc + off + (i << 4));
        const size_t b2 = i << 4;
        if (b2 + 16 <= len) b2_st16(out + off + b2, r);
        else b2_store_partial(out + off + b2, r, (int)(len - b2));
      }
    }
    if (more) {
      const size_t done = staged << 4;
      b2_copy_bytes<false>(mine + noff + done, in + noff + done, nlen - done);
      b2_barrier_arrive(c, ++e);
      e_cur = e;
    }
  }
#undef CH_OFF
#undef CH_LEN
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}


// reduce-scatter (SUM, f32 / bf16 / f16): every rank stages the P pieces of a chunk, then reads the
// in-switch sum of piece `rank` with multimem.ld_reduce straight into its output.  Next to the NVLS
// allreduce there is no multimem.st broadcast, no second barrier and no copy out.
template <int DT>
__global__ void __launch_bounds__(B2_THREADS, 2)     // <= 64 registers: two CTAs per SM (coresident_blocks)
b2_k_reduce_scatter_nvls(const B2DevComm c, const B2RSArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  const char* red = c.stage_mc + par + (size_t)c.rank * a.blk_stride;     // piece `rank`, through the switch
  const size_t nb = a.blk_bytes, st = a.blk_stride;
  const size_t nchunks = (nb + a.chunk - 1) / a.chunk;
  const int t = threadIdx.x, nt = blockDim.x, P = c.size;
#define CH_OFF(ch) ((ch) * a.chunk)
#define CH_LEN(ch) ((nb - CH_OFF(ch) < a.chunk) ? (nb - CH_OFF(ch)) : a.chunk)
  // software pipeline: the P pieces of the next chunk are staged while this one is reduced, in the
  // SAME loop as the multimem.ld_reduce, so the switch round trips and the HBM loads overlap
  size_t ch = blockIdx.x;
  unsigned e_cur = e;
  if (ch < nchunks) {
#pragma unroll 1
    for (int q = 0; q < P; ++q)
      b2_copy_bytes<false>(mine + (size_t)q * st + CH_OFF(ch), in + (size_t)q * nb + CH_OFF(ch), CH_LEN(ch));
    b2_barrier_arrive(c, ++e);
    e_cur = e;
  }
  for (; ch < nchunks; ch += gridDim.x) {
    const size_t nxt = ch + gridDim.x;
    const bool more = nxt < nchunks;
    const size_t off = CH_OFF(ch), len = CH_LEN(ch);
    const size_t noff = more ? CH_OFF(nxt) : 0, nlen = more ? CH_LEN(nxt) : 0;
    b2_barrier_wait(c, e_cur, a.opcode);              // every rank staged this chunk
    const size_t nv = (len + 15) >> 4;
    const size_t nvi = a.own_in ? (nlen >> 4) : 0;    // whole vectors of every next piece (own_in: no tails)
    const size_t nmax = nv > nvi ? nv : nvi;
    for (size_t base = 0; base < nmax; base += 2 * (size_t)nt) {
      const size_t i0 = base + t, i1 = i0 + nt;
      uint4 r0 = make_uint4(0, 0, 0, 0), r1 = r0;
      if (i0 < nv) r0 = b2_mc_ld_reduce<DT>(red + off + (i0 << 4));
      if (i1 < nv) r1 = b2_mc_ld_reduce<DT>(red + off + (i1 << 4));
#pragma unroll 1
      for (int q = 0; q < P; ++q) {
        const char* src = in + (size_t)q * nb + noff;
        char* dst = mine + (size_t)q * st + noff;
        uint4 s0 = make_uint4(0, 0, 0, 0), s1 = s0;
        if (i0 < nvi) s0 = b2_ld_stream16(src + (i0 << 4));
        if (i1 < nvi) s1 = b2_ld_stream16(src + (i1 << 4));
        if (i0 < nvi) b2_st16(dst + (i0 << 4), s0);
        if (i1 < nvi) b2_st16(dst + (i1 << 4), s1);
      }
      if (i0 < nv) {
        if ((i0 << 4) + 16 <= len) b2_st16(out + off + (i0 << 4), r0);
        else b2_store_partial(out + off + (i0 << 4), r0, (int)(len - (i0 << 4)));
      }
      if (i1 < nv) {
        if ((i1 << 4) + 16 <= len) b2_st16(out + off + (i1 << 4), r1);
        else b2_store_partial(out + off + (i1 << 4), r1, (int)(len - (i1 << 4)));
      }
    }
    if (more) {
      if (!a.own_in)                                  // unaligned blocks: stage the next chunk byte-wise
#pragma unroll 1
        for (int q = 0; q < P; ++q)
          b2_copy_bytes<false>(mine + (size_t)q * st + noff, in + (size_t)q * nb + noff, nlen);
      b2_barrier_arrive(c, ++e);
      e_cur = e;
    }
  }
#undef CH_OFF
#undef CH_LEN
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// host helpers
// ---------------------------------------------------------------------------
static size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

// How many CTAs of `kernel` (B2_THREADS threads, no dynamic shared memory) are resident at the same
// time on this GPU: occupancy x SM count, bounded by the communicator's max_blocks.  A launch of at
// most that many CTAs has every CTA resident at once whatever order the hardware dispatches them in,
// so the block-paired barriers cannot wait for a CTA that has not been scheduled yet (if other work
// owns the SMs the launch starts late, it does not deadlock: tests/test_coresidency.py).  The 64-register
// kernels (NVLS allreduce, multicast bcast, reduce-to-root) fit twice per SM -- and their bandwidth
// is proportional to the CTA count up to the link limit (profiles/r2_bw_probe_*.log).
#include <map>
static int coresident_blocks(const B2Comm* c, const void* kernel) {
  static std::map<const void*, int> per_sm;
  int n = 1;
  if (kernel != nullptr) {
    auto it = per_sm.find(kernel);
    if (it == per_sm.end()) {
      int occ = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, B2_THREADS, 0) != cudaSuccess || occ < 1) {
        cudaGetLastError();
        occ = 1;
      }
      it = per_sm.emplace(kernel, occ).first;
    }
    n = it->second;
  }
  long long cap = (long long)n * c->sm_count;
  if (cap > c->max_blocks) cap = c->max_blocks;
  if (cap > B2_MAX_BLOCKS) cap = B2_MAX_BLOCKS;
  return (int)cap;
}

// Same answer on every rank: depends only on (nbytes, size, the grid cap).
static void pick_chunks(const B2Comm* c, size_t nbytes, int cap, size_t* chunk_out, int* grid_out) {
  const size_t unit = 16 * (size_t)c->dev.size;
  const size_t min_chunk = round_up(16 * 1024, unit);
  const size_t max_chunk = round_up(512 * 1024, unit);
  const size_t target = (size_t)(cap < 1 ? 1 : cap);
  // >= 4 MiB: at least two chunks per CTA, so that the software pipeline of the kernels (stage the
  // next chunk / copy the previous one out while the flags of this one travel) has something to
  // overlap and CTAs drift to different phases; below that one chunk per CTA (latency regime)
  const size_t per_cta = nbytes >= ((size_t)64 << 20) ? 4 : nbytes >= ((size_t)4 << 20) ? 2 : 1;
  size_t chunk = round_up((nbytes + per_cta * target - 1) / (per_cta * target), unit);
  if (chunk < min_chunk) chunk = min_chunk;
  if (chunk > max_chunk) chunk = max_chunk;
  size_t nchunks = (nbytes + chunk - 1) / chunk;
  if (nchunks < 1) nchunks = 1;
  int grid = (int)(nchunks < target ? nchunks : target);
  *chunk_out = chunk;
  *grid_out = grid;
}

extern "C" size_t b2_stage_need(int opcode, int nranks, size_t blk_bytes) {
  const size_t stride = round_up(blk_bytes, 16);
  switch (opcode) {
    case B2_OPC_ALLTOALL:
    case B2_OPC_SCATTER:
    case B2_OPC_REDUCE_SCATTER:
      return stride * (size_t)nranks + 4096;
    default:
      return stride + 4096;
  }
}

static int check_stage(B2Comm* c, int opcode, size_t blk_bytes, const char* name) {
  const size_t need = b2_stage_need(opcode, c->dev.size, blk_bytes);
  if (c->stage == nullptr || need > c->dev.stage_half) {
    b2_set_error("%s: staging too small (need %zu bytes, have %zu); the Python layer must grow it",
                 name, need, c->stage ? c->dev.stage_half : (size_t)0);
    return B2_ERR_BAD_ARG;
  }
  return 0;
}

static int finish_launch(B2Comm* c, cudaError_t err, const char* name) {
  b2_count_launch(c);
  if (err != cudaSuccess) {
    b2_set_error("%s: kernel launch failed: %s", name, cudaGetErrorString(err));
    return 1000 + (int)err;
  }
  return 0;
}

extern "C" int b2_barrier(B2Comm* c, cudaStream_t stream) {
  B2DebugScope* dbg = b2_debug_begin(c, "Barrier", "", stream);
  b2_k_barrier<<<1, 32, 0, stream>>>(c->dev);
  int rc = finish_launch(c, cudaGetLastError(), "barrier");
  b2_debug_end(dbg, rc);
  return rc;
}

static int reduce_common(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                         int algo, int src_lo, int src_hi, int has_out, int opcode,
                         const char* name, cudaStream_t stream) {
  b2_ensure_tables();
  if (dtype < 0 || dtype >= B2_DTYPE_COUNT || op < 0 || op >= B2_OP_COUNT ||
      b2_reduce_table[dtype][op] == nullptr) {
    b2_set_error("%s: unsupported dtype/op combination (dtype=%d, op=%d)", name, dtype, op);
    return B2_ERR_BAD_ARG;
  }
  const size_t nbytes = count * b2_dtype_size(dtype);
  if (nbytes == 0) return 0;
  const int P = c->dev.size;
  if (algo == B2_ALGO_AUTO) {
    if (opcode != B2_OPC_ALLREDUCE) algo = B2_ALGO_ONESHOT;
    else if (P > 1 && nbytes <= c->ll_max && nbytes * 2 <= c->dev.lay.ll_cap) algo = B2_ALGO_LL;
    else if (P <= 2) algo = B2_ALGO_ONESHOT;
    else if (c->dev.stage_mc != nullptr && op == B2_SUM && nbytes >= c->nvls_min &&
             (dtype == B2_F32 || dtype == B2_BF16 || dtype == B2_F16)) algo = B2_ALGO_NVLS;
    else if (nbytes <= c->oneshot_max) algo = B2_ALGO_ONESHOT;
    else algo = B2_ALGO_TWOSHOT;
  }
  if (algo == B2_ALGO_LL) {
    if (opcode != B2_OPC_ALLREDUCE || nbytes * 2 > c->dev.lay.ll_cap) {
      b2_set_error("%s: LL algorithm needs an allreduce of <= %zu bytes", name,
                   c->dev.lay.ll_cap / 2);
      return B2_ERR_BAD_ARG;
    }
    B2LLArgs a;
    a.in = in; a.out = out; a.nbytes = nbytes; a.opcode = opcode;
    const size_t nv = (nbytes + 15) / 16;
    int grid = (int)((nv + B2_THREADS - 1) / B2_THREADS);
    if (grid > c->sm_count) grid = c->sm_count;
    if (grid < 1) grid = 1;
    return finish_launch(c, b2_ll_table[dtype][op](c->dev, a, grid, stream), name);
  }
  int rc = check_stage(c, opcode, nbytes, name);
  if (rc) return rc;
  B2ReduceArgs a;
  a.in = in; a.out = out; a.nbytes = nbytes;
  a.src_lo = src_lo; a.src_hi = src_hi; a.has_out = has_out; a.opcode = opcode;
  a.pipeline = c->nvls_pipeline;
  a.trace = c->trace; a.trace_cap = c->trace_cap;
  int grid;
  const void* kern = nullptr;
  if (algo == B2_ALGO_NVLS) {
    if (opcode == B2_OPC_REDUCE)
      kern = dtype == B2_F32 ? (const void*)b2_k_reduce_root_nvls<B2_F32>
             : dtype == B2_BF16 ? (const void*)b2_k_reduce_root_nvls<B2_BF16> : (const void*)b2_k_reduce_root_nvls<B2_F16>;
    else
      kern = dtype == B2_F32 ? (const void*)b2_k_allreduce_nvls<B2_F32>
             : dtype == B2_BF16 ? (const void*)b2_k_allreduce_nvls<B2_BF16> : (const void*)b2_k_allreduce_nvls<B2_F16>;
  }
  pick_chunks(c, nbytes, coresident_blocks(c, kern), &a.chunk, &grid);     // (typed kernels: one CTA per SM)
  if (algo == B2_ALGO_NVLS) {
    if (c->dev.stage_mc == nullptr || op != B2_SUM ||
        !(dtype == B2_F32 || dtype == B2_BF16 || dtype == B2_F16)) {
      b2_set_error("%s: NVLS path needs a multicast-bound staging segment and SUM on f32/bf16/f16",
                   name);
      return B2_ERR_BAD_ARG;
    }
    a.algo = B2_ALGO_NVLS;
    if (opcode == B2_OPC_REDUCE) {
      if (dtype == B2_F32) b2_k_reduce_root_nvls<B2_F32><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
      else if (dtype == B2_BF16) b2_k_reduce_root_nvls<B2_BF16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
      else b2_k_reduce_root_nvls<B2_F16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
      return finish_launch(c, cudaGetLastError(), name);
    }
    if (dtype == B2_F32) b2_k_allreduce_nvls<B2_F32><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else if (dtype == B2_BF16) b2_k_allreduce_nvls<B2_BF16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else b2_k_allreduce_nvls<B2_F16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    return finish_launch(c, cudaGetLastError(), name);
  }
  a.algo = (algo == B2_ALGO_TWOSHOT) ? B2_ALGO_TWOSHOT : B2_ALGO_ONESHOT;
  return finish_launch(c, b2_reduce_table[dtype][op](c->dev, a, grid, stream), name);
}

extern "C" int b2_allreduce(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                            int algo, cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "with %zu items", count);
  B2DebugScope* dbg = b2_debug_begin(c, "Allreduce", det, stream);
  int rc = reduce_common(c, in, out, count, dtype, op, algo, 0, c->dev.size, 1, B2_OPC_ALLREDUCE,
                         "allreduce", stream);
  b2_debug_end(dbg, rc);
  return rc;
}

// In-place allreduce (SUM; f32 / bf16 / f16) of a buffer inside a multicast-bound symmetric segment;
// `mc` is the buffer's multicast address (segment multicast base + the buffer's offset).
extern "C" int b2_allreduce_sym(B2Comm* c, void* mc, size_t count, int dtype, cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "with %zu items (symmetric, in place)", count);
  B2DebugScope* dbg = b2_debug_begin(c, "Allreduce", det, stream);
  int rc = 0;
  const size_t nbytes = count * b2_dtype_size(dtype);
  if (!(dtype == B2_F32 || dtype == B2_BF16 || dtype == B2_F16)) {
    b2_set_error("allreduce_: the in-switch reduction supports float32, bfloat16 and float16");
    rc = B2_ERR_BAD_ARG;
  } else if (mc == nullptr || (((uintptr_t)mc) & 15) != 0 || (nbytes & 15) != 0) {
    b2_set_error("allreduce_: the buffer must be 16-byte aligned and a multiple of 16 bytes long");
    rc = B2_ERR_BAD_ARG;
  } else if (nbytes > 0) {
    B2SymArgs a;
    a.mc = (char*)mc; a.nbytes = nbytes; a.opcode = B2_OPC_ALLREDUCE;
    const void* kern = dtype == B2_F32 ? (const void*)b2_k_allreduce_sym<B2_F32>
                       : dtype == B2_BF16 ? (const void*)b2_k_allreduce_sym<B2_BF16> : (const void*)b2_k_allreduce_sym<B2_F16>;
    // one tile of 4 x 512 vectors (32 KiB) per CTA and round at least; never more CTAs than co-resident
    const size_t slice = (nbytes / 16 + c->dev.size - 1) / c->dev.size;
    size_t want = (slice + 4 * B2_THREADS - 1) / (4 * B2_THREADS);
    int grid = coresident_blocks(c, kern);
    if (want < (size_t)grid) grid = (int)(want < 1 ? 1 : want);
    if (dtype == B2_F32) b2_k_allreduce_sym<B2_F32><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else if (dtype == B2_BF16) b2_k_allreduce_sym<B2_BF16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else b2_k_allreduce_sym<B2_F16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    rc = finish_launch(c, cudaGetLastError(), "allreduce_");
  }
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_reduce(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                         int root, cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "with %zu items to root %d", count, root);
  B2DebugScope* dbg = b2_debug_begin(c, "Reduce", det, stream);
  int rc;
  if (root < 0 || root >= c->dev.size) {
    b2_set_error("reduce: invalid root %d", root);
    rc = B2_ERR_BAD_ARG;
  } else {
    const size_t nbytes = count * b2_dtype_size(dtype);
    const bool nvls = c->dev.stage_mc != nullptr && op == B2_SUM && c->dev.size > 2 &&
                      (dtype == B2_F32 || dtype == B2_BF16 || dtype == B2_F16) && nbytes >= c->nvls_min;
    rc = reduce_common(c, in, out, count, dtype, op, nvls ? B2_ALGO_NVLS : B2_ALGO_ONESHOT, 0, c->dev.size,
                       c->dev.rank == root, B2_OPC_REDUCE, "reduce", stream);
  }
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_scan(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                       cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "with %zu items", count);
  B2DebugScope* dbg = b2_debug_begin(c, "Scan", det, stream);
  // small: rank r pulls the copies of ranks 0..r (one phase); large: rank s computes ALL prefixes of
  // sub-slice s and pushes prefix q to rank q (two phases, S bytes in and out per rank instead of
  // up to P * S into the last rank)
  const size_t nbytes = count * b2_dtype_size(dtype);
  const int algo = (c->dev.size > 2 && nbytes > c->oneshot_max) ? B2_ALGO_TWOSHOT : B2_ALGO_ONESHOT;
  int rc = reduce_common(c, in, out, count, dtype, op, algo, 0, c->dev.rank + 1, 1, B2_OPC_SCAN, "scan", stream);
  b2_debug_end(dbg, rc);
  return rc;
}

// Reduce-scatter transports.  "auto" gives the same answer on every rank: it depends only on P, the
// dtype, the op, multicast and the communicator's thresholds.  N = P x block is the input bytes per
// rank, the quantity an allreduce of the same input compares against the same thresholds.
static int reduce_scatter_common(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                                 int algo, cudaStream_t stream) {
  const char* name = "reduce_scatter";
  b2_ensure_tables();
  if (dtype < 0 || dtype >= B2_DTYPE_COUNT || op < 0 || op >= B2_OP_COUNT ||
      b2_rs_table[dtype][op] == nullptr) {
    b2_set_error("%s: unsupported dtype/op combination (dtype=%d, op=%d)", name, dtype, op);
    return B2_ERR_BAD_ARG;
  }
  const size_t blk = count * b2_dtype_size(dtype);
  if (blk == 0) return 0;
  const int P = c->dev.size;
  const size_t N = blk * (size_t)P;
  const bool nvls_ok = c->dev.stage_mc != nullptr && op == B2_SUM &&
                       (dtype == B2_F32 || dtype == B2_BF16 || dtype == B2_F16);
  if (algo == B2_ALGO_AUTO) {
    if (P > 1 && N <= c->ll_max && 2 * blk <= c->dev.lay.ll_cap) algo = B2_ALGO_LL;
    else if (P > 2 && nvls_ok && N >= c->nvls_min) algo = B2_ALGO_NVLS;
    else algo = B2_ALGO_ONESHOT;
  }
  if ((((uintptr_t)out) & 15) != 0) {
    b2_set_error("%s: the output must be 16-byte aligned", name);
    return B2_ERR_BAD_ARG;
  }
  B2RSArgs a;
  a.in = in; a.out = out; a.blk_bytes = blk; a.blk_stride = round_up(blk, 16); a.chunk = 0;
  a.own_in = ((((uintptr_t)in) & 15) == 0 && (blk & 15) == 0) ? 1 : 0;
  a.opcode = B2_OPC_REDUCE_SCATTER;
  int grid;
  if (algo == B2_ALGO_LL) {
    if (2 * blk > c->dev.lay.ll_cap) {
      b2_set_error("%s: LL algorithm needs blocks of <= %zu bytes", name, c->dev.lay.ll_cap / 2);
      return B2_ERR_BAD_ARG;
    }
    const size_t nv = (blk + 15) / 16;
    grid = (int)((nv + B2_THREADS - 1) / B2_THREADS);
    if (grid > c->sm_count) grid = c->sm_count;
    if (grid < 1) grid = 1;
    return finish_launch(c, b2_rs_ll_table[dtype][op](c->dev, a, grid, stream), name);
  }
  if (algo != B2_ALGO_ONESHOT && algo != B2_ALGO_NVLS) {
    b2_set_error("%s: unknown algorithm %d (ll, oneshot or nvls)", name, algo);
    return B2_ERR_BAD_ARG;
  }
  int rc = check_stage(c, B2_OPC_REDUCE_SCATTER, blk, name);
  if (rc) return rc;
  if (algo == B2_ALGO_NVLS) {
    if (!nvls_ok) {
      b2_set_error("%s: NVLS path needs a multicast-bound staging segment and SUM on f32/bf16/f16", name);
      return B2_ERR_BAD_ARG;
    }
    const void* kern = dtype == B2_F32 ? (const void*)b2_k_reduce_scatter_nvls<B2_F32>
                       : dtype == B2_BF16 ? (const void*)b2_k_reduce_scatter_nvls<B2_BF16>
                                          : (const void*)b2_k_reduce_scatter_nvls<B2_F16>;
    pick_chunks(c, blk, coresident_blocks(c, kern), &a.chunk, &grid);
    if (dtype == B2_F32) b2_k_reduce_scatter_nvls<B2_F32><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else if (dtype == B2_BF16) b2_k_reduce_scatter_nvls<B2_BF16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    else b2_k_reduce_scatter_nvls<B2_F16><<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
    return finish_launch(c, cudaGetLastError(), name);
  }
  pick_chunks(c, blk, coresident_blocks(c, nullptr), &a.chunk, &grid);     // (typed kernel: one CTA per SM)
  return finish_launch(c, b2_rs_table[dtype][op](c->dev, a, grid, stream), name);
}

extern "C" int b2_reduce_scatter(B2Comm* c, const void* in, void* out, size_t count, int dtype, int op,
                                 int algo, cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "with %zu items per rank", count);
  B2DebugScope* dbg = b2_debug_begin(c, "Reduce_scatter_block", det, stream);
  int rc = reduce_scatter_common(c, in, out, count, dtype, op, algo, stream);
  b2_debug_end(dbg, rc);
  return rc;
}

static int set_layout(B2MoveArgs& a, const B2Strided* lay, const char* name) {
  a.lay.nd = 0;
  a.in_blk_stride = 0;
  if (lay == nullptr || lay->nd == 0) return 0;
  const int es = lay->esize;
  if (lay->nd < 0 || lay->nd > 4 || !(es == 1 || es == 2 || es == 4 || es == 8 || es == 16)) {
    b2_set_error("%s: unsupported strided layout (nd=%d, element size %d)", name, lay->nd, es);
    return B2_ERR_BAD_ARG;
  }
  long long n = 1;
  for (int d = 0; d < lay->nd; ++d) n *= lay->shape[d];
  if ((size_t)n * (size_t)es != a.blk_bytes) {
    b2_set_error("%s: strided layout does not match the block size", name);
    return B2_ERR_BAD_ARG;
  }
  a.lay = *lay;
  a.in_blk_stride = lay->blk_stride * es;
  return 0;
}

static int move_common(B2Comm* c, B2MoveArgs& a, const char* name, cudaStream_t stream) {
  if (a.blk_bytes == 0) return 0;
  int rc = check_stage(c, a.opcode, a.blk_bytes, name);
  if (rc) return rc;
  a.blk_stride = round_up(a.blk_bytes, 16);
  a.vec_ok = ((((uintptr_t)a.out) & 15) == 0 && (a.blk_bytes % 16 == 0 || a.nsrc <= 1)) ? 1 : 0;
  int grid;
  pick_chunks(c, a.blk_bytes, coresident_blocks(c, (const void*)b2_k_move), &a.chunk, &grid);
  b2_k_move<<<grid, B2_THREADS, 0, stream>>>(c->dev, a);
  return finish_launch(c, cudaGetLastError(), name);
}

extern "C" int b2_allgather(B2Comm* c, const void* in, void* out, size_t blk_bytes, const B2Strided* lay,
                            cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "sending %zu bytes", blk_bytes);
  B2DebugScope* dbg = b2_debug_begin(c, "Allgather", det, stream);
  B2MoveArgs a;
  memset(&a, 0, sizeof a);
  a.in = in; a.out = out; a.blk_bytes = blk_bytes; a.opcode = B2_OPC_ALLGATHER;
  a.nin = 1;
  a.nsrc = c->dev.size;
  for (int q = 0; q < c->dev.size; ++q) { a.src_rank[q] = q; a.src_blk[q] = 0; a.dst_blk[q] = q; }
  int rc = set_layout(a, lay, "allgather");
  if (rc == 0) rc = move_common(c, a, "allgather", stream);
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_alltoall(B2Comm* c, const void* in, void* out, size_t blk_bytes, const B2Strided* lay,
                           cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "sending %zu bytes per peer", blk_bytes);
  B2DebugScope* dbg = b2_debug_begin(c, "Alltoall", det, stream);
  B2MoveArgs a;
  memset(&a, 0, sizeof a);
  a.in = in; a.out = out; a.blk_bytes = blk_bytes; a.opcode = B2_OPC_ALLTOALL;
  a.nin = c->dev.size;
  a.nsrc = c->dev.size;
  for (int q = 0; q < c->dev.size; ++q) {
    a.src_rank[q] = q; a.src_blk[q] = c->dev.rank; a.dst_blk[q] = q;
  }
  int rc = set_layout(a, lay, "alltoall");
  if (rc == 0) rc = move_common(c, a, "alltoall", stream);
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_bcast(B2Comm* c, const void* in, void* out, size_t nbytes, int root, const B2Strided* lay,
                        cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "%zu bytes from root %d", nbytes, root);
  B2DebugScope* dbg = b2_debug_begin(c, "Bcast", det, stream);
  int rc;
  if (root < 0 || root >= c->dev.size) {
    b2_set_error("bcast: invalid root %d", root);
    rc = B2_ERR_BAD_ARG;
  } else {
    B2MoveArgs a;
    memset(&a, 0, sizeof a);
    a.in = in; a.out = out; a.blk_bytes = nbytes; a.opcode = B2_OPC_BCAST;
    if (c->dev.rank == root) { a.nin = 1; a.nsrc = 0; }
    else { a.nin = 0; a.nsrc = 1; a.src_rank[0] = root; a.src_blk[0] = 0; a.dst_blk[0] = 0; }
    rc = set_layout(a, c->dev.rank == root ? lay : nullptr, "bcast");
    // through the switch (one multimem.st stream from the root) once the root's links would be the
    // bottleneck of P-1 pulls; contiguous 16-byte aligned root buffers only (every rank must take
    // the same path: the decision uses sizes only, the root's layout is normalised by the caller)
    const bool mc = c->dev.stage_mc != nullptr && c->dev.size > 2 && nbytes >= c->bcast_mc_min;
    if (rc == 0 && mc && nbytes > 0) {
      if ((rc = check_stage(c, a.opcode, a.blk_bytes, "bcast")) == 0) {
        if (c->dev.rank == root && (a.lay.nd > 0 || (((uintptr_t)in) & 15) != 0)) {
          b2_set_error("bcast: the multicast path needs a contiguous 16-byte aligned root buffer");
          rc = B2_ERR_BAD_ARG;
        } else {
          int grid;
          pick_chunks(c, a.blk_bytes, coresident_blocks(c, (const void*)b2_k_bcast_mc), &a.chunk, &grid);
          b2_k_bcast_mc<<<grid, B2_THREADS, 0, stream>>>(c->dev, a, root);
          rc = finish_launch(c, cudaGetLastError(), "bcast");
        }
      }
    } else if (rc == 0) {
      rc = move_common(c, a, "bcast", stream);
    }
  }
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_gather(B2Comm* c, const void* in, void* out, size_t blk_bytes, int root, const B2Strided* lay,
                         cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "sending %zu bytes to root %d", blk_bytes, root);
  B2DebugScope* dbg = b2_debug_begin(c, "Gather", det, stream);
  int rc;
  if (root < 0 || root >= c->dev.size) {
    b2_set_error("gather: invalid root %d", root);
    rc = B2_ERR_BAD_ARG;
  } else {
    B2MoveArgs a;
    memset(&a, 0, sizeof a);
    a.in = in; a.out = out; a.blk_bytes = blk_bytes; a.opcode = B2_OPC_GATHER;
    a.nin = 1;
    if (c->dev.rank == root) {
      a.nsrc = c->dev.size;
      for (int q = 0; q < c->dev.size; ++q) { a.src_rank[q] = q; a.src_blk[q] = 0; a.dst_blk[q] = q; }
    }
    rc = set_layout(a, lay, "gather");
    if (rc == 0) rc = move_common(c, a, "gather", stream);
  }
  b2_debug_end(dbg, rc);
  return rc;
}

extern "C" int b2_scatter(B2Comm* c, const void* in, void* out, size_t blk_bytes, int root, const B2Strided* lay,
                          cudaStream_t stream) {
  char det[96];
  snprintf(det, sizeof det, "%zu bytes per rank from root %d", blk_bytes, root);
  B2DebugScope* dbg = b2_debug_begin(c, "Scatter", det, stream);
  int rc;
  if (root < 0 || root >= c->dev.size) {
    b2_set_error("scatter: invalid root %d", root);
    rc = B2_ERR_BAD_ARG;
  } else {
    B2MoveArgs a;
    memset(&a, 0, sizeof a);
    a.in = in; a.out = out; a.blk_bytes = blk_bytes; a.opcode = B2_OPC_SCATTER;
    a.nin = (c->dev.rank == root) ? c->dev.size : 0;
    a.nsrc = 1;
    a.src_rank[0] = root; a.src_blk[0] = c->dev.rank; a.dst_blk[0] = 0;
    rc = set_layout(a, c->dev.rank == root ? lay : nullptr, "scatter");
    if (rc == 0) rc = move_common(c, a, "scatter", stream);
  }
  b2_debug_end(dbg, rc);
  return rc;
}
