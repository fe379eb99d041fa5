// mpi4jax_b200 -- reduction collectives over peer-mapped HBM (allreduce, reduce, scan).
//
// Replaces the reference's MPI_Allreduce / MPI_Reduce / MPI_Scan call sites
// (mpi4jax/_src/xla_bridge/mpi_ops_common.h:236-249, 310-338 and their CUDA
// callers mpi_xla_bridge_cuda.cpp:167-209, 523-632) with hand-written sm_100a
// kernels in which the reduction operator and the dtype up/down-cast are FUSED
// into the NVLink transfer: no MPI call, no host sync, no staging through host
// memory, no separate elementwise kernel.
//
// Three transports, chosen per message size by b2_allreduce():
//   * LL        flag-in-data push (8 B = 4 B payload + 4 B flag), no barrier, no
//               fence: one NVLink one-way latency.            (<= ll_max bytes)
//   * ONESHOT   stage -> barrier -> every rank pulls all P copies and reduces.
//   * TWOSHOT   stage -> barrier -> rank r reduces sub-slice r (pull) and pushes
//               the result into every peer's staging -> barrier -> copy out.
// Work is split into chunks owned by CTA (chunk mod grid) ON EVERY RANK, so all
// synchronisation is CTA<->same-CTA across GPUs (block-paired flags): CTAs are
// at different phases at any instant, which overlaps the local copy-in/copy-out
// with the NVLink reduce-scatter and all-gather phases of other chunks.
#pragma once

#include "b2_device.cuh"
#include "b2_reduce_scatter.cuh"

struct B2ReduceArgs {
  const void* in;
  void* out;
  size_t nbytes;     // payload bytes per rank
  size_t chunk;      // chunk bytes; multiple of 16 * size
  int algo;          // B2_ALGO_ONESHOT or B2_ALGO_TWOSHOT
  int src_lo;        // contributions reduced: ranks [src_lo, src_hi)
  int src_hi;
  int has_out;       // this rank materialises a result (reduce: root only)
  int opcode;
  int pipeline;      // NVLS allreduce: stage the next chunk / copy the previous one out between arrive and wait
  unsigned long long* trace;   // optional phase timeline of CTA 0 (communicator option "trace_ptr"), else null
  int trace_cap;
};

template <typename T, int OP>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_reduce_chunked(const B2DevComm c, const B2ReduceArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  const size_t nchunks = (a.nbytes + a.chunk - 1) / a.chunk;
  const int t = threadIdx.x, nt = blockDim.x;

  for (size_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const size_t off = ch * a.chunk;
    const size_t len = (a.nbytes - off < a.chunk) ? (a.nbytes - off) : a.chunk;
    const size_t nv = (len + 15) >> 4;        // vectors incl. a padded tail vector
    // 1. stage my contribution (local HBM -> local symmetric staging)
    b2_copy_bytes<false>(mine + off, in + off, len);
    // 2. everybody's copy of this chunk is staged
    b2_barrier_all(c, ++e, a.opcode);

    if (a.algo == B2_ALGO_ONESHOT) {
      if (a.has_out) {
        for (size_t i = t; i < nv; i += nt) {
          B2Vec<T> acc;
          acc.load(b2_ld_peer16(c.stage[a.src_lo] + par + off + (i << 4)));
          for (int q = a.src_lo + 1; q < a.src_hi; ++q)
            acc.template accumulate<OP>(b2_ld_peer16(c.stage[q] + par + off + (i << 4)));
          const uint4 r = acc.store();
          const size_t b = i << 4;
          if (b + 16 <= len) b2_st16(out + off + b, r);
          else b2_store_partial(out + off + b, r, (int)(len - b));
        }
      }
    } else {
      // 3. reduce-scatter by pull: rank r owns vectors [v0, v1) of this chunk
      const size_t per = (nv + c.size - 1) / c.size;
      size_t v0 = per * (size_t)c.rank;
      if (v0 > nv) v0 = nv;
      size_t v1 = v0 + per;
      if (v1 > nv) v1 = nv;
      if (a.opcode == B2_OPC_SCAN) {
        // two-phase scan: all P copies of a vector are loaded BEFORE the prefixes overwrite them
        // (prefix q lands where rank q staged its own contribution; this rank is the only reader)
        for (size_t i = v0 + t; i < v1; i += nt) {
          uint4 v[B2_MAX_RANKS];
#pragma unroll
          for (int q = 0; q < B2_MAX_RANKS; ++q)
            if (q < c.size) v[q] = b2_ld_peer16(c.stage[q] + par + off + (i << 4));
          B2Vec<T> acc;
          acc.load(v[0]);
#pragma unroll
          for (int q = 1; q < B2_MAX_RANKS; ++q)
            if (q < c.size) {
              acc.template accumulate<OP>(v[q]);
              b2_st16(c.stage[q] + par + off + (i << 4), acc.store());
            }
        }
      } else
      for (size_t i = v0 + t; i < v1; i += nt) {
        B2Vec<T> acc;
        acc.load(b2_ld_peer16(c.stage[0] + par + off + (i << 4)));
        for (int q = 1; q < c.size; ++q)
          acc.template accumulate<OP>(b2_ld_peer16(c.stage[q] + par + off + (i << 4)));
        const uint4 r = acc.store();
        // 4. all-gather by push: result goes straight into every peer's staging
        for (int q = 0; q < c.size; ++q) {
          const int p = (c.rank + q) % c.size;   // stagger destinations across ranks
          b2_st16(c.stage[p] + par + off + (i << 4), r);
        }
      }
      // 5. every sub-slice of this chunk has landed in my staging
      b2_barrier_all(c, ++e, a.opcode);
      // 6. staging -> user output
      if (a.has_out) b2_copy_bytes<true>(out + off, mine + off, len);
    }
  }
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// LL allreduce.  Wire format per 16-byte payload vector: two 16-byte stores
// {w0, flag, w1, flag} {w2, flag, w3, flag}; each 8-byte half is written
// atomically, so a reader that sees `flag` in a half sees its payload word.
// flag = ticket + 1 (never 0, unique for 2^32 launches; buffers alternate by
// ticket parity so a sender can never overwrite data that is still being read:
// to be two tickets ahead it needs this rank's contribution to the ticket in
// between, which this rank only sends after it finished reading).
// ---------------------------------------------------------------------------
struct B2LLArgs {
  const void* in;
  void* out;
  size_t nbytes;
  int opcode;
};

template <typename T, int OP>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_allreduce_ll(const B2DevComm c, const B2LLArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const unsigned flag = ticket + 1u;
  const size_t par_off = c.lay.ll_off + (size_t)(ticket & 1u) * c.size * c.lay.ll_cap;
  const size_t nv = (a.nbytes + 15) >> 4;
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  const bool aligned = (((uintptr_t)in) & 15) == 0;

  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i << 4;
    uint4 mine;
    if (aligned && b + 16 <= a.nbytes) {
      mine = *reinterpret_cast<const uint4*>(in + b);
    } else {
      alignas(16) unsigned char tmp[16];
      for (int k = 0; k < 16; ++k) tmp[k] = (b + k < a.nbytes) ? ((const unsigned char*)in)[b + k] : 0;
      mine = *reinterpret_cast<const uint4*>(tmp);
    }
    // push to every peer's LL buffer, slot [source = my rank][vector i]
    const uint4 lo = make_uint4(mine.x, flag, mine.y, flag);
    const uint4 hi = make_uint4(mine.z, flag, mine.w, flag);
    for (int q = 1; q < c.size; ++q) {
      const int p = (c.rank + q) % c.size;
      char* dst = c.heap[p] + par_off + (size_t)c.rank * c.lay.ll_cap + (i << 5);
      b2_st16_sys(dst, lo);
      b2_st16_sys(dst + 16, hi);
    }
    // gather + reduce in rank order (bitwise identical result on every rank)
    B2Vec<T> acc;
    unsigned long long t0 = 0;
    unsigned spins = 0;
    for (int q = 0; q < c.size; ++q) {
      uint4 v;
      if (q == c.rank) {
        v = mine;
      } else {
        const char* src = c.heap[c.rank] + par_off + (size_t)q * c.lay.ll_cap + (i << 5);
        uint4 l, h;
        while (true) {
          l = b2_ld_peer16(src);
          h = b2_ld_peer16(src + 16);
          if (l.y == flag && l.w == flag && h.y == flag && h.w == flag) break;
          if ((++spins & 0xfffu) == 0) {
            unsigned long long now = b2_gtime();
            if (t0 == 0) t0 = now;
            else if (now - t0 > c.timeout_ns)
              b2_fatal(c, B2_ERR_TIMEOUT, a.opcode, q, flag, l.y, 2);
          }
        }
        v = make_uint4(l.x, l.z, h.x, h.z);
      }
      if (q == 0) acc.load(v);
      else acc.template accumulate<OP>(v);
    }
    const uint4 r = acc.store();
    if (b + 16 <= a.nbytes) b2_st16(out + b, r);
    else b2_store_partial(out + b, r, (int)(a.nbytes - b));
  }
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// host-side typed dispatch.  Each instance file defines B2_INST_GROUP and gets
// the launchers for its dtype group only (keeps nvcc parallel and fast).
// ---------------------------------------------------------------------------
typedef cudaError_t (*b2_reduce_launch_fn)(const B2DevComm&, const B2ReduceArgs&, int grid,
                                           cudaStream_t);
typedef cudaError_t (*b2_ll_launch_fn)(const B2DevComm&, const B2LLArgs&, int grid, cudaStream_t);

template <typename T, int OP>
cudaError_t b2_launch_reduce(const B2DevComm& c, const B2ReduceArgs& a, int grid, cudaStream_t s) {
  b2_k_reduce_chunked<T, OP><<<grid, B2_THREADS, 0, s>>>(c, a);
  return cudaGetLastError();
}
template <typename T, int OP>
cudaError_t b2_launch_ll(const B2DevComm& c, const B2LLArgs& a, int grid, cudaStream_t s) {
  b2_k_allreduce_ll<T, OP><<<grid, B2_THREADS, 0, s>>>(c, a);
  return cudaGetLastError();
}

// tables filled by the instance files: [dtype][op] -> launcher (nullptr = invalid combo)
extern b2_reduce_launch_fn b2_reduce_table[B2_DTYPE_COUNT][B2_OP_COUNT];
extern b2_ll_launch_fn b2_ll_table[B2_DTYPE_COUNT][B2_OP_COUNT];

#define B2_REG(DT, T, OP)                               \
  b2_reduce_table[DT][OP] = &b2_launch_reduce<T, OP>;   \
  b2_ll_table[DT][OP] = &b2_launch_ll<T, OP>;           \
  b2_rs_table[DT][OP] = &b2_launch_rs<T, OP>;           \
  b2_rs_ll_table[DT][OP] = &b2_launch_rs_ll<T, OP>;

#define B2_REG_ARITH(DT, T) \
  B2_REG(DT, T, B2_SUM) B2_REG(DT, T, B2_PROD) B2_REG(DT, T, B2_MIN) B2_REG(DT, T, B2_MAX)
#define B2_REG_INT(DT, T)                                                              \
  B2_REG_ARITH(DT, T) B2_REG(DT, T, B2_LAND) B2_REG(DT, T, B2_LOR) B2_REG(DT, T, B2_LXOR) \
  B2_REG(DT, T, B2_BAND) B2_REG(DT, T, B2_BOR) B2_REG(DT, T, B2_BXOR)
