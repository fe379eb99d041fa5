// mpi4jax_b200 -- reduce-scatter (MPI_Reduce_scatter_block) over peer-mapped HBM: the typed kernels.
//
// Every rank passes `in` = P blocks of `blk_bytes`; rank r receives op over all ranks q of block r of
// q's input.  Two transports live here, instantiated for every (dtype, op) through B2_REG
// (b2_reduce.cuh); the in-switch one (SUM on f32 / bf16 / f16) is b2_k_reduce_scatter_nvls in
// b2_collectives.cu.
//   * LL       rank r pushes block q straight into rank q's flag-in-data buffer, then folds the P
//              pieces of block r as they arrive: no barrier, no staging.
//   * ONESHOT  stage the P pieces of a chunk -> barrier -> pull piece r of every rank and fold.
// Both fold in rank order 0..P-1 with the same accumulator as the allreduce kernels, so block r of
// an allreduce with the same transport is bitwise equal to this rank's result.
#pragma once

#include "b2_device.cuh"

struct B2RSArgs {
  const void* in;
  void* out;
  size_t blk_bytes;    // bytes of one block = bytes of the result
  size_t blk_stride;   // staging stride between the pieces of a chunk (blk_bytes rounded up to 16)
  size_t chunk;        // ONESHOT / NVLS: chunk bytes of a block (multiple of 16 * size)
  int own_in;          // input 16-byte aligned and blk_bytes a multiple of 16: whole-vector loads from
                       // every block (ONESHOT: this rank's own piece is read from the input, not staged)
  int opcode;
};

// Vector `b / 16` of one input block.  A block that is not a multiple of 16 bytes leaves the blocks
// after it unaligned even when the input is aligned: byte-wise load, zero padded past the block end.
__device__ __forceinline__ uint4 b2_rs_ld_vec(const char* blk, size_t b, size_t nbytes) {
  if ((((uintptr_t)blk) & 15) == 0 && b + 16 <= nbytes) return *reinterpret_cast<const uint4*>(blk + b);
  alignas(16) unsigned char tmp[16];
  for (int k = 0; k < 16; ++k) tmp[k] = (b + k < nbytes) ? ((const unsigned char*)blk)[b + k] : 0;
  return *reinterpret_cast<const uint4*>(tmp);
}

// ---------------------------------------------------------------------------
// LL reduce-scatter.  Same wire format, flag (ticket + 1) and ticket-parity buffers as
// b2_k_allreduce_ll: rank r writes vector i of block q into rank q's LL buffer, slot [source r],
// as {w0, flag, w1, flag} {w2, flag, w3, flag}; rank q polls its P - 1 slots for vector i.
// Parity argument (as for the LL allreduce): a sender reuses this launch's buffers two tickets
// later, and to finish the ticket in between it needs this rank's contribution to it -- every rank
// receives from every peer in each launch of this kernel (and every other collective kernel waits
// for every peer) -- which this rank only sends after it has finished reading this launch's data.
// ---------------------------------------------------------------------------
template <typename T, int OP>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_reduce_scatter_ll(const B2DevComm c, const B2RSArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const unsigned flag = ticket + 1u;
  const size_t par_off = c.lay.ll_off + (size_t)(ticket & 1u) * c.size * c.lay.ll_cap;
  const size_t nb = a.blk_bytes;
  const size_t nv = (nb + 15) >> 4;
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  const char* own = in + (size_t)c.rank * nb;

  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i << 4;
    // push vector i of block p to peer p, slot [source = my rank]
    for (int q = 1; q < c.size; ++q) {
      const int p = (c.rank + q) % c.size;
      const uint4 v = b2_rs_ld_vec(in + (size_t)p * nb, b, nb);
      char* dst = c.heap[p] + par_off + (size_t)c.rank * c.lay.ll_cap + (i << 5);
      b2_st16_sys(dst, make_uint4(v.x, flag, v.y, flag));
      b2_st16_sys(dst + 16, make_uint4(v.z, flag, v.w, flag));
    }
    // gather block `rank` from every peer and reduce in rank order (own piece straight from the input)
    B2Vec<T> acc;
    unsigned long long t0 = 0;
    unsigned spins = 0;
    for (int q = 0; q < c.size; ++q) {
      uint4 v;
      if (q == c.rank) {
        v = b2_rs_ld_vec(own, b, nb);
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
    if (b + 16 <= nb) b2_st16(out + b, r);
    else b2_store_partial(out + b, r, (int)(nb - b));
  }
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// ---------------------------------------------------------------------------
// One-shot reduce-scatter by pull.  Chunk k of a block is staged as P pieces, piece q (chunk k of
// block q) at staging offset q * blk_stride + k * chunk; after the barrier rank r pulls piece r of
// every rank.  One barrier per chunk is enough, as in the one-shot allreduce: nobody writes a
// chunk's staging again in this launch, and the next launch uses the other parity.
// ---------------------------------------------------------------------------
template <typename T, int OP>
__global__ void __launch_bounds__(B2_THREADS)
b2_k_reduce_scatter(const B2DevComm c, const B2RSArgs a) {
  const unsigned ticket = b2_ticket_read(c.ticket);
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;
  unsigned e = b2_ld_volatile(c.epoch + blockIdx.x);
  const char* in = (const char*)a.in;
  char* out = (char*)a.out;
  char* mine = c.stage[c.rank] + par;
  const size_t nb = a.blk_bytes, st = a.blk_stride;
  const size_t nchunks = (nb + a.chunk - 1) / a.chunk;
  const size_t piece = (size_t)c.rank * st;               // where every rank staged block `rank`
  const char* own = in + (size_t)c.rank * nb;
  const int t = threadIdx.x, nt = blockDim.x;

  for (size_t ch = blockIdx.x; ch < nchunks; ch += gridDim.x) {
    const size_t off = ch * a.chunk;
    const size_t len = (nb - off < a.chunk) ? (nb - off) : a.chunk;
    const size_t nv = (len + 15) >> 4;        // vectors incl. a padded tail vector
    // 1. stage this chunk of every block (this rank's own block only if it cannot be read in place)
    for (int q = 0; q < c.size; ++q)
      if (q != c.rank || !a.own_in)
        b2_copy_bytes<false>(mine + (size_t)q * st + off, in + (size_t)q * nb + off, len);
    // 2. every rank staged this chunk
    b2_barrier_all(c, ++e, a.opcode);
    // 3. pull piece `rank` of every rank (all P loads in flight) and fold in rank order
    for (size_t i = t; i < nv; i += nt) {
      const size_t b = i << 4;
      uint4 v[B2_MAX_RANKS];
#pragma unroll
      for (int q = 0; q < B2_MAX_RANKS; ++q)
        if (q < c.size)
          v[q] = (q == c.rank && a.own_in) ? b2_ld_stream16(own + off + b)
                                           : b2_ld_peer16(c.stage[q] + par + piece + off + b);
      B2Vec<T> acc;
      acc.load(v[0]);
#pragma unroll
      for (int q = 1; q < B2_MAX_RANKS; ++q)
        if (q < c.size) acc.template accumulate<OP>(v[q]);
      const uint4 r = acc.store();
      if (b + 16 <= len) b2_st16(out + off + b, r);
      else b2_store_partial(out + off + b, r, (int)(len - b));
    }
  }
  __syncthreads();
  if (t == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

// host-side typed dispatch (tables filled by B2_REG in the instance files)
typedef cudaError_t (*b2_rs_launch_fn)(const B2DevComm&, const B2RSArgs&, int grid, cudaStream_t);

template <typename T, int OP>
cudaError_t b2_launch_rs(const B2DevComm& c, const B2RSArgs& a, int grid, cudaStream_t s) {
  b2_k_reduce_scatter<T, OP><<<grid, B2_THREADS, 0, s>>>(c, a);
  return cudaGetLastError();
}
template <typename T, int OP>
cudaError_t b2_launch_rs_ll(const B2DevComm& c, const B2RSArgs& a, int grid, cudaStream_t s) {
  b2_k_reduce_scatter_ll<T, OP><<<grid, B2_THREADS, 0, s>>>(c, a);
  return cudaGetLastError();
}

extern b2_rs_launch_fn b2_rs_table[B2_DTYPE_COUNT][B2_OP_COUNT];
extern b2_rs_launch_fn b2_rs_ll_table[B2_DTYPE_COUNT][B2_OP_COUNT];
