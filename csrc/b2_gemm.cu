// mpi4jax_b200 -- row-parallel linear layer: GEMM + allreduce in ONE kernel.
//
//   out = allreduce_SUM_over_ranks( X_r (M x K_r, bf16)  @  W_r^T (W_r: N x K_r, bf16) )
//
// This is the tensor-parallel pattern the reference only has as a user-level test
// (column-sharded mat-vec followed by mpi4jax.allreduce,
// tests/collective_ops/test_allreduce_matvec.py:41-65).  There the product is one XLA op and
// the reduction a blocking MPI call afterwards; here both are one sm_100a kernel:
//
//   * 5th-gen tensor cores: `tcgen05.mma.cta_group::1.kind::f16` (128x256x16 UMMA, bf16 in,
//     fp32 accumulate) issued by ONE thread per CTA, operands staged by TMA
//     (`cp.async.bulk.tensor.2d`, 128-byte swizzle) through a 4-stage mbarrier ring, the
//     accumulator lives in TMEM and is read back with `tcgen05.ld`; two accumulator stages
//     (2 x 256 columns = the whole TMEM) let the MMA warp run one tile ahead of the epilogue;
//   * the epilogue warps turn a finished tile into bf16, store it into this rank's SYMMETRIC
//     staging buffer and then all-reduce that tile right there, tile by tile, while the MMA warp
//     is already multiplying the next tile: block-paired cross-GPU barrier (the same tile is
//     owned by the same CTA index on every rank), `multimem.ld_reduce.add.acc::f32.v4.bf16x2` of
//     this rank's 1/P row-slice of the tile (summed in fp32 INSIDE the NVSwitch), `multimem.st`
//     of the result to every rank, second barrier, copy of the finished tile to the output.
//     NVLink traffic equals that of a stand-alone bf16 allreduce, but it is hidden behind the
//     tensor-core work of the following tiles (first version pushed fp32 fragments to all ranks
//     with `multimem.red`: correct but P x the traffic as uncoalesced atomics, 10x slower).
//
// Warp roles (256 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM
// allocator, warps 4-7 = epilogue + per-tile collective (one TMEM lane quarter each).
// Persistent: grid = min(#tiles, #SMs), every CTA walks tiles blockIdx.x, +gridDim.x, ...
// Shapes: M, N multiples of 128, K multiple of 64 (checked by the host wrapper).
#include <cstdio>
#include <cstring>

#include <cuda.h>
#include <cuda_bf16.h>

#include "b2_device.cuh"
#include "b2_runtime.h"
#include "b2_gemm_raster.h"

extern "C" void b2_set_error(const char* fmt, ...);
extern "C" void b2_count_launch(B2Comm* c);
extern "C" int b2_tensor_map_2d_bf16(CUtensorMap* out, const void* ptr, unsigned long long rows,
                                     unsigned long long cols, unsigned box_rows, unsigned box_cols);

namespace {

constexpr int BM = 128, BK = 64, STAGES = 4, UMMA_K = 16;   // BN (128 or 256) is a template parameter
constexpr int GEMM_THREADS = 256;
constexpr uint32_t A_STAGE_BYTES = BM * BK * 2;
// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=bf16 [7,10)=1,
// B=bf16 [10,13)=1, A and B K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29)
template <int BN>
__host__ __device__ constexpr uint32_t idesc_bf16() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

struct GemmArgs {
  int M, N, K;
  __nv_bfloat16* out;
  int fused;           // > 1 rank: per-tile NVLS allreduce through the staging segment
  int raster;          // tile order: 0 = row-major, G > 0 = bands of G tile rows (b2_gemm_raster.h)
};

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t cnt) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(cnt));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t tx) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(tx) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\nbra WAIT_LOOP;\nWAIT_DONE:\n}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// K-major operand tile in shared memory, 128-byte swizzle (cute::UMMA::SmemDescriptor):
// start address >> 4 at [0,14), LBO (unused for swizzled K-major) at [16,30), SBO = 8 rows x 128 B
// = 1024 B >> 4 at [32,46), version = 1 at [46,48), layout SWIZZLE_128B = 2 at [61,64)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(1024u >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accum) {
  asm volatile(
      "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc),
      "r"(idesc), "r"(accum));
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,"
      "%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint4 mc_ld_reduce_bf16(const void* mc) {
  uint4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void mc_st16(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w) : "memory");
}
// cross-GPU barrier executed by the 128 epilogue threads only (named barrier 1), CTA b <-> CTA b
__device__ __forceinline__ void epi_barrier_all(const B2DevComm& c, unsigned e, int et) {
  asm volatile("bar.sync 1, 128;" ::: "memory");
  if (et < c.size) {
    unsigned* remote = (unsigned*)(c.heap[et] + c.lay.flags_off) + (size_t)blockIdx.x * B2_MAX_RANKS + c.rank;
    b2_st_release_sys(remote, e);
    const unsigned* local =
        (const unsigned*)(c.heap[c.rank] + c.lay.flags_off) + (size_t)blockIdx.x * B2_MAX_RANKS + et;
    b2_wait_ge(c, local, e, B2_OPC_ALLREDUCE, et);
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
}

template <int BN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
b2_k_gemm_allreduce(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                    const B2DevComm c, const GemmArgs g) {
  constexpr uint32_t B_STAGE_BYTES = BN * BK * 2, TMEM_COLS = 2 * BN, IDESC = idesc_bf16<BN>();
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], tmem_full_bar[2], tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = ((uint32_t)__cvta_generic_to_shared(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base, smem_b = smem_base + STAGES * A_STAGE_BYTES;
  auto bar = [](uint64_t* p) { return (uint32_t)__cvta_generic_to_shared(p); };

  unsigned ticket = 0, e = 0;
  if (g.fused) {
    ticket = b2_ticket_read(c.ticket);
    e = b2_ld_volatile(c.epoch + blockIdx.x);
  }
  const size_t par = (size_t)(ticket & 1u) * c.stage_half;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar(&full_bar[s]), 1); mbar_init(bar(&empty_bar[s]), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar(&tmem_full_bar[a]), 1); mbar_init(bar(&tmem_empty_bar[a]), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&tmem_base_s)), "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;");
  const uint32_t tmem_base = tmem_base_s;

  const int num_n = g.N / BN, tiles = (g.M / BM) * num_n, num_kb = g.K / BK;

  if (warp == 0 && lane == 0) {
    // ===== TMA producer =====
    uint32_t stage = 0, phase = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      int m_blk, n_blk;
      b2_gemm_tile_coords(tile, g.M / BM, num_n, g.raster, m_blk, n_blk);
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(bar(&empty_bar[stage]), phase ^ 1u);
        mbar_expect_tx(bar(&full_bar[stage]), A_STAGE_BYTES + B_STAGE_BYTES);
        tma_load_2d(smem_a + stage * A_STAGE_BYTES, &tma_a, bar(&full_bar[stage]), kb * BK, m_blk * BM);
        tma_load_2d(smem_b + stage * B_STAGE_BYTES, &tma_b, bar(&full_bar[stage]), kb * BK, n_blk * BN);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ===== MMA issuer (one thread) =====
    uint32_t stage = 0, phase = 0, it = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const uint32_t as = it & 1u, aph = (it >> 1) & 1u;        // accumulator stage / its phase
      mbar_wait(bar(&tmem_empty_bar[as]), aph ^ 1u);            // epilogue drained this accumulator
      asm volatile("tcgen05.fence::after_thread_sync;");
      const uint32_t tmem_d = tmem_base + as * (uint32_t)BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(bar(&full_bar[stage]), phase);                // TMA landed this stage
        asm volatile("tcgen05.fence::after_thread_sync;");
        const uint64_t adesc = umma_desc(smem_a + stage * A_STAGE_BYTES);
        const uint64_t bdesc = umma_desc(smem_b + stage * B_STAGE_BYTES);
#pragma unroll
        for (int k = 0; k < BK / UMMA_K; ++k)                   // +32 B per UMMA_K inside the swizzle atom
          umma_bf16(tmem_d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), IDESC, (kb | k) != 0);
        umma_commit(bar(&empty_bar[stage]));                    // frees the smem stage when the MMAs retire
        if (kb == num_kb - 1) umma_commit(bar(&tmem_full_bar[as])); // accumulator complete
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: TMEM -> bf16 -> (staging + per-tile NVLS allreduce | output) =====
    const int q = warp & 3;                                     // TMEM lane quarter of this warp
    const int et = threadIdx.x - 128;                           // 0..127 within the epilogue group
    __nv_bfloat16* stage_local = (__nv_bfloat16*)(c.stage[c.rank] + par);
    __nv_bfloat16* stage_mc = (__nv_bfloat16*)(c.stage_mc + par);
    uint32_t it = 0;
    constexpr int GROUP = 4;                                    // tiles per collective round
    int pend[GROUP], np = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const uint32_t as = it & 1u, aph = (it >> 1) & 1u;
      int m_blk, n_blk;
      b2_gemm_tile_coords(tile, g.M / BM, num_n, g.raster, m_blk, n_blk);
      mbar_wait(bar(&tmem_full_bar[as]), aph);
      asm volatile("tcgen05.fence::after_thread_sync;");
      const size_t row = (size_t)m_blk * BM + q * 32 + lane;
      __nv_bfloat16* dst_base = (g.fused ? stage_local : g.out) + row * g.N + (size_t)n_blk * BN;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        uint32_t v[32];
        tmem_ld32(tmem_base + as * (uint32_t)BN + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 32), v);
        __nv_bfloat16* dst = dst_base + ch * 32;
#pragma unroll
        for (int i = 0; i < 32; i += 8) {
          __nv_bfloat162 p0 = __floats2bfloat162_rn(__uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          __nv_bfloat162 p1 = __floats2bfloat162_rn(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
          __nv_bfloat162 p2 = __floats2bfloat162_rn(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5]));
          __nv_bfloat162 p3 = __floats2bfloat162_rn(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7]));
          uint4 pk;
          pk.x = *reinterpret_cast<uint32_t*>(&p0); pk.y = *reinterpret_cast<uint32_t*>(&p1);
          pk.z = *reinterpret_cast<uint32_t*>(&p2); pk.w = *reinterpret_cast<uint32_t*>(&p3);
          *reinterpret_cast<uint4*>(dst + i) = pk;
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(&tmem_empty_bar[as]));     // accumulator free: MMA warp runs ahead
      if (g.fused) {
        // --- all-reduce finished tiles across the ranks while the next tiles are being multiplied.
        // GROUP tiles share one pair of cross-GPU barriers; all loads of a batch are issued before
        // the first dependent store so the NVLink / L2 round trips overlap instead of adding up.
        pend[np++] = tile;
        const bool last = tile + (int)gridDim.x >= tiles;
        if (np == GROUP || last) {
          epi_barrier_all(c, ++e, et);                          // every rank staged these partial tiles
          const int per = (BM + c.size - 1) / c.size;           // my row-slice of every tile
          const int r0 = per * c.rank < BM ? per * c.rank : BM, r1 = r0 + per < BM ? r0 + per : BM;
          const int slice_vec = (r1 - r0) * (BN / 8), nred = np * slice_vec;
          for (int base = et; base < nred; base += 128 * 4) {
            uint4 v[4];
            size_t offs[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int i = base + u * 128;
              if (i < nred) {
                const int slot = i / slice_vec, w = i - slot * slice_vec;
                const int tl = pend[slot], r = r0 + w / (BN / 8), v8 = w % (BN / 8);
                int tm, tn;
                b2_gemm_tile_coords(tl, g.M / BM, num_n, g.raster, tm, tn);
                offs[u] = ((size_t)tm * BM + r) * g.N + (size_t)tn * BN + v8 * 8;
                v[u] = mc_ld_reduce_bf16(stage_mc + offs[u]);   // fp32 sum inside the NVSwitch
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (base + u * 128 < nred) mc_st16(stage_mc + offs[u], v[u]);   // broadcast to every rank
          }
          epi_barrier_all(c, ++e, et);                          // all slices of these tiles have landed
          const int ncp = np * BM * (BN / 8);
          for (int base = et; base < ncp; base += 128 * 8) {
            uint4 v[8];
            size_t offs[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int i = base + u * 128;
              if (i < ncp) {
                const int slot = i / (BM * (BN / 8)), w = i - slot * (BM * (BN / 8));
                const int tl = pend[slot], r = w / (BN / 8), v8 = w % (BN / 8);
                int tm, tn;
                b2_gemm_tile_coords(tl, g.M / BM, num_n, g.raster, tm, tn);
                offs[u] = ((size_t)tm * BM + r) * g.N + (size_t)tn * BN + v8 * 8;
                v[u] = b2_ld_peer16(stage_local + offs[u]);
              }
            }
#pragma unroll
            for (int u = 0; u < 8; ++u)
              if (base + u * 128 < ncp) b2_st16(g.out + offs[u], v[u]);
          }
          np = 0;
        }
      }
    }
    if (g.fused && et == 0) b2_st_volatile(c.epoch + blockIdx.x, e);
  }

  __syncthreads();
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
  if (g.fused) b2_finish_bump(c.ticket, c.ticket + 1, 1u, gridDim.x);
}

}  // namespace

// out (M x N, bf16) = sum over ranks of A (M x K, bf16, row-major) @ B^T (B: N x K, bf16, row-major).
// Multi-rank calls stage the bf16 partial tiles in the communicator's multicast-bound staging
// segment (M*N*2 bytes per parity; grown by the Python layer like for any other collective).
extern "C" int b2_gemm_allreduce(B2Comm* c, const void* A, const void* B, void* out, int M, int N, int K,
                                 cudaStream_t stream) {
  if (M <= 0 || N <= 0 || K <= 0 || M % BM || N % 128 || K % BK) {
    b2_set_error("gemm_allreduce: need M %% %d == 0, N %% %d == 0, K %% %d == 0 (got %d, %d, %d)", BM, 128,
                 BK, M, N, K);
    return B2_ERR_BAD_ARG;
  }
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.M = M; g.N = N; g.K = K;
  g.out = (__nv_bfloat16*)out;
  g.fused = (c->dev.size > 1) ? 1 : 0;
  // banded tile order for the stand-alone GEMM; the fused epilogue recomputes a tile's coordinates per
  // 16-byte vector (integer divisions in front of every multimem load), where the banded formula costs
  // more than it gains: 2 GPUs, 4096 x 4096 x 2048: 293 us banded vs 177 us row-major
  // (profiles/r2_gemm_fused_2gpu_banded.log, r1_gemm_allreduce_fused_2gpu.log) -- row-major there
  // until the coordinates are hoisted out of those loops
  g.raster = g.fused ? 0 : B2_GEMM_RASTER_GROUP;
  if (g.fused) {
    if (c->dev.stage_mc == nullptr) {
      b2_set_error("gemm_allreduce: multi-rank call needs a multicast-bound staging segment (NVLS)");
      return B2_ERR_BAD_ARG;
    }
    if ((size_t)M * N * 2 + 4096 > c->dev.stage_half) {
      b2_set_error("gemm_allreduce: staging too small (need %zu bytes, have %zu)", (size_t)M * N * 2 + 4096,
                   c->dev.stage_half);
      return B2_ERR_BAD_ARG;
    }
  }
  const int BN = (N % 256 == 0) ? 256 : 128;      // 128x256 tiles halve the MMA count per FLOP
  CUtensorMap ta, tb;
  if (b2_tensor_map_2d_bf16(&ta, A, (unsigned long long)M, (unsigned long long)K, BM, BK) ||
      b2_tensor_map_2d_bf16(&tb, B, (unsigned long long)N, (unsigned long long)K, BN, BK))
    return B2_ERR_BAD_ARG;
  const size_t smem = (size_t)STAGES * (A_STAGE_BYTES + (size_t)BN * BK * 2) + 1024;
  static bool attr_set[2] = {false, false};
  if (!attr_set[BN == 256]) {
    cudaError_t e = BN == 256
        ? cudaFuncSetAttribute(b2_k_gemm_allreduce<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
        : cudaFuncSetAttribute(b2_k_gemm_allreduce<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      b2_set_error("gemm_allreduce: cannot reserve %zu bytes of shared memory: %s", smem,
                   cudaGetErrorString(e));
      return 1000 + (int)e;
    }
    attr_set[BN == 256] = true;
  }
  const int tiles = (M / BM) * (N / BN);
  int grid = tiles < c->sm_count ? tiles : c->sm_count;
  if (grid > B2_MAX_BLOCKS) grid = B2_MAX_BLOCKS;
  if (BN == 256) b2_k_gemm_allreduce<256><<<grid, GEMM_THREADS, smem, stream>>>(ta, tb, c->dev, g);
  else b2_k_gemm_allreduce<128><<<grid, GEMM_THREADS, smem, stream>>>(ta, tb, c->dev, g);
  b2_count_launch(c);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    b2_set_error("gemm_allreduce: kernel launch failed: %s", cudaGetErrorString(err));
    return 1000 + (int)err;
  }
  return 0;
}
