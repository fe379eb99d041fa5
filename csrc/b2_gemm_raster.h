// mpi4jax_b200 -- tile order of the persistent GEMM kernels (csrc/b2_gemm.cu).
//
// tile index -> (m_blk, n_blk).  Group 0: row-major over the tile grid.  B2_GEMM_RASTER_GROUP = G > 0: tiles are visited in bands of G
// M-blocks, column by column inside a band, so that the ~148 tiles in flight cover G rows x ~148/G
// columns of the tile grid: A row-panels are reused ~148/G times and B column-panels G times from
// L2 instead of (148 / num_n) rows x all columns (B larger than L2 at 8192^3).  Every rank uses
// the same order (the fused all-reduce pairs tile t of all ranks).
#pragma once

#ifndef B2_GEMM_RASTER_GROUP
#define B2_GEMM_RASTER_GROUP 2     // measured (profiles/r2_gemm_raster_sweep_1gpu.log): never slower than row-major,
#endif                               // +6 % at 2048x4096x4096, +12 % at 16384x8192x4096


#ifdef __CUDACC__
#define B2_HD __host__ __device__
#else
#define B2_HD
#endif

// `group` = G of the description above (0 = row-major); a launch parameter (b2_gemm.cu picks it
// per launch), B2_GEMM_RASTER_GROUP is the compile-time default.
B2_HD inline void b2_gemm_tile_coords(int tile, int num_m, int num_n, int group, int& m_blk, int& n_blk) {
  if (group > 0) {
    const int G = group;
    const int per_band = G * num_n;
    const int band = tile / per_band;
    const int first_m = band * G;
    const int rows = (num_m - first_m) < G ? (num_m - first_m) : G;   // the last band may be thinner
    const int r = tile - band * per_band;
    m_blk = first_m + r % rows;
    n_blk = r / rows;
  } else {
    m_blk = tile / num_n;
    n_blk = tile % num_n;
  }
}
B2_HD inline void b2_gemm_tile_coords(int tile, int num_m, int num_n, int& m_blk, int& n_blk) {
  b2_gemm_tile_coords(tile, num_m, num_n, B2_GEMM_RASTER_GROUP, m_blk, n_blk);
}
