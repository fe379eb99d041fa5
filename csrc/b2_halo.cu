// mpi4jax_b200 -- fused multi-field 2-D halo exchange.
//
// The reference's flagship workload (examples/shallow_water.py:172-264,
// `enforce_boundaries`) exchanges a 1-cell halo with up to four neighbours by
// issuing, per field, 2 sendrecv + 1 send + 1 recv custom calls, each of them a
// blocking MPI call behind a full stream synchronisation, with XLA gather /
// dynamic-update-slice kernels around them for the strided column pack and the
// halo unpack (48 custom calls per model step at 8 ranks, SURVEY.md section 3.4).
//
// Here ONE kernel launch exchanges the halos of up to B2_HALO_MAX_FIELDS fields
// with all EIGHT neighbours in a single phase: strided column pack, NVLink put
// straight into the neighbour's symmetric receive buffer, halo unpack and the
// physical wall conditions, all fused.
//
// Why eight neighbours: the reference's west/north/east/south message order
// makes every corner halo cell end up with the DIAGONAL neighbour's interior
// corner value (it travels through two hops: columns first, then rows carrying
// the fresh corner).  Sending that value directly from the diagonal rank gives
// bit-identical halos with one NVLink latency instead of two.  Where a rank
// touches a y wall the wall-row cells of the halo columns come from the W/E
// neighbours' wall rows, exactly as in the reference's sequence.
//
// Every element is pushed as one 8-byte {value, flag} store and the receiver
// polls the data itself: one NVLink one-way latency (transport: b2_halo_ll.cuh).
// Receive buffers are double-buffered on device-side per-side message counters,
// so no "ready" handshake is needed and the kernel is CUDA-graph replayable.
#include <cstdio>
#include <cstring>

#include "b2_device.cuh"
#include "b2_halo_ll.cuh"
#include "b2_runtime.h"

extern "C" void b2_set_error(const char* fmt, ...);
extern "C" void b2_count_launch(B2Comm* c);

#define HALO_THREADS 256
#define HALO_MIN_CTAS 16

__global__ void __launch_bounds__(HALO_THREADS) b2_k_halo_ll(const B2DevComm c, const B2HaloDesc d,
                                                             const int fs) {
  __shared__ unsigned s_rx[FS_NSIDES], s_tx[FS_NSIDES];
  const int gt = blockIdx.x * blockDim.x + threadIdx.x, gn = gridDim.x * blockDim.x;
  const int ny = d.ny, nx = d.nx, F = d.nfields;
  const size_t pitch = (size_t)d.pitch;
  const int nb[FS_NSIDES] = {d.west, d.east, d.south, d.north, d.sw, d.se, d.nw, d.ne};
  if (threadIdx.x < FS_NSIDES) {
    s_rx[threadIdx.x] = b2_ld_volatile(c.ticket + TK_RX + threadIdx.x);
    s_tx[threadIdx.x] = b2_ld_volatile(c.ticket + TK_TX + threadIdx.x);
  }
  __syncthreads();
  // halo columns: full height where this rank (and hence its W/E neighbours) touches a y wall
  const int jlo = (d.south >= 0) ? 1 : 0, jhi = (d.north >= 0) ? ny - 1 : ny, nj = jhi - jlo;
  const bool uwall = !d.periodic_x && d.at_east_wall;

  // ---------------- push ----------------
  if (d.west >= 0) {
    uint2* dst = fz_buf(c, d.west, s_tx[FS_W] & 1u, FS_E);
    const unsigned fl = s_tx[FS_W] + 1u;
    for (int k = gt; k < F * nj; k += gn) {
      const int f = k / nj, j = jlo + k - f * nj;
      fz_put(dst + f * fs + j, d.field[f][(size_t)j * pitch + 1], fl);
    }
  }
  if (d.east >= 0) {
    uint2* dst = fz_buf(c, d.east, s_tx[FS_E] & 1u, FS_W);
    const unsigned fl = s_tx[FS_E] + 1u;
    for (int k = gt; k < F * nj; k += gn) {
      const int f = k / nj, j = jlo + k - f * nj;
      fz_put(dst + f * fs + j, d.field[f][(size_t)j * pitch + (nx - 2)], fl);
    }
  }
  if (d.south >= 0) {
    uint2* dst = fz_buf(c, d.south, s_tx[FS_S] & 1u, FS_N);
    const unsigned fl = s_tx[FS_S] + 1u;
    for (int k = gt; k < F * (nx - 2); k += gn) {
      const int f = k / (nx - 2), i = 1 + k - f * (nx - 2);
      fz_put(dst + f * fs + i, d.field[f][pitch + i], fl);
    }
  }
  if (d.north >= 0) {
    uint2* dst = fz_buf(c, d.north, s_tx[FS_N] & 1u, FS_S);
    const unsigned fl = s_tx[FS_N] + 1u;
    for (int k = gt; k < F * (nx - 2); k += gn) {
      const int f = k / (nx - 2), i = 1 + k - f * (nx - 2);
      fz_put(dst + f * fs + i, d.field[f][(size_t)(ny - 2) * pitch + i], fl);
    }
  }
  if (gt < F) {
    const int f = gt;
    if (d.sw >= 0) fz_put(fz_buf(c, d.sw, s_tx[FS_SW] & 1u, FS_NE) + f, d.field[f][pitch + 1], s_tx[FS_SW] + 1u);
    if (d.se >= 0)
      fz_put(fz_buf(c, d.se, s_tx[FS_SE] & 1u, FS_NW) + f, d.field[f][pitch + (nx - 2)], s_tx[FS_SE] + 1u);
    if (d.nw >= 0)
      fz_put(fz_buf(c, d.nw, s_tx[FS_NW] & 1u, FS_SE) + f, d.field[f][(size_t)(ny - 2) * pitch + 1],
             s_tx[FS_NW] + 1u);
    if (d.ne >= 0)
      fz_put(fz_buf(c, d.ne, s_tx[FS_NE] & 1u, FS_SW) + f,
             d.field[f][(size_t)(ny - 2) * pitch + (nx - 2)], s_tx[FS_NE] + 1u);
  }
  // every thread's edge reads are done before any halo cell of these arrays is overwritten below
  // only matters for cells that are both: none (edges are interior, halos are not) -> no barrier

  // ---------------- poll + unpack (+ wall conditions) ----------------
  if (d.east >= 0) {
    const uint2* src = fz_buf(c, c.rank, s_rx[FS_E] & 1u, FS_E);
    const unsigned fl = s_rx[FS_E] + 1u;
    for (int k = gt; k < F * nj; k += gn) {
      const int f = k / nj, j = jlo + k - f * nj;
      float val = fz_get(c, src + f * fs + j, fl, FS_E);
      if (d.kind[f] == 2 && d.at_north_wall && j == ny - 2) val = 0.f;
      d.field[f][(size_t)j * pitch + (nx - 1)] = val;
    }
  }
  if (d.west >= 0) {
    const uint2* src = fz_buf(c, c.rank, s_rx[FS_W] & 1u, FS_W);
    const unsigned fl = s_rx[FS_W] + 1u;
    for (int k = gt; k < F * nj; k += gn) {
      const int f = k / nj, j = jlo + k - f * nj;
      float val = fz_get(c, src + f * fs + j, fl, FS_W);
      if (d.kind[f] == 2 && d.at_north_wall && j == ny - 2) val = 0.f;
      d.field[f][(size_t)j * pitch] = val;
    }
  }
  if (d.south >= 0) {
    const uint2* src = fz_buf(c, c.rank, s_rx[FS_S] & 1u, FS_S);
    const unsigned fl = s_rx[FS_S] + 1u;
    for (int k = gt; k < F * (nx - 2); k += gn) {
      const int f = k / (nx - 2), i = 1 + k - f * (nx - 2);
      float val = fz_get(c, src + f * fs + i, fl, FS_S);
      if (d.kind[f] == 1 && uwall && i == nx - 2) val = 0.f;
      d.field[f][i] = val;
    }
  }
  if (d.north >= 0) {
    const uint2* src = fz_buf(c, c.rank, s_rx[FS_N] & 1u, FS_N);
    const unsigned fl = s_rx[FS_N] + 1u;
    for (int k = gt; k < F * (nx - 2); k += gn) {
      const int f = k / (nx - 2), i = 1 + k - f * (nx - 2);
      float val = fz_get(c, src + f * fs + i, fl, FS_N);
      if (d.kind[f] == 1 && uwall && i == nx - 2) val = 0.f;
      d.field[f][(size_t)(ny - 1) * pitch + i] = val;
    }
  }
  if (gt < F) {
    const int f = gt;
    if (d.sw >= 0) d.field[f][0] = fz_get(c, fz_buf(c, c.rank, s_rx[FS_SW] & 1u, FS_SW) + f, s_rx[FS_SW] + 1u, FS_SW);
    if (d.se >= 0)
      d.field[f][nx - 1] = fz_get(c, fz_buf(c, c.rank, s_rx[FS_SE] & 1u, FS_SE) + f, s_rx[FS_SE] + 1u, FS_SE);
    if (d.nw >= 0)
      d.field[f][(size_t)(ny - 1) * pitch] =
          fz_get(c, fz_buf(c, c.rank, s_rx[FS_NW] & 1u, FS_NW) + f, s_rx[FS_NW] + 1u, FS_NW);
    if (d.ne >= 0)
      d.field[f][(size_t)(ny - 1) * pitch + (nx - 1)] =
          fz_get(c, fz_buf(c, c.rank, s_rx[FS_NE] & 1u, FS_NE) + f, s_rx[FS_NE] + 1u, FS_NE);
  }
  for (int f = 0; f < F; ++f) {      // wall-row / wall-column cells that no message writes
    if (d.kind[f] == 1 && uwall)
      for (int j = gt; j < ny; j += gn)
        if ((j >= 1 && j < ny - 1) || (j == 0 && d.south < 0) || (j == ny - 1 && d.north < 0))
          d.field[f][(size_t)j * pitch + (nx - 2)] = 0.f;
    if (d.kind[f] == 2 && d.at_north_wall)
      for (int i = gt; i < nx; i += gn)
        if ((i >= 1 && i < nx - 1) || (i == 0 && d.west < 0) || (i == nx - 1 && d.east < 0))
          d.field[f][(size_t)(ny - 2) * pitch + i] = 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned old = atomicAdd(c.ticket + TK_FIN, 1u);
    if (old == gridDim.x - 1) {
      b2_st_volatile(c.ticket + TK_FIN, 0u);
      for (int k = 0; k < FS_NSIDES; ++k)
        if (nb[k] >= 0) {
          b2_st_volatile(c.ticket + TK_RX + k, s_rx[k] + 1u);
          b2_st_volatile(c.ticket + TK_TX + k, s_tx[k] + 1u);
        }
      __threadfence();
    }
  }
}

extern "C" int b2_halo_exchange(B2Comm* c, const B2HaloDesc* d, cudaStream_t stream) {
  if (d->nfields < 1 || d->nfields > B2_HALO_MAX_FIELDS) {
    b2_set_error("halo_exchange: nfields must be in [1, %d]", B2_HALO_MAX_FIELDS);
    return B2_ERR_BAD_ARG;
  }
  const size_t need = (size_t)d->nfields * (size_t)(d->ny > d->nx ? d->ny : d->nx) * sizeof(float);
  if (need > c->dev.lay.halo_cap) {
    b2_set_error("halo_exchange: halo buffers too small (%zu > %zu); raise MPI4JAX_B200_HALO_BYTES",
                 need, c->dev.lay.halo_cap);
    return B2_ERR_BAD_ARG;
  }
  if (d->pitch < d->nx) {
    b2_set_error("halo_exchange: pitch %d < nx %d", d->pitch, d->nx);
    return B2_ERR_BAD_ARG;
  }
  const int P = c->dev.size;
  const int nb[8] = {d->west, d->east, d->south, d->north, d->sw, d->se, d->nw, d->ne};
  for (int k = 0; k < 8; ++k)
    if (nb[k] < -1 || nb[k] >= P) {
      b2_set_error("halo_exchange: invalid neighbour rank %d", nb[k]);
      return B2_ERR_BAD_ARG;
    }
  const int mx = d->ny > d->nx ? d->ny : d->nx;
  const int fs = (mx + 3) / 4 * 4;
  // about one element per thread and side: the exchange is pure latency, so spread it wide
  int ctas = (d->nfields * mx + HALO_THREADS - 1) / HALO_THREADS;
  if (ctas < HALO_MIN_CTAS) ctas = HALO_MIN_CTAS;
  if (ctas > 96) ctas = 96;
  b2_k_halo_ll<<<ctas, HALO_THREADS, 0, stream>>>(c->dev, *d, fs);
  b2_count_launch(c);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    b2_set_error("halo_exchange: kernel launch failed: %s", cudaGetErrorString(err));
    return 1000 + (int)err;
  }
  return 0;
}
