// mpi4jax_b200 -- shallow-water stencil kernels (fp32), the compute side of the
// reference's demo application (examples/shallow_water.py:270-403).  The
// reference leaves this arithmetic to XLA (dozens of fused elementwise kernels
// plus pad / dynamic-update-slice copies per step, separated by 48 blocking MPI
// custom calls).  Here one model step is four stencil launches and three fused
// multi-field halo exchanges (b2_halo.cu):
//
//   K1 fluxes      (h,u,v)                 -> fe, fn, q, ke        [exchange fe,fn,q,ke]
//   K2 tendencies  (h,fe,fn,q,ke,d*_old)   -> dh,du,dv, h',u,v     [exchange h',u,v]
//   K34 friction-u (fluxes inline from u, incl. their halo) + friction-v flux -> u, fe2, fn2
//                                                                   [exchange fe2,fn2]
//   K5 friction-v apply                    -> v
//
// The physics, including the order of boundary updates, the edge-padded `hc`
// rows at the y walls and the `v - u` term of the second friction flux
// (shallow_water.py:387-392), follows the reference line by line so that the
// two programs integrate the same discrete system.  The redundant `hc` halo
// exchange of the reference (:278-279) is elided: after `enforce_boundaries(h)`
// at the end of the previous step, h's halo already holds exactly the values
// that exchange would deliver (see DESIGN.md, "shallow water").
//
// Memory layout / vectorisation: fields are (ny, pitch) with pitch a multiple of
// 4 floats, so every row starts 16-byte aligned.  One thread owns an aligned
// group of 4 cells: centre rows and the rows above/below are single 16-byte
// loads, only the two x-neighbours of the group are scalar loads (L1 hits).
// These kernels are pure streaming stencils (1 FLOP per ~2 bytes): the roofline
// is HBM bandwidth, there is no tensor-core work in this workload.
#include <cstdio>

#include "b2_runtime.h"

extern "C" void b2_set_error(const char* fmt, ...);
extern "C" void b2_count_launch(B2Comm* c);

#include "b2_swe_body.cuh"

__global__ void __launch_bounds__(SWE_THREADS)
swe_k1_fluxes(B2SweParams p, const float* __restrict__ h, const float* __restrict__ u,
              const float* __restrict__ v, float* __restrict__ fe, float* __restrict__ fn,
              float* __restrict__ q, float* __restrict__ ke) {
  int j, i0;
  bool m[4];
  if (!swe_map(p, j, i0, m)) return;
  swe_k1_body(p, h, u, v, fe, fn, q, ke, j, i0, m);
}

__global__ void __launch_bounds__(SWE_THREADS, 3)
swe_k2_tendencies(B2SweParams p, const float* __restrict__ h, float* __restrict__ h_new,
                  float* __restrict__ u, float* __restrict__ v, float* __restrict__ dh,
                  float* __restrict__ du, float* __restrict__ dv, const float* __restrict__ fe,
                  const float* __restrict__ fn, const float* __restrict__ q,
                  const float* __restrict__ ke) {
  int j, i0;
  bool m[4];
  if (!swe_map(p, j, i0, m)) return;
  swe_k2_body(p, h, h_new, u, v, dh, du, dv, fe, fn, q, ke, j, i0, m);
}

__global__ void __launch_bounds__(SWE_THREADS)
swe_k34_friction_u(B2SweParams p, const float* __restrict__ u, float* __restrict__ u_new,
                   const float* __restrict__ v, float* __restrict__ fe2, float* __restrict__ fn2,
                   int has_south) {
  int j, i0;
  bool m[4];
  if (!swe_map(p, j, i0, m)) return;
  swe_k34_body(p, u, u_new, v, fe2, fn2, j, i0, m, has_south != 0);
}

__global__ void __launch_bounds__(SWE_THREADS)
swe_k5_friction_v(B2SweParams p, float* __restrict__ v, const float* __restrict__ fe2,
                  const float* __restrict__ fn2) {
  int j, i0;
  bool m[4];
  if (!swe_map(p, j, i0, m)) return;
  swe_k5_body(p, v, fe2, fn2, j, i0, m);
}

static unsigned swe_blocks(const B2SweParams* p) {
  const long long n = (long long)(p->ny - 2) * (p->pitch / 4);
  return (unsigned)((n + SWE_THREADS - 1) / SWE_THREADS);
}

static int swe_done(B2Comm* c, const char* name) {
  b2_count_launch(c);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    b2_set_error("%s: kernel launch failed: %s", name, cudaGetErrorString(err));
    return 1000 + (int)err;
  }
  return 0;
}

static int swe_check(const B2SweParams* p) {
  if (p->pitch % 4 != 0 || p->pitch < p->nx || p->ny < 3 || p->nx < 3) {
    b2_set_error("swe: need ny,nx >= 3 and a row pitch that is a multiple of 4 floats and >= nx "
                 "(got ny=%d nx=%d pitch=%d)", p->ny, p->nx, p->pitch);
    return B2_ERR_BAD_ARG;
  }
  return 0;
}

static int b2_swe_fluxes(B2Comm* c, const B2SweParams* p, const float* h, const float* u, const float* v,
                  float* fe, float* fn, float* q, float* ke, cudaStream_t s) {
  if (int rc = swe_check(p)) return rc;
  swe_k1_fluxes<<<swe_blocks(p), SWE_THREADS, 0, s>>>(*p, h, u, v, fe, fn, q, ke);
  return swe_done(c, "swe_fluxes");
}

static int b2_swe_tendencies(B2Comm* c, const B2SweParams* p, const float* h, float* h_new, float* u,
                      float* v, float* dh, float* du, float* dv, const float* fe, const float* fn,
                      const float* q, const float* ke, cudaStream_t s) {
  if (int rc = swe_check(p)) return rc;
  swe_k2_tendencies<<<swe_blocks(p), SWE_THREADS, 0, s>>>(*p, h, h_new, u, v, dh, du, dv, fe, fn, q, ke);
  return swe_done(c, "swe_tendencies");
}

// friction-u flux + apply + friction-v flux in one kernel (no fe/fn round trip through HBM)
// (u -> u_new: out of place, u_new must not alias u)
static int b2_swe_friction_u_fused(B2Comm* c, const B2SweParams* p, const float* u, float* u_new,
                            const float* v, float* fe2, float* fn2, int has_south, cudaStream_t s) {
  if (int rc = swe_check(p)) return rc;
  if (u == u_new) {
    b2_set_error("swe_friction_u_fused: u_new must not alias u (the update reads u's neighbours)");
    return B2_ERR_BAD_ARG;
  }
  swe_k34_friction_u<<<swe_blocks(p), SWE_THREADS, 0, s>>>(*p, u, u_new, v, fe2, fn2, has_south);
  return swe_done(c, "swe_friction_u_fused");
}

static int b2_swe_friction_v(B2Comm* c, const B2SweParams* p, float* v, const float* fe2, const float* fn2,
                      cudaStream_t s) {
  if (int rc = swe_check(p)) return rc;
  swe_k5_friction_v<<<swe_blocks(p), SWE_THREADS, 0, s>>>(*p, v, fe2, fn2);
  return swe_done(c, "swe_friction_v");
}

extern "C" {

// One call = `nsteps` model steps (4 stencil launches + 3 fused halo exchanges each), all
// enqueued on `s` without touching the host again: the whole time loop of the reference's
// `do_multistep` (examples/shallow_water.py:406-411) becomes a launch sequence that CUDA-graph
// capture turns into a single replayable graph.  `h0`/`h1` ping-pong (their wall rows are
// initialised identically and never written); the state is returned in h0 (an odd step count
// ends with one device copy).
// Layout record for the import-time ABI check (mpi4jax_b200/_src/native/__init__.py): the Python
// side mirrors these structs with ctypes, so a stale library with a different layout must be
// rejected before the first call (the reference checks the MPI handle ABI the same way,
// xla_bridge/__init__.py:23-89).
int b2_abi_info(int* out, int n) {
  const int v[] = {B2_ABI_VERSION,
                   (int)sizeof(B2StatusRecord), (int)sizeof(B2HaloDesc), (int)sizeof(B2SweParams),
                   (int)sizeof(B2SweState), (int)sizeof(B2ErrorRecord), B2_MAX_RANKS, B2_P2P_NSLOT,
                   (int)sizeof(B2SweCA)};
  const int have = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n && i < have; ++i) out[i] = v[i];
  return have;
}

int b2_swe_multistep(B2Comm* c, const B2SweParams* p0, const B2SweState* st, const B2HaloDesc* topo,
                     int nsteps, int first_step, cudaStream_t s) {
  B2SweParams p = *p0;
  float* h = st->h0;
  float* hn = st->h1;
  float* u = st->u;
  float* un = st->u1;
  B2HaloDesc d = *topo;
  d.ny = p.ny;
  d.nx = p.nx;
  d.pitch = p.pitch;
  int rc = 0;
  for (int it = 0; it < nsteps && rc == 0; ++it) {
    p.first_step = (first_step && it == 0) ? 1 : 0;
    if ((rc = b2_swe_fluxes(c, &p, h, u, st->v, st->fe, st->fn, st->q, st->ke, s))) break;
    d.nfields = 4;
    d.field[0] = st->fe; d.kind[0] = 1;
    d.field[1] = st->fn; d.kind[1] = 2;
    d.field[2] = st->q;  d.kind[2] = 0;
    d.field[3] = st->ke; d.kind[3] = 0;
    if ((rc = b2_halo_exchange(c, &d, s))) break;
    if ((rc = b2_swe_tendencies(c, &p, h, hn, u, st->v, st->dh, st->du, st->dv, st->fe, st->fn,
                                st->q, st->ke, s))) break;
    d.nfields = 3;
    d.field[0] = hn;    d.kind[0] = 0;
    d.field[1] = u;     d.kind[1] = 1;
    d.field[2] = st->v; d.kind[2] = 2;
    if ((rc = b2_halo_exchange(c, &d, s))) break;
    if (p.viscosity > 0.f) {
      // friction-u fluxes are evaluated inline from u (incl. their halo, from u's fresh halo):
      // no K3 launch, no (fe, fn) exchange, no HBM round trip of the fluxes
      if ((rc = b2_swe_friction_u_fused(c, &p, u, un, st->v, st->fe2, st->fn2, topo->south >= 0, s))) break;
      { float* t = u; u = un; un = t; }
      d.nfields = 2;
      d.field[0] = st->fe2; d.kind[0] = 1;
      d.field[1] = st->fn2; d.kind[1] = 2;
      if ((rc = b2_halo_exchange(c, &d, s))) break;
      if ((rc = b2_swe_friction_v(c, &p, st->v, st->fe2, st->fn2, s))) break;
    }
    float* t = h; h = hn; hn = t;
  }
  if (rc == 0 && u != st->u) {
    cudaError_t e = cudaMemcpyAsync(st->u, u, (size_t)p.ny * p.pitch * sizeof(float),
                                    cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) {
      b2_set_error("swe_multistep: copy failed: %s", cudaGetErrorString(e));
      rc = 1000 + (int)e;
    }
  }
  if (rc == 0 && h != st->h0) {
    cudaError_t e = cudaMemcpyAsync(st->h0, h, (size_t)p.ny * p.pitch * sizeof(float),
                                    cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) {
      b2_set_error("swe_multistep: copy failed: %s", cudaGetErrorString(e));
      rc = 1000 + (int)e;
    }
  }
  return rc;
}

}  // extern "C"
