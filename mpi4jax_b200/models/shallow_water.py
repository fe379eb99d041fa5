"""Non-linear shallow-water solver on a 2-D domain decomposition -- the reference's
flagship workload (/root/reference/examples/shallow_water.py) as a reusable model.

Same discrete system as the reference: C-grid, 1-cell halos, periodic in x, walls in y,
Adams-Bashforth time stepping, lateral friction, decomposition ``nproc_y = min(P, 2)``,
``nproc_x = P // nproc_y`` (shallow_water.py:57-107), initial condition = geostrophically
balanced jet (:138-169).  Two execution paths integrate it:

``backend="native"`` (CUDA tensors)
    Hand-written sm_100a kernels, enqueued by one native call per ``multistep`` and captured
    into a CUDA graph by :func:`mpi4jax_b200.jit`.  Default schedule: the communication-avoiding
    step (csrc/b2_swe_ca.cu) -- two fused bulk kernels (16 array passes instead of 32) running
    concurrently with a thin frame pipeline that needs ONE three-cell-deep halo exchange per
    step.  This replaces the reference's per-step sequence of XLA elementwise kernels + 48
    blocking MPI custom calls.

``backend="ops"`` (any device)
    Plain torch arithmetic with halo exchange through the *public* ``sendrecv``/``send``/
    ``recv`` ops in the reference's west/north/east/south order (:172-264).  It is the
    fp32 reference implementation the native kernels are tested against, the CPU path, and
    the demonstration that reference-style user code runs unchanged on this framework.
"""

from __future__ import annotations

import ctypes
import math
import os
from collections import namedtuple
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from .. import _src as _ops
from .._src import native
from .._src.comm import Comm
from .._src.comm import flush as _flush
from .._src.decorators import env_flag
from .._src.utils import get_default_comm

ModelState = namedtuple("ModelState", "h, u, v, dh, du, dv")

SUPPORTED_NPROC = (1, 2, 4, 6, 8, 16)
_EXT_NAMES = ("hx", "upx", "vpx", "uppx", "vppx")


@dataclass
class ShallowWaterConfig:
    nx: int = 360                 # global interior cells in x (reference default 360)
    ny: int = 180                 # global interior cells in y (reference default 180)
    dx: float = 5e3
    dy: float = 5e3
    gravity: float = 9.81
    depth: float = 100.0
    coriolis_f: float = 2e-4
    coriolis_beta: float = 2e-11
    periodic_x: bool = True
    ab_a: float = 1.5 + 0.1
    ab_b: float = -(0.5 + 0.1)

    @classmethod
    def for_resolution(cls, nx: int, ny: int, **kw) -> "ShallowWaterConfig":
        """The reference demo's physical domain (360 x 180 cells of 5 km) at another
        resolution: the grid spacing shrinks so that domain size, jet and Rossby radius stay
        the same (a *larger* domain with 5 km cells, as the reference's docs benchmark used,
        makes the balanced jet's height drop exceed the 100 m depth beyond ~2000 cells)."""
        return cls(nx=nx, ny=ny, dx=360 * 5e3 / nx, dy=180 * 5e3 / ny, **kw)

    @property
    def lateral_viscosity(self) -> float:
        return 1e-3 * self.coriolis_f * self.dx**2

    @property
    def dt(self) -> float:
        return 0.125 * min(self.dx, self.dy) / math.sqrt(self.gravity * self.depth)


class ShallowWaterModel:
    def __init__(self, config: Optional[ShallowWaterConfig] = None, comm: Optional[Comm] = None,
                 device: Optional[torch.device] = None, backend: str = "auto",
                 pipeline: Optional[str] = None):
        self.cfg = cfg = config or ShallowWaterConfig()
        self.comm = comm = comm or get_default_comm()
        self.device = torch.device(device) if device is not None else comm.device
        if backend == "auto":
            # the fused kernels need the NVLink transport; a host-staged communicator (ranks on
            # several nodes) runs the same discrete system through the 12 primitives
            backend = "native" if (self.device.type == "cuda" and comm.transport == "native") else "ops"
        if backend == "native" and self.device.type != "cuda":
            raise ValueError("backend='native' needs a CUDA device")
        self.backend = backend
        # Native launch schedules (csrc/):
        #   "ca"          communication-avoiding step: ONE three-cell-deep exchange per step, the rest
        #                 recomputed on a thin frame, bulk and frame on two streams (b2_swe_ca.cu);
        #                 16 array passes per step.  Default.
        #   "standalone"  4 stencil kernels + 3 fused exchanges, 32 passes (b2_swe.cu): the oracle the
        #                 default schedule is compared with, bit for bit.
        if pipeline is None:
            pipeline = "ca"
        if pipeline not in ("ca", "standalone"):
            raise ValueError(f"unknown shallow-water pipeline {pipeline!r} (expected 'ca' or 'standalone')")
        self.pipeline = pipeline
        size, rank = comm.Get_size(), comm.Get_rank()
        if size not in SUPPORTED_NPROC:
            raise RuntimeError(
                f"Got invalid number of MPI processes: {size}. "
                f"Please choose one of these: {SUPPORTED_NPROC}."
            )
        if not cfg.periodic_x:
            raise NotImplementedError("only the reference's periodic-x configuration is built in")
        self.nproc_y = min(size, 2)
        self.nproc_x = size // self.nproc_y
        self.proc_idx = tuple(int(i) for i in np.unravel_index(rank, (self.nproc_y, self.nproc_x)))
        if cfg.nx % self.nproc_x or cfg.ny % self.nproc_y:
            raise ValueError("the process grid must divide the domain evenly")
        self.nx_global, self.ny_global = cfg.nx + 2, cfg.ny + 2
        self.nx_local = cfg.nx // self.nproc_x + 2
        self.ny_local = cfg.ny // self.nproc_y + 2
        py, px = self.proc_idx
        self.local_slice = (
            slice((self.ny_local - 2) * py, (self.ny_local - 2) * py + self.ny_local),
            slice((self.nx_local - 2) * px, (self.nx_local - 2) * px + self.nx_local),
        )

        def flat(iy, ix):
            return int(np.ravel_multi_index((iy, ix), (self.nproc_y, self.nproc_x)))

        self.neighbors = {
            "south": flat(py - 1, px) if py > 0 else None,
            "north": flat(py + 1, px) if py < self.nproc_y - 1 else None,
            "west": flat(py, (px - 1) % self.nproc_x) if (px > 0 or cfg.periodic_x) else None,
            "east": flat(py, (px + 1) % self.nproc_x) if (px < self.nproc_x - 1 or cfg.periodic_x) else None,
        }

        def diag(dy_, dx_):
            iy, ix = py + dy_, px + dx_
            if not 0 <= iy < self.nproc_y:
                return None
            if cfg.periodic_x:
                ix %= self.nproc_x
            elif not 0 <= ix < self.nproc_x:
                return None
            return flat(iy, ix)

        self.diagonals = {"sw": diag(-1, -1), "se": diag(-1, 1), "nw": diag(1, -1), "ne": diag(1, 1)}
        self.at_north_wall = py == self.nproc_y - 1
        self.at_south_wall = py == 0
        self.at_east_wall = px == self.nproc_x - 1
        self.steps_done = 0
        self._alloc()
        self.reset()

    # ------------------------------------------------------------------ setup
    def _alloc(self) -> None:
        # rows are padded to a multiple of 4 floats so that every row starts 16-byte aligned
        # (float4 loads in the stencil kernels); fields are (ny, nx) views of (ny, pitch) storage
        self.pitch = (self.nx_local + 3) // 4 * 4

        def z():
            base = torch.zeros((self.ny_local, self.pitch), dtype=torch.float32, device=self.device)
            return base[:, : self.nx_local]

        self.h, self.u, self.v = z(), z(), z()
        self.dh, self.du, self.dv = z(), z(), z()
        self._h1 = z()
        self._u1 = z()      # ping-pong partner of u for the friction update
        self._v1 = z()      # ping-pong partner of v (fused flux+tendency path only)
        self.fe, self.fn, self.q, self.ke, self.fe2, self.fn2 = z(), z(), z(), z(), z(), z()
        y_global = (np.arange(-1, self.ny_global - 1) * self.cfg.dy)
        cor = self.cfg.coriolis_f + y_global[self.local_slice[0]] * self.cfg.coriolis_beta
        self.coriolis = torch.tensor(cor, dtype=torch.float32, device=self.device)
        if self.backend == "native":
            self._params = native.B2SweParams()
            p = self._params
            p.ny, p.nx, p.pitch = self.ny_local, self.nx_local, self.pitch
            p.dx, p.dy, p.dt = self.cfg.dx, self.cfg.dy, self.cfg.dt
            p.gravity, p.viscosity = self.cfg.gravity, self.cfg.lateral_viscosity
            p.rdx = float(np.float32(1.0) / np.float32(self.cfg.dx))
            p.rdy = float(np.float32(1.0) / np.float32(self.cfg.dy))
            p.ab_a, p.ab_b = self.cfg.ab_a, self.cfg.ab_b
            # constant factors folded once, in fp32 (csrc/b2_swe_body.cuh)
            f32 = np.float32
            rdx, rdy, nu, dt = f32(p.rdx), f32(p.rdy), f32(p.viscosity), f32(p.dt)
            p.c_gx, p.c_gy = float(-f32(p.gravity) * rdx), float(-f32(p.gravity) * rdy)
            p.c_nux, p.c_nuy = float(nu * rdx), float(nu * rdy)
            p.c_fx, p.c_fy = float(dt * nu * rdx * rdx), float(dt * nu * rdy * rdy)
            p.first_step = 0
            p.south_wall, p.north_wall = int(self.at_south_wall), int(self.at_north_wall)
            p.coriolis = self.coriolis.data_ptr()
            st = self._state = native.B2SweState()
            st.h0, st.h1 = self.h.data_ptr(), self._h1.data_ptr()
            st.u1 = self._u1.data_ptr()
            st.v1 = self._v1.data_ptr()
            for name in ("u", "v", "dh", "du", "dv", "fe", "fn", "q", "ke", "fe2", "fn2"):
                setattr(st, name, getattr(self, name).data_ptr())
            t = self._topo = native.B2HaloDesc()
            nb = self.neighbors
            t.west = -1 if nb["west"] is None else nb["west"]
            t.east = -1 if nb["east"] is None else nb["east"]
            t.south = -1 if nb["south"] is None else nb["south"]
            t.north = -1 if nb["north"] is None else nb["north"]
            dg = self.diagonals
            t.sw, t.se = (-1 if dg["sw"] is None else dg["sw"]), (-1 if dg["se"] is None else dg["se"])
            t.nw, t.ne = (-1 if dg["nw"] is None else dg["nw"]), (-1 if dg["ne"] is None else dg["ne"])
            t.periodic_x = int(self.cfg.periodic_x)
            t.at_east_wall, t.at_north_wall = int(self.at_east_wall), int(self.at_north_wall)
            t.ny, t.nx, t.pitch = self.ny_local, self.nx_local, self.pitch
            # "ext" arrays of the communication-avoiding step: what lies beyond the 1-cell halo
            # (csrc/b2_swe_ca_body.cuh); only their outer cells are ever touched
            self._epitch = self.nx_local + 4
            self._ext = {name: torch.zeros((self.ny_local + 4, self._epitch), dtype=torch.float32, device=self.device)
                         for name in _EXT_NAMES}
            ca = self._ca = native.B2SweCA()
            for name in _EXT_NAMES:
                setattr(ca, name, self._ext[name].data_ptr())
            ca.epitch, ca.cb1 = self._epitch, 0

    def initial_conditions_global(self):
        """Global (ny_global, nx_global) float32 fields of the balanced jet + perturbation
        (shallow_water.py:138-164)."""
        cfg = self.cfg
        x = np.arange(-1, self.nx_global - 1) * cfg.dx
        y = np.arange(-1, self.ny_global - 1) * cfg.dy
        yy, xx = np.meshgrid(y, x, indexing="ij")
        length_x = x[-2] - x[1]
        length_y = y[-2] - y[1]
        u0 = (10 * np.exp(-((yy - 0.5 * length_y) ** 2) / (0.02 * length_x) ** 2)).astype(np.float32)
        v0 = np.zeros_like(u0)
        cor = (cfg.coriolis_f + yy * cfg.coriolis_beta).astype(np.float32)
        h_geo = np.cumsum(-cfg.dy * u0 * cor / np.float32(cfg.gravity), axis=0, dtype=np.float32)
        h0 = (
            cfg.depth + h_geo - h_geo.mean()
            + 0.2 * np.sin(xx / length_x * 10 * np.pi) * np.cos(yy / length_y * 8 * np.pi)
        ).astype(np.float32)
        return h0, u0, v0

    def reset(self) -> None:
        h0, u0, v0 = self.initial_conditions_global()
        sl = self.local_slice
        self.h.copy_(torch.from_numpy(np.ascontiguousarray(h0[sl])))
        self.u.copy_(torch.from_numpy(np.ascontiguousarray(u0[sl])))
        self.v.copy_(torch.from_numpy(np.ascontiguousarray(v0[sl])))
        for t in (self.dh, self.du, self.dv, self.fe, self.fn, self.q, self.ke, self.fe2, self.fn2):
            t.zero_()
        self.enforce_boundaries([self.h, self.u, self.v], ["h", "u", "v"])
        self._sync_partners()
        self.steps_done = 0

    def _sync_partners(self) -> None:
        """Ping-pong partners start as copies: identical wall rows / halos that no kernel writes.
        The communication-avoiding schedule also (re)derives its ext arrays from the main ones
        (collective): the neighbours' cells beyond the halo, taken as not yet touched by a
        friction step -- exact for an initial state, see :meth:`load_state` otherwise."""
        self._h1.copy_(self.h)
        self._u1.copy_(self.u)
        self._v1.copy_(self.v)
        if self.backend == "native" and self.pipeline == "ca":
            nc = self.comm._native_comm()
            rc = native.lib.b2_swe_ca_init(
                nc.handle, ctypes.byref(self._params), ctypes.byref(self._state), ctypes.byref(self._ca),
                ctypes.byref(self._topo), torch.cuda.current_stream().cuda_stream)
            nc._check(rc, "Halo")

    def load_state(self, state: ModelState, ext: Optional[dict] = None) -> None:
        """Overwrite the prognostic fields (e.g. from pinned host memory, non-blocking).

        ``ext`` (from :meth:`ext_state`) restores the communication-avoiding schedule's frame
        storage as well, which makes the continuation bit-identical to the uninterrupted run.
        Without it the frame storage is re-derived from ``state`` as for an initial condition
        (collective): the neighbours' u, v next to the block edge are then taken as fresh instead of
        stale by one friction increment -- a rounding-level difference confined to the first step."""
        for dst, src in zip((self.h, self.u, self.v, self.dh, self.du, self.dv), state):
            dst.copy_(src, non_blocking=True)
        if self.backend == "native" and self.pipeline == "ca":
            self._sync_partners()
            if ext is not None:
                for name in _EXT_NAMES:
                    self._ext_put(name, ext[name])
                # the exchange in _sync_partners refreshed the halos of u, v; the run being continued
                # had them stale by one friction step (what the frame kernels' plain path reads)
                self.u.copy_(state[1], non_blocking=True)
                self.v.copy_(state[2], non_blocking=True)

    def load_initial_condition(self, h, u, v) -> None:
        """Start from ``(h, u, v)`` (local blocks incl. their halo cells, e.g. in pinned host memory; copied
        non-blocking): the Adams-Bashforth tendencies start at zero ON THE DEVICE -- nothing but the three
        prognostic fields crosses PCIe, as in the reference's solve loop, which builds the initial state on
        the host and lets ``jnp.zeros`` create the rest (examples/shallow_water.py:414-430).  The next call
        must be ``step(first_step=True)``.  Collective on the native path (frame storage)."""
        for dst, src in zip((self.h, self.u, self.v), (h, u, v)):
            dst.copy_(src, non_blocking=True)
        for t in (self.dh, self.du, self.dv):
            t.zero_()
        self.steps_done = 0
        if self.backend == "native" and self.pipeline == "ca":
            self._sync_partners()

    # the frame storage as four strips per array (rows / columns within 4 cells of the array edge)
    def ext_state(self) -> Optional[dict]:
        if not (self.backend == "native" and self.pipeline == "ca"):
            return None
        return {name: [a[:4].clone(), a[-4:].clone(), a[:, :4].clone(), a[:, -4:].clone()]
                for name, a in self._ext.items()}

    def _ext_put(self, name: str, strips) -> None:
        a = self._ext[name]
        a[:4].copy_(strips[0], non_blocking=True)
        a[-4:].copy_(strips[1], non_blocking=True)
        a[:, :4].copy_(strips[2], non_blocking=True)
        a[:, -4:].copy_(strips[3], non_blocking=True)

    @property
    def state(self) -> ModelState:
        return ModelState(self.h, self.u, self.v, self.dh, self.du, self.dv)

    # ------------------------------------------------------------------ halo exchange
    def enforce_boundaries(self, fields, kinds) -> None:
        """In-place halo exchange + wall conditions for several fields at once."""
        if self.backend == "native":
            nb = {**self.neighbors, **self.diagonals}
            g = lambda k: -1 if nb[k] is None else nb[k]  # noqa: E731
            self.comm._native_comm().halo_exchange(
                fields, kinds, g("west"), g("east"), g("south"), g("north"),
                periodic_x=self.cfg.periodic_x, at_east_wall=self.at_east_wall,
                at_north_wall=self.at_north_wall, sw=g("sw"), se=g("se"), nw=g("nw"), ne=g("ne"))
            return
        for f, kind in zip(fields, kinds):
            self._enforce_boundaries_ops(f, kind)

    def _enforce_boundaries_ops(self, arr: torch.Tensor, grid: str) -> None:
        """Halo exchange with the public p2p ops, in the reference's message order."""
        send_order = ("west", "north", "east", "south")
        recv_order = ("east", "south", "west", "north")
        send_idx = {"south": (1, slice(None)), "west": (slice(None), 1),
                    "north": (-2, slice(None)), "east": (slice(None), -2)}
        recv_idx = {"south": (0, slice(None)), "west": (slice(None), 0),
                    "north": (-1, slice(None)), "east": (slice(None), -1)}
        for sdir, rdir in zip(send_order, recv_order):
            sp, rp = self.neighbors[sdir], self.neighbors[rdir]
            if sp is None and rp is None:
                continue
            send_arr = arr[send_idx[sdir]].contiguous()
            template = torch.empty_like(arr[recv_idx[rdir]].contiguous())
            if sp is None:
                arr[recv_idx[rdir]] = _ops.recv(template, source=rp, comm=self.comm)
            elif rp is None:
                _ops.send(send_arr, dest=sp, comm=self.comm)
            else:
                arr[recv_idx[rdir]] = _ops.sendrecv(send_arr, template, source=rp, dest=sp,
                                                    comm=self.comm)
        if not self.cfg.periodic_x and grid == "u" and self.at_east_wall:
            arr[:, -2] = 0.0
        if grid == "v" and self.at_north_wall:
            arr[-2, :] = 0.0

    # ------------------------------------------------------------------ time stepping
    def step(self, first_step: Optional[bool] = None) -> None:
        self.multistep(1, first_step=first_step)

    def multistep(self, nsteps: int, first_step: Optional[bool] = None) -> None:
        """Advance ``nsteps`` model steps (the reference's ``do_multistep``, :406-411)."""
        if first_step is None:
            first_step = self.steps_done == 0
        if self.backend == "native":
            nc = self.comm._native_comm()
            stream = torch.cuda.current_stream().cuda_stream
            if self.pipeline == "ca":
                rc = native.lib.b2_swe_multistep_ca(
                    nc.handle, ctypes.byref(self._params), ctypes.byref(self._state), ctypes.byref(self._ca),
                    ctypes.byref(self._topo), int(nsteps), int(bool(first_step)), stream)
            else:
                rc = native.lib.b2_swe_multistep(
                    nc.handle, ctypes.byref(self._params), ctypes.byref(self._state),
                    ctypes.byref(self._topo), int(nsteps), int(bool(first_step)), stream)
            nc._check(rc, "Halo")
        else:
            for it in range(nsteps):
                self._step_ops(first_step and it == 0)
        self.steps_done += nsteps

    def _step_ops(self, first: bool) -> None:
        cfg = self.cfg
        dx, dy, dt, g = cfg.dx, cfg.dy, cfg.dt, cfg.gravity
        h, u, v = self.h, self.u, self.v
        C = (slice(1, -1), slice(1, -1))          # centre
        E = (slice(1, -1), slice(2, None))        # east neighbour
        W = (slice(1, -1), slice(None, -2))
        N = (slice(2, None), slice(1, -1))
        S = (slice(None, -2), slice(1, -1))
        NE = (slice(2, None), slice(2, None))
        SE = (slice(None, -2), slice(2, None))
        NW = (slice(2, None), slice(None, -2))

        hc = torch.nn.functional.pad(h[C][None, None], (1, 1, 1, 1), mode="replicate")[0, 0]
        self._enforce_boundaries_ops(hc, "h")
        fe, fn, q, ke = self.fe, self.fn, self.q, self.ke
        fe[C] = 0.5 * (hc[C] + hc[E]) * u[C]
        fn[C] = 0.5 * (hc[C] + hc[N]) * v[C]
        self._enforce_boundaries_ops(fe, "u")
        self._enforce_boundaries_ops(fn, "v")
        dh_new = -(fe[C] - fe[W]) / dx - (fn[C] - fn[S]) / dy
        q[C] = (self.coriolis[1:-1, None] + ((v[E] - v[C]) / dx - (u[N] - u[C]) / dy)) * (
            1.0 / (0.25 * (hc[C] + hc[E] + hc[N] + hc[NE])))
        self._enforce_boundaries_ops(q, "h")
        du_new = -g * (h[E] - h[C]) / dx + 0.5 * (
            q[C] * 0.5 * (fn[C] + fn[E]) + q[S] * 0.5 * (fn[S] + fn[SE]))
        dv_new = -g * (h[N] - h[C]) / dy - 0.5 * (
            q[C] * 0.5 * (fe[C] + fe[N]) + q[W] * 0.5 * (fe[W] + fe[NW]))
        ke[C] = 0.5 * (0.5 * (u[C] ** 2 + u[W] ** 2) + 0.5 * (v[C] ** 2 + v[S] ** 2))
        self._enforce_boundaries_ops(ke, "h")
        du_new = du_new - (ke[E] - ke[C]) / dx
        dv_new = dv_new - (ke[N] - ke[C]) / dy
        if first:
            u[C] += dt * du_new
            v[C] += dt * dv_new
            h[C] += dt * dh_new
        else:
            u[C] += dt * (cfg.ab_a * du_new + cfg.ab_b * self.du[C])
            v[C] += dt * (cfg.ab_a * dv_new + cfg.ab_b * self.dv[C])
            h[C] += dt * (cfg.ab_a * dh_new + cfg.ab_b * self.dh[C])
        self.dh[C], self.du[C], self.dv[C] = dh_new, du_new, dv_new
        self._enforce_boundaries_ops(h, "h")
        self._enforce_boundaries_ops(u, "u")
        self._enforce_boundaries_ops(v, "v")
        visc = cfg.lateral_viscosity
        if visc > 0:
            fe[C] = visc * (u[E] - u[C]) / dx
            fn[C] = visc * (u[N] - u[C]) / dy
            self._enforce_boundaries_ops(fe, "u")
            self._enforce_boundaries_ops(fn, "v")
            u[C] += dt * ((fe[C] - fe[W]) / dx + (fn[C] - fn[S]) / dy)
            fe[C] = visc * (v[E] - u[C]) / dx      # sic: the reference subtracts u here
            fn[C] = visc * (v[N] - u[C]) / dy
            self._enforce_boundaries_ops(fe, "u")
            self._enforce_boundaries_ops(fn, "v")
            v[C] += dt * ((fe[C] - fe[W]) / dx + (fn[C] - fn[S]) / dy)

    # ------------------------------------------------------------------ diagnostics / IO
    def total_mass(self) -> torch.Tensor:
        """Global sum of h over interior cells (conserved up to round-off)."""
        local = self.h[1:-1, 1:-1].double().sum()
        return _ops.allreduce(local, _ops.comm.SUM, comm=self.comm)

    def gather_global(self, field: torch.Tensor, root: int = 0) -> Optional[torch.Tensor]:
        """Reassemble a decomposed field on ``root`` (shallow_water.py:466-491, 579-584)."""
        parts = _ops.gather(field.contiguous(), root, comm=self.comm)
        if self.comm.Get_rank() != root:
            return None
        out = torch.empty((self.ny_global, self.nx_global), dtype=field.dtype, device=field.device)
        for r in range(self.comm.Get_size()):
            iy, ix = np.unravel_index(r, (self.nproc_y, self.nproc_x))
            sl = (slice((self.ny_local - 2) * iy, (self.ny_local - 2) * iy + self.ny_local),
                  slice((self.nx_local - 2) * ix, (self.nx_local - 2) * ix + self.nx_local))
            out[sl] = parts[r]
        return out


    # ------------------------------------------------------------------ checkpoint / resume
    def _checkpoint_meta(self) -> dict:
        return {"ny_global": self.ny_global, "nx_global": self.nx_global, "nproc_y": self.nproc_y,
                "nproc_x": self.nproc_x, "rank": self.comm.Get_rank(), "size": self.comm.Get_size(),
                "dt": float(self.cfg.dt), "format": 1}

    def save_checkpoint(self, directory: str) -> str:
        """Write this rank's shard of the prognostic state (h, u, v and the AB2 tendencies) to
        ``directory/rank<r>.pt``; collective.  The reference keeps snapshots in a Python list only
        (shallow_water.py:421-451) -- long runs on 8 GPUs want restartability.  The file is written
        to a temporary name and renamed, so an interrupted save never leaves a torn checkpoint."""
        import os

        os.makedirs(directory, exist_ok=True)
        path = os.path.join(directory, f"rank{self.comm.Get_rank():04d}.pt")
        payload = {"meta": self._checkpoint_meta(), "steps_done": int(self.steps_done),
                   "state": {k: t.detach().to("cpu", copy=True) for k, t in self.state._asdict().items()}}
        ext = self.ext_state()
        if ext is not None:
            payload["ext"] = {k: [t.cpu() for t in v] for k, v in ext.items()}
        torch.save(payload, path + ".tmp")
        os.replace(path + ".tmp", path)
        _ops.barrier(comm=self.comm)
        _flush()
        return path

    def load_checkpoint(self, directory: str) -> int:
        """Restore a state written by :meth:`save_checkpoint` with the same decomposition; returns
        the number of steps the checkpointed run had done.  Continuing from it is bitwise identical
        to the uninterrupted run (tests/test_models.py)."""
        import os

        path = os.path.join(directory, f"rank{self.comm.Get_rank():04d}.pt")
        payload = torch.load(path, map_location="cpu", weights_only=True)
        want, have = self._checkpoint_meta(), payload["meta"]
        bad = {k: (have.get(k), v) for k, v in want.items() if have.get(k) != v}
        if bad:
            raise ValueError(f"checkpoint {path} does not match this model (checkpoint, model): {bad}")
        self.load_state(ModelState(**payload["state"]), ext=payload.get("ext"))
        if not (self.backend == "native" and self.pipeline == "ca"):
            self._sync_partners()
        self.steps_done = int(payload["steps_done"])
        return self.steps_done


def solve_shallow_water(t1: float, num_multisteps: int = 10, config: Optional[ShallowWaterConfig] = None,
                        comm: Optional[Comm] = None, device=None, backend: str = "auto",
                        use_graph: bool = True, verbose: bool = True):
    """Integrate to model time ``t1`` seconds, returning snapshots every ``num_multisteps``
    steps (the reference's ``solve_shallow_water``, shallow_water.py:414-463)."""
    import time

    from .. import jit

    model = ShallowWaterModel(config, comm, device, backend)
    dt = model.cfg.dt
    sol = [ModelState(*[t.clone() for t in model.state])]
    model.step(first_step=True)
    sol.append(ModelState(*[t.clone() for t in model.state]))
    t = dt

    def advance():
        model.multistep(num_multisteps, first_step=False)

    run = jit(advance) if (use_graph and model.backend == "native") else advance
    run()   # warm-up (the reference pre-compiles the same way, :440-441)
    t += dt * num_multisteps
    if model.device.type == "cuda":
        torch.cuda.synchronize()
    start = time.perf_counter()
    while t < t1:
        run()
        sol.append(ModelState(*[x.clone() for x in model.state]))
        t += dt * num_multisteps
    if model.device.type == "cuda":
        torch.cuda.synchronize()
    end = time.perf_counter()
    if verbose and model.comm.Get_rank() == 0:
        print(f"\nSolution took {end - start:.2f}s")
    return sol
