"""Per-world-size transport thresholds of the GPU collectives.

The native library picks a transport per call from a handful of byte thresholds
(csrc/b2_collectives.cu: reduce_common, reduce_scatter_common, b2_bcast):

* ``ll_max``        allreduce / reduce_scatter: flag-in-data (LL) kernel up to this many bytes
* ``oneshot_max``   reductions without multicast: one-shot pull up to here, two-shot beyond
* ``nvls_min``      allreduce / reduce / reduce_scatter: in-switch (NVLS) reduction from this size on
                    (world size > 2)
* ``bcast_mc_min``  bcast: one ``multimem.st`` stream from the root from this size on (world size > 2)

reduce_scatter compares its whole input per rank (P blocks) with ``ll_max`` and ``nvls_min``, the bytes an
allreduce of the same input compares; below ``nvls_min``, or without multicast, it uses its one-shot pull.
These thresholds were measured for allreduce only; ``bench/collectives_sweep.py`` records every forced
reduce_scatter transport next to them, so a later change can give reduce_scatter keys of its own.

Which transport wins where depends on the number of ranks (at 2 ranks a one-shot pull beats the
switch at every size: each GPU has to serve P + 1 streams for an in-switch allreduce) and on the box.
The table below is what was MEASURED on B200 / NVSwitch boxes (the files named next to each entry);
``bench/autotune_collectives.py`` re-measures the crossovers for the job's world size on the box at hand
and writes a JSON file that ``MPI4JAX_B200_TUNING_FILE`` (or ``mpi4jax_b200/_src/tuning_tables/<gpu>.json``)
makes every later communicator load.  The reference has no counterpart: it hands every call to MPI.
"""

from __future__ import annotations

import json
import os
from typing import Dict, Optional

KEYS = ("ll_max", "oneshot_max", "nvls_min", "bcast_mc_min")

# what csrc/b2_runtime.cpp sets when a communicator is created (b2_comm_create)
NATIVE_DEFAULTS = {"ll_max": 64 << 10, "oneshot_max": 512 << 10, "nvls_min": (64 << 10) + 1, "bcast_mc_min": 256 << 10}

# world size -> thresholds (bytes).  A world size that is not listed uses the next smaller entry.
MEASURED: Dict[str, Dict[int, Dict[str, int]]] = {
    "NVIDIA B200": {
        # profiles/r2_sweep_n2_callH.log, r2_allreduce_sym_n2.log: LL 4.2-5.3 us up to its 64 KiB buffer limit,
        # one-shot pull beyond.  (At two ranks the native selection never takes the switch paths, whatever
        # nvls_min / bcast_mc_min say: an in-switch allreduce is bounded at P / (P + 1) of a link and loses.)
        2: dict(NATIVE_DEFAULTS),
        # profiles/r2_sweep_n4.log, r2_allreduce_phases_n4.log
        4: dict(NATIVE_DEFAULTS),
        # profiles/r2_sweep_n8.log (LL 7.9-12.2 us up to 64 KiB, staged NVLS 19.7 us at 256 KiB and ahead of
        # one-shot from there on), r1_collectives_sweep_8gpu_v1.json (one-shot vs two-shot without multicast)
        8: dict(NATIVE_DEFAULTS),
    },
}
DEFAULT_GPU = "NVIDIA B200"
_TABLE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tuning_tables")


def _entry_for(table: Dict[int, Dict[str, int]], world: int) -> Dict[str, int]:
    sizes = sorted(int(k) for k in table)
    pick = sizes[0]
    for s in sizes:
        if s <= world:
            pick = s
    row = table.get(pick, table.get(str(pick)))
    return {k: int(v) for k, v in row.items() if k in KEYS}


def load_file(path: str) -> Dict[int, Dict[str, int]]:
    """A tuning file is ``{"gpu": "...", "table": {"<world size>": {"ll_max": ..., ...}, ...}}``."""
    with open(path) as fh:
        doc = json.load(fh)
    table = doc["table"] if "table" in doc else doc
    out = {}
    for world, row in table.items():
        bad = [k for k in row if k not in KEYS]
        if bad:
            raise ValueError(f"{path}: unknown tuning keys {bad} (expected a subset of {KEYS})")
        out[int(world)] = {k: int(v) for k, v in row.items()}
    if not out:
        raise ValueError(f"{path}: empty tuning table")
    return out


def thresholds(world: int, gpu_name: Optional[str] = None) -> Dict[str, int]:
    """Thresholds for a communicator of ``world`` ranks on ``gpu_name``: the measured table, overridden
    entry by entry by ``tuning_tables/<gpu name>.json`` and then by ``$MPI4JAX_B200_TUNING_FILE``."""
    base = _entry_for(MEASURED.get(gpu_name or DEFAULT_GPU, MEASURED[DEFAULT_GPU]), world)
    candidates = []
    if gpu_name:
        candidates.append(os.path.join(_TABLE_DIR, gpu_name.replace(" ", "_") + ".json"))
    env = os.environ.get("MPI4JAX_B200_TUNING_FILE")
    if env:
        candidates.append(env)
    for path in candidates:
        if path and os.path.exists(path):
            base.update(_entry_for(load_file(path), world))
        elif path == env:
            raise FileNotFoundError(f"MPI4JAX_B200_TUNING_FILE={env!r} does not exist")
    return base


def crossover(sizes, time_a, time_b) -> int:
    """Largest size up to which transport A is at least as fast as transport B, given device times at
    increasing ``sizes`` (A is expected to win at small sizes and lose at large ones; noise of a single
    sample is tolerated by requiring B to win at two consecutive sizes).  Returns 0 if A never wins and
    the last size if B never wins twice in a row."""
    best = 0
    losses = 0
    for s, a, b in zip(sizes, time_a, time_b):
        if a is None or b is None:
            continue
        if a <= b:
            best, losses = int(s), 0
        else:
            losses += 1
            if losses >= 2:
                break
    return best
