"""Package lifecycle (reference: /root/reference/mpi4jax/_src/__init__.py:1-60).

The reference imports mpi4py first (MPI_Init + finalize-atexit), gates on the JAX version,
registers the FFI targets and installs an atexit ``flush`` so that pending asynchronous
custom calls finish before MPI_Finalize.  Here: gate on the torch version, load the native
library (``native``), import the 12 ops; ``comm`` registers an atexit hook that drains
every stream / pending isend and tears the symmetric heaps down *before* the process group
is destroyed (same purpose: no deadlock or crash at interpreter exit,
tests/collective_ops/test_common.py:91-115 in the reference).
"""

from .torch_compat import check_torch_version

check_torch_version()
del check_torch_version

from . import native  # noqa: E402,F401  (loads libb2mpi.so, applies MPI4JAX_B200_DEBUG)
from . import comm  # noqa: E402,F401   (atexit flush + teardown)

from .collective_ops.allgather import allgather  # noqa: E402,F401
from .collective_ops.allreduce import allreduce  # noqa: E402,F401
from .collective_ops.alltoall import alltoall  # noqa: E402,F401
from .collective_ops.barrier import barrier  # noqa: E402,F401
from .collective_ops.bcast import bcast  # noqa: E402,F401
from .collective_ops.gather import gather  # noqa: E402,F401
from .collective_ops.recv import recv  # noqa: E402,F401
from .collective_ops.reduce import reduce  # noqa: E402,F401
from .collective_ops.reduce_scatter import reduce_scatter  # noqa: E402,F401
from .collective_ops.scan import scan  # noqa: E402,F401
from .collective_ops.scatter import scatter  # noqa: E402,F401
from .collective_ops.send import send, send_with_grad  # noqa: E402,F401
from .collective_ops.sendrecv import sendrecv  # noqa: E402,F401

from .comm import flush  # noqa: E402,F401
from .utils import allreduce_, comm_reserve, has_cuda_support, has_sycl_support, symmetric_empty  # noqa: E402,F401
