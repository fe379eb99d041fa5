"""Numeric codes shared with the native core (csrc/b2_common.h)."""

from __future__ import annotations

import torch

# enum B2DType
F32, F64, F16, BF16, I8, I16, I32, I64, U8, U16, U32, U64, BOOL, C64, C128 = range(15)

DTYPE_CODE = {
    torch.float32: F32,
    torch.float64: F64,
    torch.float16: F16,
    torch.bfloat16: BF16,
    torch.int8: I8,
    torch.int16: I16,
    torch.int32: I32,
    torch.int64: I64,
    torch.uint8: U8,
    torch.uint16: U16,
    torch.uint32: U32,
    torch.uint64: U64,
    torch.bool: BOOL,
    torch.complex64: C64,
    torch.complex128: C128,
}

# enum B2Op
SUM, PROD, MIN, MAX, LAND, LOR, LXOR, BAND, BOR, BXOR = range(10)

# enum B2Algo
ALGO_AUTO, ALGO_LL, ALGO_ONESHOT, ALGO_TWOSHOT, ALGO_NVLS = range(5)
ALGO_BY_NAME = {
    "auto": ALGO_AUTO,
    "ll": ALGO_LL,
    "oneshot": ALGO_ONESHOT,
    "twoshot": ALGO_TWOSHOT,
    "nvls": ALGO_NVLS,
}

# enum B2OpCode (subset used from Python)
OPC_ALLREDUCE, OPC_REDUCE, OPC_SCAN, OPC_ALLGATHER, OPC_ALLTOALL = 1, 2, 3, 4, 5
OPC_BCAST, OPC_GATHER, OPC_SCATTER = 6, 7, 8
OPC_REDUCE_SCATTER = 13

ANY = -1  # ANY_SOURCE / ANY_TAG on the wire
