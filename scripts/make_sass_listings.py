"""Regenerate profiles/sass/*.sass (+ opcode summary) from the built native library."""
import collections
import os
import re
import subprocess
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(REPO, "mpi4jax_b200", "_native", "libb2mpi.so")
OUT = os.path.join(REPO, "profiles", "sass")
WANT = {       # substring of the mangled name (with its length prefix where names share a stem) -> file
    "12b2_k_halo_ll": "halo_ll", "12b2_k_halo_ca": "halo_ca_deep_exchange",
    "swe_k1_fluxes": "swe_k1_fluxes", "swe_k2_tendencies": "swe_k2_tendencies", "swe_k34": "swe_k34_friction_u",
    "swe_k5": "swe_k5_friction_v", "swe_ca_bulk_k12": "swe_ca_bulk_k12", "swe_ca_bulk_fric": "swe_ca_bulk_fric",
    "swe_ca_tend_frame": "swe_ca_tend_frame", "swe_ca_fric_frame": "swe_ca_fric_frame",
    "b2_k_barrier": "barrier", "9b2_k_move": "move", "b2_k_bcast_mc": "bcast_multicast",
    "b2_k_reduce_root_nvlsILi0": "reduce_root_nvls_f32", "b2_k_allreduce_symILi0": "allreduce_symmetric_inplace_f32",
    "b2_k_p2p": "p2p", "b2_k_allreduce_nvlsILi0": "allreduce_nvls_f32",
    "b2_k_allreduce_nvlsILi3": "allreduce_nvls_bf16", "b2_k_allreduce_llIfLi0": "allreduce_ll_f32_sum",
    "b2_k_reduce_chunkedIfLi0": "reduce_chunked_f32_sum",
    "b2_k_reduce_chunkedI13__nv_bfloat16Li0": "reduce_chunked_bf16_sum",
    "b2_k_gemm": "gemm_allreduce_tcgen05",
    "b2_k_reduce_scatter_nvlsILi0": "reduce_scatter_nvls_f32", "b2_k_reduce_scatter_llIfLi0": "reduce_scatter_ll_f32_sum",
}
HEADER = """# SASS listings (cuobjdump -sass libb2mpi.so, sm_100a)

One file per kernel family (typed reduce kernels: the f32/bf16 SUM instances); instruction
encodings stripped.  What to look for: peer/multicast traffic in the same kernel as the
arithmetic -- `LDG.E.128.STRONG.SYS` (peer pulls), `STG.E.128` on peer-mapped pointers
(pushes), `LDGMC.E.ADD.F32x4` / `LDGMC.E.HPADD.BF16x8` (= `multimem.ld_reduce`, in-switch
reduction), `REDG.E.ADD.STRONG.SYS` (arrival counters), `MEMBAR.*.SYS` (release fences).
`LDGMC` / `STG` on multicast addresses in `allreduce_symmetric_inplace_f32` are the whole kernel (no staging
copies).  The collective and stencil kernels contain no UTC*MMA / UTMALDG: they are bandwidth- or
latency-bound data movers / streaming stencils (~1 FLOP per 2-4 bytes) with no GEMM-shaped work.

| file | mangled name | instructions | memory / sync opcodes |
|---|---|---|---|
"""


def main():
    txt = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
    os.makedirs(OUT, exist_ok=True)
    rows = []
    seen = set()
    for old in os.listdir(OUT) if os.path.isdir(OUT) else []:
        if old.endswith('.sass'):
            os.remove(os.path.join(OUT, old))
    for f in re.split(r"\n\s*Function : ", txt)[1:]:
        name = f.split("\n", 1)[0].strip()
        for key, out in WANT.items():
            if key in name:
                body = re.sub(r"\s*/\* 0x[0-9a-f]{16} \*/", "", f)
                ops = collections.Counter(
                    re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d\s+)?([A-Z][A-Z0-9_.]+)", body, re.M))
                keep = {k: v for k, v in ops.items()
                        if re.match(r"(LDG|STG|LDGMC|RED|ATOM|MEMBAR|CCTL|BAR|LDS|STS|UTC|UTMA|LDTM|STTM|UBLKCP|SYNCS)", k)}
                with open(os.path.join(OUT, out + ".sass"), "a" if out in seen else "w") as fh:
                    fh.write("Function : " + body)
                seen.add(out)
                rows.append((out, name, sum(ops.values()), keep))
    with open(os.path.join(OUT, "README.md"), "w") as fh:
        fh.write(HEADER)
        for out, name, n, keep in sorted(rows):
            fh.write(f"| {out}.sass | `{name[:70]}` | {n} | "
                     f"{', '.join(f'{k} x{v}' for k, v in sorted(keep.items()))} |\n")
    print(f"wrote {len(rows)} listings to {OUT}")


if __name__ == "__main__":
    sys.exit(main())
