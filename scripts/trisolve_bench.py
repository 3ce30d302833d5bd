"""Sparse triangular solve: this package's level-scheduled kernel against the reference's data flow (torch's sparse CSR
``torch.triangular_solve``, i.e. cuSPARSE with its analysis inside every call).

    python scripts/trisolve_bench.py [--steps 20] [--warmup 3] [--out FILE]

Workloads (fp32, int32 indices, values well conditioned: off-diagonal U(0,1) / row length, diagonal U(1,2)):
  stencil_k1 / stencil_k32  lower triangle of the 27-point stencil on a 128^3 volume (config 3's precision_tril)
  random_b8_k128            8 random lower triangles of 65 536 rows, 16 entries per row with the diagonal (config 2)

Per workload, one JSON line: forward and forward+backward ms (CUDA events, after warm-up) for both paths, the max
|difference| of x and of B.grad between them, the cold plan-build ms (empty pattern cache, both plans), the level
count and microseconds per level, plus the card name and power limit read in the same run.  The reference's
backward is emulated with its own steps: the transposed torch solve for B.grad and the repeat_interleave /
index_select / mul / sum sampled product for A.grad.  Batched inputs are handed to torch as the block-diagonal
operand, built once outside the timed region (the reference rebuilds it every call).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import workloads as W  # noqa: E402
from torchsparsegradutils_b200 import block_diag_operand, clear_pattern_cache, sparse_triangular_solve  # noqa: E402
from torchsparsegradutils_b200.triangular_solve import solve_plan, solve_status  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                          str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return out or torch.cuda.get_device_name()


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def ref_step(A2, B2, G2, backward):
    """The reference's SparseTriangularSolve on a 2-D CSR operand (lower triangle, no transpose)."""
    x = torch.triangular_solve(B2, A2, upper=False).solution
    if not backward:
        return x, None
    gB = torch.triangular_solve(G2, A2, upper=False, transpose=True).solution
    crow, col = A2.crow_indices(), A2.col_indices()
    row = torch.repeat_interleave(torch.arange(A2.shape[0], device=crow.device), crow[1:] - crow[:-1])
    gA = -(gB.index_select(0, row) * x.index_select(0, col)).sum(dim=1)
    return x, (gB, gA)


def run(name, A, K, steps, warmup):
    dev = A.device
    batched = A.dim() == 3
    n = A.shape[-1]
    g = torch.Generator(device=dev).manual_seed(1)
    B = torch.randn(A.shape[:-1] + (K,), generator=g, device=dev)
    G = torch.randn(A.shape[:-1] + (K,), generator=g, device=dev)

    clear_pattern_cache()
    torch.cuda.synchronize()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    plan = solve_plan(A, upper=False)
    e1.record()
    solve_plan(A, upper=False, transpose=True)
    e2.record()
    torch.cuda.synchronize()
    plan_fwd_ms, plan_bwd_ms = e0.elapsed_time(e1), e1.elapsed_time(e2)

    Ag = A.detach().requires_grad_(True)
    Bg = B.clone().requires_grad_(True)

    def ours_fwd():
        with torch.no_grad():
            return sparse_triangular_solve(A, B, upper=False)

    def ours_fwd_bwd():
        Ag.grad, Bg.grad = None, None
        x = sparse_triangular_solve(Ag, Bg, upper=False)
        x.backward(G)
        return x

    A2 = block_diag_operand(A) if batched else A
    B2, G2 = B.reshape(-1, K), G.reshape(-1, K)
    ms = dict(fwd=timed(ours_fwd, steps, warmup), fwd_bwd=timed(ours_fwd_bwd, steps, warmup),
              torch_fwd=timed(lambda: ref_step(A2, B2, G2, False), steps, warmup),
              torch_fwd_bwd=timed(lambda: ref_step(A2, B2, G2, True), steps, warmup))
    status = solve_status(dev)

    x = ours_fwd_bwd()
    xr, (gBr, _) = ref_step(A2, B2, G2, True)
    diff_x = (x.reshape(-1, K) - xr).abs().max().item()
    diff_gB = (Bg.grad.reshape(-1, K) - gBr).abs().max().item()
    return dict(workload=name, rows=A.shape[0] * n if batched else n, batch=A.shape[0] if batched else 1,
                nnz=int(A.values().numel()), K=K, levels=plan.levels,
                **{f"{k}_ms": round(v, 4) for k, v in ms.items()},
                fwd_us_per_level=round(ms["fwd"] * 1000 / plan.levels, 3),
                speedup_fwd=round(ms["torch_fwd"] / ms["fwd"], 3),
                speedup_fwd_bwd=round(ms["torch_fwd_bwd"] / ms["fwd_bwd"], 3),
                max_abs_diff_x=diff_x, max_abs_diff_gradB=diff_gB,
                cold_plan_ms=dict(forward=round(plan_fwd_ms, 3), transposed=round(plan_bwd_ms, 3)),
                status=status, card=card(), steps=steps, warmup=warmup)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated workload names")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("trisolve_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    stencil = W.triangular_values(W.stencil27_csr(128, torch.float32, torch.int32, dev, lower=True), torch.float32)
    cases = [("stencil_k1", lambda: stencil, 1), ("stencil_k32", lambda: stencil, 32),
             ("random_b8_k128", lambda: W.random_lower_csr(8, 65536, 16, torch.float32, torch.int32, dev), 128)]
    only = set(args.only.split(",")) if args.only else None
    lines = []
    for name, make, K in cases:
        if only and name not in only:
            continue
        res = run(name, make(), K, args.steps, args.warmup)
        line = json.dumps(res)
        print(line, flush=True)
        lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
