#!/usr/bin/env python
"""bench.py -- sparse_mm forward+backward throughput on B200 (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2] [--impl reference] [--dump-outputs DIR]

One step = one forward + backward of ``sparse_mm(A, B)`` (C = A B; grad_A by SDDMM; grad_B = A^T G)
over one batch of synthetic input.  Default workload = BASELINE.json configs[1] ("config 2"): batched
CSR, batch 8, 65536 x 65536, 16 nnz/row, dense 65536 x 128, fp32 / int32.  With N > 1 (launched by
torchrun, one rank per GPU) batch items are independent units with no data-path collective: by default the
8 items of BASELINE's literal config are split over the ranks (``"scaling": "strong"``); ``--scaling weak``
gives every rank a full batch of 8 of its own instead (global batch 8 N).

The timed region replays the step from a CUDA graph (fixed pattern and shapes: no host work between the
kernels); an eager region of the same K steps runs beside it and supplies the per-kernel CUDA-event durations
(`kernels`, `roofline`) and the host enqueue time.  `value` comes from the faster of the two regions
(`timed_region` says which); both do identical GPU work.

Prints ONE JSON line (rank 0).  `value` = nnz/s with inputs resident in HBM; `e2e` = the same metric
through the public API from pinned HOST buffers (H2D of A, B, G and D2H of C, grad_A, grad_B inside
the timed region); `roofline` = the dominant kernel against the measured HBM copy bandwidth;
`cpu_baseline` = the reference's CPU data flow (oracle/reference_port.py) on this host's cores.

`--dump-outputs DIR` writes what the timed region's last step computed (C, grad_A values, grad_B) as
DIR/<name>.npy, so that two builds run with the same arguments (hence the same seeded inputs) can be compared
output for output.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads as W  # noqa: E402

METRIC, UNIT = "sparse_mm_fwd_bwd_nnz_per_s", "nnz/s"

CONFIGS = {
    # name: (builder kwargs) -- see workloads.py / SURVEY.md section 8(d)
    "1": dict(kind="coo", n=4096, m=4096, nnz=167772, K=64, dtype="f32", batch=None,
              desc="COO 4096x4096 @1% x dense 4096x64 fp32 (BASELINE configs[0])"),
    "2": dict(kind="csr_uniform", n=65536, m=65536, per_row=16, K=128, dtype="f32", batch=8,
              desc="batched CSR b=8 65536x65536 16 nnz/row x dense 65536x128 fp32 int32 (BASELINE configs[1])"),
    "3": dict(kind="stencil", D=128, K=32, dtype="f32", batch=None, b_colmajor=True,
              desc="27-point 128^3 stencil CSR (55.7M nnz) x dense 2097152x32 fp32 (BASELINE configs[2])"),
    "4": dict(kind="rmat", scale=22, K=128, dtype="bf16", batch=None,
              desc="R-MAT 2^22 rows ~64M nnz x dense 2^22x128 bf16 (BASELINE configs[3])"),
    "5": dict(kind="csr_uniform", n=262144, m=262144, per_row=8, K=512, dtype="f32", batch=None,
              desc="CSR 262144^2 8 nnz/row x dense 262144x512 fp32 (BASELINE configs[4])"),
    # not a BASELINE config: the size of the reference's published suite-sparse case (Rothberg/cfd2,
    # benchmarks/results/sparse_mm_suite_results.csv:6: fwd 722 us, fwd+bwd 73.1 ms on an RTX 4090), random pattern
    "cfd2": dict(kind="csr_uniform", n=123440, m=123440, per_row=25, K=128, dtype="f32", batch=None,
                 desc="cfd2-sized synthetic CSR 123440^2, 25 nnz/row (3 086 000 nnz) x dense 123440x128 fp32"),
    # the reference's own published random cases (RTX 4090, wall clock incl. clones; BASELINE.md section 1), same sizes:
    # benchmarks/results/sparse_mm_rand_results.csv:66 ("large": fwd 10.7 ms, fwd+bwd 33.6 ms) and
    # batched_sparse_mm_rand_results.csv:31 (b=128: fwd 2.95 ms, fwd+bwd 11.8 ms)
    "rand_large": dict(kind="coo_as_csr", n=262144, m=262144, nnz=65536, K=512, dtype="f32", batch=None, idx="i64",
                       desc="reference 'large' random case: CSR int64 262144^2, nnz 65536 x dense 262144x512 fp32"),
    "batched128": dict(kind="csr_uniform", n=1024, m=1024, per_row=4, K=64, dtype="f32", batch=128,
                       desc="reference batched random case: batched CSR int32 b=128 1024^2, nnz 4096/item x dense 1024x64 fp32"),
    # one rank's share of config 2 under 8-way strong scaling (1 of the 8 batch items), for single-GPU tuning runs
    "2shard8": dict(kind="csr_uniform", n=65536, m=65536, per_row=16, K=128, dtype="f32", batch=1,
                    desc="one batch item of BASELINE configs[1] (what each of 8 ranks runs under strong scaling)"),
    "5bf16": dict(kind="csr_uniform", n=262144, m=262144, per_row=8, K=512, dtype="bf16", batch=None,
                  desc="CSR 262144^2 8 nnz/row x dense 262144x512 bf16 (BASELINE configs[4])"),
}
DT = {"f32": torch.float32, "f64": torch.float64, "bf16": torch.bfloat16}


def build_inputs(cfg, device, batch_slice=None, seed_shift=0):
    """Returns (A, B, G) on `device`.  batch_slice=(lo, hi) keeps only those batch items (rank shard /
    CPU sample); the full batch is generated with the fixed seed first so shards see identical data."""
    dt = DT[cfg["dtype"]]
    if cfg["kind"] == "coo":
        A = W.uniform_coo(cfg["n"], cfg["m"], cfg["nnz"], dt, device, seed=1 + seed_shift)
    elif cfg["kind"] == "coo_as_csr":  # uniformly random unique coordinates, handed over as CSR
        A = W.uniform_coo(cfg["n"], cfg["m"], cfg["nnz"], dt, device, seed=1 + seed_shift).to_sparse_csr()
        if cfg.get("idx") != "i64":
            A = torch.sparse_csr_tensor(A.crow_indices().int(), A.col_indices().int(), A.values(), A.shape)
    elif cfg["kind"] == "csr_uniform":
        A = W.uniform_rows_csr(cfg["batch"], cfg["n"], cfg["m"], cfg["per_row"], dt,
                               torch.int64 if cfg.get("idx") == "i64" else torch.int32, device, seed=2 + seed_shift)
    elif cfg["kind"] == "stencil":
        A = W.stencil27_csr(cfg["D"], dt, torch.int32, device, seed=3 + seed_shift)
    elif cfg["kind"] == "rmat":
        A = W.rmat_csr(cfg["scale"], 16, dt, torch.int32, device, seed=4 + seed_shift)
    else:
        raise ValueError(cfg["kind"])
    B, G = W.dense_operands(tuple(A.shape), cfg["K"], dt, device, seed=100 + seed_shift)
    if cfg.get("b_colmajor"):  # rsample hands sparse_mm eps.t(): a column-major view (SURVEY 3.4)
        B = B.t().contiguous().t()
    if batch_slice is not None and A.dim() == 3:
        lo, hi = batch_slice
        A = torch.sparse_csr_tensor(A.crow_indices()[lo:hi].contiguous(), A.col_indices()[lo:hi].contiguous(),
                                    A.values()[lo:hi].contiguous(), (hi - lo,) + tuple(A.shape[1:]))
        B, G = B[lo:hi].contiguous(), G[lo:hi].contiguous()
    return A, B, G


def problem_stats(A, K):
    batch = A.shape[0] if A.dim() == 3 else 1
    n, m = A.shape[-2], A.shape[-1]
    nnz_total = A._nnz() * batch if (A.layout == torch.sparse_csr and A.dim() == 3) else A._nnz()
    s_v = A.dtype.itemsize
    coo = A.layout == torch.sparse_coo
    s_i = 8 if coo else A.crow_indices().dtype.itemsize
    alg = W.algorithmic_bytes(batch, n, m, nnz_total // batch, K, s_v, s_i, coo=coo)
    return dict(batch=batch, n=n, m=m, nnz=nnz_total, K=K, s_v=s_v, s_i=s_i, alg=alg,
                flops=6 * nnz_total * K, gather_bytes_per_pass=nnz_total * K * s_v)


DUMP_BYTES_PER_OUTPUT = 16 << 20  # three outputs: at most 48 MiB per dump


def dump_outputs(outputs: dict, out_dir: str, max_bytes: int = DUMP_BYTES_PER_OUTPUT) -> None:
    """Write every tensor of `outputs` as out_dir/<name>.npy: float64 stays float64, other float types become float32.
    A tensor larger than `max_bytes` is cut to a fixed sample of its rows (the last dimension kept whole; elements of
    a 1-D tensor), drawn with numpy's default_rng(0) from its shape alone, so two runs with the same arguments write
    the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        if t.numel() * t.element_size() > max_bytes:
            t = t.reshape(-1, t.shape[-1]) if t.dim() > 1 else t
            keep = max(max_bytes // (t[0].numel() * t.element_size()), 1)
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """Samples SM clock / throttle reasons DURING the timed region (NVML, ~20 ms period)."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4, "hw_power_brake": 0x80}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            # honour CUDA_VISIBLE_DEVICES by resolving through the CUDA device's UUID
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in {**self.BAD, **self.NOTE}.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def report(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------ CPU baseline
def cpu_reference_run(cfg, steps, warmup, budget_s=150.0, sample_note_only=False):
    """Time the reference's CPU data flow (torch CPU ops, all host threads) on a bounded sample of the
    workload: one batch item for batched configs, a row prefix for the very large single matrices.  `steps` and
    `warmup` are honoured unless the run would exceed `budget_s` seconds (then fewer timed steps, never < 1)."""
    from oracle import reference_port as rp

    torch.set_num_threads(os.cpu_count() or 1)
    c = dict(cfg)
    sample = "full workload"
    if c.get("batch"):
        c["batch"] = 1
        sample = (f"1 of {cfg['batch']} batch items (same n, nnz/row, K); the port runs the reference's forward, SDDMM "
                  "temporaries and A^T G but skips its sparse_block_diag_split + stack_csr of grad_A (conservative: "
                  "the real reference does more work per step)")
    if c["kind"] == "stencil":
        c["D"] = 64
        sample = "64^3 volume (1/8 of the rows, same stencil)"
    if c["kind"] == "rmat":
        c["scale"] = 18
        sample = "R-MAT scale 18 (1/16 of the rows, same edge factor)"
    if c["dtype"] == "bf16":
        c["dtype"] = "f32"
        sample += "; fp32 (the reference's CPU CSR path has no bf16)"
    A, B, G = build_inputs(c, "cpu")
    nnz = problem_stats(A, c["K"])["nnz"]
    times, t_start, done_warm = [], time.perf_counter(), 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        rp.forward_backward(A, B, G)
        dt = time.perf_counter() - t0
        if i < warmup and (time.perf_counter() - t_start) < budget_s / 3:
            done_warm += 1
            continue
        times.append(dt)
        if time.perf_counter() - t_start > budget_s:
            break
    sec = statistics.median(times)
    return dict(value=nnz / sec, unit=UNIT, cores=torch.get_num_threads(), kind="port", sample=sample,
                ms_per_step=sec * 1e3, nnz_per_step=nnz, steps=len(times), warmup=done_warm)


# ------------------------------------------------------------------------------------- main
def bind_to_gpu_numa_node(local_rank: int):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, before any pinned buffer is
    allocated: with several ranks per node, first-touch then places the e2e leg's pinned staging buffers on the
    GPU's own NUMA node instead of wherever the launcher happened to start the process (cross-socket PCIe traffic
    is what limits the N > 1 e2e numbers).  Best effort: returns a description or None."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus and len(cpus) < ncpu:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} CPUs local to GPU {idx}"
    except Exception:  # noqa: BLE001 -- NVML missing / container without affinity rights: run unbound
        return None
    return None


_JSON_FD = None


def _route_library_chatter_to_stderr():
    """Keep stdout for the ONE JSON line: anything a library writes to fd 1 while the bench runs (NCCL's version
    banner under torchrun, for one) is sent to stderr instead; emit_json() writes to the real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit_json(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


def dense_mib_per_rank(cfg, world, scaling, k_sharded):
    """Dense operands + outputs one rank touches per step (B, G read; C, grad_B written), from the config alone --
    both arms print the same `config`, so nothing in it may depend on tensors only one arm builds."""
    s_v = DT[cfg["dtype"]].itemsize
    if cfg["kind"] == "stencil":
        n = m = cfg["D"] ** 3
    elif cfg["kind"] == "rmat":
        n = m = 1 << cfg["scale"]
    else:
        n, m = cfg["n"], cfg["m"]
    items = cfg.get("batch") or 1
    if cfg.get("batch") and world > 1 and scaling == "strong":
        items = max(items // world, 1)
    K = cfg["K"] // world if (k_sharded and world > 1) else cfg["K"]
    return items * (m * K + 3 * n * K) * s_v / 2**20


def describe_config(cfg, args, world):
    batched = bool(cfg.get("batch"))
    k_sharded = world > 1 and not batched and args.sharding == "k"
    scaling = args.scaling if batched else "strong"
    if batched and world > 1 and scaling == "strong":
        sharding = f"strong: {cfg['batch']} batch items split over {world} ranks, no collective"
    elif batched and world > 1:
        sharding = f"weak: {cfg['batch']} batch items per rank, global batch {cfg['batch'] * world}, no collective"
    elif batched:
        sharding = "single GPU: all batch items on one rank"
    elif world == 1:
        sharding = "single GPU"
    elif k_sharded:
        sharding = f"dense columns K split over {world} ranks, A replicated, grad_A values all-reduce (NCCL)"
    else:
        sharding = (f"nnz-balanced row blocks over {world} ranks, B replicated, grad_B {args.grad_b} (NCCL"
                    f"{', not overlapped' if args.no_overlap else ', overlapped with the SDDMM'})")
    mib = dense_mib_per_rank(cfg, world, scaling, k_sharded)
    flush = mib <= 252
    l2 = (f"dense operands + outputs of one step = {mib:.0f} MiB per rank fit L2 (126 MB): an L2 flush "
          "(a 256 MiB write, then a 256 MiB read that leaves clean lines) runs between timed steps, outside the per-step event pair" if flush else
          f"inputs larger than L2: dense operands + outputs of one step = {mib:.0f} MiB per rank vs 126 MB L2; no explicit flush")
    return ({"workload": cfg["desc"], "config_id": args.config, "K": cfg["K"], "l2": l2, "sharding": sharding},
            scaling, k_sharded, flush)


def reference_methodology_ms(A, B, op, repeats=10):
    """The reference's own timing method (benchmarks/benchmark_utils.py:194-199, :258-264): host wall clock around
    clone(A) + clone(B) + op (+ out.sum().backward()) + synchronize, empty_cache before every repeat.  Cloning A gives
    it new index tensors, so the sparsity pattern is cold on every repeat.  Reported next to the CUDA-event numbers
    for comparability with the reference's published (RTX 4090) rows; mean over `repeats` after 3 warm-ups."""
    def one(backward):
        torch.cuda.empty_cache()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        A1 = A.detach().clone().requires_grad_(True)
        B1 = B.detach().clone().requires_grad_(True)
        out = op(A1, B1)
        if backward:
            out.sum().backward()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    res = {}
    for name, bw in (("fwd_ms", False), ("fwd_bwd_ms", True)):
        for _ in range(3):
            one(bw)
        res[name] = statistics.mean(one(bw) for _ in range(repeats))
    res["method"] = "wall clock: clone A, clone B, op, sum().backward(), synchronize (reference benchmark_utils.py:194-199,258-264); pattern cold every repeat"
    return res


def _positive_int(text: str) -> int:
    value = int(text)
    if value < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {value}")
    return value


def main():
    _route_library_chatter_to_stderr()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=50, help="timed steps of every timed region (e2e included)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-steps", type=_positive_int, default=None, help="timed steps of the e2e leg (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed region's last-step outputs (C, grad_A values, grad_B; rank 0's share at N > 1) "
                         f"as DIR/<name>.npy; an output over {DUMP_BYTES_PER_OUTPUT >> 20} MiB is cut to a fixed seeded "
                         "sample of its rows")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--sharding", default="k", choices=["rows", "k"],
                    help="one large (unbatched) matrix at N > 1: rows = nnz-balanced row blocks, B replicated, grad_B "
                         "reduce-scatter (north_star's scheme); k = dense columns split, A replicated, grad_A all-reduce")
    ap.add_argument("--grad-b", default="all_reduce", choices=["all_reduce", "reduce_scatter"],
                    help="row sharding: collective for grad_B (reduce_scatter leaves each rank its block of rows)")
    ap.add_argument("--no-overlap", action="store_true", help="row sharding: run the SDDMM after the collective finished")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"],
                    help="batched configs at N > 1: strong (default) = BASELINE's literal config, its batch items split over "
                         "the ranks; weak = every rank runs a full batch of its own (global batch = batch x N)")
    ap.add_argument("--no-graph", action="store_true",
                    help="time eager steps only (default: the timed region replays the step from a CUDA graph, the eager "
                         "region beside it gives the per-kernel durations and the host enqueue time)")
    ap.add_argument("--ref-methodology", action="store_true",
                    help="also report the reference's wall-clock methodology (default on for cfd2 / rand_large / batched128)")
    args = ap.parse_args()
    cfg = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3)
    config_out, scaling, k_sharded, flush = describe_config(cfg, args, world)

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        base = cpu_reference_run(cfg, steps=max(args.steps, 1), warmup=max(args.warmup, 1), budget_s=150.0)
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": base["steps"], "warmup": base["warmup"], "ms_per_step": base["ms_per_step"], "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config_out,
                "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit_json(line)
        return

    # ------------------------------------------------------------------------- B200 arm
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200 import _ops, sparse_mm

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    if not os.path.exists(nat.LIB_PATH) and rank == 0:  # normally shipped prebuilt with the snapshot
        from torchsparsegradutils_b200.csrc.build import build as _build_native

        _build_native(verbose=True)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    shard, seed_shift = None, 0
    if cfg.get("batch") and world > 1:
        if scaling == "strong":  # BASELINE's literal reading: batch 8 split over the ranks
            assert cfg["batch"] % world == 0, "batch must divide across ranks"
            per = cfg["batch"] // world
            shard = (rank * per, (rank + 1) * per)
        else:  # independent batch items: every rank owns a full batch of its own (weak scaling)
            seed_shift = 1000 * rank
    A, B, G = build_inputs(cfg, dev, shard, seed_shift)
    row_sharded = world > 1 and not cfg.get("batch") and A.layout == torch.sparse_csr and not k_sharded
    from torchsparsegradutils_b200 import distributed as D

    if k_sharded:
        # one large matrix, alternative: shard the dense K columns; A replicated; forward and grad_B local,
        # grad_A values all-reduced (nnz elements) over NVLink
        klo, khi = D.k_shard_bounds(cfg["K"], world, rank, align=16 // B.element_size())
        assert khi > klo, "more ranks than 128-bit column blocks"
        B = B[:, klo:khi].contiguous()
        G = G[:, klo:khi].contiguous()
    if row_sharded:
        # one large matrix: nnz-balanced row blocks, B replicated, grad_B reduced over NVLink
        bounds = D.nnz_balanced_row_blocks(A.crow_indices(), world)
        A = D.shard_rows_csr(A, bounds[rank], bounds[rank + 1])
        G = G[bounds[rank]:bounds[rank + 1]].contiguous()
    st = problem_stats(A, cfg["K"])
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flush else None
    flush_src = torch.zeros(64 << 20, dtype=torch.int32, device=dev) if flush else None

    def flush_l2():
        # evict the step's operands: write a 256 MiB buffer (> 126 MB L2), then stream a second 256 MiB buffer through L2
        # by reading it, so the cache is left holding clean lines -- after the write alone it holds 126 MB of dirty lines
        # whose write-back would be charged to the first kernels of the timed step
        flush_buf.zero_()
        flush_src.sum()

    A.requires_grad_(True)
    B.requires_grad_(True)
    if row_sharded:
        def op(a, b):
            return D.sparse_mm_row_sharded(a, b, grad_b=args.grad_b, overlap=not args.no_overlap)
    else:
        op = D.sparse_mm_k_sharded if k_sharded else sparse_mm

    last_C = [None]

    def step():
        A.grad = None
        B.grad = None
        C = op(A, B)
        C.backward(G)
        # detached: a reference to C itself would keep this step's autograd graph alive, and a CUDA graph capture on
        # the side stream fails while it is.  Inside a capture this is the static output every replay rewrites.
        last_C[0] = C.detach()
        return C

    def step_outputs():
        """What a caller of the step receives from its latest run (the captured one's tensors after graph replays);
        grad_A values flattened in storage order, so that a sample of them is drawn per entry, not per batch item."""
        gA = A.grad.values() if A.grad.layout == torch.sparse_csr else A.grad._values()
        return {"C": last_C[0], "grad_A_values": gA.reshape(-1), "grad_B": B.grad}

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # cold first call: empty pattern cache (COO sort / CSR transpose / padding are built here)
    torch.cuda.synchronize()
    t_cold = time.perf_counter()
    step()
    torch.cuda.synchronize()
    cold_ms = (time.perf_counter() - t_cold) * 1e3
    for _ in range(warmup):
        step()
    barrier()
    # cold pattern, warm process: drop the cached COO order / transposes / plans and time the step that rebuilds them
    # (median of 3: a single sample also catches one-off allocator growth and lazy module loads of the builder kernels)
    import torchsparsegradutils_b200 as _tsgu

    cold_samples = []
    for _ in range(3):
        _tsgu.clear_pattern_cache()
        torch.cuda.synchronize()
        t_cp = time.perf_counter()
        step()
        torch.cuda.synchronize()
        cold_samples.append((time.perf_counter() - t_cp) * 1e3)
    cold_pattern_ms = statistics.median(cold_samples)
    for _ in range(warmup):  # back to the steady state: from its second use on the pattern has its final layout
        step()
    barrier()

    # the reference's own wall-clock methodology, measured while the process is still in the state the reference's
    # benchmark script would be in (no captured graph, no flush buffers in use): it empties the allocator cache before
    # every repeat, so its cost depends on what else the process holds
    ref_meth = None
    if (args.ref_methodology or args.config in ("cfd2", "rand_large", "batched128")) and world == 1:
        ref_meth = reference_methodology_ms(A, B, sparse_mm)
        step()
        barrier()

    def timed_region(run_step, with_kernel_timer):
        """K steps between a barrier + synchronize on both sides; returns (ms of the K steps, host ms to enqueue one,
        clocks, per-kernel summary).  Small configs: L2 flush before every step, per-step event pairs."""
        launches0 = nat.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kt_cm = _ops.KernelTimer() if with_kernel_timer else _ops._NULL
        barrier()
        with ClockSampler(local_rank) as clk, kt_cm as kt:
            e0.record()
            t_host = time.perf_counter()
            pairs = []
            for _ in range(args.steps):
                if flush_buf is not None:
                    flush_l2()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    run_step()
                    b.record()
                    pairs.append((a, b))
                else:
                    run_step()
            host_ms = (time.perf_counter() - t_host) * 1e3 / args.steps  # time to ENQUEUE a step (no sync)
            e1.record()
            barrier()
        ms_total = sum(a.elapsed_time(b) for a, b in pairs) if pairs else e0.elapsed_time(e1)
        return ms_total, host_ms, clk.report(), (kt.summary() if with_kernel_timer else None), nat.launch_count() - launches0

    # region A: eager steps through the public op, with per-kernel CUDA events (roofline) and the host enqueue time
    eager_total, host_ms, clocks, ksum, launches = timed_region(step, True)
    timed = {"region": "eager", "ms_total": eager_total}
    timed_outputs = step_outputs() if args.dump_outputs else None
    # region B: the same step replayed from a CUDA graph (fixed pattern, fixed shapes): no host work between kernels
    graph_note = None
    if (row_sharded or k_sharded) and not args.no_graph:
        # a step with a collective inside is not captured: a capture failure on ONE rank would desynchronise the ranks
        graph_note = {"unavailable": "step contains a NCCL collective: eager region only"}
    elif not args.no_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):
                    step()
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            cap0 = nat.launch_count()
            with torch.cuda.graph(graph):
                step()
            graph_launches = nat.launch_count() - cap0  # kernels of ours inside one replay
            for _ in range(warmup):
                graph.replay()
            g_total, g_host_ms, g_clocks, _, _ = timed_region(graph.replay, False)
            graph_note = {"ms_per_step": g_total / args.steps, "host_enqueue_ms_per_step": g_host_ms}
            if g_total <= eager_total:
                timed = {"region": "cuda_graph", "ms_total": g_total}
                clocks, launches = g_clocks, graph_launches * args.steps
                timed_outputs = step_outputs() if args.dump_outputs else None
        except Exception as exc:  # noqa: BLE001 -- capture not possible (e.g. a collective that refuses capture): eager stands
            graph_note = {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}
            torch.cuda.synchronize()
    ms_total = timed["ms_total"]
    timed_region_note = (
        "CUDA-graph replay of the step (pattern and shapes fixed); per-kernel durations and host enqueue time from the "
        "eager region run beside it (same K steps, same work)" if timed["region"] == "cuda_graph" else
        "eager steps through the public op")
    if timed_outputs is not None and rank == 0:
        dump_outputs(timed_outputs, args.dump_outputs)
    timed_outputs = None
    if dist is not None:
        t = torch.tensor([ms_total, eager_total, host_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, eager_total, host_ms_max = float(t[0]), float(t[1]), float(t[2])
        # K-sharding: every rank walks all nnz entries over its 1/N of the dense columns -- the job's units are nnz once
        cnt = torch.tensor([0 if (k_sharded and rank != 0) else st["nnz"], launches], device=dev, dtype=torch.int64)
        dist.all_reduce(cnt)
        nnz_all, launches_all = int(cnt[0]), int(cnt[1])
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {"kernels_ms": {k: round(v["ms"], 4) for k, v in ksum.items()},
                                           "nnz": st["nnz"], "rows": st["n"] * st["batch"],
                                           "host_enqueue_ms": round(host_ms, 4)})
    else:
        nnz_all, launches_all, host_ms_max, per_rank = st["nnz"], launches, host_ms, None
    ms_step = ms_total / args.steps
    value = nnz_all / (ms_step * 1e-3)

    # ---- roofline of the dominant kernel (live CUDA-event durations from the eager region)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    kernels = {}
    for tag, rec in ksum.items():
        alg = st["alg"].get(tag)
        if alg is None:
            kernels[tag] = {"ms": rec["ms"], "launches": rec["launches"]}
            continue
        gbs = alg / (rec["ms"] * 1e-3) / 1e9
        kernels[tag] = {"ms": rec["ms"], "launches": rec["launches"], "alg_bytes": alg, "achieved_gbs": gbs,
                        "frac": gbs / peak, "gather_gbs": st["gather_bytes_per_pass"] / (rec["ms"] * 1e-3) / 1e9}
    # measured DRAM traffic per launch from the committed ncu --set full capture of this workload
    traffic = {}
    for rnd in ("r2", "r1"):
        tpath = os.path.join(ROOT, "profiles", f"{rnd}_cfg{args.config}_traffic.json")
        if os.path.exists(tpath) and world == 1:
            traffic = {k: v["dram_bytes"] for k, v in json.load(open(tpath))["kernels"].items()}
            break
    main_k = {k: v for k, v in kernels.items() if "alg_bytes" in v}
    dom = max(main_k, key=lambda k: main_k[k]["ms"]) if main_k else None
    roofline = None
    if dom:
        d = kernels[dom]
        l2_peak = 20000.0  # GB/s: measured ceiling of a 512-B-row LDG gather out of L2 (profiles/r1_gather_ceilings.txt)
        roofline = {"bound": "hbm", "kernel": dom, "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": d["frac"], "frac_of_nominal_8000": d["achieved_gbs"] / 8000.0, "traffic": traffic.get(dom),
                    "alg_bytes": d["alg_bytes"], "peak_source": peak_src,
                    "share_of_step": d["ms"] / (eager_total / args.steps), "l2_gather_gbs": d["gather_gbs"],
                    "l2_peak": l2_peak, "l2_ceiling_frac": d["gather_gbs"] / l2_peak}
    step_gbs = st["alg"]["total"] / (ms_step * 1e-3) / 1e9

    # ---- e2e: same step through the public API from pinned host buffers
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(A.detach(), B.detach(), G, args.e2e_steps or args.steps, dev, dist, op)
        e2e["value"] = (nnz_all / (e2e.pop("ms_per_step_max") * 1e-3))

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_run(cfg, steps=5, warmup=1, budget_s=30.0)
        cpu_base = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic", "config": config_out,
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches_all, "roofline": roofline,
                "cpu_baseline": cpu_base, "gflops": st["flops"] * (nnz_all / st["nnz"]) / (ms_step * 1e-3) / 1e9,
                "step_alg_gbs": step_gbs * (nnz_all / st["nnz"]), "step_frac_of_hbm_peak": step_gbs / peak,
                "kernels": kernels, "nnz_per_step": nnz_all,
                "timed_region": timed_region_note, "eager_ms_per_step": eager_total / args.steps, "cuda_graph": graph_note,
                "host_enqueue_ms_per_step": host_ms_max, "cold_first_step_ms": cold_ms,
                "cold_pattern_step_ms": cold_pattern_ms, "cold_pattern_step_ms_samples": [round(x, 3) for x in cold_samples], "reference_methodology": ref_meth, "host_affinity": numa, "per_rank": per_rank}
        emit_json(line)
    if dist is not None:
        dist.destroy_process_group()


def run_e2e(A, B, G, steps, dev, dist, sparse_mm):
    """Public-API step from HOST memory, everything inside the timed region: pinned H2D of A's index and
    value arrays, B and the upstream gradient G; the op (forward + backward); D2H of C, grad_A values
    and grad_B into pinned buffers.

    Batched inputs are independent per item (no cross-item data flow), so the step walks the items on
    three streams -- H2D of item i+1, compute of item i, D2H of item i-1 overlap (PCIe is full duplex) -- and
    the pipeline keeps running across steps (a data loader prefetching the next batch): at most two steps are in
    flight, the host waits for step s-1's last D2H before it enqueues step s+1, and the timed region ends when
    the last step's results are in host memory.  Device index tensors are rewritten every step, so the pattern cache misses and the transpose is
    rebuilt per item per step (cold-pattern cost is part of e2e)."""
    pin = lambda t: t.detach().cpu().contiguous().pin_memory()  # noqa: E731
    is_csr = A.layout == torch.sparse_csr
    batched = A.dim() == 3 and is_csr
    if is_csr:
        hA = [pin(A.crow_indices()), pin(A.col_indices()), pin(A.values())]
    else:
        hA = [pin(A._indices()), pin(A._values())]
    hB, hG = pin(B), pin(G)
    outC = torch.empty(tuple(G.shape), dtype=G.dtype).pin_memory()
    outgB = torch.empty(tuple(B.shape), dtype=B.dtype).pin_memory()
    outgA = torch.empty(hA[-1].shape, dtype=hA[-1].dtype).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in hA + [hB, hG])
    d2h = sum(t.numel() * t.element_size() for t in (outC, outgB, outgA))
    items = A.shape[0] if batched else 1
    item_shape = tuple(A.shape[1:]) if batched else tuple(A.shape)
    sl = (lambda t, i: t[i]) if batched else (lambda t, i: t)
    s_in, s_cmp, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    NSLOT = int(os.environ.get("TSGU_E2E_SLOTS", "4"))
    LOOKAHEAD = NSLOT - 1  # items whose H2D is queued ahead of the one being enqueued for compute: the host blocks in the
                           # pattern builds (host syncs), PCIe must not run dry meanwhile
    slots = [dict(A=[torch.empty_like(sl(t, 0), device=dev) for t in hA], B=torch.empty_like(sl(hB, 0), device=dev),
                  G=torch.empty_like(sl(hG, 0), device=dev), free=torch.cuda.Event()) for _ in range(NSLOT)]

    from torchsparsegradutils_b200 import clear_pattern_cache, prepare_pattern

    # diagnostics only (scripts/e2e_probe.py): where the host's time goes, and two what-if switches
    trace = {"prepare": 0.0, "enqueue": 0.0, "d2h": 0.0, "wait": 0.0} if os.environ.get("TSGU_E2E_TRACE") else None
    what_if_warm = os.environ.get("TSGU_E2E_WHATIF_WARM") == "1"      # keep the (stale) cached patterns: the r1 behaviour
    what_if_no_d2h = os.environ.get("TSGU_E2E_WHATIF_NO_D2H") == "1"  # skip the result copies

    def make_A(slot):
        if is_csr:
            return torch.sparse_csr_tensor(slot["A"][0], slot["A"][1], slot["A"][2], item_shape)
        return torch.sparse_coo_tensor(slot["A"][0], slot["A"][1], item_shape, is_coalesced=True)

    def upload(i):
        """H2D of item i: the sparse operand first, then the dense ones; returns (A is on the device, all is)."""
        slot = slots[i % NSLOT]
        ev_A, ev_in = torch.cuda.Event(), torch.cuda.Event()
        with torch.cuda.stream(s_in):
            s_in.wait_event(slot["free"])  # the compute that last used this slot is done
            for d, h in zip(slot["A"], hA):
                d.copy_(sl(h, i), non_blocking=True)
            ev_A.record(s_in)
            slot["B"].copy_(sl(hB, i), non_blocking=True)
            slot["G"].copy_(sl(hG, i), non_blocking=True)
            ev_in.record(s_in)
        return ev_A, ev_in

    inflight = collections.deque()  # (all results of the step are in host memory, tensors its D2H still reads)

    def one_step():
        keep = []
        pending = collections.deque(upload(j) for j in range(min(LOOKAHEAD, items)))
        for i in range(items):
            slot = slots[i % NSLOT]
            if i + LOOKAHEAD < items:
                pending.append(upload(i + LOOKAHEAD))
            (ev_A, ev_in), ev_cmp = pending.popleft(), torch.cuda.Event()
            with torch.cuda.stream(s_cmp):
                # the pattern-only work (transpose, plans) starts as soon as A's index arrays are on the device, while
                # the dense operands of this item are still crossing PCIe
                s_cmp.wait_event(ev_A)
                # a data loader delivers a NEW matrix into this device slot: its pattern is not the cached one.  The slot's
                # index buffers were rewritten in place (which the cache key cannot see), so the cache is dropped here and
                # every item of every step pays its pattern build inside the timed region.
                t_a = time.perf_counter()
                if not what_if_warm:
                    clear_pattern_cache()
                As = make_A(slot).requires_grad_(True)
                prepare_pattern(As, reuse=False)  # this matrix lives for one step
                t_b = time.perf_counter()
                s_cmp.wait_event(ev_in)
                dB = slot["B"].requires_grad_(True)
                dB.grad = None
                C = sparse_mm(As, dB)
                C.backward(slot["G"])
                gv = As.grad.values() if is_csr else As.grad._values()
                gB = dB.grad
                dB.requires_grad_(False)
                ev_cmp.record(s_cmp)
                slot["free"].record(s_cmp)
            t_c = time.perf_counter()
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_cmp)
                if not what_if_no_d2h:
                    sl(outC, i).copy_(C.detach(), non_blocking=True)
                    sl(outgB, i).copy_(gB, non_blocking=True)
                    sl(outgA, i).copy_(gv.reshape(sl(outgA, i).shape), non_blocking=True)
            if trace is not None:
                trace["prepare"] += t_b - t_a
                trace["enqueue"] += t_c - t_b
                trace["d2h"] += time.perf_counter() - t_c
            keep.append((C, gB, gv, As))  # outputs live until their D2H is done
        ev_done = torch.cuda.Event()
        ev_done.record(s_out)
        inflight.append((ev_done, keep))
        t_w = time.perf_counter()
        while len(inflight) > 1:  # two steps in flight at most: the older one's results must have landed
            ev, k = inflight.popleft()
            ev.synchronize()
            k.clear()
        if trace is not None:
            trace["wait"] += time.perf_counter() - t_w

    def drain():
        while inflight:
            ev, k = inflight.popleft()
            ev.synchronize()
            k.clear()

    for _ in range(2):
        one_step()
    drain()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    if trace is not None:
        trace.update(dict.fromkeys(trace, 0.0))
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    drain()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / steps  # host wall clock; every step's copies and results inside
    if trace is not None:
        print("e2e host ms/step:", {k: round(v * 1e3 / steps, 3) for k, v in trace.items()}, "total", round(ms, 3),
              file=sys.stderr)
    # what landed in host memory is the op's result (outside the timed region): compare with a device-resident run
    clear_pattern_cache()
    Ad = A.detach().requires_grad_(True)
    Bd = B.detach().requires_grad_(True)
    Cd = sparse_mm(Ad, Bd)
    Cd.backward(G)
    gAd = Ad.grad.values() if is_csr else Ad.grad._values()
    tol = dict(rtol=2e-2, atol=2e-2) if B.dtype == torch.bfloat16 else dict(rtol=1e-4, atol=1e-3)
    verified = bool(torch.allclose(outC.to(dev), Cd.detach(), **tol) and torch.allclose(outgB.to(dev), Bd.grad, **tol)
                    and torch.allclose(outgA.to(dev).reshape(-1), gAd.reshape(-1), **tol))
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return {"value": None, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms,
            "ms_per_step_max": ms, "steps": steps, "results_verified": verified, "pipeline": f"{items} item(s) on 3 streams (H2D | fwd+bwd | D2H), H2D queued {LOOKAHEAD} items ahead, 2 steps in flight",
            "note": "every item of every step is a NEW matrix for the library (pattern cache dropped per item): transpose / plan builds "
                    "are inside the timed region, issued (prepare_pattern(reuse=False)) as soon as A's arrays have arrived, under "
                    "the H2D of the dense operands; results_verified compares what landed in host memory with a device-resident run"}


if __name__ == "__main__":
    main()
