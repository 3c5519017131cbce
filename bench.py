#!/usr/bin/env python
"""bench.py — the hot-path benchmark (driver contract).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|...] [--dump-outputs DIR]

One "step" = one CSR SpMM (sum) pass over the synthetic matrix of BASELINE.json configs[1]:
1M x 1M (per GPU), ~16 nnz/row, dense operand F=128 bf16 (SURVEY §8d generator G2 / G5).
Rank 0 prints ONE JSON line. `value` = whole-job GFLOP/s (2*E*F per SpMM) with inputs resident in HBM;
`e2e` = the same metric through the C-ABI host-buffer call (pinned host tensors in, host tensors out,
H2D/D2H inside the timed region); `roofline` = algorithmic HBM bytes / step time vs the measured copy
peak; `cpu_baseline` = the reference's own CPU spmm (oracle/_ref) on this box's host cores.

`--impl reference` times the reference's CPU operator itself on the same config (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

WORKLOADS = {
    # name: (rows per GPU, avg nnz/row, F, dtype, reduce, generator)
    "c2": dict(M=1_000_000, deg=16, F=128, dtype="bf16", reduce="sum", gen="uniform",
               desc="SpMM_sum CSR 1Mx1M, avg 16 nnz/row, F=128 bf16 (BASELINE configs[1])"),
    "c2_f32": dict(M=1_000_000, deg=16, F=32, dtype="bf16", reduce="sum", gen="uniform",
                   desc="SpMM_sum CSR 1Mx1M, avg 16 nnz/row, F=32 bf16"),
    "c2_f256": dict(M=1_000_000, deg=16, F=256, dtype="bf16", reduce="sum", gen="uniform",
                    desc="SpMM_sum CSR 1Mx1M, avg 16 nnz/row, F=256 bf16"),
    "c2_fp32": dict(M=1_000_000, deg=16, F=128, dtype="f32", reduce="sum", gen="uniform",
                    desc="SpMM_sum CSR 1Mx1M, avg 16 nnz/row, F=128 fp32"),
    "c1": dict(M=10_000, deg=5, F=32, dtype="f32", reduce="sum", gen="uniform",
               desc="spmm_sum random COO 10kx10k, 50k nnz, F=32 fp32 (BASELINE configs[0])"),
    "c3": dict(M=500_000, deg=16, F=256, dtype="f32", reduce="max", gen="powerlaw",
               desc="SpMM_max CSR 500kx500k power-law degree, F=256 fp32 (BASELINE configs[2], forward)"),
}


def torch_dtype(name):
    import torch
    return {"bf16": torch.bfloat16, "f32": torch.float32, "f16": torch.float16}[name]


# ---------------------------------------------------------------------------------------------------
# synthetic inputs (identical on both arms: generated on the CPU from fixed seeds)
# ---------------------------------------------------------------------------------------------------
def gen_matrix(w, rank, world):
    """Row block `rank` of the (world*M) x (world*M) matrix: returns rowptr, col, value(float32), Ncols."""
    import torch
    M, N = w["M"], w["M"] * world
    g = torch.Generator().manual_seed(1 if world == 1 else 10 + rank)
    if w["gen"] == "uniform":
        E0 = w["deg"] * M
        row = torch.randint(M, (E0,), generator=g)
        col = torch.randint(N, (E0,), generator=g)
        key = torch.unique(row * N + col)
        row, col = key // N, key % N
    else:  # power-law degrees (SURVEY §8d G3): deg_i = min(floor(d0 * u^(-1/alpha)), N/10), alpha = 1.5
        u = torch.rand(M, generator=g).clamp_(min=1e-9)
        deg = (w["deg"] / 3.0 * u.pow(-1.0 / 1.5)).floor().long().clamp_(max=N // 10)
        deg[torch.rand(M, generator=g) < 0.02] = 0          # some empty rows by design
        row = torch.repeat_interleave(torch.arange(M), deg)
        col = torch.randint(N, (row.numel(),), generator=g)
        key = torch.unique(row * N + col)
        row, col = key // N, key % N
    rowptr = torch.zeros(M + 1, dtype=torch.long)
    rowptr[1:] = torch.cumsum(torch.bincount(row, minlength=M), 0)
    value = torch.rand(col.numel(), generator=g) + 0.5     # U(0.5, 1.5)
    return rowptr, col, value, N


def gen_dense(w, rank, rows):
    import torch
    g = torch.Generator().manual_seed(1000 + rank)
    return torch.randn(rows, w["F"], generator=g)


def algorithmic_bytes(M, N, E, F, s, arg):
    """compulsory model, SURVEY §8d: 8(M+1) + 8E + sE + s*N*F + s*M*F (+ 8*M*F arg_out)."""
    return 8 * (M + 1) + 8 * E + s * E + s * N * F + s * M * F + (8 * M * F if arg else 0)


# ---------------------------------------------------------------------------------------------------
# clocks sampling (NVML, in-process thread)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.power = [], set(), []
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_mhz = None

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.ok:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.ok:
            self.t.join(timeout=1)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s),
                "power_w_max": max(self.power) if self.power else None}


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU operator (oracle/_ref), all host threads
# ---------------------------------------------------------------------------------------------------
def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _numa_nodes():
    try:
        return len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except OSError:
        return 1


def _interleaved(t):
    """First-touch placement spread over all NUMA nodes (the numactl --interleave equivalent available without
    the tool): the tensor is re-created by a multi-threaded copy, so its pages are first touched by the OpenMP
    threads that are bound across the sockets instead of all landing on the generating thread's node."""
    import torch
    out = torch.empty_like(t)
    out.copy_(t)
    return out


def run_reference(args, w):
    # OpenMP placement must be fixed before libgomp starts: bind the threads and spread them over the cores, so the
    # CPU baseline does not depend on where the scheduler happens to put 128 unbound threads (VERDICT r01: the same
    # code measured 10 vs 35 GFLOP/s on two boxes)
    if os.environ.get("OMP_PROC_BIND") is None and os.environ.get("TSB200_NO_REEXEC") is None:
        env = dict(os.environ, OMP_PROC_BIND="spread", OMP_PLACES="cores", TSB200_NO_REEXEC="1")
        os.execve(sys.executable, [sys.executable] + sys.argv, env)
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(len(os.sched_getaffinity(0)) or 1)
    cores = torch.get_num_threads()
    from oracle import build_ref
    kind = "reference"
    if build_ref.available():
        build_ref.load()

        def cpu_spmm(rowptr, col, value, x):
            if w["reduce"] == "max":
                return torch.ops.torch_sparse.spmm_max(rowptr, col, value, x)[0]
            return torch.ops.torch_sparse.spmm_sum(None, rowptr, col, value, None, None, x)
    else:  # the reference could not be compiled here: time the oracle port instead
        import oracle
        kind = "port"
        os.environ.setdefault("OMP_NUM_THREADS", str(cores))

        def cpu_spmm(rowptr, col, value, x):
            return oracle.spmm(rowptr, col, value, x, w["reduce"])[0]

    dt = torch_dtype(w["dtype"])
    rowptr, col, value, N = gen_matrix(w, 0, 1)
    x = _interleaved(gen_dense(w, 0, N).to(dt))
    value = _interleaved(value.to(dt))
    col = _interleaved(col)
    M, F = w["M"], w["F"]

    def sample(rows):
        rp = rowptr[:rows + 1]
        e = int(rp[-1])
        return rp, col[:e], value[:e]

    # calibrate a bounded sample: whole run (warmup + steps) within ~150 s of CPU time
    rp, c, v = sample(M)
    cpu_spmm(rp, c, v, x)          # untimed: thread pool start-up, page faults of the output allocator
    t0 = time.perf_counter()
    cpu_spmm(rp, c, v, x)
    t_full = time.perf_counter() - t0
    total = args.steps + args.warmup
    frac = min(1.0, 150.0 / max(t_full * total, 1e-9))
    rows = M if frac >= 1.0 else max(1024, int(M * frac))
    rp, c, v = sample(rows)
    E = c.numel()
    for _ in range(args.warmup):
        cpu_spmm(rp, c, v, x)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        cpu_spmm(rp, c, v, x)
        times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    ts_sorted = sorted(times)
    gflops = 2.0 * E * F / t / 1e9
    sample_desc = f"rows [0,{rows}) of the {M}-row workload ({E} nnz), all {N} dense rows, mean of {args.steps} steps"
    line = {
        "impl": "reference", "metric": "spmm_gflops", "value": gflops, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
        "config": {"workload": w["desc"], "rows": rows, "nnz": E, "F": F, "reduce": w["reduce"],
                   "device": "host CPU", "cpu_model": _cpu_model(), "numa_nodes": _numa_nodes(),
                   "placement": "OMP_PROC_BIND=%s OMP_PLACES=%s, operands first-touched by the bound thread pool"
                                % (os.environ.get("OMP_PROC_BIND"), os.environ.get("OMP_PLACES"))},
        "cpu_baseline": {"value": gflops, "unit": "GFLOP/s", "cores": cores, "kind": kind, "sample": sample_desc,
                         "best_ms": ts_sorted[0] * 1e3, "median_ms": ts_sorted[len(ts_sorted) // 2] * 1e3,
                         "best_value": 2.0 * E * F / ts_sorted[0] / 1e9, "cpu_model": _cpu_model()},
        "e2e": {"value": gflops, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "hbm_gbs_equiv": algorithmic_bytes(rows, N, E, F, x.element_size(), w["reduce"] == "max") / t / 1e9,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def _time_cuda(fn, steps, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _kernel_sha():
    """Hash of the sources of the headline kernel: an ncu traffic figure is only quoted for the code it was taken on."""
    import hashlib
    h = hashlib.sha256()
    for f in ("spmm_fw.cu", "spmm_common.cuh", "common.cuh"):
        h.update((ROOT / "pytorch_sparse_b200" / "csrc" / f).read_bytes())
    return h.hexdigest()[:16]


def _spmm_parity(oracle, rowptr_h, col_h, value_h, x_h, out_rows, rows, rel):
    """|out - ref| <= rel * (|A||B|) on the first `rows` rows, ref from the oracle in fp32 (north_star tolerance:
    1e-5 fp32, 1e-2 bf16, both against the |A||B| normaliser of SURVEY §8d)."""
    rp = rowptr_h[:rows + 1]
    e = int(rp[-1])
    c, v = col_h[:e], value_h[:e].float()
    xf = x_h.float()
    ref, _ = oracle.spmm(rp, c, v, xf, "sum")
    bound, _ = oracle.spmm(rp, c, v.abs(), xf.abs(), "sum")
    err = (out_rows.float() - ref).abs()
    return bool((err <= rel * bound + 1e-30).all()), float((err / bound.clamp_min(1e-30)).max())


def run_ours(args, w):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import oracle
    import pytorch_sparse_b200 as ts
    from pytorch_sparse_b200 import ops
    from pytorch_sparse_b200.parallel import PipelinedRowShardedSpMM, RowShardedSpMM

    dt = torch_dtype(w["dtype"])
    M, F, reduce = w["M"], w["F"], w["reduce"]
    rowptr_h, col_h, value_h, N = gen_matrix(w, rank, world)
    value_h = value_h.to(dt)
    x_local_h = gen_dense(w, rank, M).to(dt)   # this rank's row block of the dense operand
    E = col_h.numel()
    s = x_local_h.element_size()
    rel_tol = 1e-2 if s == 2 else 1e-5

    a_local = ts.SparseTensor(rowptr=rowptr_h.to(dev), col=col_h.to(dev), value=value_h.to(dev),
                              sparse_sizes=(M, N), is_sorted=True, trust_data=True)
    sharded = RowShardedSpMM(a_local, reduce=reduce)
    # dense operand made resident on every GPU ONCE over NVLink (north_star: "broadcast once")
    x_local = x_local_h.to(dev)
    if world > 1:  # NCCL communicator setup is not part of the gather time
        dist.all_reduce(torch.zeros(1, device=dev))
        sharded.gather_dense(x_local)
    gather_ms = _time_cuda(lambda: sharded.gather_dense(x_local), 5, 1) if world > 1 else 0.0
    x_full = sharded.gather_dense(x_local)

    def step():
        return sharded.local_spmm(x_full)

    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    torch.cuda.synchronize()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        out = step()
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank, world)
    if world > 1:
        dist.barrier()

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    def all_ranks(flag):
        t = torch.tensor([1.0 if flag else 0.0], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    ms_step = max_over_ranks(ev0.elapsed_time(ev1)) / args.steps
    launches_per_step = 1 if ops._auto_plan(a_local.storage.rowptr(), E) is not None else 3

    # ---- the same step INCLUDING the gather of the dense operand (it changes every step: chained layers) ----
    multi = None
    if world > 1 and reduce == "sum":
        steps_g = max(5, min(args.steps, 20))

        def step_serial():
            return sharded.local_spmm(sharded.gather_dense(x_local))
        dist.barrier()
        ms_serial = max_over_ranks(_time_cuda(step_serial, steps_g, 2))
        multi = {"gather_ms": max_over_ranks(gather_ms), "ms_per_step_incl_gather_serial": ms_serial,
                 "steps": steps_g, "collective": "NCCL all_gather_into_tensor over NVLink, inside the timed step"}
        out_pipe = None
        try:
            chunks = int(os.environ.get("TSB200_PIPE_CHUNKS", "2"))
            split = os.environ.get("TSB200_PIPE_SPLIT", "feature")
            transport = os.environ.get("TSB200_PIPE_TRANSPORT", "auto")
            pipe = PipelinedRowShardedSpMM(a_local, block=M, chunks=chunks, split=split, transport=transport)
            if split == "feature":   # slice-major layout on both sides (what a chain of layers keeps between steps)
                x_in = pipe.to_sliced(x_local)
                if pipe.transport == "peer":   # the producer writes straight into the symmetric buffers (both of
                    for _ in range(2):         # them: the steps alternate), so no staging copy is inside the step
                        pipe.input_buffer(x_in, x_in.size(-1)).copy_(x_in)
                        pipe._step += 1
                    pipe._step = 0
                    run_pipe = lambda: pipe.forward_sliced(pipe.input_buffer(x_in, x_in.size(-1)))
                else:
                    run_pipe = lambda: pipe.forward_sliced(x_in)
                as_rows = pipe.from_sliced
            else:
                run_pipe = lambda: pipe(x_local)
                as_rows = lambda t: t
            dist.barrier()
            ms_pipe = max_over_ranks(_time_cuda(run_pipe, steps_g, 2))
            out_pipe = as_rows(run_pipe())
            multi.update({"ms_per_step_incl_gather_pipelined": ms_pipe, "pipeline_chunks": chunks,
                          "pipeline_split": split,
                          "pipeline_transport": pipe.transport + (
                              " (cudaMemcpyAsync pulls over NVLink from symmetric memory, copy engines only, "
                              f"{pipe.peer_streams} DMA stream)" if pipe.transport == "peer" else "")})
        except Exception as e:  # e.g. no symmetric-memory allocator on this box: the serial numbers still stand
            multi["pipelined_error"] = repr(e)[:300]

    # ---- parity of the timed results against the oracle (outside the timed regions), every rank ----
    rows_chk = min(M, 65536)
    x_full_h = x_full.cpu()
    ok_steady, worst = _spmm_parity(oracle, rowptr_h, col_h, value_h, x_full_h, out[:rows_chk].cpu(), rows_chk,
                                    rel_tol) if reduce == "sum" else (True, 0.0)
    parity = {"rows_per_rank": rows_chk, "tolerance": f"{rel_tol:g} * |A||B|", "steady_state": all_ranks(ok_steady),
              "worst_ratio": max_over_ranks(worst)}
    if multi is not None and out_pipe is not None:
        ok_pipe, worst_p = _spmm_parity(oracle, rowptr_h, col_h, value_h, x_full_h, out_pipe[:rows_chk].cpu(),
                                        rows_chk, rel_tol)
        parity["pipelined"] = all_ranks(ok_pipe)
        parity["worst_ratio_pipelined"] = max_over_ranks(worst_p)
        del out_pipe
    del x_full_h

    # ---- end to end through the C-ABI host-buffer call (pinned host in, host out) ------------------
    pin = lambda t: t.pin_memory()
    rp_p, col_p, val_p = pin(rowptr_h), pin(col_h), pin(value_h)
    x_full_p = pin(x_full.cpu())
    e2e_steps = max(3, min(args.steps, 10))
    # warm-up: device staging buffers + BOTH pinned output buffers the steady-state loop alternates between
    w1 = ops.spmm_fw_host(rp_p, col_p, val_p, x_full_p, reduce)
    w2 = ops.spmm_fw_host(rp_p, col_p, val_p, x_full_p, reduce)
    del w1, w2
    ops.spmm_fw_host(rp_p, col_p, val_p, x_full_p, reduce)
    if world > 1:
        dist.barrier()
    te = time.perf_counter()
    for _ in range(e2e_steps):
        out_h, _ = ops.spmm_fw_host(rp_p, col_p, val_p, x_full_p, reduce)
    e2e_ms = max_over_ranks((time.perf_counter() - te) * 1e3 / e2e_steps)
    arg = reduce in ("min", "max")
    h2d = 8 * (M + 1) + 8 * E + s * E + s * N * F
    d2h = s * M * F + (8 * M * F if arg else 0)
    # the host-buffer path runs the same kernel: bit-identical to the device-resident result
    parity["e2e_equals_device_result"] = all_ranks(torch.equal(out_h, out.cpu()))
    del rp_p, col_p, val_p, x_full_p, out_h

    flops = 2.0 * E * F
    tot = torch.tensor([flops], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot)
    gflops = tot.item() / (ms_step * 1e-3) / 1e9
    e2e_gflops = tot.item() / (e2e_ms * 1e-3) / 1e9
    if multi is not None:
        multi["value_incl_gather_serial"] = tot.item() / (multi["ms_per_step_incl_gather_serial"] * 1e-3) / 1e9
        if "ms_per_step_incl_gather_pipelined" in multi:
            multi["value_incl_gather_pipelined"] = tot.item() / (multi["ms_per_step_incl_gather_pipelined"] * 1e-3) / 1e9
        multi["unit"] = "GFLOP/s"

    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    peak = float(peaks.get("hbm_gbs", 6650.0))

    secondary = None
    if world == 1 and not args.no_secondary and args.workload == "c2":
        del a_local, sharded, x_full, x_local, out
        torch.cuda.empty_cache()
        secondary = run_secondary(dev, peak, local_rank)

    if rank == 0:
        abytes = algorithmic_bytes(M, N, E, F, s, arg)
        achieved = abytes / (ms_step * 1e-3) / 1e9
        traffic, traffic_note = None, None
        tf = ROOT / "profiles" / "ncu_traffic.json"
        if tf.exists() and world == 1:  # ncu capture of the N=1 launch; quoted only for the kernel it was taken on
            rec = json.loads(tf.read_text()).get(args.workload)
            if isinstance(rec, dict):
                if rec.get("kernel_sha") == _kernel_sha():
                    traffic = rec.get("bytes")
                    traffic_note = f"ncu dram__bytes_read+write per launch, {rec.get('capture', '')}"
                else:
                    traffic_note = (f"stale: capture taken on kernel sources {rec.get('kernel_sha')}, "
                                    f"current {_kernel_sha()}")
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_subprocess(args)
        line = {
            "metric": "spmm_gflops", "value": gflops, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": {"workload": w["desc"], "rows_per_gpu": M, "cols": N, "nnz_per_gpu": E, "F": F,
                       "reduce": reduce, "parallelism": f"row-block x{world}; headline = steady state (dense operand "
                       f"already gathered); the including-gather step is in `multi_gpu`" if world > 1 else "single GPU",
                       "l2": "inputs larger than L2 (dense operand %d MB + indices %d MB vs 126 MB L2); no flush"
                             % (s * N * F >> 20, (8 * E + s * E) >> 20),
                       "accumulate": "fp32",
                       "plan": "segment structure of the matrix planned once (tsb200_spmm_plan, cached per rowptr "
                               "like csr2csc): every timed step is one memset + one kernel"},
            "hbm_gbs": achieved, "gather_counted_gbs": (abytes - s * N * F + s * E * F) / (ms_step * 1e-3) / 1e9,
            "clocks": clocks,
            "e2e": {"value": e2e_gflops, "unit": "GFLOP/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "path": "tsb200_spmm_fw_host (pinned host buffers)"},
            # planned SpMM (the structure plan of the matrix is cached after its first use): one kernel per step;
            # unplanned: main + segment + combine kernels
            "gpu_launches": launches_per_step * args.steps,
            "parity": parity,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_note,
                         "peak_source": "measured" if peaks else "fallback", "algorithmic_bytes": abytes},
            "cpu_baseline": cpu,
        }
        if multi is not None:
            line["multi_gpu"] = multi
        if secondary is not None:
            line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 48 << 20   # all ranks together; row indices add 8 bytes a row


def dump_outputs(out_dir, out, rank, world):
    """What the last timed step returned to its caller, as float32 .npy files: a fixed, seeded sample of its rows
    (`out.npy`) and their indices (`out_rows.npy`, float64); with several ranks, one pair per rank (`out_rank<r>`).
    The inputs depend on the arguments only, so two builds can be compared file by file."""
    import numpy as np
    import torch
    M, F = out.size(0), out[0].numel()
    n = min(M, max(1, DUMP_BYTES // (4 * F * world)))
    rows = torch.randperm(M, generator=torch.Generator().manual_seed(0))[:n].sort().values
    tag = "out" if world == 1 else f"out_rank{rank}"
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / f"{tag}.npy", out[rows.to(out.device)].float().cpu().numpy())
    np.save(d / f"{tag}_rows.npy", rows.double().numpy())


# ---------------------------------------------------------------------------------------------------
# secondary north_star targets, measured in the same run after the headline (N = 1)
# ---------------------------------------------------------------------------------------------------
def run_secondary(dev, peak, gpu_index):
    """F=32 / F=256 bf16 SpMM, C3 SpMM_max forward and forward+backward, C4 SpSpMM, coalesce of 8.4M entries, C1 —
    each with its own clocks sample and an oracle spot check (`parity_ok`) taken outside the timed region."""
    import torch
    import oracle
    import pytorch_sparse_b200 as ts
    from pytorch_sparse_b200 import ops
    res = {}

    def timed(fn, steps, warm=3):
        sampler = ClockSampler(gpu_index)
        sampler.start()
        ms = _time_cuda(fn, steps, warm)
        ck = sampler.stop()
        return ms, {"sm_mhz": ck["sm_mhz"], "sm_max_mhz": ck["sm_max_mhz"], "reasons": ck["reasons"]}

    def guarded(name, fn):
        try:
            res[name] = fn()
        except Exception as e:  # one failing entry must not take the headline line down
            res[name] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    # ---- C2 at F = 32 and F = 256 (bf16, same matrix recipe as the headline) ----
    w = WORKLOADS["c2"]
    rowptr_h, col_h, value_h, N = gen_matrix(w, 0, 1)
    value_h = value_h.bfloat16()
    rowptr, col, value = rowptr_h.to(dev), col_h.to(dev), value_h.to(dev)
    M, E = w["M"], col_h.numel()
    for F in (32, 256):
        def one(F=F):
            x_h = torch.randn(N, F, generator=torch.Generator().manual_seed(1000)).bfloat16()
            x = x_h.to(dev)
            ms, ck = timed(lambda: ops.spmm_fw(rowptr, col, value, x, "sum"), 50)
            out = ops.spmm_fw(rowptr, col, value, x, "sum")[0]
            ok, worst = _spmm_parity(oracle, rowptr_h, col_h, value_h, x_h, out[:65536].cpu(), 65536, 1e-2)
            ab = algorithmic_bytes(M, N, E, F, 2, False)
            return {"workload": f"SpMM_sum CSR 1Mx1M, {E} nnz, F={F} bf16", "ms": ms, "gflops": 2.0 * E * F / ms / 1e6,
                    "hbm_gbs": ab / ms / 1e6, "frac": ab / ms / 1e6 / peak, "algorithmic_bytes": ab,
                    "parity_ok": ok, "parity": f"65536 rows vs oracle, worst |err|/(|A||B|) = {worst:.2e} (tol 1e-2)",
                    "clocks": ck}
        guarded(f"c2_f{F}", one)
    del rowptr, col, value, rowptr_h, col_h, value_h

    # ---- C3: SpMM_max forward and forward + backward, power-law 500k x 500k, F = 256 fp32 ----
    def c3():
        w3 = WORKLOADS["c3"]
        rp_h, c_h, v_h, N3 = gen_matrix(w3, 0, 1)
        M3, F3, E3 = w3["M"], w3["F"], c_h.numel()
        g = torch.Generator().manual_seed(7)
        x_h = torch.randn(N3, F3, generator=g)
        go_h = torch.randn(M3, F3, generator=g)
        a = ts.SparseTensor(rowptr=rp_h.to(dev), col=c_h.to(dev), value=v_h.to(dev), sparse_sizes=(M3, N3),
                            is_sorted=True, trust_data=True).requires_grad_()
        x = x_h.to(dev).requires_grad_()
        go = go_h.to(dev)
        ms_f, ck_f = timed(lambda: a.matmul(x.detach(), "max"), 20)

        def fb():
            x.grad = None
            a.storage.value().grad = None
            a.matmul(x, "max").backward(go)
        ms_fb, ck_fb = timed(fb, 10)
        out, arg_out = ops.spmm_fw(a.storage.rowptr(), a.storage.col(), a.storage.value().detach(), x.detach(), "max")
        R = 32768
        e = int(rp_h[R])
        ref, ref_arg = oracle.spmm(rp_h[:R + 1], c_h[:e], v_h[:e], x_h, "max")
        ref_arg = torch.where(ref_arg == e, torch.full_like(ref_arg, E3), ref_arg)   # sentinel of the sliced problem
        ok_f = bool(torch.equal(out[:R].cpu(), ref) and torch.equal(arg_out[:R].cpu(), ref_arg))
        # backward: both gradients against the oracle's restatement of SPMMMax::backward on the full problem
        gv_ref, gm_ref = oracle.spmm_minmax_bw(c_h, v_h, x_h, go_h, arg_out.cpu(), True, True)
        gv, gm = a.storage.value().grad.cpu(), x.grad.cpu()
        nv = oracle.spmm_minmax_bw(c_h, v_h.abs(), x_h.abs(), go_h.abs(), arg_out.cpu(), True, True)
        ok_b = bool(((gv - gv_ref).abs() <= 1e-5 * nv[0] + 1e-30).all() and
                    ((gm - gm_ref).abs() <= 1e-5 * nv[1] + 1e-30).all())
        ab_f = algorithmic_bytes(M3, N3, E3, F3, 4, True)
        ab_b = 4 * M3 * F3 + 8 * M3 * F3 + 4 * N3 * F3 + 4 * E3 + 8 * E3 + 4 * E3 + 4 * N3 * F3
        deg = rp_h[1:] - rp_h[:-1]
        res["c3_max_fwd"] = {"workload": w3["desc"], "nnz": E3, "max_degree": int(deg.max()),
                             "empty_rows": int((deg == 0).sum()), "ms": ms_f, "hbm_gbs": ab_f / ms_f / 1e6,
                             "frac": ab_f / ms_f / 1e6 / peak, "algorithmic_bytes": ab_f, "parity_ok": ok_f,
                             "parity": f"first {R} rows: values and arg_out bit-exact vs oracle", "clocks": ck_f}
        return {"workload": "SpMM_max forward + backward (grad_value and grad_mat), same inputs", "ms": ms_fb,
                "backward_ms": ms_fb - ms_f, "hbm_gbs": (ab_f + ab_b) / ms_fb / 1e6,
                "frac": (ab_f + ab_b) / ms_fb / 1e6 / peak, "algorithmic_bytes": ab_f + ab_b, "parity_ok": ok_b,
                "parity": "both gradients vs oracle.spmm_minmax_bw on the full problem, 1e-5 * |A||B|-style bound",
                "clocks": ck_fb}
    guarded("c3_max_fwd_bwd", c3)

    # ---- C4: SpSpMM 262 144^2, ~32 nnz/row, fp32 ----
    def c4():
        Mq = 262_144

        def rnd_csr(seed):
            g = torch.Generator(device=dev).manual_seed(seed)
            r = torch.randint(Mq, (32 * Mq,), generator=g, device=dev)
            c = torch.randint(Mq, (32 * Mq,), generator=g, device=dev)
            key = torch.unique(r * Mq + c)
            r, c = key // Mq, key % Mq
            rp = torch.zeros(Mq + 1, dtype=torch.long, device=dev)
            rp[1:] = torch.cumsum(torch.bincount(r, minlength=Mq), 0)
            return rp, c
        rpa, ca = rnd_csr(3)
        rpb, cb = rnd_csr(4)
        g = torch.Generator(device=dev).manual_seed(9)
        va = torch.randn(ca.numel(), generator=g, device=dev)
        vb = torch.randn(cb.numel(), generator=g, device=dev)
        keep = {}

        def run():
            keep["c"] = ops.spspmm(rpa, ca, va, rpb, cb, vb, Mq, Mq, Mq, True)
        ms, ck = timed(run, 5, 3)   # three warm-ups: the caching allocator must own both output sets
        rp_c, r_c, c_c, v_c = keep["c"]
        nnz = c_c.numel()
        R = 2048
        ea = int(rpa[R])
        orp, orow, oc, ov = oracle.spspmm(rpa[:R + 1], ca[:ea], va[:ea], rpb, cb, vb, R, Mq, Mq)
        _, _, _, ob = oracle.spspmm(rpa[:R + 1], ca[:ea], va[:ea].abs(), rpb, cb, vb.abs(), R, Mq, Mq)
        n = oc.numel()
        ok = bool(torch.equal(rp_c[:R + 1].cpu(), orp) and torch.equal(c_c[:n].cpu(), oc) and
                  torch.equal(r_c[:n].cpu(), orow) and ((v_c[:n].cpu() - ov).abs() <= 1e-5 * ob + 1e-30).all())
        out_bytes = nnz * 20
        alg = out_bytes + (ca.numel() + cb.numel()) * 12 + 2 * (Mq + 1) * 8
        return {"workload": "SpSpMM CSRxCSR 262144^2, ~32 nnz/row, fp32 (BASELINE configs[3]); whole op incl. output "
                            "allocation and nnz read-back", "nnz_a": ca.numel(), "nnz_b": cb.numel(), "nnz_c": nnz,
                "mode": os.environ.get("TSB200_SPSPMM", "auto"), "ms": ms, "gnnz_per_s": nnz / ms / 1e6,
                "out_gbs": out_bytes / ms / 1e6, "hbm_gbs": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak,
                "algorithmic_bytes": alg, "parity_ok": ok,
                "parity": f"first {R} rows of A times the full B vs oracle: structure bit-exact, values 1e-5 * |A||B|",
                "clocks": ck}
    guarded("c4_spspmm", c4)

    # ---- coalesce of 8.4M shuffled entries, every key duplicated once ----
    def co():
        Mq = 262_144
        g = torch.Generator().manual_seed(5)
        E0 = 4_194_304
        row = torch.randint(Mq, (E0,), generator=g)
        col = torch.randint(Mq, (E0,), generator=g)
        perm = torch.randperm(2 * E0, generator=g)
        row2_h, col2_h = torch.cat([row, row])[perm], torch.cat([col, col])[perm]
        val_h = torch.randn(2 * E0, generator=g, dtype=torch.float64)
        row2, col2, val = row2_h.to(dev), col2_h.to(dev), val_h.to(dev)
        ms, ck = timed(lambda: ops.coalesce(row2, col2, val, Mq, Mq, "add"), 10)
        r, c, v = ops.coalesce(row2, col2, val, Mq, Mq, "add")
        orow, ocol, oval = oracle.coalesce(row2_h, col2_h, val_h, Mq, Mq, "add")
        ok = bool(torch.equal(r.cpu(), orow) and torch.equal(c.cpu(), ocol) and
                  torch.allclose(v.cpu(), oval, rtol=1e-12, atol=1e-12))
        alg = 2 * E0 * (16 + 8) + r.numel() * (16 + 8)
        return {"workload": "coalesce(add) of 8 388 608 shuffled COO entries over 262144^2, every key twice, fp64 values",
                "entries": 2 * E0, "unique": r.numel(), "ms": ms, "mkeys_per_s": 2 * E0 / ms / 1e3,
                "hbm_gbs": alg / ms / 1e6, "frac": alg / ms / 1e6 / peak, "algorithmic_bytes": alg, "parity_ok": ok,
                "parity": "full result vs oracle.coalesce: indices bit-exact, values 1e-12", "clocks": ck}
    guarded("coalesce_8m", co)

    # ---- C1: the reference's own test configuration (10k x 10k, 50k nnz, F = 32 fp32) ----
    def c1():
        w1 = WORKLOADS["c1"]
        rp_h, c_h, v_h, N1 = gen_matrix(w1, 0, 1)
        x_h = gen_dense(w1, 0, N1)
        rp, c, v, x = rp_h.to(dev), c_h.to(dev), v_h.to(dev), x_h.to(dev)
        ms, ck = timed(lambda: ops.spmm_fw(rp, c, v, x, "sum"), 200, 10)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def cold():
            flush.zero_()
            ops.spmm_fw(rp, c, v, x, "sum")
        ms_cold = _time_cuda(cold, 20, 3) - _time_cuda(lambda: flush.zero_(), 20, 3)
        out = ops.spmm_fw(rp, c, v, x, "sum")[0]
        # the same call replayed from a CUDA graph (20 SpMMs per graph): what a launch-bound caller should do
        ms_graph = None
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    ops.spmm_fw(rp, c, v, x, "sum")
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for _ in range(20):
                    og = ops.spmm_fw(rp, c, v, x, "sum")[0]
            ms_graph = _time_cuda(graph.replay, 20, 3) / 20
            if not torch.equal(og, out):
                ms_graph = None
        except Exception:
            ms_graph = None
        ok, worst = _spmm_parity(oracle, rp_h, c_h, v_h, x_h, out.cpu(), w1["M"], 1e-5)
        E1 = c_h.numel()
        ab = algorithmic_bytes(w1["M"], N1, E1, 32, 4, False)
        return {"workload": w1["desc"], "nnz": E1, "ms": ms, "ms_l2_flushed": ms_cold, "ms_cuda_graph": ms_graph, "gflops": 2.0 * E1 * 32 / ms / 1e6,
                "hbm_gbs": ab / ms / 1e6, "frac": ab / ms / 1e6 / peak, "algorithmic_bytes": ab,
                "note": "fits in L2 (3 MB): launch-latency bound; `ms` is the L2-hot figure", "parity_ok": ok,
                "parity": f"all rows vs oracle, worst |err|/(|A||B|) = {worst:.2e} (tol 1e-5)", "clocks": ck}
    guarded("c1", c1)
    return res


def cpu_baseline_subprocess(args):
    """Time the reference's CPU operator in a clean process (its torch_sparse op namespace must not
    collide with ours); bounded sample chosen by run_reference()."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1",
           "--workload", args.workload]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        line = [l for l in res.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)["cpu_baseline"]
    except Exception as e:  # pragma: no cover
        return {"value": None, "error": repr(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary north_star targets (N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded row sample of the last step's output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":   # that arm times a row prefix sized by a clock calibration
        ap.error("--dump-outputs writes what the GPU path computed; it is not available with --impl reference")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
