#!/usr/bin/env python3
"""bench.py -- proof-gen seconds for the guest-keccak APC segment shape (2^20 rows x 2022 columns, 187 constraints of
degree <= 3, 1734 bus interactions: /root/reference/openvm-riscv/src/lib.rs:1377-1386) on N B200s, through the C ABI of
include/powdr_b200.h.

  python bench.py --gpus N --steps K --warmup W                 # native CUDA arm (torchrun launches N ranks for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W  # the CPU implementation on the host cores (rank 0 only)
  python bench.py ... --dump-outputs DIR                          # also write the last timed step's proof and openings as DIR/*.npy

One step = one segment per GPU through the whole path: main trace commit (LDE + Poseidon2 Merkle) -> LogUp permutation trace
(generate, LDE, commit) -> quotient -> quotient commit -> openings at zeta / zeta*w -> FRI commit phase -> proof of work (16 bits)
-> 100 queries.  `value` = device-timed seconds per segment with the trace already resident in HBM (max over ranks, divided by
the N segments proved concurrently); `e2e` = the same through pb_prove_segment + pb_query_segment with the trace in pinned
HOST memory (H2D inside the timed region, proof and query openings read back).  Inputs (8.5 GB/segment) exceed the 126 MB
L2, so no L2 flush is needed between iterations.  torch is plumbing only: device memory, the stream, events, NCCL.
"""
import argparse
import math
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "proof-gen sec for guest-keccak APC segment @2^20 rows"
P = 2013265921


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--width", type=int, default=2022)          # keccak APC: 2022 main columns
    ap.add_argument("--constraints", type=int, default=187)     # ... 187 constraints (openvm-riscv/src/lib.rs:1377-1386)
    ap.add_argument("--interactions", type=int, default=1734)   # ... 1734 bus interactions (same test)
    ap.add_argument("--queries", type=int, default=100)
    ap.add_argument("--pow-bits", type=int, default=16)
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="wall-clock budget of the CPU arm (full-size runs until it is spent)")
    ap.add_argument("--cpu-log-n", type=int, default=-1, help="rows of the CPU run (default: the full 2^log_n if host memory allows)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--metrics-out", default="", help="write the last step's stage times as an OpenVM-1 metrics JSON (basic_metrics.py schema)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the one-segment-on-all-GPUs (strong scaling) measurement at N > 1")
    ap.add_argument("--one-transcript", action="store_true",
                    help="multichip workload: prove all 50 chips under ONE transcript on one GPU (pb_prove_chips) instead of one proof per chip")
    ap.add_argument("--workload", default="keccak", choices=["keccak", "multichip", "pairing", "stage0"],
                    help="keccak: one APC chip per segment (the BASELINE metric); multichip: 50 independent chips of one segment "
                         "sharded over the ranks by LPT (BASELINE.json configs[3] shape, strong scaling); pairing: ONE wide segment "
                         "(default 2^20 x 16384, BASELINE.json configs[4]) column-sharded over all ranks -- the case that needs sharding")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (proof fields, query openings, opened values) as "
                         "DIR/<name>.npy in float64, so that two builds can be compared output for output (keccak workload, native arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "native" or a.workload != "keccak"):
        ap.error("--dump-outputs is implemented for the keccak workload of the native arm")
    return a


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, proof, arrays):
    """proof dict + named arrays -> path/<name>.npy, float64 (every value is a field element or a 32-bit word: exact).  Over
    DUMP_LIMIT_BYTES in all, a fixed seeded sample of the query rows is kept, with their indices in query_rows.npy."""
    import numpy as np
    out = {k: np.asarray(v, dtype=np.float64) for k, v in proof.items()}
    out.update({k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()})
    total = sum(v.nbytes for v in out.values())
    if total > DUMP_LIMIT_BYTES:
        q = out["queries"]
        keep = (DUMP_LIMIT_BYTES - (total - q.nbytes)) // (8 * (q.shape[1] + 1))      # a row and its index
        assert keep > 0, "outputs other than the query rows exceed %d bytes" % DUMP_LIMIT_BYTES
        rows = np.sort(np.random.default_rng(0).choice(q.shape[0], keep, replace=False))
        out["queries"], out["query_rows"] = q[rows], rows.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v)


def workload_name(a):
    shape = (a.log_n, a.width, a.constraints, a.interactions)
    name = {(20, 2022, 187, 1734): "guest-keccak APC shape", (16, 12035, 3770, 9539): "guest-sha256 largest-APC shape"}.get(shape, "custom APC shape")
    return ("%s: 2^%d rows x %d cols, %d constraints deg<=3, %d bus interactions (LogUp), log_blowup 1, "
            "%d queries, %d PoW bits (synthetic AIR + uniform trace)" % (name, a.log_n, a.width, a.constraints, a.interactions, a.queries, a.pow_bits))


def machine_for(a):
    """-> (machine, constraint bytecode, spans, bus) ; bus = compile_bus(machine, 1) or None"""
    from powdr_b200 import machine as M
    base = M.synthetic_machine(a.width, a.constraints, seed=0xB2000001)
    mach = M.SymbolicMachine(base.constraints, M.synthetic_bus(base, a.interactions, seed=0xB2000002)) if a.interactions else base
    assert mach.width == base.width
    bc, spans = M.compile_constraints(mach)
    return mach, bc, spans, (M.compile_bus(mach, 1) if a.interactions else None)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self):
        """start of the timed region (the sampler is started before the warm-up steps: nvidia-smi needs ~0.5 s to deliver its
        first sample, longer than a short timed region)"""
        self.t_mark = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        t_mark = getattr(self, "t_mark", 0.0)
        timed = [r for t, r in self.rows if t >= t_mark]
        window = "timed region"
        if not timed:                                   # region shorter than the sampling latency: the warm-up steps ran the same load
            timed, window = [r for _, r in self.rows], "warm-up + timed region"
        sm, mx, reasons = [], None, set()
        for r in timed:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


CPU_STAGES = ("lde", "merkle", "logup_gen", "logup_commit", "quotient", "quotient_commit", "openings", "fri_commit", "pow", "query")


def _mem_available_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 0.0


def cpu_prepare(a):
    """pins OpenMP before the CPU library loads; returns (orc, threads)"""
    n_cpu = os.cpu_count() or 1
    try:        # one OpenMP thread per PHYSICAL core: the AVX-512 kernels do not gain from the second hyperthread
        sib = set()
        for i in range(n_cpu):
            sib.add(open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % i).read().strip())
        n_cpu = max(1, len(sib))
    except Exception:
        pass
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_NUM_THREADS", str(n_cpu))
    from oracle import orc
    orc.build()
    return orc, orc.num_threads()


def cpu_run(a, orc, mach, bc, spans, bus, log_n):
    """one whole-segment proof on the host cores: the CPU implementation of the same path (oracle/prove.c driving the AVX-512
    Montgomery primitives of oracle/fast.c; falls back to the scalar ones without AVX-512) -> (seconds, stage seconds)"""
    import numpy as np
    rng = np.random.default_rng(0xB2000001)
    trace = orc.big_array((mach.width, 1 << log_n))                 # huge-page backed like the prover's own buffers
    for c0 in range(0, mach.width, 64):
        trace[c0:c0 + 64] = rng.integers(0, P, size=trace[c0:c0 + 64].shape, dtype=np.uint32)
    air = orc.Air(bc, spans, bus)
    t0 = time.time()
    _, _, _, st = orc.prove(trace, bc, spans, air, n_queries=a.queries, pow_bits=a.pow_bits, fast=True)
    return time.time() - t0, st


def cpu_baseline(a, mach, bc, spans, bus, budget_s=None, max_runs=1):
    """Times the CPU arm at the FULL configuration when host memory allows (trace + LDE + permutation trace + its LDE, ~4.6x the
    trace bytes), else on the largest power-of-two row count that fits, scaled by rows (said in `sample`)."""
    orc, threads = cpu_prepare(a)
    wp = orc.Air(bc, spans, bus).perm_width
    need_gb = lambda ln: 4.0 * (1 << ln) * (3.2 * mach.width + 3.2 * wp + 64) / 1e9
    ln = a.log_n if a.cpu_log_n < 0 else min(a.cpu_log_n, a.log_n)
    avail = _mem_available_gb()
    while ln > 12 and avail and need_gb(ln) > 0.8 * avail:
        ln -= 1
    cpu_run(a, orc, mach, bc, spans, bus, min(ln, 12))                      # warm-up: library load, thread pool
    runs, stages = [], None
    t_start = time.time()
    while len(runs) < max_runs and (not runs or budget_s is None or (time.time() - t_start) + runs[-1] < budget_s):
        dt, stages = cpu_run(a, orc, mach, bc, spans, bus, ln)
        runs.append(dt)
    scale = float(1 << (a.log_n - ln))
    v = sum(runs) / len(runs) * scale
    simd = "avx512" if orc.fast_available() else "scalar"
    sample = ("full configuration: 2^%d rows x %d cols, %d constraints, %d interactions; %d timed run(s) %s s" % (
        ln, mach.width, len(spans), a.interactions, len(runs), ["%.2f" % r for r in runs])) if scale == 1.0 else (
        "2^%d rows x %d cols (host memory %.0f GB does not hold the full 2^%d-row working set of %.0f GB), %d run(s) %s s, scaled x%d by rows" % (
            ln, mach.width, avail, a.log_n, need_gb(a.log_n), len(runs), ["%.2f" % r for r in runs], int(scale)))
    return {"value": v, "unit": "s", "cores": threads, "kind": "port", "simd": simd, "sample": sample, "runs": len(runs),
            "omp": {k: os.environ.get(k) for k in ("OMP_PROC_BIND", "OMP_PLACES", "OMP_NUM_THREADS")},
            "stages_s": {k: stages[k] * scale for k in CPU_STAGES}}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mach, bc, spans, bus = machine_for(a)
    # full-size runs until the budget is spent (at most --steps of them); `steps` in the line = the runs actually timed
    base = cpu_baseline(a, mach, bc, spans, bus, budget_s=a.cpu_budget_s, max_runs=max(1, a.steps))
    v = base["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "s", "n_gpus": a.gpus, "steps": base["runs"], "warmup": 1,
        "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (BabyBear, Montgomery, AVX-512 lanes)",
        "data": "synthetic", "config": {"workload": workload_name(a), "note": "CPU implementation of the same path (same proof bit for bit) on all host "
                                        "cores; the reference's own prover is an un-vendored Rust crate and cannot be built here (DESIGN.md §5)",
                                        "steps_requested": a.steps},
        "cpu_baseline": base, "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_native(a):
    import numpy as np
    import torch
    import powdr_b200
    from powdr_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL's version banner goes to stdout by default: keep stdout = the JSON line
        dist.init_process_group("nccl", device_id=dev)

    stream = torch.cuda.current_stream()
    ctx = powdr_b200.Context(local, stream.cuda_stream)      # raises without the CUDA library / a GPU: no fallback
    ctx.set_fri_params(a.queries, a.pow_bits)
    mach, bc, spans, bus = machine_for(a)
    t_key = time.time()
    if world > 1 and rank != 0:
        dist.barrier()                                        # rank 0 compiles first; the others then hit the on-disk cubin cache
    air = ctx.air(bc, spans, mach.width, bus)                # key generation: NVRTC builds of the constraint and LogUp kernels
    if world > 1 and rank == 0:
        dist.barrier()
    keygen_s = time.time() - t_key
    wp = air.perm_width
    n, w = 1 << a.log_n, mach.width
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB2000000 + 1 + rank)
    # uniform field elements; the buffer is read as Montgomery-form words (uniform either way)
    trace = torch.randint(0, P, (w, n), dtype=torch.int32, device=dev, generator=gen)
    caps = torch.zeros(16, dtype=torch.int32, device=dev)

    def step_device():
        proof = ctx.prove_segment(air, trace.data_ptr(), a.log_n, w, on_device=True)
        queries, ys = ctx.query_segment(a.log_n, w, wp)      # query phase: 100 openings gathered on the device, read back
        if world > 1:   # the path's one exchange: all-gather of the segment commitments (Merkle caps) over NCCL/NVLink
            caps.copy_(torch.tensor(proof["trace_root"] + proof["quotient_root"], dtype=torch.int64).to(torch.int32), non_blocking=True)
            parallel.all_gather_caps(caps.view(2, 8), dist)
        return proof, queries, ys

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(a.warmup):
        step_device()
    sync_all()
    ctx.leaf_kernel_profile()                                  # reset
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    sampler.mark()
    e0.record(stream)
    for _ in range(a.steps):
        proof, queries, ys = step_device()
    e1.record(stream)
    sync_all()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count() - launches0
    n_leaf, leaf_ms, leaf_bytes = ctx.leaf_kernel_profile()
    stage_ms = ctx.last_stage_ms()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / a.steps
    value = ms_per_step / 1e3 / world                           # seconds per segment, N segments proved per step

    from powdr_b200.capi import SegmentProof
    import ctypes
    C_sizeof_proof = ctypes.sizeof(SegmentProof)
    e2e = None
    if not a.no_e2e:
        host = torch.empty((w, n), dtype=torch.int32, pin_memory=True)
        host.copy_(trace)
        torch.cuda.synchronize()
        for _ in range(min(2, a.warmup)):
            ctx.prove_segment(air, host.data_ptr(), a.log_n, w, on_device=False)
        sync_all()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.time()
        f0.record(stream)
        for _ in range(a.steps):
            p2 = ctx.prove_segment(air, host.data_ptr(), a.log_n, w, on_device=False)
            q2, ys2 = ctx.query_segment(a.log_n, w, wp)
        f1.record(stream)
        sync_all()
        wall = (time.time() - t_wall) / a.steps
        ems = f0.elapsed_time(f1)
        te = torch.tensor([max(ems / 1e3 / a.steps, wall)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": float(te.item()) / world, "unit": "s", "h2d_bytes_per_step": 4 * w * n * world,
               "proof_equals_device_path": p2 == proof,           # same trace through the host-input pipeline: same proof
               "d2h_bytes_per_step": (C_sizeof_proof + int(q2.nbytes) + int(ys2.nbytes)) * world,
               "stages_ms": ctx.last_stage_ms()}

    last = (proof, {"queries": queries, "opened_values": ys})
    sharded = None
    if world > 1 and not a.no_sharded:
        sharded, last = sharded_segment(a, ctx, air, dist, dev, stream, world, rank)

    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, *last)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = (leaf_bytes / 1e9) / (leaf_ms / 1e3) if leaf_ms > 0 else 0.0
        traffic = None
        try:
            # one `ncu --set full` capture of this kernel gives DRAM bytes / algorithmic bytes of a launch; the timed launches differ in
            # width (main, permutation, quotient matrices), so the ratio is applied to their average algorithmic size
            traffic = json.load(open(os.path.join(ROOT, "profiles", "leaf_kernel_traffic.json")))["dram_over_algorithmic"] * leaf_bytes / max(1, n_leaf)
        except Exception:
            pass
        nn, ww, wpp = float(n), float(w), float(wp)
        alg = {"lde": 12 * nn * ww, "merkle": 8 * nn * ww + 64 * nn, "quotient": 8 * nn * (ww + (2 * wpp if wp else 0)) + 32 * nn,
               "logup_gen": 4 * nn * (ww + wpp), "logup_commit": 12 * nn * wpp + 8 * nn * wpp + 64 * nn}
        out = {
            "metric": METRIC, "value": value, "unit": "s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 (BabyBear, Montgomery)", "data": "synthetic",
            "config": {"workload": workload_name(a), "segments_per_step": world, "l2": "inputs (%.1f GB) exceed L2, no flush" % (4 * nn * ww / 1e9),
                       "timed_region": "pb_prove_segment + pb_query_segment per step",
                       "parallelism": "1 segment per GPU, NCCL all-gather of Merkle caps" if world > 1 else "single GPU"},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "p2::leaf_hash_cols_kernel (Poseidon2 leaf hashing)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "launches_timed": n_leaf,
                         "avg_launch_ms": leaf_ms / max(1, n_leaf), "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                         "note": "integer-ALU-bound kernel (~22 mulmod per byte); HBM fraction is reported as the contract asks"},
            # the same kernel against the roof that actually binds it: the integer multiplier pipe.  One Poseidon2 permutation
            # is 564 Montgomery products (10 pipe cycles each) + 117 constant products (8 cycles) = 657.6 Montgomery-product
            # equivalents; peak = 12.6 products/clk/SM measured by scripts/microbench.cu (profiles/r01_microbench.txt)
            "roofline_integer": (lambda perms, peak_i: {"bound": "imad pipe", "achieved": perms * 657.6 / (leaf_ms / 1e3) / 1e12 if leaf_ms > 0 else 0.0,
                                                        "peak": peak_i / 1e12, "unit": "T mulmod/s",
                                                        "frac": (perms * 657.6 / (leaf_ms / 1e3)) / peak_i if leaf_ms > 0 else 0.0})(
                (leaf_bytes / (4.0 * ww + 32.0)) * math.ceil(ww / 8.0) if n_leaf else 0.0,
                12.6 * 148 * ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6),
            "stages_ms": stage_ms, "keygen_s": keygen_s, "perm_width": wp,
            "stage_roofline_frac": {k: (alg[k] / 1e9) / (stage_ms[k] / 1e3) / peak for k in alg if stage_ms.get(k, 0) > 0},
            "segments_per_s": world / (ms_per_step / 1e3),
        }
        if a.metrics_out:
            from powdr_b200 import metrics
            metrics.write(a.metrics_out, metrics.segment_metrics(stage_ms, n, w, wp, len(spans), a.interactions))
        if e2e:
            out["e2e"] = e2e
        if sharded:
            # N > 1: the headline is ONE segment proved by all N GPUs together (strong scaling, same workload as N = 1); the
            # one-segment-per-GPU replicas measured above stay as an extra key
            out["replicas"] = {"value": value, "unit": "s", "scaling": "weak", "ms_per_step": ms_per_step, "segments_per_step": world,
                               "segments_per_s": world / (ms_per_step / 1e3), "stages_ms": stage_ms, "e2e": e2e}
            out["value"], out["ms_per_step"], out["scaling"] = sharded["value"], sharded["value"] * 1e3, "strong"
            out["stages_ms"] = sharded["stages_ms"]
            out["config"]["segments_per_step"] = 1
            out["config"]["parallelism"] = ("one segment on %d GPUs: column-sharded trace -> all-to-all -> row-sharded LDE / Merkle / LogUp / quotient / FRI "
                                            "(pb_prove_segment_sharded, NCCL over NVLink); proof identical to the single-GPU proof" % world)
            out["segments_per_s"] = 1.0 / sharded["value"]
            if "e2e" in sharded:
                out["e2e"] = sharded["e2e"]
            out["one_segment_on_all_gpus"] = sharded
        if world == 1 and not a.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(a, mach, bc, spans, bus)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def sharded_segment(a, ctx, air, dist, dev, stream, world, rank):
    """Strong scaling of ONE segment: the N ranks prove the same segment together (pb_prove_segment_sharded: column-sharded
    trace in, one all-to-all of folded coefficients, row-sharded LDE / Merkle / quotient / FRI; NCCL through
    powdr_b200.sharded.TorchComm).  Reported next to the weak-scaling headline; the proof is checked against the
    single-GPU proof of the same trace on every rank.  -> (result dict, (proof, query openings) of the last device-input step)"""
    import torch
    from powdr_b200.sharded import TorchComm, shard_columns
    n, w = 1 << a.log_n, air.width
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB2000000)                                   # the same trace on every rank
    full = torch.randint(0, P, (w, n), dtype=torch.int32, device=dev, generator=gen)
    single = ctx.prove_segment(air, full.data_ptr(), a.log_n, w, on_device=True)
    single_ms = ctx.last_stage_ms()["total"]
    single_q = ctx.query_segment(a.log_n, w, air.perm_width)[0] if a.queries else None
    first, count = shard_columns(w, world, rank)
    mine = full[first:first + count].clone()
    del full
    torch.cuda.empty_cache()
    comm = TorchComm()

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for _ in range(max(2, min(3, a.warmup))):
            fn()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(stream)
        for _ in range(a.steps):
            pr = fn()
        e1.record(stream)
        sync_all()
        wall = (time.time() - t0) / a.steps
        t = torch.tensor([max(e0.elapsed_time(e1) / 1e3 / a.steps, wall)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), pr

    q_state = {"on": bool(a.queries), "error": None}

    def sharded_queries():
        # a library error here is symmetric across ranks (same arguments, same state): record it once and keep the proof-only line
        if not q_state["on"]:
            return None
        try:
            return ctx.query_segment_sharded(comm, a.log_n, w, air.perm_width)
        except Exception as e:      # noqa: BLE001
            q_state["on"], q_state["error"] = False, repr(e)
            return None

    def step_dev():
        # the same unit of work as the N = 1 step: proof AND the query openings (pb_query_segment_sharded: one more all-gather)
        pr = ctx.prove_segment_sharded(air, mine.data_ptr() if count else 0, a.log_n, w, comm, on_device=True)
        return pr, sharded_queries()

    sec, (proof, queries) = timed(step_dev)
    stages = ctx.last_stage_ms()
    calls, nbytes = comm.calls, comm.bytes
    same = proof == single and (queries is None or bool((queries == single_q).all())) and q_state["error"] is None
    ok = torch.tensor([1 if same else 0], dtype=torch.int32, device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    out = {"value": sec, "unit": "s", "scaling": "strong", "single_gpu_s": single_ms / 1e3, "speedup": single_ms / 1e3 / sec,
           "proof_equals_single_gpu": bool(ok.item()), "stages_ms": stages,
           "collectives_per_segment": calls // max(1, a.steps + max(2, min(3, a.warmup))),
           "collective_bytes_per_rank_per_segment": nbytes // max(1, a.steps + max(2, min(3, a.warmup)))}
    if q_state["error"]:
        out["query_phase_error"] = q_state["error"]
    if not a.no_e2e:
        host = torch.empty((max(1, count), n), dtype=torch.int32, pin_memory=True)
        if count:
            host.copy_(mine)
        torch.cuda.synchronize()
        def step_host():
            pr = ctx.prove_segment_sharded(air, host.data_ptr() if count else 0, a.log_n, w, comm, on_device=False)
            sharded_queries()
            return pr

        esec, eproof = timed(step_host)
        import ctypes
        from powdr_b200.capi import SegmentProof
        out["e2e"] = {"value": esec, "unit": "s", "h2d_bytes_per_step": 4 * w * n, "d2h_bytes_per_step": (ctypes.sizeof(SegmentProof) + (4 * int(single_q.size) if single_q is not None else 0)) * world,
                      "proof_equals_single_gpu": eproof == single,
                      "stages_ms": ctx.last_stage_ms()}
    return out, (proof, {} if queries is None else {"queries": queries})


def multichip_shapes():
    """50 synthetic chips shaped like the guest-ecrecover APC set: widths sum to 18508, constraints to 10511
    (/root/reference/openvm-riscv/src/lib.rs:1332-1339); heights 2^12..2^18 by decreasing width rank (deterministic)."""
    s = [0xEC0EC0]

    def rnd():
        s[0] = (s[0] * 6364136223846793005 + 1442695040888963407) & (2**64 - 1)
        return (s[0] >> 33) / float(1 << 31)

    raw = sorted((2.718281828 ** (4.5 + 1.2 * (rnd() + rnd() + rnd() - 1.5)) for _ in range(50)), reverse=True)
    tot = sum(raw)
    widths = [max(8, int(round(x / tot * 18508))) for x in raw]
    widths[0] += 18508 - sum(widths)
    cons = [max(2, int(round(w * 10511 / 18508))) for w in widths]
    logs = [18 - (i * 7) // 50 for i in range(50)]          # widest chips are also the tallest: 2^18 ... 2^12
    return list(zip(logs, widths, cons))


def run_multichip(a):
    """strong scaling of ONE multi-chip segment: chips are independent until the transcript, so they are sharded by LPT
    on height*width; each rank proves its chips back to back; one all-gather of the per-chip Merkle caps ends the step."""
    import torch
    import powdr_b200
    from powdr_b200 import machine as M, parallel
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL's version banner goes to stdout by default: keep stdout = the JSON line
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream()
    ctx = powdr_b200.Context(local, stream.cuda_stream)
    shapes = multichip_shapes()
    costs = [w * (1 << ln) for ln, w, _ in shapes]
    plan = parallel.lpt_assign(costs, world)
    mine = plan[rank]
    kmax = max(len(p) for p in plan)
    chips = []
    ctx.set_fri_params(a.queries, a.pow_bits)
    n_ints_total = 0
    for i in mine:
        ln, w, c = shapes[i]
        base = M.synthetic_machine(w, c, seed=0xEC000 + i)
        # bus interactions in the keccak proportion (1734 per 2022 columns); the reference pins only their sum for this guest family
        n_ints = max(1, (w * 1734) // 2022) if a.interactions else 0
        mach = M.SymbolicMachine(base.constraints, M.synthetic_bus(base, n_ints, seed=0xEC200 + i)) if n_ints else base
        n_ints_total += n_ints
        bc, spans = M.compile_constraints(mach)
        air = ctx.air(bc, spans, mach.width, M.compile_bus(mach, 1) if n_ints else None)
        gen = torch.Generator(device=dev)
        gen.manual_seed(0xEC100 + i)
        chips.append((ln, mach.width, air, torch.randint(0, P, (mach.width, 1 << ln), dtype=torch.int32, device=dev, generator=gen)))
    caps = torch.zeros((kmax, 8), dtype=torch.int32, device=dev)
    one = bool(a.one_transcript)
    if one and world > 1:
        raise SystemExit("--one-transcript proves all chips of the segment on ONE GPU (pb_prove_chips); run it with --gpus 1")
    chip_args = [(air, tr.data_ptr(), ln, w) for ln, w, air, tr in chips]

    def step():
        if one:
            # every chip under one transcript: three mixed-height commitments, shared challenges, ONE FRI instance, one PoW, one query set
            ctx.prove_chips(chip_args)
            return
        roots = []
        for ln, w, air, tr in chips:
            roots.append(ctx.prove_segment(air, tr.data_ptr(), ln, w, on_device=True)["trace_root"])
            ctx.query_segment(ln, w, air.perm_width)
        if roots:
            caps[:len(roots)].copy_(torch.tensor(roots, dtype=torch.int64).to(torch.int32), non_blocking=True)
        parallel.all_gather_caps(caps, dist)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(a.warmup):
        step()
    sync_all()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(a.steps):
        step()
    e1.record(stream)
    sync_all()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / a.steps
    if rank == 0:
        mx, mean = parallel.plan_summary(costs, world)
        print(json.dumps({
            "metric": "proof-gen sec for a 50-chip APC segment (ecrecover-shaped), " + ("one transcript (pb_prove_chips)" if one else "chips sharded over GPUs"),
            "value": ms / 1e3, "unit": "s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 (BabyBear, Montgomery)", "data": "synthetic",
            "config": {"workload": "50 chips, widths sum 18508, constraints sum 10511, bus interactions ~0.86 per column (LogUp per chip), heights 2^12..2^18, "
                                   + ("%d queries + %d PoW bits for the segment; all chips in one proof: mixed-height MMCS x3, one FRI" if one else
                                      "%d queries + %d PoW bits per chip; LPT by height*width") % (a.queries, a.pow_bits),
                       "stages_ms": ctx.last_stage_ms() if one else None,
                       "lpt_max_over_mean": mx / mean, "chips_per_rank": [len(p) for p in plan]},
            "gpu_launches": ctx.launch_count() - l0}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def run_stage0(a):
    """Stage 0 (trace generation on the device, SURVEY §8 a5) at the keccak shape through the reference's own three entry points
    (_apc_tracegen, _apc_apply_bus; cuda_abi.rs:8-64): gather of W substituted columns out of a dummy original-AIR trace, then the
    periphery histograms of the AIR's bus interactions.  Reports the gather against the HBM roof (8 B per cell: read + write), the bus
    kernel's time, and the whole segment with the trace BORN on the device (stage 0 + pb_prove_segment + pb_query_segment) -- the flow of
    /root/reference/openvm/src/powdr_extension/trace_generator/cuda/mod.rs:201-421, where no host copy of the trace ever exists."""
    import ctypes as C
    import numpy as np
    import torch
    import powdr_b200
    from powdr_b200 import capi, machine as M
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream()                      # the reference symbols launch on the default stream
    ctx = powdr_b200.Context(0, stream.cuda_stream)
    ctx.set_fri_params(a.queries, a.pow_bits)
    mach, bc, spans, bus = machine_for(a)
    air = ctx.air(bc, spans, mach.width, bus)
    H, W = 1 << a.log_n, mach.width
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB2000007)
    src = torch.randint(0, 256, (W, H), dtype=torch.int32, device=dev, generator=gen)      # byte-valued cells, as most APC columns are
    ctx.lib.pb_to_monty(ctx.h, C.c_void_p(src.data_ptr()), C.c_size_t(W * H))
    out = torch.empty((W, H), dtype=torch.int32, device=dev)
    airs = (capi.OriginalAir * 1)()
    airs[0].width, airs[0].height, airs[0].buffer, airs[0].row_block_size = W, H, src.data_ptr(), 1
    subs = (capi.Subst * W)()
    for i in range(W):
        subs[i].air_index, subs[i].col, subs[i].row, subs[i].apc_col = 0, (i * 7919) % W, 0, i
    ints, isp, ibc = M.compile_bus(mach, H)                   # absolute-offset convention of the reference kernels (col * H)
    di = (capi.DevInteraction * len(ints))()
    for i, (b, k, o) in enumerate(ints):
        di[i].bus_id, di[i].num_args, di[i].args_index_off = b, k, o
    spn = (capi.Span * len(isp))()
    for i, (o, l) in enumerate(isp):
        spn[i].off, spn[i].len = o, l

    def up(raw):
        t = torch.from_numpy(np.frombuffer(bytes(raw), dtype=np.uint8).copy()).to(dev)
        return t
    d_airs, d_subs, d_ints, d_spans = up(airs), up(subs), up(di), up(spn)
    d_bc = torch.tensor(np.array(ibc, dtype=np.uint32).astype(np.int64), dtype=torch.int64, device=dev).to(torch.int32)
    var_hist = torch.zeros(1 << 18, dtype=torch.int32, device=dev)
    t2_hist = torch.zeros(256 * 2048, dtype=torch.int32, device=dev)
    bw_hist = torch.zeros(1 << 17, dtype=torch.int32, device=dev)

    def gather():
        ctx.apc_tracegen(out.data_ptr(), H, d_airs.data_ptr(), d_subs.data_ptr(), W, H)

    def busk():
        ctx.apc_apply_bus(out.data_ptr(), H, d_bc.data_ptr(), len(ibc), d_ints.data_ptr(), len(ints), d_spans.data_ptr(), len(isp), 3, var_hist.data_ptr(),
                          1 << 18, 7, t2_hist.data_ptr(), 256, 2048, 6, bw_hist.data_ptr())

    def timed(fn, reps):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    handle = ctx.bus_compile(bus, W)                           # per-AIR generated periphery kernel (bus_jit.cuh)

    def busj():
        ctx.bus_apply(handle, out.data_ptr(), H, H, var_hist.data_ptr(), 1 << 18, t2_hist.data_ptr(), 256, 2048, bw_hist.data_ptr())

    gather()
    var_hist.zero_(); t2_hist.zero_(); bw_hist.zero_()
    busk()
    ref = (var_hist.clone(), t2_hist.clone(), bw_hist.clone())
    var_hist.zero_(); t2_hist.zero_(); bw_hist.zero_()
    busj()
    same = bool((ref[0] == var_hist).all() and (ref[1] == t2_hist).all() and (ref[2] == bw_hist).all())
    g_ms, b_ms, j_ms = timed(gather, a.steps), timed(busk, a.steps), timed(busj, a.steps)

    def whole():
        gather()
        busj()
        ctx.prove_segment(air, out.data_ptr(), a.log_n, W, on_device=True)
        ctx.query_segment(a.log_n, W, air.perm_width)
    w_ms = timed(whole, max(1, a.steps // 2))
    peak = 6575.1
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    gbs = 8.0 * H * W / 1e9 / (g_ms / 1e3)
    n_periph = sum(1 for b, _, _ in ints if b in (3, 6, 7))
    print(json.dumps({
        "metric": "stage 0 (device trace generation) ms for the guest-keccak APC shape", "value": (g_ms + j_ms) / 1e3, "unit": "s", "n_gpus": 1, "steps": a.steps,
        "warmup": 2, "higher_is_better": False, "dtype": "u32 (BabyBear, Montgomery)", "data": "synthetic",
        "config": {"workload": "2^%d rows: gather of %d substituted columns from a dummy original-AIR trace, periphery histograms of %d of %d bus interactions" % (
            a.log_n, W, n_periph, len(ints))},
        "gather": {"ms": g_ms, "algorithmic_bytes": 8.0 * H * W, "achieved_GBps": gbs, "peak_GBps": peak, "frac": gbs / peak},
        "apply_bus_dropin": {"ms": b_ms, "interactions_evaluated_per_row": n_periph, "G_interaction_rows_per_s": n_periph * H / (b_ms / 1e3) / 1e9,
                             "note": "_apc_apply_bus: the reference's symbol and shape (row-serial bytecode interpreter)"},
        "apply_bus_generated": {"ms": j_ms, "G_interaction_rows_per_s": n_periph * H / (j_ms / 1e3) / 1e9, "histograms_equal_dropin": same,
                                "note": "pb_bus_apply: per-AIR NVRTC kernel, (row tile) x (interaction group) grid"},
        "segment_with_trace_born_on_device": {"ms": w_ms, "note": "stage 0 + pb_prove_segment + pb_query_segment, no host copy of the trace"}}))
    ctx.close()


def run_pairing(a):
    """BASELINE.json configs[4]: one segment too wide for one GPU's comfort (2^20 x 16384 = 68.7 GB of trace, 137 GB of LDE)
    proved by all ranks together (pb_prove_segment_sharded).  Every rank generates only its own column block; the proofs of
    all ranks must be identical.  Constraints only (the sharded prover has no LogUp phase yet)."""
    import torch
    import torch.distributed as dist
    import powdr_b200
    from powdr_b200 import machine as M
    from powdr_b200.sharded import TorchComm, shard_columns
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world > 1, "--workload pairing shards one segment over the ranks: launch with torchrun, N >= 2"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.current_stream()
    ctx = powdr_b200.Context(local, stream.cuda_stream)
    ctx.set_fri_params(a.queries, a.pow_bits)
    width = a.width if a.width != 2022 else 16384
    ncons = a.constraints if a.constraints != 187 else 4096
    mach = M.synthetic_machine(width, ncons, seed=0xB2000005)
    bc, spans = M.compile_constraints(mach)
    t_key = time.time()
    air = ctx.air(bc, spans, mach.width)
    keygen_s = time.time() - t_key
    n, w = 1 << a.log_n, mach.width
    first, count = shard_columns(w, world, rank)
    gen = torch.Generator(device=dev)
    gen.manual_seed(0xB2000500 + rank)
    mine = torch.randint(0, P, (max(1, count), n), dtype=torch.int32, device=dev, generator=gen)
    comm = TorchComm()

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def step():
        pr = ctx.prove_segment_sharded(air, mine.data_ptr() if count else 0, a.log_n, w, comm, on_device=True)
        if a.queries:
            ctx.query_segment_sharded(comm, a.log_n, w, 0)       # the query openings belong to the unit of work, as at N = 1
        return pr

    for _ in range(a.warmup):
        step()
    sync_all()
    l0 = ctx.launch_count()
    c0, b0 = comm.calls, comm.bytes
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record(stream)
    for _ in range(a.steps):
        proof = step()
    e1.record(stream)
    sync_all()
    wall = (time.time() - t0) / a.steps
    t = torch.tensor([max(e0.elapsed_time(e1) / 1e3 / a.steps, wall)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sig = torch.tensor(proof["trace_root"] + proof["quotient_root"] + proof["final_poly"][0] + [proof["pow_witness"]], dtype=torch.int64, device=dev)
    lo, hi = sig.clone(), sig.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    same = bool((lo == hi).all().item())
    if rank == 0:
        print(json.dumps({
            "metric": "proof-gen sec for ONE wide APC segment (guest-pairing shape) column-sharded over N B200", "value": float(t.item()), "unit": "s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": float(t.item()) * 1e3, "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32 (BabyBear, Montgomery)", "data": "synthetic",
            "config": {"workload": "2^%d rows x %d cols, %d constraints deg<=3, no bus interactions (sharded prover), log_blowup 1; trace %.1f GB, LDE %.1f GB "
                                   "in total, column block per rank resident in HBM" % (a.log_n, w, ncons, 4.0 * n * w / 1e9, 8.0 * n * w / 1e9),
                       "parallelism": "column-sharded trace -> one all-to-all -> row-sharded LDE/Merkle/quotient/FRI; NCCL over NVLink"},
            "proof_identical_on_all_ranks": same, "final_poly_constant": proof["final_poly"][0] == proof["final_poly"][1],
            "stages_ms": ctx.last_stage_ms(), "keygen_s": keygen_s, "gpu_launches": ctx.launch_count() - l0,
            "collectives_per_segment": (comm.calls - c0) // a.steps, "collective_bytes_per_rank_per_segment": (comm.bytes - b0) // a.steps}))
    dist.barrier()
    dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "multichip":
        run_multichip(args)
    elif args.workload == "pairing":
        run_pairing(args)
    elif args.workload == "stage0":
        run_stage0(args)
    else:
        run_native(args)
