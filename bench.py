#!/usr/bin/env python3
"""bench.py — headline benchmark of the hot path (BASELINE.json metric).

Metric   field-muls/s on a 2^24-coefficient forward NTT over the 64-bit prime 2^64-2^32+1
         (algorithmic count (n/2)·log2 n = 201 326 592 per transform, independent of the radix used).
Step     one in-place forward NTT of one 2^24-coefficient polynomial per GPU, operands resident in
         HBM (`value`), or pinned host → HBM → NTT → pinned host through the C ABI (`e2e`).
N > 1    one process per GPU (torchrun), independent transforms per rank, no data-path collective
         (SURVEY §8e "batched NTTs"): weak scaling, value = N·muls / max-over-ranks time.  The line also
         carries a `multi` block with the other multi-GPU modes of the path, all through the C ABI
         (ronk_dist_* in include/ronk_b200.h, NCCL inside the library): BASELINE config 5 (4096 × 2^16) sharded
         with no collective and as the all-to-all variant (top log2 N stages across GPUs, NCCL and fused
         peer-memory flavours), ONE 2^24 transform across the N GPUs, and kzg::commit of 2^20 terms over
         index-range shards — each with a bit_exact flag from an in-run check against the oracle.
N = 1    the line carries a `configs` block: BASELINE configs 2, 3, 4 and one GPU's share of config 5, each
         checked against the oracle and with its own roofline fraction.
--impl reference   the reference's own algorithm (oracle/ronk_oracle.c: faithful recursive
         fft_recursive, src/polynomial/mod.rs:295-323) on the box's host cores, one independent
         2^24 transform per thread.

The oracle (oracle/) is used here only as the checker (spot checks outside every timed region) and as the
CPU baseline; nothing timed on the GPU arm runs through it.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GL = 0xFFFFFFFF00000001
LOG_N = 24
N = 1 << LOG_N
MULS_PER_NTT = (N // 2) * LOG_N          # 201 326 592 (SURVEY §8d)
ALG_BYTES_PER_NTT = 16 * N               # one read + one write of the data (SURVEY §8d)
METRIC = "field-muls/s on 2^24-coeff 64-bit-prime NTT"
UNIT = "field-muls/s"
DUMP_SAMPLE = 1 << 20                    # output coefficients --dump-outputs writes, over all ranks


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
            }
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report, never fake
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def bind_to_gpu_numa(index: int):
    """Pin this rank's host threads and (preferred) memory policy to the NUMA node its GPU hangs off, BEFORE the
    pinned staging buffers are allocated: in round 1 un-bound torchrun ranks allocated them wherever the kernel had
    put the process, and the 8-GPU end-to-end step doubled in time.  Returns what was done (reported in the line)."""
    info = {"bound": False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        if len(bus.split(":")[0]) == 8:      # NVML prints an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus.lower()}/numa_node") as f:
            node = int(f.read().strip())
        info["numa_node"] = node
        if node < 0:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        os.sched_setaffinity(0, cpus)
        info["cpus"] = len(cpus)
        libc = ctypes.CDLL(None, use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(65))  # set_mempolicy(MPOL_PREFERRED, node)
        info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
        info["bound"] = True
    except Exception as e:
        info["error"] = f"{type(e).__name__}: {e}"
    return info


def run_reference(args):
    """--impl reference: the reference algorithm on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, args.ref_threads or cores))
    for _ in range(args.warmup):
        oracle.bench_fft_threads(GL, N, threads)
    t = 0.0
    for _ in range(args.steps):
        secs, _ = oracle.bench_fft_threads(GL, N, threads)
        t += secs
    ms = 1e3 * t / args.steps
    value = threads * MULS_PER_NTT / (t / args.steps)
    sample = f"{threads} independent 2^24-point transforms per step, one per host thread (faithful recursive fft_recursive)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic (splitmix64 mod p, seed 42+thread)",
        "config": {"workload": "2^24-coeff forward NTT, Goldilocks p=2^64-2^32+1, g=7", "parallelism": f"{threads} host threads"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------
# helpers shared by the N = 1 `configs` block and the N > 1 `multi` block
# ------------------------------------------------------------------------------------------------------------
def msm_terms(n, seed_pts=44, seed_sc=45):
    """SURVEY §8d inputs of config 4: points k·G1 + l·G2 with (k, l) from splitmix(seed 44) mod 17 (on the curve by
    construction, Infinity when both are 0), scalars from seed 45 mod 17.  Input synthesis only."""
    import numpy as np
    import oracle
    g1, g2 = bytes([1, 0, 2, 0]), bytes([36, 0, 0, 31])
    lut = np.zeros((17, 17, 4), dtype=np.uint8)
    for k in range(17):
        for l in range(17):
            lut[k, l] = np.frombuffer(oracle.point_add(oracle.point_smul(g1, k), oracle.point_smul(g2, l)), dtype=np.uint8)
    kl = oracle.splitmix(17, seed_pts, 2 * n).astype(np.int64)
    return np.ascontiguousarray(lut[kl[0::2], kl[1::2]]), oracle.splitmix(17, seed_sc, n).astype(np.uint8)


def horner_spots(a_host, X_host, log_n, ks):
    """X[k] == a(ω^k) for the listed k (oracle Horner, O(n) each) — a size-independent check of a transform."""
    import oracle
    w = oracle.root_of_unity(GL, 1 << log_n)
    return all(int(X_host[k]) == oracle.poly_eval_horner(GL, a_host, pow(w, k, GL)) for k in ks)


def dump_outputs(out_dir, x, rank, world):
    """--dump-outputs: what the last timed step left in the 2^24-coefficient operand (u64 mod p), as a fixed sample
    of DUMP_SAMPLE coefficients over all ranks (seed 0, sorted): the indices and values as float64 (values rounded
    to 53 bits) and the values exactly as four 16-bit limbs, least significant first, in float32."""
    import numpy as np
    idx = np.sort(np.random.default_rng(0).choice(N, DUMP_SAMPLE // world, replace=False))
    v = x[idx]
    limbs = np.stack([(v >> np.uint64(16 * k)) & np.uint64(0xFFFF) for k in range(4)], axis=1)
    suffix = "" if world == 1 else f"_rank{rank}"
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"ntt_out_index{suffix}.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, f"ntt_out{suffix}.npy"), v.astype(np.float64))
    np.save(os.path.join(out_dir, f"ntt_out_u16{suffix}.npy"), limbs.astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `configs` / `multi` blocks (A/B timing runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of the last timed step's output to DIR/*.npy (32 MiB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    numa = bind_to_gpu_numa(local_rank)   # before torch creates its threads and before any pinned allocation

    # This program's stdout is ONE JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its
    # version banner there when NCCL_DEBUG is set in the environment): everything before the JSON line goes to stderr.
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from ronkathon_b200 import Context, ops
    ctx = Context(local_rank, torch.cuda.current_stream().cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, iters, warm=3):
        """CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks (ms per call)."""
        for _ in range(warm):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / iters)

    # synthetic operand, generated on the device (splitmix64 mod p, seed 42 + rank)
    data = ops.splitmix_fill(ctx, N, 42 + rank, GL, dev)
    ctx.sync()
    for _ in range(args.warmup):
        ops.ntt_(ctx, data, LOG_N)
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.05)

    # ---- timed region 1: whole-job throughput, operands resident in HBM -------------------------
    launches0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        ops.ntt_(ctx, data, LOG_N)
    e1.record()
    barrier()
    launches = ctx.launches - launches0
    ms_per_step = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    value = world * MULS_PER_NTT / (ms_per_step * 1e-3)
    last_output = ops.to_host(data) if args.dump_outputs else None   # region 2 transforms `data` again

    # ---- timed region 2: per-kernel durations (CUDA events around every launch, same stream) ----
    ctx.prof_enable(True)
    barrier()
    for _ in range(args.steps):
        ops.ntt_(ctx, data, LOG_N)
    recs = ctx.prof_fetch()
    ctx.prof_enable(False)
    per = {}
    for name, ms in recs:
        per.setdefault(name, []).append(ms)
    kern = {k: sum(v) / len(v) for k, v in per.items()}
    dom = max(kern, key=kern.get)
    stages = {"ntt_pass1": 12, "ntt_pass2": 12, "ntt3_pass1": 8, "ntt3_pass2": 8, "ntt3_pass3": 8}
    peak, peak_src = measured_peaks()
    # algorithmic bytes of one launch = 16·n · (butterfly stages this launch does / 24)
    alg_bytes = ALG_BYTES_PER_NTT * stages.get(dom, 24) / 24
    achieved = alg_bytes / (kern[dom] * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(dom)
    whole_ms = sum(kern.values())
    roofline = {
        "bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "peak_source": peak_src,
        "alg_bytes_per_launch": alg_bytes, "kernel_ms": kern,
        "whole_ntt": {"alg_bytes": ALG_BYTES_PER_NTT, "ms": whole_ms,
                      "achieved": ALG_BYTES_PER_NTT / (whole_ms * 1e-3) / 1e9,
                      "frac": ALG_BYTES_PER_NTT / (whole_ms * 1e-3) / 1e9 / peak},
    }

    # ---- what was timed is correct: fresh input, two outputs against the oracle's Horner (outside any timed region)
    spot = None
    if rank == 0:
        fresh = ops.splitmix_fill(ctx, N, 7, GL, dev)
        a_host = ops.to_host(fresh)
        ops.ntt_(ctx, fresh, LOG_N)
        ctx.sync()
        ks = [1, N // 2 + 3]
        spot = {"ok": bool(horner_spots(a_host, ops.to_host(fresh), LOG_N, ks)), "indices": ks,
                "how": "X[k] == a(ω^k), oracle Horner over the 2^24 coefficients of a fresh input"}
        del fresh, a_host

    # ---- timed region 3: end to end through the C ABI with HOST buffers -------------------------
    # Every step uploads its own pinned host buffer, transforms it and downloads the result
    # (ronk_ntt_u64_host_submit / _wait).  Three steps are in flight (three device slots): the upload
    # of step i+1, the kernels of step i and the download of step i-1 overlap on the full-duplex link.
    SLOTS = 3
    hosts = [torch.empty(N, dtype=torch.int64).pin_memory() for _ in range(SLOTS)]
    for h in hosts:
        h.copy_(data.cpu())

    def e2e_run(steps):
        for i in range(steps):
            ctx.call("ronk_ntt_u64_host_submit", GL, 7, hosts[i % SLOTS].data_ptr(), LOG_N, 1, 0, i % SLOTS)
            if i >= SLOTS - 1:
                ctx.call("ronk_ntt_u64_host_wait", (i - (SLOTS - 1)) % SLOTS)
        for s in range(SLOTS):
            ctx.call("ronk_ntt_u64_host_wait", s)

    e2e_run(4)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps)
    torch.cuda.synchronize()
    e2e_mine = (time.perf_counter() - t0) / args.steps
    e2e_s = max_over_ranks(e2e_mine)
    e2e_value = world * MULS_PER_NTT / e2e_s
    copy_gbs = 2 * 8 * N / e2e_mine / 1e9   # this rank's H2D + D2H bytes per second while all N ranks copy
    gbs = [copy_gbs]
    if world > 1:
        g = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(g, torch.tensor([copy_gbs], dtype=torch.float64, device=dev))
        gbs = [float(x.item()) for x in g]
    # single-step latency (no overlap) for reference
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        ctx.call("ronk_ntt_u64_host", GL, 7, hosts[0].data_ptr(), LOG_N, 1, 0)
    e2e_latency_ms = 1e3 * (time.perf_counter() - t0) / 3
    del hosts

    sampler.stop_flag = True
    sampler.join(timeout=2)
    clocks = sampler.result()

    # ---- N = 1: the other BASELINE configs, each checked against the oracle ---------------------------------
    configs = None
    if world == 1 and not args.no_extras:
        try:
            configs = run_configs(ctx, ops, dev, timed, peak)
        except Exception as e:  # never lose the headline line
            configs = {"error": f"{type(e).__name__}: {e}"}

    # ---- N > 1: the other multi-GPU modes, through the C ABI -------------------------------------------------
    multi = None
    if world > 1 and not args.no_extras:
        try:
            multi = run_multi(ctx, ops, dev, timed, rank, world, peak)
        except Exception as e:
            multi = {"error": f"{type(e).__name__}: {e}"}

    # ---- CPU baseline beside it (rank 0, N = 1 only) ---------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        secs, _ = oracle.bench_fft_threads(GL, N, 1)
        cpu_baseline = {"value": MULS_PER_NTT / secs, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": "one full 2^24-point faithful recursive fft (polynomial/mod.rs:295-323 restated in C), "
                                  f"single thread as in the reference, {secs:.2f} s; host has {os.cpu_count()} cores"}

    if last_output is not None:
        dump_outputs(args.dump_outputs, last_output, rank, world)
        del last_output

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic (splitmix64 mod p generated on device, seed 42+rank)",
            "config": {"workload": "2^24-coeff forward NTT, Goldilocks p=2^64-2^32+1, g=7, in place, natural order in/out",
                       "per_gpu": "1 transform per step", "parallelism": f"independent transforms × {world} GPU(s), no collective",
                       "l2": "working set 256 MiB (data + workspace) > 126 MB L2; no flush needed"},
            "roofline": roofline,
            "spot_check": spot,
            "cpu_baseline": cpu_baseline,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 8 * N, "d2h_bytes_per_step": 8 * N,
                    "ms_per_step": 1e3 * e2e_s, "single_step_latency_ms": e2e_latency_ms,
                    "api": "ronk_ntt_u64_host_submit/_wait, pinned host buffers, 3 steps in flight",
                    "copy_gbs_per_rank": [round(x, 1) for x in gbs], "numa": numa},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if configs is not None:
            line["configs"] = configs
        if multi is not None:
            line["multi"] = multi
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_configs(ctx, ops, dev, timed, peak):
    """BASELINE configs 2, 3, 4 and one GPU's share of config 5 on one GPU: check against the oracle, then time with
    CUDA events; `frac` = algorithmic bytes (SURVEY §8d) / time / measured HBM peak."""
    import numpy as np
    import torch
    import oracle
    out = {}

    def frac(nbytes, ms):
        return nbytes / (ms * 1e-3) / 1e9 / peak

    # config 2: 2^20-coefficient forward NTT, bit-exact vs the oracle
    lg = 20
    a = oracle.splitmix(GL, 42, 1 << lg)
    d = ops.to_device(a, dev)
    ops.ntt_(ctx, d, lg)
    ctx.sync()
    ok = bool(np.array_equal(ops.to_host(d), oracle.ntt_fast(GL, a)))
    ms = timed(lambda: ops.ntt_(ctx, d, lg), 50)
    out["config2_ntt_2^20"] = {"bit_exact": ok, "ms": ms, "field_muls_per_s": (1 << (lg - 1)) * lg / (ms * 1e-3),
                               "alg_bytes": 16 << lg, "frac": frac(16 << lg, ms)}

    # config 3: 2^23 × 2^23 coefficients (2 forward + fused point-wise + 1 inverse 2^24-point transform)
    n3 = 1 << 23
    pa, pb = ops.splitmix_fill(ctx, n3, 42, GL, dev), ops.splitmix_fill(ctx, n3, 43, GL, dev)
    pc = ops.poly_mul(ctx, pa, pb)
    ctx.sync()
    ha, hb, hc = ops.to_host(pa), ops.to_host(pb), ops.to_host(pc)
    x = 0x123456789ABCDEF1 % GL
    ev = lambda c: oracle.poly_eval_horner(GL, c, x)  # noqa: E731
    ok = bool(ev(hc) == oracle.mul(GL, ev(ha), ev(hb)) and int(hc[0]) == oracle.mul(GL, int(ha[0]), int(hb[0]))
              and int(hc[-1]) == oracle.mul(GL, int(ha[-1]), int(hb[-1])) and len(hc) == 2 * n3 - 1)
    ms = timed(lambda: ops.poly_mul(ctx, pa, pb), 10)
    muls = 3 * (N // 2) * LOG_N + 2 * N
    out["config3_poly_mul_2^23x2^23"] = {"identity_checks": ok, "ms": ms, "field_muls_per_s": muls / (ms * 1e-3),
                                         "alg_bytes": 24 * N, "frac": frac(24 * N, ms),
                                         "check": "c(x) = a(x)·b(x) at one point (oracle Horner), first / last coefficient, length"}
    del pa, pb, pc, ha, hb, hc

    # config 4: kzg::commit of 2^20 (point, scalar) pairs
    n4 = 1 << 20
    pts, sc = msm_terms(n4)
    P, S = torch.from_numpy(pts).to(dev), torch.from_numpy(sc).to(dev)
    got = ops.msm(ctx, P, S)
    ok = bool(got == oracle.commit(sc, pts, fast=True))
    ms = timed(lambda: ops.msm(ctx, P, S), 30)
    out["config4_commit_2^20"] = {"bit_exact": ok, "ms_per_call": ms, "point_adds_per_s": n4 / (ms * 1e-3),
                                  "alg_bytes": 5 * n4, "bytes_per_s": 5 * n4 / (ms * 1e-3), "frac": frac(5 * n4, ms),
                                  "note": "whole synchronous call incl. the 4-byte result back on the host"}

    # one GPU's share of config 5: 512 × 2^16
    bt, lg5 = 512, 16
    buf = ops.splitmix_fill(ctx, bt << lg5, 100, GL, dev)
    first = ops.to_host(buf[: 1 << lg5])
    last = ops.to_host(buf[(bt - 1) << lg5:])
    ops.ntt_(ctx, buf, lg5, bt)
    ctx.sync()
    ok = bool(np.array_equal(ops.to_host(buf[: 1 << lg5]), oracle.ntt_fast(GL, first))
              and np.array_equal(ops.to_host(buf[(bt - 1) << lg5:]), oracle.ntt_fast(GL, last)))
    ms = timed(lambda: ops.ntt_(ctx, buf, lg5, bt), 20)
    out["config5_share_512x2^16"] = {"bit_exact_sampled": ok, "ms": ms, "field_muls_per_s": bt * (1 << (lg5 - 1)) * lg5 / (ms * 1e-3),
                                     "alg_bytes": 16 * (bt << lg5), "frac": frac(16 * (bt << lg5), ms)}
    return out


def run_multi(ctx, ops, dev, timed, rank, world, peak):
    """The multi-GPU modes other than independent replicas, through the C ABI's ronk_dist_* entry points."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import oracle
    from ronkathon_b200 import dist as rd

    # NCCL prints its version banner on STDOUT when a communicator is created with NCCL_DEBUG=VERSION/INFO in the
    # environment; this program's stdout is one JSON line, so the banner goes to stderr
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dctx = rd.DistContext(ctx)
        ctx.sync()
    finally:
        os.dup2(saved, 1)
        os.close(saved)
    out = {"abi": "ronk_dist_init / ronk_ntt_u64_batch_sharded / ronk_ntt_u64_dist / ronk_msm_pluto_ext_dist", "n_gpus": world}

    def gather_host(t):
        """all ranks' tensors (equal shapes) → list of numpy uint64 arrays on every rank"""
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous())
        return [ops.to_host(p) for p in parts]

    # ---- BASELINE config 5, contiguous shards, no collective (strong scaling: 4096 × 2^16 in total)
    total, lg = 4096, 16
    lo, hi = dctx.shard_range(total)
    buf = ops.splitmix_fill(ctx, (hi - lo) << lg, 100 + rank, GL, dev)
    first = ops.to_host(buf[: 1 << lg])
    dctx.ntt_batch_sharded(buf, lg, total)
    ctx.sync()
    ok = bool(np.array_equal(ops.to_host(buf[: 1 << lg]), oracle.ntt_fast(GL, first)))
    ms = timed(lambda: dctx.ntt_batch_sharded(buf, lg, total), 10)
    muls5 = total * (1 << (lg - 1)) * lg
    out["config5_sharded"] = {"ms": ms, "field_muls_per_s": muls5 / (ms * 1e-3), "bit_exact": ok,
                              "scaling": "strong", "collective": "none",
                              "check": "first transform of every rank's shard == oracle (rank 0 reports its own)"}
    del buf

    # ---- the same 4096 transforms with the top log2(N) stages across the GPUs: ONE exchange (all-to-all)
    m = (1 << lg) // world
    blk = m // world
    for name, flavour in (("nccl", rd.DIST_NCCL), ("fused_p2p", rd.DIST_FUSED)):
        loc = ops.splitmix_fill(ctx, total * m, 1000 + rank, GL, dev)
        probe = [0, total - 1]
        ins = {b: gather_host(loc[b * m:(b + 1) * m]) for b in probe}
        dctx.ntt_dist(loc, lg, total, flavour)
        ctx.sync()
        ok = True
        for b in probe:
            outs = gather_host(loc[b * m:(b + 1) * m])
            a = np.empty(1 << lg, dtype=np.uint64)
            for r in range(world):
                a[r::world] = ins[b][r]
            X = np.empty(1 << lg, dtype=np.uint64)
            for s in range(world):
                o = outs[s].reshape(world, blk)
                for q in range(world):
                    X[s * blk + m * q: s * blk + m * q + blk] = o[q]
            ok = ok and bool(np.array_equal(X, oracle.ntt_fast(GL, a)))
        ms = timed(lambda: dctx.ntt_dist(loc, lg, total, flavour), 10)
        out[f"config5_alltoall_{name}"] = {"ms": ms, "field_muls_per_s": muls5 / (ms * 1e-3), "bit_exact": ok,
                                           "scaling": "strong", "exchange_bytes_per_gpu": 8 * total * m * (world - 1) // world,
                                           "check": "transforms 0 and 4095 reassembled from all ranks == oracle"}
        del loc

    # ---- ONE 2^24-point transform across the N GPUs
    lgn = 24
    mm = (1 << lgn) // world
    bb = mm // world
    for name, flavour in (("nccl", rd.DIST_NCCL), ("fused_p2p", rd.DIST_FUSED)):
        loc = ops.splitmix_fill(ctx, mm, 5 + rank, GL, dev)
        src = loc.clone()
        ins = gather_host(loc)
        dctx.ntt_dist(loc, lgn, 1, flavour)
        ctx.sync()
        outs = gather_host(loc)
        ok = None
        if rank == 0:
            a = np.empty(1 << lgn, dtype=np.uint64)
            for r in range(world):
                a[r::world] = ins[r]
            X = np.empty(1 << lgn, dtype=np.uint64)
            for s in range(world):
                o = outs[s].reshape(world, bb)
                for q in range(world):
                    X[s * bb + mm * q: s * bb + mm * q + bb] = o[q]
            ok = bool(horner_spots(a, X, lgn, [0, 1, (1 << 23) + 3, (1 << lgn) - 1]))
            del a, X
        del ins, outs

        def one():
            loc.copy_(src)
            dctx.ntt_dist(loc, lgn, 1, flavour)
        ms = timed(one, 10)
        out[f"dist_ntt_2^24_{name}"] = {"ms": ms, "field_muls_per_s": MULS_PER_NTT / (ms * 1e-3), "bit_exact": ok,
                                        "check": "X[k] == a(ω^k) at 4 indices (oracle Horner on the gathered input)",
                                        "note": "timed step includes a device copy of the n/N-word input"}
        del loc, src

    # ---- kzg::commit of 2^20 terms over index-range shards
    n4 = 1 << 20
    pts, sc = msm_terms(n4)
    i0, i1 = dctx.shard_range(n4)
    P, S = torch.from_numpy(pts[i0:i1].copy()).to(dev), torch.from_numpy(sc[i0:i1].copy()).to(dev)
    got = dctx.msm(P, S)
    ok = bool(got == oracle.commit(sc, pts, fast=True)) if rank == 0 else None
    ms = timed(lambda: dctx.msm(P, S), 10)
    out["commit_2^20_sharded"] = {"ms_per_call": ms, "point_adds_per_s": n4 / (ms * 1e-3), "bit_exact": ok,
                                  "collective": "one 4-byte-per-rank ncclAllGather"}
    dctx.close()
    return out


if __name__ == "__main__":
    main()
