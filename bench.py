#!/usr/bin/env python
"""bench.py -- throughput of the batched 1-D complex FFT hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c1] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  The default workload is
BASELINE.json configs[1]: batched N=2^20 complex-f32 forward FFT, batch 4096, on one B200.  With
--gpus N>1 (launched by torchrun, one rank per GPU) every rank transforms its own batch of the same
size (independent transforms, no data-path collective): weak scaling.

Prints ONE JSON line (rank 0).  `value` is whole-job complex samples/s with inputs resident in HBM;
`e2e` is the same metric through the C-ABI call with HOST (pinned) buffers, copies inside the timed
region; `roofline` relates the dominant kernel's algorithmic bytes (16 B/sample f32, 32 B/sample
f64: read once + write once, SURVEY.md 8d) to the measured HBM peak; `cpu_baseline` is the oracle
(C restatement of the reference CPU algorithm; the Rust reference cannot be built in this image)
timed on the host cores on a bounded sample.

--dump-outputs DIR writes what the last timed step returned (rank 0's share) to DIR as .npy files, so that two
builds can be compared output for output: the inputs are the same hash-generated data in every run.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N, per-GPU batch, real, description)
    "c1": (1024, 1, "f32", "single 1024-pt c-f32 forward (BASELINE configs[0], correctness gate)"),
    "c2": (1 << 20, 4096, "f32", "batched N=2^20 c-f32 forward, batch 4096 per GPU (BASELINE configs[1])"),
    "c3": (1 << 16, 65536, "f64", "batched N=2^16 c-f64 forward, batch 65536 (BASELINE configs[2])"),
    "c4": (1009, 1 << 20, "f32", "prime N=1009 Bluestein c-f32 forward, batch 2^20 (BASELINE configs[3])"),
    "c5": (1 << 30, 1, "f32", "single distributed N=2^30 c-f32 over all ranks, six-step with NCCL all-to-all "
                              "transposes (BASELINE configs[4])"),
}
BYTES_PER_SAMPLE = {"f32": 16, "f64": 32}  # algorithmic: read once + write once


def measured_traffic(workload):
    """DRAM bytes per sample of the dominant kernel from the committed ncu capture (profiles/), or None."""
    try:
        for name in ("r02_traffic.json", "r01_traffic.json"):
            path = os.path.join(ROOT, "profiles", name)
            if os.path.exists(path):
                with open(path) as f:
                    d = json.load(f)
                if workload in d:
                    return d[workload]
        return None
    except Exception:
        return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (pynvml)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


def cpu_baseline(n, real, seconds_target=12.0, threads=None):
    """Oracle (C restatement of the reference CPU path) on the host cores, bounded sample."""
    from oracle import oracle as O
    threads = threads or os.cpu_count() or 1
    dt = np.complex64 if real == "f32" else np.complex128
    # probe one transform per thread, then size the sample for ~seconds_target of CPU work
    x = O.fill_input(threads, n, dt)
    _, sec = O.transform_batch(x, O.FFT, threads, timing=True)
    per_thread = max(1, min(int(seconds_target / max(sec, 1e-6)), max(1, (1 << 31) // (n * threads))))
    batch = per_thread * threads
    x = O.fill_input(batch, n, dt)
    _, sec = O.transform_batch(x, O.FFT, threads, timing=True)
    return {"value": batch * n / sec, "unit": "complex samples/s", "cores": threads, "kind": "port",
            "build": O.timing_build(),
            "sample": f"{batch} transforms of N={n} ({real}), {per_thread} per thread, out-of-place forward, "
                      f"{sec:.2f} s; oracle/ = C restatement of the reference algorithm (rustc absent)"}


def workload_config(desc, n, batch, world, real):
    """The `config` of a batched workload: identical in the CUDA arm and in the --impl reference arm (the driver
    compares them); what is specific to an implementation goes into its own keys (`plan`, `cpu_baseline`)."""
    bps = 16 if real == "f32" else 32
    return {"workload": desc, "N": n, "batch_per_gpu": batch, "transform": "Fft (forward, out of place)",
            "l2": "inputs larger than L2 (no flush needed)" if batch * n * bps // 2 > (256 << 20)
            else "inputs smaller than L2: numbers are L2-warm",
            "parallelism": f"batch-sharded x{world}, no collective"}


def run_reference(args, n, batch, real, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port), host cores."""
    if rank != 0:
        return
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    dt = np.complex64 if real == "f32" else np.complex128
    x = O.fill_input(threads, n, dt)
    _, sec = O.transform_batch(x, O.FFT, threads, timing=True)
    # each step: bounded sample so that steps+warmup finish within a few minutes
    budget = 120.0 / max(1, args.steps + args.warmup)
    per_thread = max(1, min(int(budget / max(sec, 1e-6)), max(1, (1 << 27) // (n * threads))))
    sample = per_thread * threads
    x = O.fill_input(sample, n, dt)
    for _ in range(args.warmup):
        O.transform_batch(x, O.FFT, threads, timing=True)
    total = 0.0
    for _ in range(args.steps):
        y, s = O.transform_batch(x, O.FFT, threads, timing=True)
        total += s
    dumped = None
    if args.dump_outputs:
        import torch
        dumped = dump_outputs(args.dump_outputs, torch.from_numpy(y))
    value = sample * n * args.steps / total
    base = {"value": value, "unit": "complex samples/s", "cores": threads, "kind": "port", "build": O.timing_build(),
            "sample": f"{sample} transforms of N={n} per step ({per_thread} per thread)"}
    print(json.dumps({
        "impl": "reference", "metric": "batched 1D FFT complex-samples/sec", "value": value,
        "unit": "complex samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": real, "data": "synthetic",
        "config": workload_config(WORKLOADS[args.workload][3], n, batch, world, real),
        "note": "reference CPU algorithm (oracle port: rustc/cargo absent from the image), all host threads, bounded "
                "sample of the workload per step",
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "complex samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        **({"dump": dumped} if dumped else {}),
    }))


def nvml_handle(local_rank):
    """NVML handle of the CUDA device `local_rank` (by PCI bus id: NVML ignores CUDA_VISIBLE_DEVICES)."""
    import pynvml
    import torch
    pynvml.nvmlInit()
    pr = torch.cuda.get_device_properties(local_rank)
    try:
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        return pynvml, pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
    except Exception:
        return pynvml, pynvml.nvmlDeviceGetHandleByIndex(local_rank)


def numa_bind(local_rank):
    """Pins this process to the CPUs next to its GPU (NVML's ideal affinity = the GPU's NUMA node) so that the
    pinned staging buffers it allocates afterwards are first-touched on that node and the copy threads run
    there.  Returns (previous affinity, description); a no-op description when NVML cannot tell."""
    prev = os.sched_getaffinity(0)
    try:
        nv, h = nvml_handle(local_rank)
        words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1} & prev
        if not cpus:
            return prev, "NVML reported no usable CPU affinity: not bound"
        os.sched_setaffinity(0, cpus)
        return prev, f"bound to the {len(cpus)} CPUs NVML lists as local to the GPU ({min(cpus)}..{max(cpus)})"
    except Exception as e:  # no NVML, or a container without the call
        return prev, f"not bound ({type(e).__name__})"


DUMP_BYTES = 48 << 20   # sample budget of --dump-outputs: with the .npy headers the files stay below 64 MB in all


def dump_outputs(out_dir, rows):
    """Writes the complex tensor `rows` ([count, length], device or host) to out_dir: output.npy, float32 or float64
    [k, length, 2] (real, imaginary), and output_rows.npy, float64 [k], the index of each row written.  All rows
    when they fit DUMP_BYTES, else k rows drawn with a fixed seed, in ascending order.  Returns the JSON record."""
    import torch
    count, length = rows.shape
    k = max(1, min(count, DUMP_BYTES // (length * rows.element_size())))
    idx = np.arange(count) if k == count else np.sort(np.random.default_rng(0).choice(count, k, replace=False))
    sample = torch.view_as_real(rows[torch.from_numpy(idx).to(rows.device)]).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output.npy"), sample)
    np.save(os.path.join(out_dir, "output_rows.npy"), idx.astype(np.float64))
    return {"dir": out_dir, "files": ["output.npy", "output_rows.npy"], "rows": k, "of_rows": count,
            "row_length": length, "dtype": str(sample.dtype)}


def run_distributed(args, rank, local_rank, world, barrier, log2n=None, steps=None, dump_dir=None):
    """BASELINE configs[4]: ONE transform of N = 2^30 (or 2^--log2n) samples block-distributed over the ranks.
    Returns the record (rank 0) or None."""
    import torch
    import torch.distributed as dist
    import fourier_b200 as fb
    from fourier_b200.distributed import CudaBackend, DistributedFft
    k = log2n or args.log2n
    steps = steps or args.steps
    # N = n1 * n2: rows of length n2 = 2^16 run on the persistent two-pass kernel (0.60 ms per batch of N/P samples on
    # 8 GPUs, against 0.87 ms for 2^15-point rows on the two-launch tile kernels: profiles/r02_c5_sweep_8gpu.json)
    k2 = 16 if k >= 26 else k - k // 2
    n1, n2 = 1 << (k - k2), 1 << k2
    n = n1 * n2
    blk = n // world
    be = CudaBackend("f32")
    plan = DistributedFft(n1, n2, rank, world, be, exchange=args.exchange, chunks=args.chunks or None)
    x, s = plan.buffers()
    fb.fill_input(x.view(1, blk), first_transform=rank)
    cur, oth = x, s
    natural = not args.transposed_output
    for _ in range(args.warmup):
        out = plan.transform(cur, oth, natural_order=natural)
        cur, oth = (out, oth if out is cur else cur)
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        start.record()
        for _ in range(steps):
            out = plan.transform(cur, oth, natural_order=natural)
            cur, oth = (out, oth if out is cur else cur)
        stop.record()
        barrier()
    # rank 0's block of the last step's result, in rows of n2 samples
    dumped = dump_outputs(dump_dir, cur.view(-1, n2)) if dump_dir and rank == 0 else None
    ms = torch.tensor([start.elapsed_time(stop)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    n_exchanges = 3 if natural else 2
    wire = plan.wire_bytes_per_exchange(8) * n_exchanges
    be.launches = 0          # one more, untimed transform to count this library's kernel launches per step
    out = plan.transform(cur, oth, natural_order=natural)
    launches_per_step, be.launches = be.launches, None
    exchange, chunks, fused = plan.exchange, plan.chunks, plan.fused
    plan.close()
    del x, s, cur, oth, out
    if rank != 0:
        return None
    ms_per_step = float(ms.item()) / steps
    peak, peak_src = measured_peak()
    # per GPU and step, read + write each: 2 FFT batches and 3 exchanges (one sweep each over NVLink peer memory;
    # pack + all_to_all + unpack = 3 sweeps with NCCL)
    # fused: the exchanges that follow row FFTs ride on the FFTs' stores -- exchange 1, then 2 (FFT + exchange)
    # sweeps, or FFT + exchange and a plain FFT for transposed output
    sweeps = 3 if fused else 2 + n_exchanges * (1 if exchange == "peer" else 3)
    local_bytes = blk * 8 * 2 * sweeps
    achieved = local_bytes / (ms_per_step * 1e-3) / 1e9
    return {
        "metric": "distributed 1D FFT complex-samples/sec (one N=2^%d transform)" % k, "value": n / (ms_per_step * 1e-3),
        "unit": "complex samples/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS["c5"][3], "N": n, "n1": n1, "n2": n2,
                   "parallelism": (f"block-distributed over {world} ranks, {n_exchanges} exchanges over NVLink peer memory (CUDA IPC), "
                                   f"{n_exchanges - 1} of them folded into the last register stage of the row FFTs that precede "
                                   "them (the FFT kernel stores straight into the peers' buffers), the first one a "
                                   "transposing kernel; stream-ordered barriers between the steps"
                                   if fused else
                                   f"block-distributed over {world} ranks, {n_exchanges} exchanges, each ONE transposing kernel storing "
                                   "into the peers' buffers over NVLink (CUDA IPC) + a stream-ordered barrier"
                                   + (f"; the exchange of a row block overlaps the FFTs of the next ({chunks} blocks)"
                                      if chunks > 1 else "")
                                   if exchange == "peer" else
                                   f"block-distributed over {world} ranks, {n_exchanges} NCCL all-to-all transposes, each "
                                   f"pipelined in {chunks} pieces"),
                   "output": "natural order" if natural else "transposed (Y[k1][k2] = X[k1 + n1*k2], last exchange skipped)",
                   "note": "successive steps transform the previous result (ping-pong buffers)"},
        "nvlink": {"bytes_sent_per_gpu_per_step": wire,
                   "achieved_gbs_per_gpu_per_direction_if_exchanges_were_the_whole_step": wire / (ms_per_step * 1e-3) / 1e9,
                   "reference_gbs": 770, "reference": "measured peer copy per direction (B200_PROFILING.md)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "peak_source": peak_src,
                     "note": f"local sweeps only: {sweeps} read+write sweeps of the rank's block per step"},
        "gpu_launches": launches_per_step * steps, "clocks": clocks.summary(),
        **({"dump": dumped} if dumped else {}),
    }


# nominal f32 FMA peak of one B200: 148 SMs x 128 lanes x 2 flop x 1.965 GHz; the packed FFMA2 rate measured by
# tools/ubench.cu (profiles/r01_ubench_fp_pipes.txt) is 113.4 of those 128 lanes per clock and SM
FP32_PEAK_TFLOPS_NOMINAL = 148 * 128 * 2 * 1.965e9 / 1e12
FP32_PEAK_TFLOPS_MEASURED = 148 * 113.4 * 2 * 1.965e9 / 1e12
C4_FLOP_PER_SAMPLE = 230.0   # SURVEY.md 8(d) / BASELINE.md: two 2048-point FFTs + 3 pointwise passes per 1009 samples


def run_batched(args, workload, batch, rank, local_rank, world, barrier, steps, scaling, keep_output=False):
    """One batched workload on every rank (each its own shard of the global synthetic batch, no collective).
    Returns (record or None on rank != 0, plan, x, y) -- the buffers only when keep_output."""
    import torch
    import torch.distributed as dist
    import fourier_b200 as fb
    n, _, real, desc = WORKLOADS[workload]
    cdt = torch.complex64 if real == "f32" else torch.complex128
    plan = fb.create_fft_f32(n) if real == "f32" else fb.create_fft_f64(n)
    info = plan.info()
    # this rank's shard: transforms [rank*batch, (rank+1)*batch) of the global synthetic batch
    x = torch.empty((batch, n), dtype=cdt, device="cuda")
    y = torch.empty_like(x)
    fb.fill_input(x, first_transform=rank * batch)
    torch.cuda.synchronize()
    for _ in range(args.warmup):
        plan.transform(x, y, fb.Transform.Fft)
    barrier()
    launches_per_step = plan.info()["last_launches"]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        start.record()
        for _ in range(steps):
            plan.transform(x, y, fb.Transform.Fft)
        stop.record()
        barrier()
    ms = torch.tensor([start.elapsed_time(stop)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    ms_per_step = ms_total / steps
    value = world * batch * n * steps / (ms_total * 1e-3)

    rec = None
    if rank == 0:
        # parity spot-check of the timed output against the oracle (identical hash-generated input)
        verify = {}
        if args.verify > 0:
            from oracle import oracle as O
            dt = np.complex64 if real == "f32" else np.complex128
            picks = sorted({0, 1 % batch, batch // 2, batch - 1})[: args.verify]
            worst = 0.0
            for b in picks:
                want = O.transform(O.fill_input(1, n, dt, first_transform=b)[0], O.FFT)
                got = y[b].cpu().numpy()
                worst = max(worst, float(np.abs(got - want).max() / np.abs(want).max()))
            verify = {"transforms_checked": picks, "max_rel_err_vs_oracle": worst,
                      "tolerance": 1e-5 if real == "f32" else 1e-12}
        peak, peak_src = measured_peak()
        bps = BYTES_PER_SAMPLE[real]
        achieved = batch * n * bps / (ms_per_step * 1e-3) / 1e9  # per GPU
        tr = measured_traffic(workload)
        one_kernel = int(launches_per_step) == 1
        rec = {
            "metric": "batched 1D FFT complex-samples/sec", "value": value, "unit": "complex samples/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": real, "data": "synthetic",
            "config": workload_config(desc, n, batch, world, real),
            "plan": {"path": info["path_name"], "inner_path": info["inner_path_name"]},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (tr["dram_bytes_per_sample"] * batch * n) if tr else None,
                         "traffic_source": tr["source"] if tr else None,
                         "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                         "algorithmic_bytes_per_sample": bps,
                         "algorithmic_bytes_per_launch": batch * n * bps,
                         "kernel": (plan.kernel_name() + " -- one launch = one step (whole batch)") if one_kernel
                         else f"whole step ({int(launches_per_step)} launches; dominant kernel {plan.kernel_name()})",
                         "launch_ms": ms_per_step},
            "gpu_launches": int(launches_per_step) * steps,
            "clocks": clocks.summary(),
            "verify": verify,
        }
        if workload == "c4":
            # above the f32 ridge (14 flop/B): report the FMA-pipe fraction next to the HBM fraction
            tf = C4_FLOP_PER_SAMPLE * (value / world) / 1e12
            rec["roofline"].update({
                "hbm_frac": achieved / peak, "flop_per_sample_nominal": C4_FLOP_PER_SAMPLE, "achieved_tflops": tf,
                "fma_frac": tf / FP32_PEAK_TFLOPS_MEASURED, "fma_frac_of_nominal": tf / FP32_PEAK_TFLOPS_NOMINAL,
                "fma_peak_tflops": FP32_PEAK_TFLOPS_MEASURED,
                "fma_peak_source": "packed FFMA2 issue rate measured by tools/ubench.cu (113.4 of 128 lanes/clk/SM)"})
    if keep_output:
        return rec, plan, x, y
    plan.close()
    del x, y
    torch.cuda.empty_cache()
    return rec, None, None, None


def run_e2e(args, plan, x, y, n, real, batch, rank, local_rank, world, barrier):
    """The same metric through the C-ABI call with HOST (pinned) buffers, copies inside the timed region."""
    import torch
    import torch.distributed as dist
    import fourier_b200 as fb
    cdt = torch.complex64 if real == "f32" else torch.complex128
    prev_aff, numa = numa_bind(local_rank)
    eb = args.e2e_batch or max(1, min(batch, (2 << 30) // (n * (8 if real == "f32" else 16))))
    hx = torch.empty((eb, n), dtype=cdt).pin_memory()
    hy = torch.empty((eb, n), dtype=cdt).pin_memory()
    hx.copy_(x[:eb])
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(2):
        plan.transform(hx, hy, fb.Transform.Fft)  # warm-up (allocates staging)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        plan.transform(hx, hy, fb.Transform.Fft)
    barrier()
    dt_s = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt_s, op=dist.ReduceOp.MAX)
    bytes_step = eb * n * (8 if real == "f32" else 16)
    e2e = {"value": world * eb * n * e2e_steps / float(dt_s.item()), "unit": "complex samples/s",
           "h2d_bytes_per_step": bytes_step, "d2h_bytes_per_step": bytes_step,
           "batch_per_step": eb, "steps": e2e_steps, "host_numa": numa,
           "pcie_gbs_each_way_per_gpu": bytes_step * e2e_steps / float(dt_s.item()) / 1e9,
           "note": "fourier_b200_transform_batch_* on pinned host buffers: chunked H2D -> FFT -> D2H pipeline"}
    if rank == 0 and args.verify > 0:
        e2e["matches_device_path"] = bool(torch.equal(hy[:1], y[:1].cpu()))
    os.sched_setaffinity(0, prev_aff)
    return e2e


def run_latency(sizes=(256, 1024, 3125), reps=200):
    """Single-transform latency through the LEGACY 8-symbol ABI (fourier_transform_float on host buffers), the
    only thing the reference itself benchmarks (fourier-bench/benches/fft_bench.rs:18-37: one out-of-place
    fft.transform of 256..3125 points), next to one oracle call on one host core."""
    import fourier_b200 as fb
    from oracle import oracle as O
    out = []
    for n in sizes:
        plan = fb.create_fft_f32(n)
        x = O.fill_input(1, n, np.complex64)[0]
        y = np.empty_like(x)
        for _ in range(20):
            plan.c_transform(x, y, fb.Transform.Fft)
        t0 = time.perf_counter()
        for _ in range(reps):
            plan.c_transform(x, y, fb.Transform.Fft)
        gpu_us = (time.perf_counter() - t0) / reps * 1e6
        op = O.Plan(n, np.complex64)
        want = op.transform(x)
        t0 = time.perf_counter()
        for _ in range(reps):
            op.transform(x)
        cpu_us = (time.perf_counter() - t0) / reps * 1e6
        err = float(np.abs(y - want).max() / np.abs(want).max())
        out.append({"N": n, "path": plan.info()["path_name"], "gpu_us_per_call": gpu_us, "cpu_oracle_us_per_call": cpu_us,
                    "rel_err": err})
        plan.close()
        op.close()
    return {"what": "one fourier_transform_float call on host buffers (ctypes call overhead included on both "
                    "sides); cpu = oracle port on one core (plain -O2 build)", "calls_timed": reps, "sizes": out,
            "note": "a single small transform is latency-bound (two PCIe copies + one launch): the CPU path wins "
                    "here; the GPU library is for batches"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch")
    ap.add_argument("--e2e-batch", type=int, default=0, help="transforms per e2e step (host buffers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--also", default=None,
                    help="comma list of the other BASELINE configs appended to the JSON line as `also` "
                         "(c3,c4,c5,latency; 'none'); default: all that apply to this GPU count when the "
                         "workload is the default c2 at its full batch")
    ap.add_argument("--verify", type=int, default=4, help="transforms checked against the oracle")
    ap.add_argument("--log2n", type=int, default=30, help="c5 only: log2 of the distributed transform length")
    ap.add_argument("--transposed-output", action="store_true",
                    help="c5 only: leave the result transposed (2 exchanges instead of 3)")
    ap.add_argument("--chunks", type=int, default=0, help="c5 only: row blocks per pipelined exchange (0 = plan default)")
    ap.add_argument("--exchange", default="fused", choices=["fused", "peer", "nccl"],
                    help="c5 only: exchanges folded into the row FFTs' stores over NVLink peer memory, as one kernel "
                         "each over peer memory, or pack + NCCL all_to_all + unpack")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's output (rank 0; a fixed, seeded sample of its rows when larger "
                         "than 48 MB) to DIR/output.npy, the indices of those rows to DIR/output_rows.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n, batch, real, desc = WORKLOADS[args.workload]
    default_run = args.workload == "c2" and not args.batch
    if args.batch:
        batch = args.batch

    if args.impl == "reference":
        run_reference(args, n, batch, real, rank, world)
        return

    import torch
    import torch.distributed as dist
    import fourier_b200 as fb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    fb.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.workload == "c5":
        rec = run_distributed(args, rank, local_rank, world, barrier, dump_dir=args.dump_outputs)
        if rank == 0:
            print(json.dumps(rec))
        if world > 1:
            dist.destroy_process_group()
        return

    if args.workload == "c3" and not args.batch:
        batch = max(1, batch // world)   # BASELINE configs[2]: the batch of 65536 is sharded over the GPUs
    out, plan, x, y = run_batched(args, args.workload, batch, rank, local_rank, world, barrier, args.steps,
                                  "strong" if args.workload == "c3" else "weak", keep_output=True)
    if args.dump_outputs and rank == 0:
        out["dump"] = dump_outputs(args.dump_outputs, y)
    e2e = None if args.no_e2e else run_e2e(args, plan, x, y, n, real, batch, rank, local_rank, world, barrier)
    plan.close()
    del x, y
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, appended to the same JSON line ------------------------------------------------
    if args.also is None:
        wanted = ["c3", "c4", "c5", "latency"] if default_run else []
    else:
        wanted = [w for w in args.also.split(",") if w and w != "none"]
    also = []
    sub_steps = max(3, min(args.steps, 10))
    for w in wanted:
        rec = None
        if w == "c3":       # configs[2]: batch 65536 sharded over the GPUs (strong scaling)
            rec, _, _, _ = run_batched(args, "c3", max(1, WORKLOADS["c3"][1] // world), rank, local_rank, world, barrier,
                                       sub_steps, "strong")
        elif w == "c4" and world == 1:   # configs[3]: 1 x B200
            rec, _, _, _ = run_batched(args, "c4", WORKLOADS["c4"][1], rank, local_rank, world, barrier, sub_steps, "weak")
        elif w == "c5" and world >= 2:   # configs[4]: one N = 2^30 transform over all ranks
            rec = run_distributed(args, rank, local_rank, world, barrier, log2n=30, steps=sub_steps)
        elif w == "latency" and world == 1 and rank == 0:
            rec = {"config": {"workload": WORKLOADS["c1"][3] + " + the reference's own bench sizes"},
                   "latency": run_latency()}
        if rec is not None and rank == 0:
            rec["name"] = w
            also.append(rec)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    if e2e:
        out["e2e"] = e2e
    if also:
        out["also"] = also
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(n, real)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
