#!/usr/bin/env python
"""bench.py -- headline benchmark: 256-channel fir_decimate_cc bank (decim 10, 199-tap HAMMING), BASELINE config 2,
plus one leg per other BASELINE config (3: fastddc, 4: fused NFM bank, 5: overlap-add bank) in `extra`.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch: 256 channels x 2.4 M cf32 samples per GPU (1 s of a
2.4 Msps stream per channel).  Multi-GPU: a 256*N-channel bank, one contiguous 256-channel slice per device,
no data-path collective (independent inputs, SURVEY 8(e)) -> weak scaling.

Prints ONE JSON line (rank 0):
  value      whole-job Msamples/s of complex input, inputs resident in HBM, device-timed (CUDA events), max over ranks;
             the K timed steps follow a >= 0.7 s pre-heat of the same kernel, so they run at the power-capped clock the
             `clocks` record shows; `sustained` repeats the measurement over >= 1 s
  e2e        same metric through the host-buffer C-ABI call (csdrb_fir_decimate_bank_cc_host): pinned host input,
             H2D + kernel + D2H of the outputs inside the timed region, every step;  e2e_u8: the same bank fed with
             rtl_sdr-style u8 IQ (csdrb_fir_decimate_bank_u8_host, conversion fused into the FIR kernel)
  roofline   algorithmic bytes (8 B/sample in + 8 B/output) / measured kernel time vs MEASURED_PEAKS.json hbm_gbs
  extra      configs 3, 4, 5 (and the strong-scaling split of config 2 at N > 1): value, kernel_ms, roofline, clocks per leg,
             timed with CUDA events around the C-ABI calls over >= 1 s each.  Config 4 at N > 1 moves the wideband block from
             rank 0 to every rank with an NCCL broadcast per step (double-buffered against the previous block's kernel)
  cpu_baseline  the compiled reference (oracle/_ref) or the oracle port on this box's host cores, bounded sample
--impl reference: the reference's own CPU implementation of the same step on all host threads (rank 0 only).

--dump-outputs DIR (rank 0): after the K timed steps, what the last step handed its caller, for comparing two builds output for output
(the inputs are seeded, so they are the same in every run):
  fir_bank_out.npy       float32 (256, 16384, 2): I,Q of every channel at DUMP_COLS fixed output positions (all 239 981 would be 491 MB)
  fir_bank_out_cols.npy  float64 (16384,): those positions -- the first and last 1024 outputs and a seeded sample in between
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CHANNELS, N_IN, TAPS, DECIM = 256, 2_400_000, 199, 10
WORKLOAD = "256-channel fir_decimate_cc bank, decim=10, 199-tap HAMMING, 2.4 Msps/ch synthetic cf32 (BASELINE configs[1])"
METRIC = "Msamples/s in, 256-ch fir_decimate_cc d=10"
ALGO_BYTES_PER_SAMPLE = 8.0 + 8.0 / DECIM            # SURVEY 8(d): 8 B read per input sample + 8 B written per output
DUMP_COLS, DUMP_EDGE = 16384, 1024


def dump_columns(n_out: int) -> np.ndarray:
    """output positions --dump-outputs keeps: both ends of the stream (filter start-up and the last complete window) and a seeded sample between"""
    mid = np.random.default_rng(0).choice(np.arange(DUMP_EDGE, n_out - DUMP_EDGE), DUMP_COLS - 2 * DUMP_EDGE, replace=False)
    return np.sort(np.concatenate([np.arange(DUMP_EDGE), mid, np.arange(n_out - DUMP_EDGE, n_out)]))


def dump_outputs(out_dir: str, arrays: dict) -> None:
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(d / f"{name}.npy", a)


def base_config(world: int) -> dict:
    """the `config` object of BOTH arms (the driver compares the key sets)"""
    return {"workload": WORKLOAD, "channels_per_gpu": CHANNELS, "samples_per_channel": N_IN, "taps": TAPS, "decimation": DECIM,
            "parallelism": f"channel slices, {CHANNELS} per GPU x {world} GPUs, no collective",
            "l2": "inputs (4.9 GB per GPU) exceed the 126 MB L2; no flush needed", "timing": "CUDA events on the launch stream, max over ranks"}


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


FP32_PEAK_TFLOPS = 72.0      # 148 SMs x 128 lanes x 2 flop x 1.9 GHz: context for the FP32-bound legs (tools/bin/microbench measured 71 with FFMA)


def ncu_traffic():
    for name in ("r02_fir_bank_ncu_summary.json", "fir_bank_ncu_summary.json"):
        p = ROOT / "profiles" / name
        if p.exists():
            try:
                return json.loads(p.read_text()).get("dram_bytes_per_launch"), f"ncu --set full capture, profiles/{name} (static: not re-measured in this run)"
            except Exception:
                pass
    return None, None


# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, pw, reasons = [], 0, [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm          # samples taken under load (power), not the idle edges
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw)}


def physical_gpu_index(local: int) -> int:
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    parts = [p for p in cvd.split(",") if p.strip()]
    if parts and local < len(parts) and parts[local].strip().isdigit():
        return int(parts[local])
    return local


# ----------------------------------------------------------------------------------------------------
def cpu_reference_runner():
    """(callable, kind): fir_decimate_cc of the compiled reference if oracle/_ref is there, else the oracle port."""
    from oracle import pyoracle
    if pyoracle.have_ref():
        L = C.CDLL(str(pyoracle.REF_SO)); fn = L.fir_decimate_cc; kind = "reference"
    else:
        pyoracle.build(ref=False)
        L = C.CDLL(str(pyoracle.ORACLE_SO)); fn = L.oracle_fir_decimate_cc; kind = "port"
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
    fn.restype = C.c_int
    return fn, kind


def cpu_fir_threads(fn, taps, n_threads, channels_per_thread, reps=1):
    """Every thread filters `channels_per_thread` synthetic channels of N_IN samples; returns (seconds, samples)."""
    rng = np.random.default_rng(0)
    x = (rng.uniform(-1, 1, 2 * N_IN).astype(np.float32))          # one shared read-only input (interleaved I,Q)
    outs = [np.empty(2 * (N_IN // DECIM + 1), np.float32) for _ in range(n_threads)]
    start = threading.Barrier(n_threads + 1)

    def work(k):
        start.wait()
        for _ in range(channels_per_thread * reps):
            fn(x.ctypes.data, outs[k].ctypes.data, N_IN, DECIM, taps.ctypes.data, TAPS)

    th = [threading.Thread(target=work, args=(k,)) for k in range(n_threads)]
    [t.start() for t in th]
    start.wait(); t0 = time.perf_counter()
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    return dt, n_threads * channels_per_thread * reps * N_IN


def host_taps():
    """Taps for the CPU arms, designed by the CPU library itself (no GPU library needed)."""
    from oracle import pyoracle
    o = pyoracle.Ref() if pyoracle.have_ref() else pyoracle.Oracle()
    return np.ascontiguousarray(o.firdes_lowpass_f(TAPS, 0.5 / DECIM, "HAMMING"), np.float32)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fn, kind = cpu_reference_runner()
    taps = host_taps()
    cores = os.cpu_count() or 1
    for _ in range(max(args.warmup, 1)):
        cpu_fir_threads(fn, taps, cores, 1)
    times, samples = [], 0
    for _ in range(args.steps):
        dt, s = cpu_fir_threads(fn, taps, cores, 1)
        times.append(dt); samples += s
    total = sum(times)
    value = samples / total / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(max(args.gpus, 1)),
            "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": kind,
                             "sample": f"{args.steps} steps x {cores} channels x {N_IN} samples of the workload (one channel per host thread; a bounded sample of the "
                                       f"{CHANNELS}-channel bank), reference fir_decimate_cc, {cores} threads"},
            "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import csdr_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = csdr_b200.lib()
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    cur_stream = lambda: torch.cuda.current_stream().cuda_stream
    peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def check(rc, what):
        if rc < 0:
            raise SystemExit(f"bench.py: {what} failed: {L.csdrb_last_error().decode()}")
        return rc

    def timed_loop(step, steps):
        """`steps` calls bracketed by barrier + synchronize; (total ms, mean per-call ms), both max over ranks"""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record()
        for k in range(steps):
            step(k)
            ev[k + 1].record()
        barrier()
        total = max_over_ranks(ev[0].elapsed_time(ev[steps]))
        per = max_over_ranks(float(np.mean([ev[k].elapsed_time(ev[k + 1]) for k in range(steps)])))
        return total, per

    def sustained(step, min_seconds=1.0, probe=3, cap=4000):
        """run `step` back to back for >= min_seconds; ms per call over that stretch (max over ranks)"""
        _, per = timed_loop(step, probe)
        n = int(min(cap, max(probe, np.ceil(min_seconds * 1e3 / max(per, 1e-3)))))
        if world > 1:                                              # every rank must run the same number of collective steps
            t = torch.tensor([n], dtype=torch.int64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); n = int(t.item())
        total, _ = timed_loop(step, n)
        return total / n, n

    def leg(name, step, warm, units_per_step, algo_bytes_per_step, flops_per_step, bound, note, config, total_units_factor=1):
        """one `extra` entry: warm-up, then >= 1 s of back-to-back steps under the clock sampler"""
        for k in range(max(warm, 3)):
            step(k)
        l0 = csdr_b200.kernel_launches()
        with ClockSampler(physical_gpu_index(local)) as clk:
            ms, n = sustained(step)
        launches = (csdr_b200.kernel_launches() - l0)
        gbs = algo_bytes_per_step / (ms * 1e-3) / 1e9
        tf = flops_per_step / (ms * 1e-3) / 1e12
        roof = {"bound": bound, "unit": "GB/s" if bound == "hbm" else "TFLOP/s"}
        if bound == "hbm":
            roof.update(achieved=gbs, peak=peak, frac=gbs / peak, fp32_tflops=tf, peak_source=peak_src)
        else:
            roof.update(achieved=tf, peak=FP32_PEAK_TFLOPS, frac=tf / FP32_PEAK_TFLOPS, algorithmic_gbs=gbs, frac_of_hbm=gbs / peak,
                        peak_source="FP32 FMA peak 148 SMs x 128 lanes x 2 x 1.9 GHz (nominal; no tensor cores on this path)")
        return {"name": name, "value": total_units_factor * units_per_step / ms / 1e3, "unit": "Msamples/s", "kernel_ms": ms, "steps": n,
                "gpu_launches": int(launches), "roofline": roof, "clocks": clk.summary(), "config": config, "note": note}

    extra = []
    taps = csdr_b200.firdes_lowpass_f(TAPS, 0.5 / DECIM, "HAMMING")
    n_out = csdr_b200.fir_out_len(N_IN, DECIM, TAPS)
    ostride = n_out + (n_out & 1)
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    x = torch.rand((CHANNELS, N_IN, 2), generator=g, device=dev, dtype=torch.float32) * 2 - 1      # 4.9 GB >> 126 MB L2
    y = torch.empty((CHANNELS, ostride), dtype=torch.complex64, device=dev)

    # ---- config 2, device-resident leg (the headline) ---------------------------------------------------
    def fir_step(_k, ch=CHANNELS):
        check(L.csdrb_fir_decimate_bank_cc(x.data_ptr(), N_IN, y.data_ptr(), ostride, ch, N_IN, DECIM, fp(taps), TAPS, -1, cur_stream()), "csdrb_fir_decimate_bank_cc")

    for k in range(args.warmup):
        fir_step(k)
    barrier()              # the first collective sets the communicator up (hundreds of ms): do it here, or the timed loop's own barrier lets the GPU cool off after the pre-heat
    with ClockSampler(physical_gpu_index(local)) as clk:
        if not args.quick:
            t_hold = time.perf_counter()                         # pre-heat: the timed steps below run at the clock the GPU settles to under this kernel
            while time.perf_counter() - t_hold < 0.7:
                for k in range(8):
                    fir_step(k)
                torch.cuda.synchronize()
        launches0 = csdr_b200.kernel_launches()
        total_ms, per_kernel_ms = timed_loop(fir_step, args.steps)
        launches = csdr_b200.kernel_launches() - launches0
        if args.dump_outputs and rank == 0:                      # before the sustained run below overwrites y
            cols = dump_columns(n_out)
            dumped = {"fir_bank_out": torch.view_as_real(y[:, torch.from_numpy(cols).to(dev)]).cpu().numpy(), "fir_bank_out_cols": cols.astype(np.float64)}
        sus_ms, sus_n = (per_kernel_ms, args.steps) if args.quick else sustained(fir_step)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dumped)
    samples_per_step = CHANNELS * N_IN
    value = world * samples_per_step * args.steps / total_ms / 1e3                                   # Msamples/s, whole job
    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "value": value, "unit": "Msamples/s", "kernel_ms": per_kernel_ms, "gpu_launches": int(launches)}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    main_clocks = clk.summary()

    # ---- config 2, strong-scaling split (256 / N channels per GPU): SURVEY 8(e)'s partition next to the weak one ----------
    if world > 1 and not args.no_extra:
        chs = max(1, CHANNELS // world)
        e = leg("cfg2_strong", lambda k: fir_step(k, chs), args.warmup, chs * N_IN, chs * (N_IN * 8.0 + n_out * 8.0), chs * n_out * TAPS * 4.0, "hbm",
                "the same 256-channel bank split 256/N per GPU (strong scaling; the headline above is the weak form, 256 per GPU)",
                {"workload": WORKLOAD, "channels_per_gpu": chs, "channels_total": chs * world, "scaling": "strong"}, total_units_factor=world)
        extra.append(e)

    # ---- end-to-end legs: pinned host buffers through the C-ABI host calls ----------------------------------
    hin = csdr_b200.PinnedArray((CHANNELS, N_IN), np.complex64)
    hout = csdr_b200.PinnedArray((CHANNELS, n_out), np.complex64)
    stage = torch.from_numpy(hin.array.view(np.float32).reshape(CHANNELS, N_IN, 2))
    stage.copy_(x)                                                                                     # same synthetic data, now on the host
    del x, y
    torch.cuda.empty_cache()
    e2e_steps = max(2, min(args.steps, 5))

    def e2e_run(call):
        call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            call()
        torch.cuda.synchronize()
        s = max_over_ranks(time.perf_counter() - t0)
        if world > 1:
            dist.barrier(device_ids=[local])
        return world * samples_per_step * e2e_steps / s / 1e6, s

    e2e_value, e2e_s = e2e_run(lambda: csdr_b200.fir_decimate_bank_cc_host(hin.array, DECIM, taps, out=hout.array))
    checksum = float(np.abs(hout.array[:, :: max(1, n_out // 64)]).sum())                            # the step's result is read on the host
    hin.close()
    hu8 = csdr_b200.PinnedArray((CHANNELS, N_IN, 2), np.uint8)
    rng = np.random.default_rng(rank)
    hu8.array[:] = rng.integers(0, 256, (1, N_IN, 2), dtype=np.uint8)                                  # rtl_sdr-style bytes (same row in every channel: content does not matter here)
    e2e_u8_value, _ = e2e_run(lambda: csdr_b200.fir_decimate_bank_u8_host(hu8.array, DECIM, taps, out=hout.array))
    checksum_u8 = float(np.abs(hout.array[:, :: max(1, n_out // 64)]).sum())
    hu8.close(); hout.close()

    # ---- BASELINE configs 3, 4, 5 ---------------------------------------------------------------------------
    if not args.no_extra:
        extra += other_configs(torch, dist, csdr_b200, L, dev, world, rank, local, leg, check, cur_stream, fp, args, sustained=sustained, barrier=barrier)

    # ---- CPU baseline beside it (rank 0, N=1 only, bounded) --------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fn, kind = cpu_reference_runner()
        cores = os.cpu_count() or 1
        cpu_fir_threads(fn, taps, cores, 1)
        dt, s = 0.0, 0
        reps = 0
        while dt < 8.0 and reps < 64:
            d, n = cpu_fir_threads(fn, taps, cores, 1)
            dt += d; s += n; reps += 1
        cpu = {"value": s / dt / 1e6, "unit": "Msamples/s", "cores": cores, "kind": kind,
               "sample": f"{reps} x {cores} channels x {N_IN} samples of the same workload, fir_decimate_cc of "
                         f"{'oracle/_ref (unmodified reference build)' if kind == 'reference' else 'oracle port'}, {cores} host threads, {dt:.1f} s"}

    if rank == 0:
        algo_bytes = samples_per_step * 8.0 + CHANNELS * n_out * 8.0
        achieved = algo_bytes / (per_kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic()
        line = {"metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": base_config(world),
                "e2e": {"value": e2e_value, "unit": "Msamples/s", "h2d_bytes_per_step": samples_per_step * 8, "d2h_bytes_per_step": CHANNELS * n_out * 8,
                        "steps": e2e_steps, "api": "csdrb_fir_decimate_bank_cc_host (pinned host buffers on the GPU's NUMA node, 3-stream chunked pipeline)",
                        "checksum": checksum, "h2d_gbs_per_rank": samples_per_step * 8 * e2e_steps / e2e_s / 1e9},
                "e2e_u8": {"value": e2e_u8_value, "unit": "Msamples/s", "h2d_bytes_per_step": samples_per_step * 2, "d2h_bytes_per_step": CHANNELS * n_out * 8,
                           "steps": e2e_steps, "api": "csdrb_fir_decimate_bank_u8_host (u8 IQ in, convert_u8_f fused into the FIR kernel; csdr-fm:41)",
                           "checksum": checksum_u8, "vs_cf32_e2e": e2e_u8_value / e2e_value},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": per_kernel_ms,
                             "fp32_tflops": CHANNELS * n_out * TAPS * 4 / (per_kernel_ms * 1e-3) / 1e12,
                             "note": "8.8 algorithmic B/sample at 79.6 flop/sample sits on the FP32/HBM ridge; both are reported"},
                "sustained": {"value": world * samples_per_step / sus_ms / 1e3, "unit": "Msamples/s", "kernel_ms": sus_ms, "steps": sus_n,
                              "frac": algo_bytes / (sus_ms * 1e-3) / 1e9 / peak, "note": ">= 1 s of back-to-back launches right after the timed steps, same clock record"},
                "cpu_baseline": cpu, "clocks": main_clocks, "extra": extra}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def other_configs(torch, dist, cb, L, dev, world, rank, local, leg, check, cur_stream, fp, args, sustained=None, barrier=None):
    """BASELINE configs 3, 4, 5 as `extra` entries.  Shared-input banks (3, 4) move the wideband block with an NCCL broadcast per step at N > 1."""
    out = []
    vp = C.c_void_p

    class Bcast:
        """double-buffered broadcast of a wideband block from rank 0: block k+1 travels on a side stream while block k is processed"""
        def __init__(self, src):
            self.bufs = [src, torch.empty_like(src) if world > 1 else src]
            if world > 1 and rank == 0:
                self.bufs[1].copy_(src)
            self.comm = torch.cuda.Stream() if world > 1 else None
            self.ready = [torch.cuda.Event(), torch.cuda.Event()]
            self.done = [torch.cuda.Event(), torch.cuda.Event()]
            self.k = 0
            if world > 1:
                self._post(0)

        def _post(self, slot):
            self.comm.wait_event(self.done[slot])                 # the kernel that last read this buffer
            with torch.cuda.stream(self.comm):
                dist.broadcast(self.bufs[slot], src=0)
                self.ready[slot].record(self.comm)

        def next(self):
            """the buffer holding this step's block (ordered on the current stream); the following block's broadcast is already in flight"""
            if world == 1:
                return self.bufs[0]
            slot = self.k & 1
            torch.cuda.current_stream().wait_event(self.ready[slot])
            self._post(slot ^ 1)
            self.k += 1
            return self.bufs[slot]

        def release(self, buf):
            if world > 1:
                self.done[0 if buf is self.bufs[0] else 1].record(torch.cuda.current_stream())

    # ---- config 4: 128 channels per GPU of ONE wideband stream: shift | fir_decimate 50 (801 taps) | fmdemod, fused ------------------------
    Cg, N, D, bw = 128, 1 << 21, 50, 0.005
    T = cb.firdes_filter_len(bw)
    taps = cb.firdes_lowpass_f(T, 0.5 / D)
    n_out = cb.fir_out_len(N, D, T)
    gen = torch.Generator(device=dev).manual_seed(4)
    wide = torch.view_as_complex(torch.rand((N, 2), generator=gen, device=dev) * 2 - 1)
    rates_all = np.linspace(-0.45, 0.45, Cg * world).astype(np.float32)
    rates = np.ascontiguousarray(rates_all[rank * Cg:(rank + 1) * Cg])
    bank = cb.DdcBank(rates, D, taps, demod=True, chunk=1024)
    fo = torch.empty((Cg, n_out + (n_out & 1)), dtype=torch.float32, device=dev)
    bc = Bcast(wide)

    def step4(_k):
        w = bc.next()
        check(L.csdrb_ddc_bank_process(bank.h, w.data_ptr(), N, fo.data_ptr(), fo.stride(0), cur_stream()), "csdrb_ddc_bank_process")
        bc.release(w)

    M = (T + D - 1) // D
    out.append(leg("cfg4_nfm_bank", step4, 4, N, N * 8.0 + Cg * n_out * 4.0, Cg * N * (10.0 + 4.0 * M), "fp32",
                   "value = wideband Msamples/s through ALL channels of the job (every GPU sees the whole stream for its own 128 channels); "
                   "flops = (10 + 4*17) per channel-sample (rotation 4, phasor recursion 6, 17 tap FMAs on I and Q)"
                   + ("; the block reaches ranks 1.. by NCCL broadcast from rank 0 each step, overlapped with the previous block's kernel" if world > 1 else ""),
                   {"workload": "1024-ch-class shift+fir_decimate_cc+fmdemod NFM bank, decim=50, 801 taps, 128 ch/GPU (BASELINE configs[3])", "channels_per_gpu": Cg,
                    "channels_total": Cg * world, "block_samples": N, "nco_chunk": 1024, "collective": "ncclBroadcast of the 16 MiB IQ block per step" if world > 1 else "none (1 GPU)",
                    "scaling": "weak"}))
    if world > 1:
        # the overlap in numbers (no nsys in this image): the broadcast alone, the kernel alone (every rank on its own copy of the block), and the leg above
        # where block k+1 travels while block k is processed
        def only_bcast(_k):
            dist.broadcast(bc.bufs[_k & 1], src=0)

        def only_kernel(_k):
            check(L.csdrb_ddc_bank_process(bank.h, bc.bufs[0].data_ptr(), N, fo.data_ptr(), fo.stride(0), cur_stream()), "csdrb_ddc_bank_process")
        torch.cuda.synchronize(); barrier()
        b_ms, _ = sustained(only_bcast, min_seconds=0.3)
        k_ms, _ = sustained(only_kernel, min_seconds=0.3)
        out[-1]["overlap"] = {"broadcast_alone_ms": b_ms, "kernel_alone_ms": k_ms, "step_ms": out[-1]["kernel_ms"], "sum_ms": b_ms + k_ms,
                              "broadcast_gbs": N * 8.0 / (b_ms * 1e-3) / 1e9, "hidden_ms": b_ms + k_ms - out[-1]["kernel_ms"],
                              "note": "hidden_ms = sum - step: how much of the broadcast of block k+1 runs under the kernel of block k (the bank kernel fills every SM in one wave, "
                                      "NCCL's copy kernel gets SMs as CTAs of the bank kernel retire)"}
    torch.cuda.synchronize()
    bank.close()
    del wide, fo, bc
    torch.cuda.empty_cache()

    # ---- config 3: fastddc, 16384-pt forward FFT, 64 channels (64 / N per GPU) of one wideband stream ---------------------------------------
    bw3, dec3, C3 = 0.002, 64, 64
    c3 = max(1, C3 // world)
    ddc = cb.fastddc_init(bw3, dec3, 0.0)
    nblocks = 592                                                          # 4 x 148 SMs: whole waves for the forward FFT (a CTA per block) and for the fold (a CTA per 16 blocks x 16 ch x 64 bins)
    nsamp = nblocks * ddc.input_size
    gen = torch.Generator(device=dev).manual_seed(3)
    xw = torch.view_as_complex(torch.rand((nsamp, 2), generator=gen, device=dev) * 2 - 1)
    shifts_all = list(np.linspace(-0.45, 0.45, c3 * world))
    shifts = shifts_all[rank * c3:(rank + 1) * c3]
    sp, ov = cb.fastddc_fwd_cc(xw, ddc)
    plan3 = cb.FastddcInvPlan(shifts, dec3, bw3, nblocks, device=dev)      # csdrb_fastddc_inv_plan_*: the state chain + phasors of step k+1 are prepared during step k
    o3, counts = plan3.out, plan3.counts
    bc3 = Bcast(xw)

    def step3(_k):
        w = bc3.next()
        check(L.csdrb_fastddc_fwd_cc(w.data_ptr(), sp.data_ptr(), ov.data_ptr(), ddc.fft_size, ddc.input_size, nblocks, cur_stream()), "csdrb_fastddc_fwd_cc")
        bc3.release(w)
        check(L.csdrb_fastddc_inv_plan_run(plan3.h, sp.data_ptr(), plan3.taps_fft.data_ptr(), o3.data_ptr(), o3.stride(0), counts.data_ptr(), cur_stream()),
              "csdrb_fastddc_inv_plan_run")

    per_blk = ddc.post_input_size // ddc.post_decimation
    flops3 = nblocks * (5.0 * ddc.fft_size * 14 + c3 * (8.0 * ddc.fft_size + 5.0 * ddc.fft_inv_size * 9))
    out.append(leg("cfg3_fastddc", step3, 3, nsamp, nsamp * 8.0 + c3 * nblocks * per_blk * 8.0, flops3, "fp32",
                   "forward 16384-pt FFT + inverse bank (csdrb_fastddc_inv_plan_run: fold + IFFT, the post-shift state chain of the next step prepared meanwhile) per step; algorithmic bytes = wideband samples in + channel outputs (SURVEY 8(d): 16 B/sample at 64 ch); "
                   "the dominant kernel is the fold (8*N flop per channel and block, FFMA2 on the FMA pipe), hence the FP32 roofline; flops = 5*N*log2(N) forward + per channel 8*N fold + 5*M*log2(M) inverse",
                   {"workload": "fastddc overlap-save: 16384-pt FFT, 64 output channels from one 61.44 Msps wideband stream (BASELINE configs[2])", "channels_per_gpu": c3,
                    "channels_total": c3 * world, "blocks_per_step": nblocks, "block_samples": ddc.input_size, "fft_size": ddc.fft_size, "fft_inv_size": ddc.fft_inv_size,
                    "collective": "ncclBroadcast of the time-domain block per step; every rank runs the forward FFT for its own channel slice" if world > 1 else "none (1 GPU)",
                    "scaling": "strong" if world > 1 else "n/a", "x_real_time_at_61.44_Msps": None}))
    out[-1]["config"]["x_real_time_at_61.44_Msps"] = out[-1]["value"] / 61.44
    torch.cuda.synchronize()
    plan3.close()
    del xw, sp, o3, bc3
    torch.cuda.empty_cache()

    # ---- config 5: bandpass_fir_fft_cc overlap-add bank, 4096-pt, 512 channels (512 / N per GPU), block-size sweep -------------------------
    T5, NF, isz, ov5 = cb.bandpass_geometry(0.002)
    tf = cb.bandpass_taps_fft(-0.05, 0.05, 0.002)
    C5 = max(1, 512 // world)
    sweep = []
    best = None
    for Lsz in (65536, 262144, 1048576, 4194304):
        nb = Lsz // isz
        n5 = nb * isz
        try:
            x5 = torch.view_as_complex(torch.rand((C5, n5, 2), device=dev) * 2 - 1)
            y5 = torch.empty((C5, n5), dtype=torch.complex64, device=dev)
        except torch.OutOfMemoryError:
            break
        tail = torch.zeros((C5, NF), dtype=torch.complex64, device=dev)

        def step5(_k):
            check(L.csdrb_bandpass_fir_fft_bank_cc(x5.data_ptr(), n5, y5.data_ptr(), n5, C5, NF, isz, nb, tf.data_ptr(), 0, tail.data_ptr(), cur_stream()),
                  "csdrb_bandpass_fir_fft_bank_cc")

        e = leg(f"cfg5_olafir_L{Lsz}", step5, 3, C5 * n5, C5 * n5 * 16.0, C5 * nb * (2 * 5.0 * NF * 12 + 8.0 * NF), "fp32",
                "16 algorithmic B/sample (8 in + 8 out) and ~250 flop/sample (two 4096-point transforms per 2098 new samples): the FP32 roof is the lower one (frac_of_hbm beside it)",
                {"workload": "bandpass_fir_fft_cc overlap-add, 4096-pt, 512 channels (BASELINE configs[4])", "channels_per_gpu": C5, "channels_total": C5 * world,
                 "samples_per_channel": n5, "fft_size": NF, "input_size": isz, "taps": T5, "scaling": "strong" if world > 1 else "n/a"}, total_units_factor=world)
        sweep.append({"block_samples": Lsz, "value": e["value"], "kernel_ms": e["kernel_ms"], "algorithmic_gbs": e["roofline"]["algorithmic_gbs"], "frac_of_hbm": e["roofline"]["frac_of_hbm"], "fp32_tflops": e["roofline"]["achieved"], "frac": e["roofline"]["frac"],
                      "sm_mhz": e["clocks"].get("sm_mhz")})
        best = e
        del x5, y5, tail
        torch.cuda.empty_cache()
    if best is not None:
        best["name"] = "cfg5_olafir_bank"
        best["sweep"] = sweep
        out.append(best)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 3/4/5 legs")
    ap.add_argument("--quick", action="store_true", help="device-resident leg only (for ncu runs): no clock hold loop, no e2e, no CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output (sampled, float32) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's output: it needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
