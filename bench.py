#!/usr/bin/env python
"""
bench.py -- REPET separation throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference on the host cores
    python bench.py --probe-host-link [--gpus N]                    # copy-only ceiling of the host<->device links
    python bench.py --steps K --dump-outputs DIR                    # also write what the last timed step computed

Workload (BASELINE.json configs[1]): `repet.original` on a batch of synthetic 30 s stereo
44.1 kHz clips, 512 clips per GPU (4096 over 8 GPUs; weak scaling, clips are independent, no
collective on the data path).  One "step" = one pass of the whole hot path (STFT, beat
spectrum, period, median model, mask, ISTFT) over the rank's 512 clips.

Printed JSON line (rank 0):
  value     audio-seconds separated per second, all ranks, inputs/outputs resident in HBM,
            timed with CUDA events on the launching stream, max over ranks
  e2e       same metric through the public API (`repet.separate_batch`) with page-locked HOST
            arrays, fp32 in and out: H2D of the inputs and D2H of the results inside the timed region
  e2e_pcm16 the same with int16 PCM (WAV order) on both sides: 2 + 2 bytes per sample over the link
  e2e_numpy_f64  the drop-in call `repet.original(float64 (S, C) ndarray, fs)` clip by clip (pageable NumPy)
  host_link the copy-only ceiling measured in the same run (the e2e bytes, no kernels, both directions at once)
  roofline  the dominant kernel's algorithmic bytes / its event-timed duration vs the measured
            HBM copy bandwidth (MEASURED_PEAKS.json)
  configs   (N = 1) the other BASELINE.json configs on this GPU: cfg1 `original` on the bundled clip, cfg3 `adaptive`
            on 32 ten-minute tracks, cfg4 `sim` on a ten-minute track (with the similarity GEMM's tensor fraction),
            cfg5 `extended` and `simonline` on one hour + streaming latency per 1 s block
  cpu_baseline  the reference algorithm timed on this box's host cores on a bounded sample of the same clips
            (N=1, rank 0 only); its periods are compared with the GPU's on those clips
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "repet-python_b200"))

import numpy as np  # noqa: E402

FS = 44100
CLIP_SECONDS = 30
CLIP_SAMPLES = CLIP_SECONDS * FS  # 1 323 000
CHANNELS = 2
METRIC = "audio-seconds separated/sec (x realtime), repet.original, 30 s stereo 44.1 kHz clips"
UNIT = "audio-s/s"
TUNABLES = dict(
    cutoff_frequency=100, period_range=[1, 10], segment_length=10, segment_step=5, filter_order=5,
    similarity_threshold=0, similarity_distance=1, similarity_number=100, buffer_length=10,
)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--clips-per-gpu", type=int, default=512)
    ap.add_argument("--cpu-sample-clips", type=int, default=0, help="clips of the CPU sample (0 = automatic)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--configs", default="auto", help="'auto' (all of them at N = 1, none at N > 1), 'none', or a comma "
                    "separated subset of cfg1,cfg3,cfg4,cfg5")
    ap.add_argument("--cfg3-tracks", type=int, default=32, help="10-minute tracks of BASELINE configs[2] per GPU")
    ap.add_argument("--probe-host-link", action="store_true", help="copy-only probe: pinned H2D + D2H, no kernels")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not bind the rank to the GPU's NUMA-local CPUs")
    ap.add_argument("--workspace-mb", type=int, default=0, help="per-chunk workspace cap of the library (0 = default)")
    ap.add_argument("--tune", default="", help="comma separated knob=value pairs for repet_set_tuning (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.probe_host_link):
        ap.error("--dump-outputs writes the outputs of the CUDA arm's separation")
    return args


# --------------------------------------------------------------------------------------------
# CPU side: the reference algorithm on the host cores
# --------------------------------------------------------------------------------------------
_CPU_KIND = None  # "reference" (unmodified repet.py through oracle/reference_shim.py) or "port" (oracle/repet_oracle.py)


def _cpu_worker_init():
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["MKL_NUM_THREADS"] = "1"
    sys.path.insert(0, os.path.join(ROOT, "oracle"))


def cpu_kind():
    """The unmodified reference when /root/reference exists (the build container), else the oracle port (the GPU
    box has no /root/reference)."""
    global _CPU_KIND
    if _CPU_KIND is None:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import reference_shim

        _CPU_KIND = "reference" if reference_shim.available() else "port"
    return _CPU_KIND


def _cpu_worker(job):
    index, kind = job
    import warnings

    import repet_synth

    warnings.simplefilter("ignore")
    clip = repet_synth.make_clip(index, CLIP_SAMPLES, CHANNELS, FS)
    x = clip.T.astype(np.float64)
    if kind == "reference":
        import reference_shim

        ref = reference_shim.load()
        seen = []
        inner = ref._periods

        def periods(*a, **k):
            r = inner(*a, **k)
            seen.append(int(r))
            return r

        ref._periods = periods
        try:
            t0 = time.perf_counter()
            ref.original(x, FS)
            dt = time.perf_counter() - t0
        finally:
            ref._periods = inner
        return dt, seen[0]
    import repet_oracle

    t0 = time.perf_counter()
    _, det = repet_oracle.original(x, FS, return_details=True)
    return time.perf_counter() - t0, det["period"]


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_pool_size():
    cores = host_cores()
    try:
        import psutil

        by_memory = int(psutil.virtual_memory().available / (1.5 * (1 << 30)))  # ~1 GB peak per worker
        return max(1, min(cores, by_memory))
    except Exception:
        return max(1, min(cores, 64))


class CpuArm:
    """The reference algorithm on a process pool, one clip per task, BLAS/OpenMP pinned to one thread per worker
    (clip-parallel: the fair analogue of GPU batching, SURVEY.md 8(d))."""

    def __init__(self):
        import multiprocessing

        self.kind = cpu_kind()
        self.workers = cpu_pool_size()
        self.pool = multiprocessing.get_context("fork").Pool(self.workers, initializer=_cpu_worker_init)

    def run(self, first_index, number_clips):
        """Returns (seconds of separation per busy worker, wall seconds, audio seconds, periods)."""
        t0 = time.perf_counter()
        jobs = [(i, self.kind) for i in range(first_index, first_index + number_clips)]
        results = self.pool.map(_cpu_worker, jobs, chunksize=1)
        wall = time.perf_counter() - t0
        # clip synthesis runs inside the workers too: the figure is the sum of the per-clip separation times
        # divided by the workers actually busy
        compute = sum(r[0] for r in results)
        busy = min(self.workers, number_clips)
        return compute / busy, wall, number_clips * CLIP_SECONDS, [r[1] for r in results]

    def describe(self):
        return ("unmodified repet.py (oracle/reference_shim.py)" if self.kind == "reference"
                else "oracle port of repet.original (oracle/repet_oracle.py; /root/reference is absent on this box)")

    def close(self):
        self.pool.close()
        self.pool.join()


def run_reference_arm(args, rank, world):
    """--impl reference: rank 0 alone times the CPU implementation; other ranks exit."""
    if rank != 0:
        return
    arm = CpuArm()
    sample = args.cpu_sample_clips or max(64, 4 * arm.workers)  # BASELINE.md section 3: >= 64 clips
    for w in range(args.warmup):
        arm.run(10_000 + w * arm.workers, arm.workers)
    total_time = 0.0
    total_audio = 0.0
    for k in range(args.steps):
        compute, wall, audio, _ = arm.run(20_000 + k * sample, sample)
        total_time += compute
        total_audio += audio
    arm.close()
    value = total_audio / total_time
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_time / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.workers, "kind": arm.kind,
                         "sample": "%d clips of 30 s per step (the full step is %d clips per GPU), %s, one clip per core"
                                   % (sample, args.clips_per_gpu, arm.describe())},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def config_dict(args):
    return {
        "workload": "BASELINE configs[1]: repet.original, synthetic 30 s stereo 44.1 kHz clips, %d clips per GPU "
                    "(4096 over 8 GPUs), 2048-pt STFT" % args.clips_per_gpu,
        "clips_per_gpu": args.clips_per_gpu, "clip_seconds": CLIP_SECONDS, "channels": CHANNELS,
        "sampling_frequency": FS, "parallelism": "clip-sharded, no collective",
        "l2": "inputs larger than L2 (%.1f GB of audio per step per GPU)" % (args.clips_per_gpu * CHANNELS * CLIP_SAMPLES * 4 / 1e9),
    }


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every few ms DURING the timed region."""

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.samples = []
        self.reasons = set()
        self.running = False
        self.thread = None
        self.max_mhz = None
        self.error = None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # pragma: no cover
            self.error = "nvml unavailable: %r" % (exc,)
            return
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        n = self.nvml
        flags = {
            "hw_slowdown": n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown") else 0x8,
            "hw_thermal_slowdown": 0x40,
            "sw_thermal_slowdown": 0x20,
            "sw_power_cap": 0x4,
        }
        while self.running:
            try:
                self.samples.append(float(n.nvmlDeviceGetClockInfo(self.dev, n.NVML_CLOCK_SM)))
                try:
                    mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.dev)
                except AttributeError:
                    mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev)
                for name, bit in flags.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception as exc:  # pragma: no cover
                self.error = repr(exc)
                break
            time.sleep(0.001)

    def stop(self):
        self.running = False
        if self.thread:
            self.thread.join(timeout=2)
        out = {
            "sm_mhz": float(np.median(self.samples)) if self.samples else None,
            "sm_max_mhz": self.max_mhz,
            "samples": len(self.samples),
            "reasons": sorted(self.reasons),
        }
        if self.error:
            out["error"] = self.error
        return out


# --------------------------------------------------------------------------------------------
# peaks and committed ncu figures
# --------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            data = json.load(f)
        return {"hbm_gbs": float(data["hbm_gbs"]), "bf16_tflops": float(data["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1650.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(kernel, clips_per_launch):
    """dram__bytes_read + dram__bytes_write per launch of `kernel`, scaled from the committed
    ncu --set full capture (profiles/traffic.json holds bytes per clip), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f)[kernel]["dram_bytes_per_clip"] * clips_per_launch
    except Exception:
        return None


def ncu_figure(*keys):
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            node = json.load(f)
        for k in keys:
            node = node[k]
        return node
    except Exception:
        return None


def bind_to_gpu_numa_node(gpu_index):
    """Pin this process (and the pinned host buffers it allocates next: first touch) to the CPUs NVML reports
    as local to the GPU.  With several ranks per box the host-buffer copies otherwise cross the socket
    interconnect.  Best effort: returns a description, or why it was skipped."""
    try:
        import pynvml

        pynvml.nvmlInit()
        handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        after = len(os.sched_getaffinity(0))
        if after == 0:
            raise RuntimeError("empty affinity")
        return "bound to %d of %d cpus (NVML affinity of GPU %d)" % (after, before, gpu_index)
    except Exception as exc:  # not fatal: containers may forbid it
        return "not bound: %r" % (exc,)


# --------------------------------------------------------------------------------------------
# copy-only probe of the host <-> device links
# --------------------------------------------------------------------------------------------
def host_link_probe(torch, device, host_in, host_out, dev_in, dev_out, reps, barrier):
    """Pinned H2D of `host_in` and D2H into `host_out` with NO kernels: each direction alone, then both at once
    on two streams (what the e2e pipeline asks of the link).  Returns seconds per repetition (this rank)."""
    s_up, s_down = torch.cuda.Stream(device), torch.cuda.Stream(device)

    def timed(up, down):
        barrier()
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        for _ in range(reps):
            if up:
                with torch.cuda.stream(s_up):
                    dev_in.copy_(host_in, non_blocking=True)
            if down:
                with torch.cuda.stream(s_down):
                    host_out.copy_(dev_out, non_blocking=True)
        torch.cuda.synchronize(device)
        dt = (time.perf_counter() - t0) / reps
        barrier()
        return dt

    timed(True, True)  # warm-up
    return {"h2d_s": timed(True, False), "d2h_s": timed(False, True), "duplex_s": timed(True, True)}


def run_host_link_probe(args, rank, local_rank, world):
    numa = "disabled" if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    number_bytes = 2 << 30
    host_in = torch.empty(number_bytes, dtype=torch.uint8).pin_memory()
    host_out = torch.empty(number_bytes, dtype=torch.uint8).pin_memory()
    host_in.fill_(1)
    dev_in = torch.empty(number_bytes, dtype=torch.uint8, device=device)
    dev_out = torch.ones(number_bytes, dtype=torch.uint8, device=device)
    t = host_link_probe(torch, device, host_in, host_out, dev_in, dev_out, max(3, args.steps), barrier)
    times = torch.tensor([t["h2d_s"], t["d2h_s"], t["duplex_s"]], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    if rank == 0:
        h2d, d2h, duplex = (float(v) for v in times)
        gb = number_bytes / 1e9
        print(json.dumps({
            "probe": "host_link", "n_gpus": world, "bytes_per_direction_per_rank": number_bytes, "numa": numa,
            "h2d_gbs_per_rank": gb / h2d, "d2h_gbs_per_rank": gb / d2h,
            "duplex_gbs_per_rank_each_way": gb / duplex,
            "aggregate_h2d_gbs": world * gb / h2d, "aggregate_d2h_gbs": world * gb / d2h,
            "aggregate_duplex_gbs_both_ways": 2 * world * gb / duplex,
            "how": "pinned host memory, cudaMemcpyAsync on two streams, no kernels, wall clock between device "
                   "synchronisations, max over ranks",
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------
# the other BASELINE configs (N = 1)
# --------------------------------------------------------------------------------------------
def frames_of(samples):
    return -(-samples // 1024) + 1


def config_algorithmic_bytes(driver, samples):
    """SURVEY.md 8(d) byte model per track (fp32 / complex64 intermediates, each tensor once per kernel that must
    touch it)."""
    T = frames_of(samples)
    audio = samples * CHANNELS * 4
    X = T * CHANNELS * 1025 * 8
    P = T * 1025 * 4
    per_kernel = {"k_stft": audio + X + P, "k_mask_istft": X + audio}
    if driver == "original":
        per_kernel.update({"k_beat": P, "k_model": X})
        total = 2 * audio + 2 * X + 2 * P
    elif driver == "adaptive":
        per_kernel.update({"k_beat": 2 * P, "k_model": X})  # P re-read with 2x overlap
        total = 2 * audio + 2 * X + 3 * P
    elif driver == "extended":
        # `original` on 2x overlapped segments + one audio pass for the cross-fade
        per_kernel = {k: 2 * v for k, v in per_kernel.items()}
        per_kernel.update({"k_beat": 2 * P, "k_model": 2 * X, "k_xfade": 3 * audio})
        total = 2 * (2 * audio + 2 * X + 2 * P) + audio
    else:
        total = None
    return per_kernel, total


def run_configs(args, torch, repet, handle, stream, device, wanted, peaks):
    """Device-resident throughput of BASELINE configs 1, 3, 4, 5 on this GPU, each with its per-kernel times
    (CUDA events, repet_set_profiling) and roofline fractions."""
    import repet_synth

    out = {}
    tun = TUNABLES
    hbm = peaks["hbm_gbs"]

    def measure(driver, audio_host, steps):
        B, C, S = audio_host.shape
        params, _ = repet._host.derive_params(FS, tun, driver)
        handle.ensure_window(params.window_length)
        audio = torch.from_numpy(audio_host).to(device)
        background = torch.empty_like(audio)
        fn = getattr(handle.lib, "repet_%s_batch_dev" % driver)

        def step():
            handle.check(fn(handle.h, ctypes.c_void_p(audio.data_ptr()), B, C, S, ctypes.byref(params),
                            ctypes.c_void_p(background.data_ptr()), None, None))

        for _ in range(3):
            step()
        torch.cuda.synchronize(device)
        handle.profile_read(reset=True)
        handle.set_profiling(True)
        launches = handle.launch_count()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(steps):
            step()
        end.record(stream)
        torch.cuda.synchronize(device)
        ms = start.elapsed_time(end) / steps
        prof = handle.profile_read(reset=True)
        handle.set_profiling(False)
        launches = handle.launch_count() - launches
        per_kernel, total = config_algorithmic_bytes(driver, S)
        kernels = {}
        for name, (t_ms, count) in prof.items():
            entry = {"ms_per_step": t_ms / steps, "share_of_step": t_ms / steps / ms}
            if name in per_kernel and t_ms > 0:
                entry["achieved_gbs"] = per_kernel[name] * B / (t_ms / steps / 1e3) / 1e9
                entry["frac_of_hbm_peak"] = entry["achieved_gbs"] / hbm
            kernels[name] = entry
        line = {"driver": driver, "tracks": B, "seconds_each": S / FS, "steps": steps, "ms_per_step": ms,
                "x_realtime": B * S / FS / (ms / 1e3), "gpu_launches_per_step": launches // steps, "kernels": kernels}
        if total:
            line["whole_path_algorithmic_gbs"] = total * B / (ms / 1e3) / 1e9
            line["whole_path_frac_of_hbm_peak"] = line["whole_path_algorithmic_gbs"] / hbm
        del audio, background
        torch.cuda.empty_cache()
        return line, prof

    if "cfg1" in wanted:
        # BASELINE configs[0]: the reference's bundled 23 s stereo clip (int16 PCM committed under tests/golden/)
        data = np.load(os.path.join(ROOT, "tests", "golden", "audio_file_int16.npz"))
        pcm = data["pcm"]
        x = pcm / pow(2, pcm.itemsize * 8 - 1)  # repet.wavread (repet.py:929)
        planar = np.ascontiguousarray(x.T[None].astype(np.float32))
        line, _ = measure("original", planar, 20)
        handle.set_stream(None)
        repet._host.original_f64(x, FS, tun, handle=handle)
        t0 = time.perf_counter()
        reps = 10
        for _ in range(reps):
            y, period = repet._host.original_f64(x, FS, tun, handle=handle, return_period=True)
        dt = (time.perf_counter() - t0) / reps
        handle.set_stream(stream.cuda_stream)
        line.update({"workload": "BASELINE configs[0]: repet.original on the bundled audio_file.wav (23.0 s stereo)",
                     "period": int(period), "period_reference": 286,
                     "drop_in_call_ms": 1e3 * dt, "drop_in_x_realtime": len(x) / FS / dt,
                     "drop_in_api": "repet.original(float64 (S, C) ndarray, fs) -> float64 ndarray, pageable host memory"})
        out["cfg1"] = line

    if "cfg3" in wanted:
        B = args.cfg3_tracks
        t0 = time.perf_counter()
        tracks = repet_synth.make_batch(7000, B, 600 * FS, redraw_seconds=(60, 120))
        t_gen = time.perf_counter() - t0
        line, _ = measure("adaptive", tracks, 3)
        del tracks
        line.update({"workload": "BASELINE configs[2]: repet.adaptive, %d synthetic 10-min stereo tracks per GPU "
                                 "(256 over 8 GPUs)" % B, "synthesis_seconds": t_gen})
        out["cfg3"] = line

    if "cfg4" in wanted:
        track = repet_synth.make_batch(7100, 1, 600 * FS, redraw_seconds=(60, 120))
        line, prof = measure("sim", track, 3)
        T = frames_of(600 * FS)
        gemm_ms = prof.get("k_simgemm", (0.0, 0))[0] / 3
        topk_ms = prof.get("k_topk", (0.0, 0))[0] / 3
        tf32_peak = peaks["bf16_tflops"] / 2.0
        if gemm_ms > 0:
            useful = float(T) * (T + 1) * 1025 / (gemm_ms / 1e3) / 1e12
            issued = 3.0 * float(T) * (T + 1) * 1056 / (gemm_ms / 1e3) / 1e12
            line["gemm"] = {
                "ms": gemm_ms, "useful_tflops": useful, "issued_tflops": issued,
                "tf32_peak_tflops": tf32_peak, "frac_of_tf32_peak": useful / tf32_peak,
                "issued_frac_of_tf32_peak": issued / tf32_peak,
                "dram_bytes": ncu_figure("k_simgemm", "dram_bytes_per_launch"),
                "useful_flops": "T (T + 1) F: only the triangle of S = A A^T is formed (SURVEY.md 8(d))",
                "issued_flops": "3 TF32 MMAs per useful one (hi hi^T + hi lo^T + lo hi^T split for fp32-class accuracy) on "
                                "K padded 1025 -> 1056: the split caps useful/peak at 0.32",
                "peak": "half the measured dense bf16 rate (%s)" % peaks["source"],
            }
        if topk_ms > 0:
            line["kernels"]["k_topk"]["achieved_gbs"] = float(T) * T * 4 / (topk_ms / 1e3) / 1e9
            line["kernels"]["k_topk"]["frac_of_hbm_peak"] = line["kernels"]["k_topk"]["achieved_gbs"] / hbm
        line["workload"] = "BASELINE configs[3]: repet.sim on a synthetic 10-min stereo track (T = %d, %dx%d similarity)" % (T, T, T)
        out["cfg4"] = line

    if "cfg5" in wanted:
        hour = repet_synth.make_batch(7200, 1, 3600 * FS, redraw_seconds=(60, 120))
        line, _ = measure("extended", hour, 3)
        line["workload"] = "BASELINE configs[4]: repet.extended on one hour of synthetic stereo audio (719 segments)"
        out["cfg5_extended"] = line
        S_online = 155038 * 1024 + 2048
        padded = np.zeros((1, CHANNELS, S_online), dtype=np.float32)
        padded[:, :, : hour.shape[2]] = hour
        padded[:, :, hour.shape[2]:] = hour[:, :, : S_online - hour.shape[2]]
        del hour
        line, _ = measure("simonline", padded, 3)
        line["workload"] = ("BASELINE configs[4]: repet.simonline on one hour (S = 155 038 * 1024 + 2048), all frames in "
                            "parallel")
        out["cfg5_simonline"] = line
        # streaming: latency per 1 s block of the stateful stream (host float64 blocks in, final samples out)
        seconds = 150
        x = padded[0, :, : seconds * FS].T.astype(np.float64)
        del padded
        handle.set_stream(None)
        saved = repet._host._handles.get(device.index)
        repet._host._handles[device.index] = handle
        try:
            streamer = repet._host.SimOnlineStream(FS, CHANNELS, tun, handle=handle)
            latencies = []
            for k in range(0, len(x), FS):
                t0 = time.perf_counter()
                streamer.process(x[k : k + FS])
                latencies.append(1e3 * (time.perf_counter() - t0))
            streamer.flush()
            streamer.close()
        finally:
            if saved is not None:
                repet._host._handles[device.index] = saved
            handle.set_stream(stream.cuda_stream)
        steady = np.array(latencies[12:])  # after the 10 s warm-up of the algorithm
        out["cfg5_simonline_stream"] = {
            "workload": "BASELINE configs[4]: repet.SimOnline stream, 1 s blocks of float64 (S, C) samples in host memory",
            "blocks": int(len(steady)), "latency_ms_p50": float(np.percentile(steady, 50)),
            "latency_ms_p99": float(np.percentile(steady, 99)), "latency_ms_max": float(steady.max()),
            "x_realtime_per_stream": 1e3 / float(np.mean(steady)),
        }
    return out


# --------------------------------------------------------------------------------------------
# the CUDA arm
# --------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20


def dump_positions(number_clips, number_channels, number_samples):
    """The sample positions dump_outputs writes for `number_clips` clips over all ranks: a fixed seeded draw, as
    many as keep its four files within DUMP_LIMIT_BYTES."""
    fixed = number_clips * 8 + number_channels * number_samples * 4 + 4 * 4096  # periods, clip 0, four .npy headers
    count = (DUMP_LIMIT_BYTES - fixed) // (number_clips * number_channels * 4 + 8)
    count = max(1, min(number_samples, count))
    return np.sort(np.random.default_rng(0).choice(number_samples, size=count, replace=False))


def write_dump(directory, periods, background_clip0, background_sample, positions):
    os.makedirs(directory, exist_ok=True)
    for name, array in (("periods", periods.astype(np.float64)), ("background_clip0", background_clip0),
                        ("background_sample", background_sample),
                        ("background_sample_positions", positions.astype(np.float64))):
        np.save(os.path.join(directory, name + ".npy"), array)


def dump_outputs(directory, torch, dist, world, rank, out_dev, periods_dev):
    """Write what the timed path returned in its last step, so that two builds can be compared output for output
    on the same seeded clips.  The whole background of all ranks is GBs, so rank 0 gathers and writes, in at most
    64 MB for the whole run (every rank must call this):
      periods                       (N,) float64, the repeating period of each of the N clips, in frames
      background_clip0              (C, S) float32, the whole background of clip 0
      background_sample             (N, C, K) float32, every clip's background at K sample positions
      background_sample_positions   (K,) float64, those positions: a fixed seeded draw, the same on every run"""
    B, C, S = out_dev.shape
    positions = dump_positions(world * B, C, S)
    periods = periods_dev.to(torch.float64)
    sample = out_dev.index_select(2, torch.from_numpy(positions).to(out_dev.device))
    if world > 1:
        def gathered(part):
            parts = [torch.empty_like(part) for _ in range(world)]
            dist.all_gather(parts, part)
            return torch.cat(parts)

        periods, sample = gathered(periods), gathered(sample)
    if rank == 0:
        write_dump(directory, periods.cpu().numpy(), out_dev[0].cpu().numpy(), sample.cpu().numpy(), positions)


def run_b200_arm(args, rank, local_rank, world):
    import repet_synth

    numa = "disabled" if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)
    B = args.clips_per_gpu
    # 1) synthesise this rank's clips on the host BEFORE CUDA is initialised (fork pool)
    t_gen = time.perf_counter()
    workers = max(1, host_cores() // max(1, world))
    host_audio = repet_synth.make_batch(rank * B, B, CLIP_SAMPLES, CHANNELS, FS, processes=True, workers=workers)
    t_gen = time.perf_counter() - t_gen

    import torch
    import torch.distributed as dist

    import repet

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    handle = repet._host.Handle(local_rank)
    if args.tune:
        repet._host.set_tuning(**{k: int(v) for k, v in (kv.split("=") for kv in args.tune.split(","))})
    if args.workspace_mb:
        handle.set_workspace_limit(args.workspace_mb << 20)
    stream = torch.cuda.Stream(device)  # everything below is enqueued on this one stream
    torch.cuda.set_stream(stream)
    handle.set_stream(stream.cuda_stream)

    pinned_in = torch.from_numpy(host_audio).pin_memory()
    del host_audio
    pinned_out = torch.empty_like(pinned_in).pin_memory()
    audio_dev = pinned_in.to(device, non_blocking=True)
    out_dev = torch.empty_like(audio_dev)
    periods_dev = torch.zeros(B, dtype=torch.int32, device=device)
    torch.cuda.synchronize(device)

    def step_device():
        repet._host.original_batch_device(
            audio_dev.data_ptr(), out_dev.data_ptr(), B, CHANNELS, CLIP_SAMPLES, FS, TUNABLES, handle=handle,
            periods_ptr=periods_dev.data_ptr())

    # ---- device-resident timing ---------------------------------------------------------------
    for _ in range(max(3, args.warmup)):
        step_device()
    torch.cuda.synchronize(device)
    handle.profile_read(reset=True)
    handle.set_profiling(True)
    sampler = ClockSampler(local_rank)
    launches_before = handle.launch_count()
    barrier()
    torch.cuda.synchronize(device)
    sampler.start()
    start = torch.cuda.Event(enable_timing=True)
    end = torch.cuda.Event(enable_timing=True)
    start.record(stream)
    t_host = time.perf_counter()
    for _ in range(args.steps):
        step_device()
    t_host = time.perf_counter() - t_host  # host time to ENQUEUE the steps (no synchronisation inside)
    end.record(stream)
    torch.cuda.synchronize(device)
    barrier()
    clocks = sampler.stop()
    elapsed_ms = start.elapsed_time(end)
    launches = handle.launch_count() - launches_before
    profile = handle.profile_read(reset=True)
    handle.set_profiling(False)
    periods_first = periods_dev.cpu().numpy().copy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, dist, world, rank, out_dev, periods_dev)

    # ---- end to end through the public API: page-locked host arrays in and out --------------------
    host_in = pinned_in.numpy()
    host_out = pinned_out.numpy()
    e2e_ms = pcm_ms = link = None
    f64 = None
    if not args.no_e2e:
        def step_host():
            return repet._host.separate_batch("original", host_in, FS, TUNABLES, handle=handle, out=host_out)

        def timed(step):
            step()
            barrier()
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            for _ in range(args.steps):
                result = step()
            torch.cuda.synchronize(device)
            ms = 1e3 * (time.perf_counter() - t0)
            barrier()
            return ms, result

        e2e_ms, (_, ints) = timed(step_host)
        assert np.array_equal(ints[:, 0], periods_first), "host-buffer and device-resident paths disagree"
        assert np.array_equal(host_out, out_dev.cpu().numpy()), "host-buffer and device-resident outputs differ"

        # the same with int16 PCM on both sides (what WAVE files hold): a quarter of the bytes of float64 NumPy
        pcm_in = torch.empty((B, CLIP_SAMPLES, CHANNELS), dtype=torch.int16).pin_memory()
        pcm_out = torch.empty((B, CLIP_SAMPLES, CHANNELS), dtype=torch.int16).pin_memory()
        for lo in range(0, B, 32):  # quantise the same clips to 16 bits, WAV sample order
            block = pinned_in[lo : lo + 32].transpose(1, 2)
            pcm_in[lo : lo + 32] = torch.clamp(torch.round(block * 32768.0), -32768, 32767).to(torch.int16)
        pcm_in_np, pcm_out_np = pcm_in.numpy(), pcm_out.numpy()

        def step_pcm():
            return repet._host.separate_batch("original", pcm_in_np, FS, TUNABLES, handle=handle, in_format="pcm16",
                                              out_format="pcm16", out=pcm_out_np)

        pcm_ms, _ = timed(step_pcm)

        # copy-only ceiling: the e2e bytes over the same link with no kernels, both directions at once
        link = host_link_probe(torch, device, pinned_in, pinned_out, audio_dev, out_dev, max(2, min(args.steps, 5)), barrier)
        del pcm_in, pcm_out

        # the drop-in call itself: repet.original(float64 (S, C) ndarray, fs), clip by clip, pageable NumPy
        if rank == 0:
            n64 = min(B, 32)
            clips64 = [np.ascontiguousarray(host_in[i].T.astype(np.float64)) for i in range(n64)]
            repet._host.original_f64(clips64[0], FS, TUNABLES, handle=handle)
            t0 = time.perf_counter()
            per64 = [repet._host.original_f64(c, FS, TUNABLES, handle=handle, return_period=True)[1] for c in clips64]
            dt = time.perf_counter() - t0
            assert per64 == periods_first[:n64].tolist(), "float64 drop-in path and batch path disagree"
            f64 = {"value": n64 * CLIP_SECONDS / dt, "unit": UNIT, "clips": n64, "ms_per_clip": 1e3 * dt / n64,
                   "h2d_bytes_per_clip": CLIP_SAMPLES * CHANNELS * 8, "d2h_bytes_per_clip": CLIP_SAMPLES * CHANNELS * 8,
                   "api": "repet.original(float64 (S, C) ndarray, fs) -> float64 (S, C) ndarray, one clip per call, "
                          "pageable host memory (the reference's own calling convention)"}

    # ---- reduce over ranks: max time -------------------------------------------------------------
    vals = [elapsed_ms, e2e_ms or 0.0, pcm_ms or 0.0] + ([link["h2d_s"], link["d2h_s"], link["duplex_s"]] if link else [0.0] * 3)
    times = torch.tensor(vals, dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    elapsed_ms, e2e_max_ms, pcm_max_ms, link_h2d, link_d2h, link_duplex = (float(v) for v in times)

    if rank == 0:
        peaks = measured_peaks()
        audio_seconds_per_step = world * B * CLIP_SECONDS
        value = audio_seconds_per_step * args.steps / (elapsed_ms / 1e3)
        T = frames_of(CLIP_SAMPLES)
        audio_bytes = CLIP_SAMPLES * CHANNELS * 4
        x_bytes = T * CHANNELS * 1025 * 8
        p_bytes = T * 1025 * 4
        algorithmic, _ = config_algorithmic_bytes("original", CLIP_SAMPLES)  # bytes per clip, DESIGN.md section 3
        peak, peak_source = peaks["hbm_gbs"], peaks["source"] + " hbm_gbs"
        kernels = {}
        for name, (ms, count) in profile.items():
            entry = {"ms_total": ms, "launches": count, "share_of_step": ms / elapsed_ms if elapsed_ms else None}
            if name in algorithmic and ms > 0:
                gbs = algorithmic[name] * B * args.steps / (ms / 1e3) / 1e9
                entry.update({"achieved_gbs": gbs, "frac": gbs / peak,
                              "algorithmic_bytes_per_launch": algorithmic[name] * B * args.steps / max(1, count)})
            kernels[name] = entry
        dominant = max((k for k in kernels if "achieved_gbs" in kernels[k]), key=lambda k: kernels[k]["ms_total"], default=None)
        roofline = None
        if dominant:
            d = kernels[dominant]
            whole = (2 * audio_bytes + 2 * x_bytes + 2 * p_bytes) * B * args.steps / (elapsed_ms / 1e3) / 1e9
            roofline = {"bound": "hbm", "kernel": dominant, "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s",
                        "frac": d["frac"],
                        "traffic": ncu_traffic(dominant, B * args.steps / max(1, d["launches"])), "peak_source": peak_source,
                        "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_launch"],
                        "avg_launch_ms": d["ms_total"] / max(1, d["launches"]), "kernels": kernels,
                        "whole_path_algorithmic_gbs": whole, "whole_path_frac": whole / peak}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(args), "clocks": clocks,
            "gpu_launches": int(launches), "roofline": roofline,
            "periods_sample": periods_first[:8].tolist(), "synthesis_seconds": t_gen,
            "host_enqueue_ms_per_step": 1e3 * t_host / args.steps, "numa": numa,
        }
        if e2e_ms is not None:
            step_bytes = world * B * audio_bytes
            duplex_gbs = 2 * step_bytes / link_duplex / 1e9
            line["host_link"] = {
                "h2d_gbs": step_bytes / link_h2d / 1e9, "d2h_gbs": step_bytes / link_d2h / 1e9,
                "duplex_gbs_both_ways": duplex_gbs, "duplex_ms_per_step": 1e3 * link_duplex,
                "how": "the fp32 e2e bytes of one step (all ranks at once) over pinned cudaMemcpyAsync on two streams, no "
                       "kernels, max over ranks: the ceiling of any host-buffer path on this box",
            }
            line["e2e"] = {"value": audio_seconds_per_step * args.steps / (e2e_max_ms / 1e3), "unit": UNIT,
                           "h2d_bytes_per_step": B * audio_bytes, "d2h_bytes_per_step": B * audio_bytes + B * 4,
                           "ms_per_step": e2e_max_ms / args.steps,
                           "frac_of_host_link": (1e3 * link_duplex) / (e2e_max_ms / args.steps),
                           "api": "repet.separate_batch(method='original') on page-locked fp32 planar NumPy arrays, in and out"}
            line["e2e_pcm16"] = {"value": audio_seconds_per_step * args.steps / (pcm_max_ms / 1e3), "unit": UNIT,
                                 "h2d_bytes_per_step": B * audio_bytes // 2, "d2h_bytes_per_step": B * audio_bytes // 2 + B * 4,
                                 "ms_per_step": pcm_max_ms / args.steps,
                                 "frac_of_host_link": (1e3 * link_duplex / 2) / (pcm_max_ms / args.steps),
                                 "api": "repet.separate_batch(in_format='pcm16', out_format='pcm16'): int16 PCM in WAV order "
                                        "on both sides; the output is round(y * 2^15), <= 2^-16 of quantisation error"}
            if f64:
                line["e2e_numpy_f64"] = f64
        wanted = []
        if args.configs == "auto":
            wanted = ["cfg1", "cfg3", "cfg4", "cfg5"] if world == 1 else []
        elif args.configs != "none":
            wanted = [c for c in args.configs.split(",") if c]
        if wanted:
            del pinned_in, pinned_out, audio_dev, out_dev, host_in, host_out
            torch.cuda.empty_cache()
            line["configs"] = run_configs(args, torch, repet, handle, stream, device, wanted, peaks)
        if world == 1 and not args.no_cpu_baseline:
            # fork the CPU pool only now; workers never touch CUDA
            arm = CpuArm()
            sample = args.cpu_sample_clips or max(2 * arm.workers, min(64, B))
            compute, wall, audio, cpu_periods = arm.run(0, sample)
            arm.close()
            same = cpu_periods == periods_first[:sample].tolist()
            line["cpu_baseline"] = {"value": audio / compute, "unit": UNIT, "cores": arm.workers, "kind": arm.kind,
                                    "sample": "%d of the %d clips (30 s each), %s, one clip per core"
                                              % (sample, B, arm.describe()), "wall_seconds": wall,
                                    "periods_equal_gpu": bool(same)}
            assert same, "CPU and GPU periods differ on the benchmark's own clips: %s vs %s" % (
                cpu_periods, periods_first[:sample].tolist())
        print(json.dumps(line), flush=True)
    handle.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1 and args.gpus > 1 and args.impl == "b200":
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
    elif args.probe_host_link:
        run_host_link_probe(args, rank, local_rank, world)
    else:
        run_b200_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
