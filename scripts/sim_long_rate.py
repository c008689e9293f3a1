#!/usr/bin/env python
"""repet.sim on long tracks, one GPU, device resident (repet_sim_batch_dev, CUDA events).

Cases are "<minutes>" (the default workspace limit) or "<minutes>p<n>" (a workspace limit that forms the similarity
matrix in about n row panels; "<minutes>w" forces the whole matrix with a limit that holds it).  Cases of the same
length share one synthetic stereo track (repet_synth, background redrawn every 60-120 s), so "10w,10p8,10w,10p8"
alternates the whole-matrix and the panel path on the same input in one process.

Per case, one JSON line: ms per call and x realtime (warm-up, then --steps calls between two events), per-kernel ms
(a separate profiled call), row panels and their height, columns settled by the exact fallback (a separate
REPET_DEBUG_TOPK call), the handle's workspace bytes, and the similarity GEMM's rate.  The card's name, power limit
and maximum SM clock are read in the same process.

    python scripts/sim_long_rate.py --cases 10w,10p8,10w,10p8,30,60,120 --out profiles/r3_sim_long.jsonl
    python scripts/sim_long_rate.py --lib <other librepet_b200.so> --cases 10w,30   # another build, same inputs
"""
import argparse
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "repet-python_b200"))
import numpy as np  # noqa: E402

FS = 44100
HOP = 1024


def sim_linear_bytes(T, nch, number, sm_count):
    """Workspace of one `sim` track besides S (make_plan in csrc/repet_drivers.cu, 44.1 kHz instantiation)."""
    def al(v):
        return (v + 255) // 256 * 256

    XPITCH, PPITCH, KPAD = 1024, 1032, 1056
    b = al(T * nch * XPITCH * 8) + al(T * PPITCH * 4) + al(T * PPITCH * 8) + al(T * number * 4) + al(T * 4)
    b += al(nch * T * PPITCH * 4)
    if number > 32:
        b += al(nch * T * PPITCH * 4)
    b += 2 * al(T * KPAD * 4) + al(T * 4)
    b += al((T * 12 + 255) // 256 * 256 * sm_count * 2)
    return b + 2048


def limit_for_panels(T, n_panels, nch, number, sm_count):
    """A workspace limit under which S is formed in row panels of ceil(T / n / 128) * 128 rows."""
    P = -(-T // (n_panels * 128)) * 128
    return sim_linear_bytes(T, nch, number, sm_count) + 256 + P * T * 4 + 4096


def parse_debug(text):
    m = re.search(r"k_topk: (\d+) columns \((\d+) through the exact fallback\), (\d+) candidates", text)
    out = {"exact_fallback_columns": int(m.group(2)), "candidates": int(m.group(3))} if m else {"debug": text}
    m = re.search(r"(\d+) row panels of (\d+)", text)
    if m:
        out["panels"], out["panel_rows"] = int(m.group(1)), int(m.group(2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="10w,10p8,10w,10p8,30,60,120")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--lib", default="", help="another build of librepet_b200.so (default: the tree's)")
    ap.add_argument("--out", default="", help="append the JSON lines to this file as well")
    args = ap.parse_args()
    import repet_synth

    cases = []
    for c in args.cases.split(","):
        m = re.fullmatch(r"(\d+)(w|p\d+)?", c.strip())
        if not m:
            raise SystemExit("bad case %r" % c)
        cases.append((c.strip(), int(m.group(1)), m.group(2) or ""))
    tracks = {}
    for _, minutes, _ in cases:
        if minutes not in tracks:
            t0 = time.perf_counter()
            tracks[minutes] = repet_synth.make_clip(7300 + minutes, minutes * 60 * FS, redraw_seconds=(60, 120))[None]
            print("# synthesised %d min in %.1f s" % (minutes, time.perf_counter() - t0), file=sys.stderr, flush=True)

    import torch

    import repet

    if args.lib:
        repet._host.LIB_PATH = os.path.abspath(args.lib)
        try:
            ctypes.CDLL(repet._host.LIB_PATH).repet_workspace_bytes
        except AttributeError:
            del repet._host.SIGNATURES["repet_workspace_bytes"]
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    handle = repet._host.Handle(0)
    stream = torch.cuda.Stream(device)
    torch.cuda.set_stream(stream)
    handle.set_stream(stream.cuda_stream)
    params, _ = repet._host.derive_params(FS, repet._tunables(), "sim")
    handle.ensure_window(params.window_length)
    fn = handle.lib.repet_sim_batch_dev
    on_device = {}
    for name, minutes, mode in cases:
        if minutes not in on_device:
            on_device.clear()
            torch.cuda.empty_cache()
            audio = torch.from_numpy(tracks[minutes]).to(device)
            on_device[minutes] = (audio, torch.empty_like(audio))
        audio, out = on_device[minutes]
        S = audio.shape[-1]
        T = (S + HOP - 1) // HOP + 1
        if mode.startswith("p"):
            limit = limit_for_panels(T, int(mode[1:]), 2, params.similarity_number, sm_count)
        elif mode == "w":
            limit = sim_linear_bytes(T, 2, params.similarity_number, sm_count) + T * T * 4 + (1 << 20)
        else:
            limit = 0
        handle.set_workspace_limit(limit)

        def step():
            handle.check(fn(handle.h, ctypes.c_void_p(audio.data_ptr()), 1, 2, S, ctypes.byref(params),
                            ctypes.c_void_p(out.data_ptr()), None, None))

        step()
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(args.steps):
            step()
        end.record(stream)
        torch.cuda.synchronize()
        ms = start.elapsed_time(end) / args.steps
        handle.profile_read(reset=True)
        handle.set_profiling(True)
        step()
        prof = handle.profile_read(reset=True)
        handle.set_profiling(False)
        # statistics of k_topk: printed to stderr by the library, captured at the file-descriptor level
        os.environ["REPET_DEBUG_TOPK"] = "1"
        saved = os.dup(2)
        with tempfile.TemporaryFile(mode="w+") as tmp:
            os.dup2(tmp.fileno(), 2)
            try:
                step()
                torch.cuda.synchronize()
            finally:
                os.dup2(saved, 2)
                os.close(saved)
                del os.environ["REPET_DEBUG_TOPK"]
            tmp.seek(0)
            debug = tmp.read()
        line = {"case": name, "gpu": gpu, "lib": "tree" if not args.lib else os.path.basename(os.path.dirname(os.path.abspath(args.lib))),
                "seconds": S / FS, "T": T, "workspace_limit": limit, "ms_per_call": ms, "x_realtime": S / FS / (ms / 1e3),
                "kernels_ms": {k: v[0] for k, v in prof.items()}}
        line.update(parse_debug(debug))
        if "repet_workspace_bytes" in repet._host.SIGNATURES:
            line["workspace_bytes"] = handle.workspace_bytes()
        gemm_ms = prof.get("k_simgemm", (0.0, 0))[0]
        if gemm_ms:
            panels = line.get("panels", 1) > 1
            # issued TF32 MMA flops of the 3xTF32 split product (K padded to 1056): the full rectangle of every
            # panel, or the tiles on and above the diagonal of the whole matrix
            issued = 6.0 * T * T * 1056 if panels else 3.0 * T * (T + 1) * 1056
            line["gemm_tf32_tflops_issued"] = issued / (gemm_ms / 1e3) / 1e12
            line["gemm_full_product_equivalent_tflops"] = 2.0 * T * T * 1025 / (gemm_ms / 1e3) / 1e12
        text = json.dumps(line)
        print(text, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(text + "\n")
    handle.set_workspace_limit(0)


if __name__ == "__main__":
    main()
