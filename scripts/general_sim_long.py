#!/usr/bin/env python
"""repet.sim on long 96 kHz mono tracks through the general float64 path (repet_general_f64), one GPU.

Cases are "<minutes>" (the default workspace limit) or "<minutes>g<GiB>" (a workspace limit of that many GiB).  Cases
of the same length share one synthetic track (repet_synth, background redrawn every 60-120 s), so "10,10g1,10,10g1"
alternates the whole matrix and row panels on the same input in one process.

Per case, one JSON line: wall seconds of one sim_f64 call (host clock; the call ends in a stream synchronise) after
one warm-up call of the same case, x realtime, T, the panel height the call used and its number of panels (from the
handle's launch count: each panel is one Gram and one selection launch), and a digest of the lists and background.
The card's name, power limit and maximum SM clock are read in the same process.

    python scripts/general_sim_long.py --cases 10,10g1,10,10g1,60 --out profiles/r3_general_sim_long.jsonl
    python scripts/general_sim_long.py --lib <other librepet_b200.so> --cases 10    # another build, same input
"""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "repet-python_b200"))
import numpy as np  # noqa: E402

FS = 96000
HOP = 2048
TILE = 64


def need(P, T, sm_count):
    """Bytes of one S panel of P rows and of the selection's per-CTA kept lists (gen_run, csrc/repet_generic.cu)."""
    return P * T * 8 + min(P, 2 * sm_count) * T * 4


def panel_rows(T, limit, sm_count):
    """The panel height gen_run picks under `limit` (T: the whole matrix)."""
    if need(T, T, sm_count) <= limit:
        return T
    P = min(T, limit // (T * 8)) // TILE * TILE
    while P > TILE and need(P, T, sm_count) > limit:
        P -= TILE
    return min(T, max(P, TILE))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="10,10g1,10,10g1,60")
    ap.add_argument("--lib", default="", help="another build of librepet_b200.so (default: the tree's)")
    ap.add_argument("--out", default="", help="append the JSON lines to this file as well")
    args = ap.parse_args()
    import torch

    import repet
    import repet_synth

    if args.lib:
        repet._host.LIB_PATH = os.path.abspath(args.lib)
    cases = []
    for c in args.cases.split(","):
        m = re.fullmatch(r"(\d+)(?:g(\d+))?", c.strip())
        if not m:
            raise SystemExit("bad case %r" % c)
        cases.append((c.strip(), int(m.group(1)), int(m.group(2) or 0)))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    handle = repet._host.Handle(0)
    tunables = repet._tunables()

    def call(x, limit):
        handle.set_workspace_limit(limit)
        try:
            before = handle.launch_count()
            t0 = time.perf_counter()
            y, lists = repet._host.sim_f64(x, FS, tunables, handle=handle, return_indices=True)
            wall = time.perf_counter() - t0
            return y, lists, wall, handle.launch_count() - before
        finally:
            handle.set_workspace_limit(0)

    # the launches of a call with one Gram + selection pair (a 20 s track holds its whole matrix on any limit)
    probe = repet_synth.make_clip(9600, 20 * FS, 1, FS, HOP).T.astype(np.float64)
    launches_one = call(probe, 0)[3]
    tracks = {}
    out = open(args.out, "a") if args.out else None
    for name, minutes, gib in cases:
        if minutes not in tracks:
            tracks[minutes] = repet_synth.make_clip(9600 + minutes, minutes * 60 * FS, 1, FS, HOP,
                                                    redraw_seconds=(60, 120)).T.astype(np.float64)
        x = tracks[minutes]
        limit = gib << 30
        T = repet._host.number_of_frames(len(x), 2 * HOP, HOP)
        call(x, limit)  # warm-up: module load, pool growth
        y, lists, wall, launches = call(x, limit)
        n_panels = 1 + (launches - launches_one) // 2
        digest = hashlib.sha256()
        for v in lists:
            digest.update(np.int32(len(v)).tobytes() + v.astype(np.int32).tobytes())
        digest.update(np.ascontiguousarray(y).tobytes())
        line = {"case": name, "gpu": gpu, "lib": "tree" if not args.lib else os.path.basename(os.path.dirname(os.path.abspath(args.lib))),
                "seconds_of_audio": minutes * 60, "fs": FS, "channels": 1, "T": T,
                "workspace_limit": limit or "default", "panels": n_panels,
                "panel_rows": panel_rows(T, limit, sm_count) if limit else None,
                "wall_s": round(wall, 4), "x_realtime": round(minutes * 60 / wall, 1),
                "digest": digest.hexdigest()[:16]}
        if not limit:  # the default limit is 24 GiB unless the device has less than 60 GiB free
            P = panel_rows(T, 24 << 30, sm_count)
            line["panel_rows"] = P if -(-T // P) == n_panels else None
        print(json.dumps(line), flush=True)
        if out:
            out.write(json.dumps(line) + "\n")
    if out:
        out.close()
    handle.close()


if __name__ == "__main__":
    main()
