"""Cost of the 64-APSK frame source on the device (nbgpu_source_frames_apsk64) on one B200, against the BPSK source
(nbgpu_source_frames) on the same code, and what it buys the Monte-Carlo driver.

    python scripts/source_apsk64_cost.py [--reps 7] [--warmup 2] [--out FILE]   (default FILE: profiles/r03b_source_apsk64_cost.json)

Workload: config 3 (MatDeclercq_R12_GF64, N = 10800, GF(64); the seeded stand-in of tests/common.code_path when the file is
absent), n_m = 20, 10 iterations, batches of two whole waves of the persistent grid (geometry()), as bench.py runs it.
  * source: one call = encoder + noise kernel + flag read-back (+ host fix-up), timed by CUDA events around the call and by
    the host clock (the call ends in a stream synchronise); the two channels alternate inside every repetition, each call on
    a new block of frames.  The decode kernel time of the same batch (fixed-iteration mode) is given for scale.
  * driver: frames/s of `nbldpc_mc ... channel 1` with the device source (1) and the host source (0), three batches.
Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nbldpc                      # noqa: E402
from common import MATRIX_DIRS, code_path       # noqa: E402

REL, N_M, NB_OPER, OFFSET, NB_ITER_MAX = "matrices/MatDeclercq_R12_GF64", 20, 25, 0.3, 10
EBN = {"bpsk": 1.2, "apsk64": 12.0}          # bench.py's point for config 3; a 64-APSK point where the frames converge
WAVES = 2
EXE = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def source_cost(code, reps, warmup):
    d = nbldpc.Decoder(code, N_M, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=1 << 14)
    g = d.geometry()
    B = WAVES * g["grid"] * g["frames_per_cta"]
    d.close()
    d = nbldpc.Decoder(code, N_M, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=B)
    calls = {"bpsk": d.source_frames, "apsk64": d.source_frames_apsk64}
    ev, host, fix, dec = ({ch: [] for ch in calls} for _ in range(4))
    for r in range(warmup + reps):
        for ch, fn in calls.items():
            d.sync()
            d.timer_begin()
            t0 = time.perf_counter()
            fn(r * B, B, EBN[ch])
            t1 = time.perf_counter()
            ms = d.timer_end()
            d.run()
            d.sync()
            if r < warmup:
                continue
            ev[ch].append(ms); host[ch].append((t1 - t0) * 1e3); fix[ch].append(d.source_fixups()); dec[ch].append(d.last_kernel_ms())
    out = {"frames": B, "geometry": g, "reps": reps, "channels": {}}
    for ch in calls:
        samples = B * code.N * (2 if ch == "apsk64" else code.logq)
        out["channels"][ch] = {"ebn": EBN[ch], "samples": samples, "source_event_ms": spread(ev[ch]), "source_host_ms": spread(host[ch]),
                               "source_ns_per_frame": statistics.median(ev[ch]) * 1e6 / B, "fixups": fix[ch],
                               "decode_kernel_ms": spread(dec[ch])}
    out["apsk64_over_bpsk_source_time"] = statistics.median(ev["apsk64"]) / statistics.median(ev["bpsk"])
    d.close()
    return out


def driver(path, B):
    """frames/s of the C driver, 64-APSK channel, device and host frame source"""
    res = {}
    for source in (1, 0):
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "data"))
            args = [EXE, str(3 * B), str(NB_ITER_MAX), path, "%g" % EBN["apsk64"], str(N_M), str(OFFSET), str(NB_OPER), str(B), "0", "0",
                    str(source), "1"]
            r = subprocess.run(args, cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=3000)
            if r.returncode != 0:
                raise SystemExit("nbldpc_mc failed:\n" + r.stdout[-2000:])
            m = re.search(r"frame source: (\d+) frames in ([\d.]+) s = ([\d.]+) frames/s", r.stdout)
            last = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+).*?avr_it=([\d.]+)", r.stdout)[-1]
            res["device_source" if source else "host_source"] = {
                "frames": int(m.group(1)), "seconds": float(m.group(2)), "frames_per_s": float(m.group(3)),
                "err_frames": int(last[1]), "avr_it": float(last[3])}
    res["args"] = "nbldpc_mc %d %d <matrix> %g %d %g %d %d 0 0 <source> 1" % (3 * B, NB_ITER_MAX, EBN["apsk64"], N_M, OFFSET, NB_OPER, B)
    res["device_over_host"] = res["device_source"]["frames_per_s"] / res["host_source"]["frames_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03b_source_apsk64_cost.json"))
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("source_apsk64_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    path = code_path(REL)
    code = nbldpc.Code(path)
    standin = all(os.path.join(m, REL) != path for m in MATRIX_DIRS)
    src = source_cost(code, max(3, args.reps), args.warmup)
    line = {"card": name, "power_limit": limit,
            "matrix": "seeded stand-in for %s (tests/common.code_path)" % REL if standin else REL,
            "N": code.N, "q": code.q, "n_m": N_M, "iterations": NB_ITER_MAX,
            "source": src, "driver": driver(path, src["frames"])}
    code.close()
    s = json.dumps(line)
    print(s)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
