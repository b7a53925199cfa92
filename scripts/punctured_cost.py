"""Cost of puncturing on one B200: the decode kernel and the device frame source of the same build with no puncturing pattern
bound and with a pattern of 10 % of the variables (nbgpu_set_puncturing), BPSK over AWGN.

    python scripts/punctured_cost.py [--reps 7] [--warmup 2] [--out FILE]   (default FILE: profiles/r03f_punctured_cost.json)

Workloads: config 5 (AD_64800_R12_GF256) and config 4 (Ahmed_64800_R34_GF16), as seeded stand-ins of tests/common.code_path
when the files are absent; n_m and iterations as bench.py, 592 frames, fixed-iteration mode, so the decode time does not depend
on the channel's quality.  The pattern is a seeded random 10 % of the variables.
  * decode: nbgpu_run on the resident batch (generated on the device), CUDA events, median of the repetitions; the two
    settings alternate inside every repetition.  Only the frame initialisation reads the pattern (one map load per variable
    and frame, a zero row for a punctured one); the pass loop is the same code.
  * source: one nbgpu_source_frames call (encoder + noise kernel + flag read-back + host fix-up), CUDA events around the call,
    alternated the same way, each call on a new block of frames.  With the pattern the noise kernel runs one thread per
    transmitted symbol, 10 % fewer.
  * slow selects: selection rows per launch that needed the exact scan (nbgpu_slow_selects), with and without the pattern.
Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nbldpc                      # noqa: E402
from common import MATRIX_DIRS, code_path       # noqa: E402

# (matrix, n_m, Eb/N0 in dB)
CONFIGS = {"config5": ("matrices/AD_64800_R12_GF256", 20, 1.5), "config4": ("matrices/Ahmed_64800_R34_GF16", 16, 3.0)}
NB_OPER, OFFSET, NB_ITER_MAX = 25, 0.3, 10
FRAMES = 592
FRACTION = 0.10


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def cost(code, n_m, ebn, reps, warmup):
    B = FRAMES
    d = nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=B)
    g = d.geometry()
    pattern = np.random.default_rng(1).choice(code.N, int(FRACTION * code.N), replace=False).astype(np.int32)
    settings = {"none": (), "punctured": pattern}
    src, dec, slow = ({s: [] for s in settings} for _ in range(3))
    for r in range(warmup + reps):
        for s, pv in settings.items():
            d.set_puncturing(pv)                         # outside the timed window; the previous batch has been run
            d.sync()
            d.timer_begin()
            d.source_frames(r * B, B, ebn)
            ms = d.timer_end()
            s0 = d.slow_selects()
            d.run()
            d.sync()
            if r < warmup:
                continue
            src[s].append(ms); dec[s].append(d.last_kernel_ms()); slow[s].append(d.slow_selects() - s0)
    out = {"frames": B, "geometry": g, "reps": reps, "n_m": n_m, "ebn": ebn, "punctured": int(pattern.size), "settings": {}}
    for s in settings:
        out["settings"][s] = {"decode_kernel_ms": spread(dec[s]), "source_event_ms": spread(src[s]),
                              "source_ns_per_frame": statistics.median(src[s]) * 1e6 / B, "slow_selects_per_launch": slow[s]}
    out["punctured_over_none_decode_time"] = statistics.median(dec["punctured"]) / statistics.median(dec["none"])
    out["punctured_over_none_source_time"] = statistics.median(src["punctured"]) / statistics.median(src["none"])
    d.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03f_punctured_cost.json"))
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("punctured_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    line = {"card": name, "power_limit": limit, "iterations": NB_ITER_MAX, "channel": "BPSK over AWGN"}
    for key, (rel, n_m, ebn) in CONFIGS.items():
        path = code_path(rel)
        code = nbldpc.Code(path)
        standin = all(os.path.join(m, rel) != path for m in MATRIX_DIRS)
        line[key] = {"matrix": "seeded stand-in for %s (tests/common.code_path)" % rel if standin else rel, "N": code.N, "q": code.q,
                     "cost": cost(code, n_m, ebn, max(3, args.reps), args.warmup)}
        code.close()
    s = json.dumps(line)
    print(s)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
