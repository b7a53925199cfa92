"""Cost of the split channel (every GF(q) symbol sent as P points of Gray QPSK or 16-QAM, noisy[B][N][P][2]) on one B200, against
the mapped channel (one point of Gray square q-QAM, noisy[B][N][2]) on the same code: the decode kernel with the split intake,
and the device frame source.

    python scripts/split_channel_cost.py [--reps 7] [--warmup 2] [--out FILE]   (default FILE: profiles/r03e_split_channel_cost.json)

Workloads: config 5 (AD_64800_R12_GF256, GF(256): P = 2 (16-QAM) and P = 4 (QPSK) against 256-QAM) and config 4
(Ahmed_64800_R34_GF16, GF(16): P = 2 (QPSK) against 16-QAM), as seeded stand-ins of tests/common.code_path when the files are
absent; n_m and iterations as bench.py, 592 frames, fixed-iteration mode, so the decode time does not depend on the channel's
quality.
  * decode: nbgpu_run on the resident batch (generated on the device), CUDA events, median of the repetitions; the channels
    alternate inside every repetition.  The split intake computes P*M table entries per variable (2*P*M f64 divisions) and
    sums P of them per symbol, where the mapped intake divides 2q times.
  * source: one nbgpu_source_frames_mapped / nbgpu_source_frames_split call (encoder + noise kernel + flag read-back + host
    fix-up), CUDA events around the call, with the fix-up count; alternated the same way, each call on a new block of frames.
Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nbldpc                      # noqa: E402
from common import MATRIX_DIRS, code_path       # noqa: E402

# (matrix, n_m, Es/N0 of the mapped channel, {points: Es/N0 per point})
CONFIGS = {"config5": ("matrices/AD_64800_R12_GF256", 20, 20.0, {2: 10.0, 4: 4.0}),
           "config4": ("matrices/Ahmed_64800_R34_GF16", 16, 12.0, {2: 6.0})}
NB_OPER, OFFSET, NB_ITER_MAX = 25, 0.3, 10
FRAMES = 592


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def cost(code, n_m, esn, split_esn, reps, warmup):
    B = FRAMES
    d = nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=B)
    g = d.geometry()
    d.set_constellation(nbldpc.constellation(nbldpc.MAP_QAM, code.q))

    # per channel: (table binding outside the timed window, source call)
    calls = {"mapped": (lambda: None, lambda f0: d.source_frames_mapped(f0, B, esn))}
    for P, e in split_esn.items():
        calls["split_p%d" % P] = (lambda P=P: d.set_split_constellation(nbldpc.split_qam(code.q, P), P),
                                  lambda f0, e=e: d.source_frames_split(f0, B, e))
    src, fix, dec = ({ch: [] for ch in calls} for _ in range(3))
    for r in range(warmup + reps):
        for ch, (bind, fn) in calls.items():
            bind()                                   # the previous batch has been run: re-binding drops nothing needed
            d.sync()
            d.timer_begin()
            fn(r * B)
            ms = d.timer_end()
            d.run()
            d.sync()
            if r < warmup:
                continue
            src[ch].append(ms); fix[ch].append(d.source_fixups()); dec[ch].append(d.last_kernel_ms())
    out = {"frames": B, "geometry": g, "reps": reps, "n_m": n_m, "esn_mapped": esn, "esn_per_point_split": split_esn, "channels": {}}
    for ch in calls:
        out["channels"][ch] = {"decode_kernel_ms": spread(dec[ch]), "source_event_ms": spread(src[ch]),
                               "source_ns_per_frame": statistics.median(src[ch]) * 1e6 / B, "fixups": fix[ch]}
        if ch != "mapped":
            out[ch + "_over_mapped_decode_time"] = statistics.median(dec[ch]) / statistics.median(dec["mapped"])
            out[ch + "_over_mapped_source_time"] = statistics.median(src[ch]) / statistics.median(src["mapped"])
    d.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03e_split_channel_cost.json"))
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("split_channel_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    line = {"card": name, "power_limit": limit, "iterations": NB_ITER_MAX}
    for key, (rel, n_m, esn, split_esn) in CONFIGS.items():
        path = code_path(rel)
        code = nbldpc.Code(path)
        standin = all(os.path.join(m, rel) != path for m in MATRIX_DIRS)
        line[key] = {"matrix": "seeded stand-in for %s (tests/common.code_path)" % rel if standin else rel, "N": code.N, "q": code.q,
                     "mapped": "Gray square %d-QAM" % code.q,
                     "split": {"p%d" % P: "Gray %s" % ("QPSK" if (code.logq // P) == 2 else "16-QAM") for P in split_esn},
                     "cost": cost(code, n_m, esn, split_esn, max(3, args.reps), args.warmup)}
        code.close()
    s = json.dumps(line)
    print(s)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
