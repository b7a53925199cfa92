"""Cost and error rate of the Min-Max check node (ecn_kind = 4) next to the sum-product node (ecn_kind = 2) and L-Bubble
(ecn_kind = 0) on one B200.

    python scripts/minmax_cost.py [--reps 5] [--warmup 1] [--out FILE]   (default FILE: profiles/r03h_minmax_cost.json)

  * throughput: configs 3, 4 and 5 (seeded stand-ins of tests/common.code_path when the matrices are absent), 592 frames
    generated on the device and resident, 10 iterations in fixed-iteration mode (no early stop), n_m as bench.py.  nbgpu_run
    timed with CUDA events; the three nodes alternate inside every repetition; median, min and max.  Decoded Mbit/s counts
    information bits (K log2 q per frame).
  * FER: the three nodes on the same device-generated frames (the reference's stream, BPSK over AWGN, 10 iterations, early stop)
    at three Eb/N0 points of N96_K48_GF64 (2000 frames) and two of config 3 (1184 frames); every frame counted (no stop at
    40 erroneous frames).
Reads the card's name and power limit in the same call.  Prints one JSON line and writes it to --out."""
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

import nbldpc                                   # noqa: E402
from common import MATRIX_DIRS, code_path, multigpu      # noqa: E402

CONFIGS = {"config3": ("matrices/MatDeclercq_R12_GF64", 20, 1.5), "config4": ("matrices/Ahmed_64800_R34_GF16", 16, 3.0),
           "config5": ("matrices/AD_64800_R12_GF256", 20, 1.5)}
NODES = {"Min-Max": 4, "sum-product": 2, "L-Bubble": 0}
NB_OPER, OFFSET, NB_ITER_MAX = 25, 0.3, 10
FRAMES = 592
FER_POINTS = {"N96_K48_GF64": ("matrices/N96_K48_GF64", 20, 2000, (2.0, 2.5, 3.0)), "config3": ("matrices/MatDeclercq_R12_GF64", 20, 1184, (1.2, 1.4))}


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def matrix_name(rel, path):
    standin = all(os.path.join(m, rel) != path for m in MATRIX_DIRS)
    return "seeded stand-in for %s (tests/common.code_path)" % rel if standin else rel


def throughput(code, n_m, ebn, reps, warmup):
    decs = {k: nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, ecn_kind=e, max_batch=FRAMES)
            for k, e in NODES.items()}
    for d in decs.values():
        d.source_frames(0, FRAMES, ebn)
    ms = {k: [] for k in decs}
    for r in range(warmup + reps):
        for k, d in decs.items():
            d.run()
            d.sync()
            if r >= warmup:
                ms[k].append(d.last_kernel_ms())
    bits = FRAMES * code.K * code.logq
    out = {"frames": FRAMES, "ebn": ebn, "n_m_l_bubble": n_m}
    for k, d in decs.items():
        out[k] = {"decode_kernel_ms": spread(ms[k]), "mbit_per_s": bits / (statistics.median(ms[k]) * 1e3), "geometry": d.geometry()}
        d.close()
    out["min_max_over_l_bubble_time"] = statistics.median(ms["Min-Max"]) / statistics.median(ms["L-Bubble"])
    out["min_max_over_sum_product_time"] = statistics.median(ms["Min-Max"]) / statistics.median(ms["sum-product"])
    return out


def fer(code, n_m, frames, points):
    out = {"frames": frames, "points": {}}
    for ebn in points:
        row = {}
        for k, e in NODES.items():
            d = nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, ecn_kind=e, max_batch=592)
            st = multigpu.monte_carlo(code, frames, ebn, decoder=d, batch=592, max_err_frames=10 ** 9)
            row[k] = {"err_frames": st["err_frames"], "bit_errors": st["bit_errors"], "avr_it": st["sum_it"] / st["frames"]}
            d.close()
        out["points"]["%.2f" % ebn] = row
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03h_minmax_cost.json"))
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("minmax_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    line = {"card": name, "power_limit": limit, "iterations": NB_ITER_MAX, "channel": "BPSK over AWGN", "throughput": {}, "fer": {}}
    for key, (rel, n_m, ebn) in CONFIGS.items():
        path = code_path(rel)
        code = nbldpc.Code(path)
        line["throughput"][key] = dict(matrix=matrix_name(rel, path), N=code.N, q=code.q, **throughput(code, n_m, ebn, args.reps, args.warmup))
        code.close()
    for key, (rel, n_m, frames, points) in FER_POINTS.items():
        path = code_path(rel)
        code = nbldpc.Code(path)
        line["fer"][key] = dict(matrix=matrix_name(rel, path), N=code.N, q=code.q, **fer(code, n_m, frames, points))
        code.close()
    s = json.dumps(line)
    print(s)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
