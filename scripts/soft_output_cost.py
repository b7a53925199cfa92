"""Cost of the soft output (nbgpu_set_soft_output) on one B200: kernel time of nbgpu_run with soft output NONE, LIST k = 1,
LIST k = n_m and BITS, alternated over the repetitions, and the host time of bringing the whole batch's soft output back.

    python scripts/soft_output_cost.py [--reps 7] [--warmup 2] [--out FILE]

Workloads as bench.py runs them: fixed-iteration mode (10 iterations, early termination off), whole waves of the persistent
grid; the 64800-bit matrices are the seeded stand-ins of tests/common.code_path when the files are absent.  Prints one JSON
line (and writes it to --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nbldpc                      # noqa: E402
from common import MATRIX_DIRS, code_path       # noqa: E402

# name -> (matrix, n_m, nb_oper, offset, Eb/N0, frames): bench.py's configs 5 and 4
WORKLOADS = {"AD_64800_R12_GF256": ("matrices/AD_64800_R12_GF256", 20, 25, 0.3, 2.0, 2368),
             "Ahmed_64800_R34_GF16": ("matrices/Ahmed_64800_R34_GF16", 16, 25, 0.3, 3.0, 4144)}
NB_ITER_MAX = 10


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def frames(code, B, ebn, pool=8, seed=5):
    """pool codewords of the product's encoder, BPSK, white Gaussian noise of the reference's sigma (one draw per frame)"""
    code.prepare_encoder()
    code.rng_default()
    bits = np.stack([code.random_codeword()[1] for _ in range(pool)])
    sigma = code.sigma(ebn)
    rng = np.random.default_rng(seed)
    tx = 1.0 - 2.0 * bits[rng.integers(0, pool, B)].astype(np.float32)
    return (tx + np.float32(sigma) * rng.standard_normal(tx.shape, dtype=np.float32)).astype(np.float32), sigma


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def measure(wl, reps, warmup):
    rel, n_m, nb_oper, offset, ebn, B = WORKLOADS[wl]
    path = code_path(rel)
    code = nbldpc.Code(path)
    noisy, sigma = frames(code, B, ebn)
    d = nbldpc.Decoder(code, n_m, nb_oper, NB_ITER_MAX, offset, early_stop=False, max_batch=B)
    kinds = [("none", nbldpc.SOFT_NONE, 0), ("list_k1", nbldpc.SOFT_LIST, 1), ("list_k%d" % n_m, nbldpc.SOFT_LIST, n_m),
             ("bits", nbldpc.SOFT_BITS, 0)]
    d.upload_noisy(noisy, sigma)
    d.sync()
    ms = {name: [] for name, _, _ in kinds}
    dl = {name: [] for name, kind, _ in kinds if kind != nbldpc.SOFT_NONE}
    for r in range(warmup + reps):
        for name, kind, k in kinds:                     # alternate the kinds inside every repetition
            d.set_soft_output(kind, k)                  # (re)allocates the output: outside the timed launch
            d.run()
            d.sync()
            if r < warmup:
                continue
            ms[name].append(d.last_kernel_ms())
            if kind != nbldpc.SOFT_NONE:
                t0 = time.perf_counter()
                d.soft_list() if kind == nbldpc.SOFT_LIST else d.soft_bits()
                dl[name].append((time.perf_counter() - t0) * 1e3)
    info_bits = code.info_bits * B
    standin = all(os.path.join(m, rel) != path for m in MATRIX_DIRS)
    res = {"matrix": "seeded stand-in for %s (tests/common.code_path)" % rel if standin else rel,
           "N": code.N, "q": code.q, "n_m": n_m, "frames": B, "iterations": NB_ITER_MAX, "early_stop": False, "reps": reps,
           "geometry": d.geometry(), "kinds": {}}
    for name, kind, k in kinds:
        per = k if kind == nbldpc.SOFT_LIST else code.logq if kind == nbldpc.SOFT_BITS else 0
        e = {"kernel_ms": spread(ms[name]), "mbit_s": spread([info_bits / (x * 1e3) for x in ms[name]]),
             "overhead_vs_none_pct": spread([100.0 * (x / y - 1.0) for x, y in zip(ms[name], ms["none"])]),
             "soft_bytes_per_frame": code.N * per * (5 if kind == nbldpc.SOFT_LIST else 4)}
        if name in dl:
            e["download_host_ms"] = spread(dl[name])
        res["kinds"][name] = e
    d.close(); code.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("soft_output_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    line = {"card": name, "power_limit": limit, "workloads": {wl: measure(wl, max(5, args.reps), args.warmup) for wl in WORKLOADS}}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
