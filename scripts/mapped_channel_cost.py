"""Cost of the mapped channel (one GF(q) symbol per point of a q-point constellation) on one B200, against BPSK on the same
code: the decode kernel with the mapped intake, the device frame source, and the Monte-Carlo driver.

    python scripts/mapped_channel_cost.py [--reps 7] [--warmup 2] [--out FILE]   (default FILE: profiles/r03c_mapped_channel_cost.json)

Workloads: config 5 (AD_64800_R12_GF256, GF(256), 256-QAM) and config 4 (Ahmed_64800_R34_GF16, GF(16), 16-QAM), as seeded
stand-ins of tests/common.code_path when the files are absent; n_m and iterations as bench.py, batches of two whole waves of
the persistent grid (geometry()), fixed-iteration mode.
  * decode: nbgpu_run on the resident batch (generated on the device), CUDA events, median of the repetitions; the mapped and
    the BPSK batch alternate inside every repetition.  The mapped intake does 2q f64 divisions per symbol.
  * source: one nbgpu_source_frames_mapped / nbgpu_source_frames call (encoder + noise kernel + flag read-back + host fix-up),
    CUDA events around the call, with the fix-up count; alternated the same way, each call on a new block of frames.
  * driver: frames/s of `nbldpc_mc ... <source 1> <channel>` with channel 2 (square QAM) and channel 0 (BPSK), three batches.
Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import nbldpc                      # noqa: E402
from common import MATRIX_DIRS, code_path       # noqa: E402

# (matrix, n_m, Eb/N0 of BPSK, Es/N0 of QAM): points where most frames converge; fixed-iteration mode makes the decode time
# independent of them
CONFIGS = {"config5": ("matrices/AD_64800_R12_GF256", 20, 1.5, 20.0), "config4": ("matrices/Ahmed_64800_R34_GF16", 16, 3.0, 12.0)}
NB_OPER, OFFSET, NB_ITER_MAX = 25, 0.3, 10
WAVES = 2
EXE = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    name, limit = [x.strip() for x in out.split(",")]
    return name, limit


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs)}


def cost(code, n_m, ebn, esn, reps, warmup):
    d = nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=1 << 14)
    g = d.geometry()
    B = WAVES * g["grid"] * g["frames_per_cta"]
    d.close()
    d = nbldpc.Decoder(code, n_m, NB_OPER, NB_ITER_MAX, OFFSET, early_stop=False, max_batch=B)
    d.set_constellation(nbldpc.constellation(nbldpc.MAP_QAM, code.q))
    calls = {"bpsk": (d.source_frames, ebn), "mapped": (d.source_frames_mapped, esn)}
    src, fix, dec = ({ch: [] for ch in calls} for _ in range(3))
    for r in range(warmup + reps):
        for ch, (fn, e) in calls.items():
            d.sync()
            d.timer_begin()
            fn(r * B, B, e)
            ms = d.timer_end()
            d.run()
            d.sync()
            if r < warmup:
                continue
            src[ch].append(ms); fix[ch].append(d.source_fixups()); dec[ch].append(d.last_kernel_ms())
    out = {"frames": B, "geometry": g, "reps": reps, "n_m": n_m, "channels": {}}
    for ch, (_, e) in calls.items():
        out["channels"][ch] = {"ebn": e, "decode_kernel_ms": spread(dec[ch]), "source_event_ms": spread(src[ch]),
                               "source_ns_per_frame": statistics.median(src[ch]) * 1e6 / B, "fixups": fix[ch]}
    out["mapped_over_bpsk_decode_time"] = statistics.median(dec["mapped"]) / statistics.median(dec["bpsk"])
    out["mapped_over_bpsk_source_time"] = statistics.median(src["mapped"]) / statistics.median(src["bpsk"])
    d.close()
    return out


def driver(path, n_m, ebn, esn, B):
    """frames/s of the C driver with the device source: channel 2 (square QAM) against channel 0 (BPSK)"""
    res = {}
    for channel, e in ((2, esn), (0, ebn)):
        with tempfile.TemporaryDirectory() as tmp:
            os.makedirs(os.path.join(tmp, "data"))
            args = [EXE, str(3 * B), str(NB_ITER_MAX), path, "%g" % e, str(n_m), str(OFFSET), str(NB_OPER), str(B), "0", "0", "1", str(channel)]
            r = subprocess.run(args, cwd=tmp, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=3000)
            if r.returncode != 0:
                raise SystemExit("nbldpc_mc failed:\n" + r.stdout[-2000:])
            m = re.search(r"frame source: (\d+) frames in ([\d.]+) s = ([\d.]+) frames/s", r.stdout)
            last = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+).*?avr_it=([\d.]+)", r.stdout)[-1]
            res["channel%d" % channel] = {"ebn": e, "frames": int(m.group(1)), "seconds": float(m.group(2)), "frames_per_s": float(m.group(3)),
                                          "err_frames": int(last[1]), "avr_it": float(last[3])}
    res["args"] = "nbldpc_mc %d %d <matrix> <EbN> %d %g %d %d 0 0 1 <channel>" % (3 * B, NB_ITER_MAX, n_m, OFFSET, NB_OPER, B)
    res["qam_over_bpsk_frames_per_s"] = res["channel2"]["frames_per_s"] / res["channel0"]["frames_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03c_mapped_channel_cost.json"))
    args = ap.parse_args()
    if nbldpc.device_count() < 1:
        raise SystemExit("mapped_channel_cost.py needs a B200: nothing is measured without one")
    name, limit = card()
    line = {"card": name, "power_limit": limit, "iterations": NB_ITER_MAX}
    for key, (rel, n_m, ebn, esn) in CONFIGS.items():
        path = code_path(rel)
        code = nbldpc.Code(path)
        standin = all(os.path.join(m, rel) != path for m in MATRIX_DIRS)
        c = cost(code, n_m, ebn, esn, max(3, args.reps), args.warmup)
        line[key] = {"matrix": "seeded stand-in for %s (tests/common.code_path)" % rel if standin else rel, "N": code.N, "q": code.q,
                     "constellation": "Gray square %d-QAM" % code.q, "cost": c, "driver": driver(path, n_m, ebn, esn, c["frames"])}
        code.close()
    s = json.dumps(line)
    print(s)
    with open(args.out, "w") as f:
        f.write(s + "\n")


if __name__ == "__main__":
    main()
