#!/usr/bin/env python3
"""bench.py -- decoded info Mbit/s of the EMS NB-LDPC decode path at fixed iterations (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--frames B]

A *step* is one pass of the hot path (NB_LDPC.c:266-474: intake, NbIterMax-1 layered EMS passes, decision,
syndrome) over one batch of B synthetic frames per GPU.  One process per GPU (torchrun for N > 1); frames are
independent, so the batch shards by frame with no data-path collective ("weak" scaling: B per GPU is fixed) and
NCCL is used only for the barrier, the max-over-ranks time and one final all-reduce of the frame counters.

`value`    whole-job info Mbit/s with the noisy frames already resident in HBM (device time, CUDA events).
`e2e`      the same metric through the reference-facing C-ABI call nbgpu_decode_noisy with HOST buffers: H2D of the
           received samples from pinned memory, decode, D2H of decisions/syndromes/iteration counts, every step.
`roofline` HBM model of DESIGN.md section 4 for the decode kernel (the only kernel in a step).
`cpu_baseline` / `--impl reference`  the reference's own CPU decoder (oracle/_ref/essai_probe = unmodified
           NB_LDPC.c main loop, decode time only, Syndrom forced non-zero so all passes run) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)          # the product binding (nbldpc.py); tests/ and oracle/ stay off the product arm's path

# name -> (matrix, n_m, nb_oper, offset, Eb/N0, default frames per GPU per step)        (SURVEY.md section 8d)
# The default batch is a whole number of waves of the persistent grid (296 CTAs x frames per CTA group: 1 for the 64800-bit
# GF(256) / GF(16) codes, 8 for MatDeclercq, 4 for Mat24): a partial last wave leaves SMs idle (MatDeclercq at 4096 frames =
# 1.73 waves measured 197 Mbit/s, at 2368 or 4736 frames 226).
WORKLOADS = {
    "AD_64800_R12_GF256": ("matrices/AD_64800_R12_GF256", 20, 25, 0.3, 2.0, 2368),
    "Ahmed_64800_R34_GF16": ("matrices/Ahmed_64800_R34_GF16", 16, 25, 0.3, 3.0, 4144),
    "MatDeclercq_R12_GF64": ("matrices/MatDeclercq_R12_GF64", 20, 25, 0.3, 1.2, 4736),
    "Mat24_N480_M240": ("matrices/Mat24_N480_M240", 16, 25, 0.3, 1.5, 66304),
    "N96_K48_GF64": ("matrices/N96_K48_GF64", 20, 25, 0.3, 3.0, 1 << 20),
    # full-alist file shipped with the reference, which its own LoadCode cannot read (SURVEY.md 8f.4): no CPU arm for it
    "KN_64800_R34_GF256": ("matrices/KN/N64800_K48600_GF256.txt", 20, 25, 0.3, 3.4, 2368),
}
NO_REFERENCE = {"KN_64800_R34_GF256"}
# index of the workload in BASELINE.json "configs" (1-based, as SURVEY.md section 8d numbers them)
BASELINE_CONFIG = {"N96_K48_GF64": 1, "Mat24_N480_M240": 2, "MatDeclercq_R12_GF64": 3, "Ahmed_64800_R34_GF16": 4, "AD_64800_R12_GF256": 5}
NB_ITER_MAX = 10
# syndrome_ems parameters (d1, d2, d3, truncation, n_cv): the shapes of the commented call site NB_LDPC.c:185-201 with
# d1 capped at n_m-1 (its d_1 = 40 overruns the n_m-wide message rows); see DESIGN.md "Syndrome path"
SYND = {20: (19, 15, 5, 1000, 25), 16: (15, 15, 5, 1000, 25)}
SYND_FRAMES = {"AD_64800_R12_GF256": 592, "MatDeclercq_R12_GF64": 592, "Mat24_N480_M240": 16384, "N96_K48_GF64": 1 << 18}
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
# (N, M, GF, dc) of each workload's code, all with column degree 2.  Only the small matrices ship in matrices/ (see its README);
# a workload whose file is absent decodes a seeded random code of this shape instead, so that the kernels see the same sizes,
# degrees and field.  The JSON line names the code that ran under "matrix".
STANDIN = {"AD_64800_R12_GF256": (8100, 4050, 256, 4), "Ahmed_64800_R34_GF16": (16200, 4050, 16, 8),
           "MatDeclercq_R12_GF64": (10800, 5400, 64, 4), "Mat24_N480_M240": (480, 240, 64, 4),
           "KN_64800_R34_GF256": (8100, 2025, 256, 8)}
STANDIN_SEED = 2024
_standin_dir = None


def find_matrix(rel):
    for d in (ROOT, REF_DIR):
        p = os.path.join(d, rel)
        if os.path.exists(p):
            return p
    raise FileNotFoundError("%s found neither in matrices/ nor in oracle/_ref" % rel)


def write_standin(path, N, M, q, dc, seed):
    """UBS alist of a random code, every column in 2 checks, no column twice in a check, non-zero coefficients."""
    rng = np.random.default_rng(seed)
    rows = rng.permutation(np.repeat(np.arange(N), 2)).reshape(M, dc)
    while True:
        bad = [m for m in range(M) if len(set(rows[m])) < dc]
        if not bad:
            break
        for m in bad:                                  # swap one slot of the row with a random slot anywhere
            k, m2, k2 = int(rng.integers(dc)), int(rng.integers(M)), int(rng.integers(dc))
            rows[m, k], rows[m2, k2] = rows[m2, k2], rows[m, k]
    val = rng.integers(1, q, (M, dc))
    with open(path, "w") as f:
        f.write("%d %d %d\n%s\n%s\n" % (N, M, q, " ".join(["2"] * N), " ".join([str(dc)] * M)))
        f.write("".join(" ".join(map(str, r)) + "\n" for r in rows))
        f.write("".join(" ".join(map(str, r)) + "\n" for r in val))


def workload_matrix(wl):
    """(path, description) of the code of workload wl: its matrix file, or the seeded stand-in written to a temporary directory."""
    rel = WORKLOADS[wl][0]
    try:
        return find_matrix(rel), rel
    except FileNotFoundError:
        pass
    global _standin_dir
    if _standin_dir is None:
        import atexit
        import shutil
        _standin_dir = tempfile.mkdtemp(prefix="nbldpc_bench_")
        atexit.register(shutil.rmtree, _standin_dir, True)
    N, M, q, dc = STANDIN[wl]
    path = os.path.join(_standin_dir, wl)
    if not os.path.exists(path):
        write_standin(path, N, M, q, dc, STANDIN_SEED)
    return path, "random stand-in for %s (absent): N=%d, M=%d, GF(%d), dv=2, dc=%d, seed %d" % (rel, N, M, q, dc, STANDIN_SEED)


def bytes_per_frame(N, E, q, n_m, passes, ecn="bubble"):
    """Algorithmic HBM bytes of one frame (SURVEY.md 8d / DESIGN.md 4): dense f32 APP rows read+written once per edge
    visit, CtoV read+written once per edge visit (lossless record for the bubble check node, dense row for syndrome_ems
    whose output is not a truncated list), intake write, decisions."""
    ctov = q * 4 if ecn == "syndrome" else min(q * 4, 5 * n_m + 4)
    return N * q * 4 + passes * E * (2 * q * 4 + 2 * ctov) + N


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.3 and len(r) >= 7] or [r for (_, r) in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == "Active" for r in rows)]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(rows[0][1]) if rows[0][1].isdigit() else None,
                "power_w_max": max(pw) if pw else None, "samples": len(rows), "reasons": reasons}


# -----------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the unmodified reference main loop on the host cores
# -----------------------------------------------------------------------------------------------------------------
def run_reference_cpu(wl, frames_per_proc, procs, seconds_hint=None, ecn="bubble"):
    """Runs `procs` concurrent copies of the reference (it is single-threaded; start.sh does the same) and returns
    (aggregate frames/s over decode time, kind, sample description, wall seconds)."""
    matrix, n_m, nb_oper, offset, ebn, _ = WORKLOADS[wl]
    exe = os.path.join(REF_DIR, "essai_probe")
    if os.path.exists(exe):
        with tempfile.TemporaryDirectory() as td:
            os.makedirs(os.path.join(td, "data"), exist_ok=True)
            os.symlink(os.path.join(REF_DIR, "matrices"), os.path.join(td, "matrices"))
            ps = []
            t0 = time.time()
            for i in range(procs):
                env = dict(os.environ, NBREF_FORCE="1", NBREF_LEVEL="0", NBREF_DIALECT="ubs",
                           NBREF_SUMMARY=os.path.join(td, "sum%d.txt" % i))
                env.pop("NBREF_TRACE", None)
                env.pop("NBREF_ECN", None)
                if ecn == "syndrome":
                    env["NBREF_ECN"] = "syndrome"
                    env["NBREF_SYND"] = ",".join(str(x) for x in SYND[n_m])
                ps.append(subprocess.Popen([exe, str(frames_per_proc), str(NB_ITER_MAX), matrix, str(ebn), str(n_m), str(offset),
                                            str(nb_oper)], cwd=td, env=env, stdin=subprocess.DEVNULL, stdout=subprocess.DEVNULL,
                                           stderr=subprocess.DEVNULL))
            for p in ps:
                p.wait()
            wall = time.time() - t0
            rate = 0.0
            nfr = 0
            for i in range(procs):
                fr, dec_s, ch_s, passes = open(os.path.join(td, "sum%d.txt" % i)).read().split()[:4]
                assert int(passes) == int(fr) * (NB_ITER_MAX - 1), "reference did not run the fixed number of passes"
                rate += int(fr) / float(dec_s)
                nfr += int(fr)
        sample = "%d concurrent single-thread runs of the unmodified reference main loop (oracle/_ref/essai_probe%s), %d frames each, " \
                 "decode time only (channel return -> last Syndrom), Syndrom forced non-zero -> %d passes/frame" % (
                     procs, ", check node = the reference's syndrome_ems" if ecn == "syndrome" else "", frames_per_proc, NB_ITER_MAX - 1)
        return rate, "reference", sample, wall, nfr
    # fallback: the oracle port (plain-C restatement), same sampling
    import multiprocessing as mp
    t0 = time.time()
    with mp.Pool(procs) as pool:
        res = pool.map(_port_worker, [(wl, frames_per_proc, i, ecn) for i in range(procs)])
    wall = time.time() - t0
    rate = sum(f / s for f, s in res)
    sample = "%d processes of the oracle port (oracle/liboracle.so), %d frames each, decode time only, %d passes/frame" % (
        procs, frames_per_proc, NB_ITER_MAX - 1)
    return rate, "port", sample, wall, procs * frames_per_proc


def _port_worker(arg):
    wl, frames, idx, ecn = arg
    sys.path.insert(0, os.path.join(ROOT, "tests"))          # the oracle port: cpu_baseline fallback only, never the product arm
    import oracle_lib as ol
    matrix, n_m, nb_oper, offset, ebn, _ = WORKLOADS[wl]
    o = ol.Oracle(workload_matrix(wl)[0])
    kw = {}
    if ecn == "syndrome":
        d1, d2, d3, trunc, n_cv = SYND[n_m]
        kw = dict(ecn=1, cfg=o.build_config_table(int(o.row_deg[0]), d1, d2, d3, trunc), n_cv=n_cv)
    rng = np.random.default_rng(idx)
    sigma = o.sigma(ebn)
    tot = 0.0
    for _ in range(frames):
        noisy = (1.0 + sigma * rng.standard_normal((o.N, o.logGF))).astype(np.float32)
        llr = o.channel_llr(noisy, sigma)
        t0 = time.perf_counter()
        o.decode_frame(llr, n_m, nb_oper, NB_ITER_MAX, offset, force=True, **kw)
        tot += time.perf_counter() - t0
    return frames, tot


def cpu_sample_size(wl, ecn="bubble"):
    """frames per process so that one concurrent batch is roughly 10-30 s of CPU work per core"""
    n = {"AD_64800_R12_GF256": 4, "Ahmed_64800_R34_GF16": 10, "MatDeclercq_R12_GF64": 10, "Mat24_N480_M240": 400,
         "N96_K48_GF64": 10000}[wl]
    return max(1, n // 6) if ecn == "syndrome" else n


class AlistHeader:
    """N, M, GF and the check degree read from the matrix file itself: the reference arm must not load the product library."""
    def __init__(self, path):
        tok = open(path).read().split()
        self.N, self.M, self.q = int(tok[0]), int(tok[1]), int(tok[2])
        self.logq = self.q.bit_length() - 1
        self.info_bits = (self.N - self.M) * self.logq          # the reference exits when H is rank deficient (tools.c:181-185)
        self.dc_max = max(int(x) for x in tok[3 + self.N:3 + self.N + self.M])
        self.dc_min = min(int(x) for x in tok[3 + self.N:3 + self.N + self.M])


def reference_arm(args, rank, world):
    """The reference's own CPU decoder (unmodified main loop) on all host cores; rank 0 only.  --steps/--warmup are honoured:
    a step is one concurrent batch of `cores` single-thread processes, sized after a calibration run so that the whole
    arm ends within a few minutes."""
    if rank != 0:
        return
    wl = args.workload
    matrix, n_m, nb_oper, offset, ebn, _ = WORKLOADS[wl]
    code = AlistHeader(workload_matrix(wl)[0])
    cores = host_cores()
    budget_s = float(os.environ.get("NBLDPC_REF_BUDGET_S", "240"))
    # calibration (also the first warm-up step): one frame per process
    c0 = time.time()
    run_reference_cpu(wl, 1, cores, ecn=args.ecn)
    per_frame_s = max(time.time() - c0, 1e-3)
    warm = max(args.warmup, 1)
    fpp = int(max(1, min(cpu_sample_size(wl, args.ecn) * 4, (budget_s - warm * per_frame_s) / (args.steps * per_frame_s))))
    for _ in range(warm - 1):
        run_reference_cpu(wl, 1, cores, ecn=args.ecn)
    rates, walls, frames = [], [], 0
    for _ in range(args.steps):
        rate, kind, sample, wall, nfr = run_reference_cpu(wl, fpp, cores, ecn=args.ecn)
        rates.append(rate); walls.append(wall); frames += nfr
    fps = statistics.mean(rates)
    val = fps * code.info_bits / 1e6
    sample += "; %d timed steps (%d frames per process in total, %d frames over all cores), %d warm-up steps of 1 frame per process" % (
        args.steps, fpp * args.steps, frames, warm)
    line = {"impl": "reference", "metric": "decoded info Mbit/s at fixed iterations (%d passes)" % (NB_ITER_MAX - 1), "value": val,
            "unit": "Mbit/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(walls),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (reference's own drand48 frame stream)",
            "frames_per_s": fps,
            "config": config_dict(wl, code, fpp * cores, "host CPU only", args.ecn),
            "cpu_baseline": {"value": val, "unit": "Mbit/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "Mbit/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(line)


def config_dict(wl, code, frames, note, ecn="bubble"):
    matrix, n_m, nb_oper, offset, ebn, _ = WORKLOADS[wl]
    if ecn == "syndrome":
        cn = "syndrome-based check node (syndrome_ems with presorting, d=(%d,%d,%d), %d configurations max, n_cv=%d)" % SYND[n_m]
    else:
        cn = "L-Bubble forward/backward EMS check node (CheckPassLogEMS), nbOper=%d" % nb_oper
    idx = BASELINE_CONFIG.get(wl)
    which = "BASELINE.json configs[%d] (config %d of SURVEY.md 8d) = " % (idx - 1, idx) if idx else "extra workload (not in BASELINE.json) = "
    if idx == 5:
        which += "as written (syndrome_decoder path) " if ecn == "syndrome" else "with the reference's shipped check node (NB_LDPC.c:392) "
    return {"workload": which + "%s: N=%d symbols over GF(%d) (%d code bits, %d info bits), M=%d, dc=%d, %s, n_m=%d, offset=%.1f, "
                        "NbIterMax=%d (= %d passes, early termination off), AWGN BPSK Eb/N0=%.1f dB"
                        % (wl, code.N, code.q, code.N * code.logq, code.info_bits, code.M, code.dc_max, cn, n_m, offset, NB_ITER_MAX,
                           NB_ITER_MAX - 1, ebn),
            "baseline_config": idx, "check_node": ecn, "frames_per_step_per_gpu": frames, "cache": note}


# -----------------------------------------------------------------------------------------------------------------
# our arm
# -----------------------------------------------------------------------------------------------------------------
def synth_frames(code, B, ebn, seed, pool=8):
    """B received frames: `pool` codewords from the product's encoder (reference frame source), BPSK, plus white Gaussian
    noise of the reference's sigma drawn with numpy (distinct per frame and per rank)."""
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(seed * 7919)
    bits = np.stack([code.random_codeword()[1] for _ in range(pool)])            # [pool, N, logq]
    sigma = code.sigma(ebn)
    rng = np.random.default_rng(1000 + seed)
    idx = rng.integers(0, pool, B)
    noisy = np.empty((B, code.N, code.logq), np.float32)
    for lo in range(0, B, 256):
        hi = min(B, lo + 256)
        tx = 1.0 - 2.0 * bits[idx[lo:hi]].astype(np.float32)
        noisy[lo:hi] = tx + np.float32(sigma) * rng.standard_normal(tx.shape, dtype=np.float32)
    return noisy, bits[idx], sigma


def git_head():
    """Commit of the tree when .git is there; on the GPU box (a snapshot without history) a hash of the kernel sources,
    so that a traffic capture can still be tied to the code it measured."""
    try:
        h = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short=12", "HEAD"], capture_output=True, text=True).stdout.strip()
        if h:
            return h
    except OSError:
        pass
    return "src-" + source_id()


def source_id():
    import glob
    import hashlib
    m = hashlib.sha1()
    for f in sorted(glob.glob(os.path.join(ROOT, "ems-decoder-of-nb-ldpc-codes_b200", "csrc", "*.[ch]*")) +
                    glob.glob(os.path.join(ROOT, "include", "*.h"))):
        m.update(open(f, "rb").read())
    return m.hexdigest()[:12]


def measured_traffic(wl, ecn, B, kernel_ms):
    """DRAM bytes per launch of the decode kernel from an ncu capture (profiles/traffic_<workload>_<ecn>.json, written by
    scripts/gpu_traffic.sh).  Only a capture of THIS kernel counts: same workload, check node and frames per launch, and a
    kernel duration within 3 % of the one measured live, and the same kernel sources (hash of csrc/ + include/) -- otherwise the
    figure is stale and null is reported."""
    tp = os.path.join(ROOT, "profiles", "traffic_%s_%s.json" % (wl, ecn))
    if not os.path.exists(tp):
        return None, None
    tj = json.load(open(tp))
    if tj.get("frames") != B or tj.get("ecn") != ecn or not tj.get("kernel_ms"):
        return None, {"capture": os.path.basename(tp), "rejected": "other launch size or check node"}
    dev = abs(tj["kernel_ms"] - kernel_ms) / kernel_ms
    info = {"capture": os.path.basename(tp), "git": tj.get("git"), "source_id": tj.get("source_id"), "source_id_now": source_id(),
            "kernel_ms_at_capture": tj["kernel_ms"], "kernel_ms_deviation": dev}
    if dev > 0.03:
        info["rejected"] = "kernel duration differs by more than 3 % from the live measurement: capture is stale"
        return None, info
    if tj.get("source_id") and tj["source_id"] != info["source_id_now"]:
        info["rejected"] = "captured from other kernel sources (hash of csrc/ + include/ differs): capture is stale"
        return None, info
    return tj.get("dram_bytes_per_launch"), info


def measure_leg(nbldpc, code, wl, ecn, B, args, rank, local_rank, world, dist, noisy, bits, sigma, out, with_sim):
    """One check node on one workload: resident-input throughput, end-to-end throughput through the C ABI with host buffers,
    roofline of the decode kernel, counters.  Same steps / warm-up for every leg."""
    matrix, n_m, nb_oper, offset, ebn, _ = WORKLOADS[wl]
    passes = NB_ITER_MAX - 1
    kw = {}
    if ecn == "syndrome":
        d1, d2, d3, trunc, n_cv = SYND[n_m]
        kw = dict(ecn_kind=1, d1=d1, d2=d2, d3=d3, cfg_trunc=trunc, n_cv=n_cv)
    dec = nbldpc.Decoder(code, n_m, nb_oper, NB_ITER_MAX, offset, early_stop=False, device=local_rank, max_batch=B,
                         frames_per_cta=args.frames_per_cta, cns_per_step=args.cns_per_step, **kw)
    geo = dec.geometry()
    noisy = noisy[:B]
    out = tuple(o[:B] for o in out)

    def barrier():
        if dist is not None:
            dist.barrier()

    def maxr(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- resident-input throughput (`value`) ----------------
    dec.upload_noisy(noisy, sigma)
    dec.sync()
    for _ in range(args.warmup):
        dec.run()
    dec.sync()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    l0 = dec.launch_count()
    t0 = time.time()
    kms = []
    dec.timer_begin()
    for _ in range(args.steps):
        dec.run()
    ms = dec.timer_end()
    t1 = time.time()
    barrier()
    d_res, s_res, it_res = dec.download()              # what the last timed step computed
    launches = dec.launch_count() - l0
    clocks = sampler.stop(t0, t1) if sampler else None
    ms = maxr(ms)
    # per-launch duration of the decode kernel (CUDA events on the launching stream), outside the timed region
    for _ in range(min(3, args.steps)):
        dec.run()
        kms.append(dec.last_kernel_ms())
    kernel_ms = statistics.mean(kms)
    frames_total = world * B * args.steps
    fps = frames_total / (ms / 1e3)
    value = fps * code.info_bits / 1e6

    # ---------------- end to end through the C ABI with host buffers (`e2e`) ----------------
    for _ in range(max(1, min(args.warmup, 2))):
        dec.decode_noisy_into(noisy, sigma, out)
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        dec.decode_noisy_into(noisy, sigma, out)
    e2e_s = maxr(time.perf_counter() - e0)
    barrier()
    e2e_val = frames_total / e2e_s * code.info_bits / 1e6
    assert (out[0] == d_res).all() and (out[2] == it_res).all(), "e2e and resident runs disagree"

    # ---------------- whole simulation step on the device (SURVEY 8f.1): frame source -> decode -> error count ----------------
    sim = None
    if with_sim:
        dec.source_frames(rank * B, B, ebn)
        dec.run(); dec.source_results()
        nsim = min(args.steps, 3)
        barrier()
        s0 = time.perf_counter()
        for i in range(nsim):
            dec.source_frames((world * (i + 1) + rank) * B, B, ebn)
            dec.run()
            dec.source_results()
        sim_s = maxr(time.perf_counter() - s0)
        barrier()
        sim = {"value": world * B * nsim / sim_s * code.info_bits / 1e6, "unit": "Mbit/s", "steps": nsim, "ms_per_step": 1e3 * sim_s / nsim,
               "d2h_bytes_per_step": 12 * B, "h2d_bytes_per_step": 0, "host_fixups_last_step": dec.source_fixups(),
               "note": "Monte-Carlo step with the frames of the reference's drand48 stream generated, decoded (fixed iterations) and scored on the "
                       "device: nbgpu_source_frames + nbgpu_run + nbgpu_source_results"}

    # ---------------- counters: one all-reduce (the only collective of the path) ----------------
    bit_err = int((bits[:B, :code.K, :] != np.stack([code_bits(code, d_res[:, k]) for k in range(code.K)], axis=1)).sum()) if args.count_errors else -1
    counters = np.array([B, int((s_res != 0).sum()), int(it_res.sum()), bit_err], np.int64)
    counters = nbldpc.multigpu.allreduce_counters(counters, device="cuda" if dist is not None else None)

    # ---------------- sharding check (N > 1): frames [0, N*Bc) of the reference's stream generated on the devices, one block per
    # rank, early termination on; the all-reduced counters must equal those of ONE GPU decoding the same range ----------------
    shard = None
    if world > 1 and ecn == "bubble":
        Bc = min(B, 296)
        dchk = nbldpc.Decoder(code, n_m, nb_oper, NB_ITER_MAX, offset, early_stop=True, device=local_rank, max_batch=Bc)

        def block(r):
            dchk.source_frames(r * Bc, Bc, ebn)
            dchk.run()
            e, sy, it = dchk.source_results()
            return np.array([Bc, int((e != 0).sum()), int(((e != 0) & (sy == 0)).sum()), int(e.sum()), int(it.sum())], np.int64)

        mine = nbldpc.multigpu.allreduce_counters(block(rank), device="cuda")
        if rank == 0:
            alone = sum(block(r) for r in range(world))
            shard = {"frames": int(world * Bc), "counters": ["frames", "erroneous_frames", "undetected", "bit_errors", "sum_iterations"],
                     "all_reduced": [int(x) for x in mine], "single_gpu_same_range": [int(x) for x in alone],
                     "equal": bool((np.asarray(mine) == alone).all())}
        dchk.close()
        barrier()

    leg = None
    if rank == 0:
        bpf = bytes_per_frame(code.N, code.E, code.q, n_m, passes, ecn)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = bpf * B / (kernel_ms / 1e3) / 1e9
        traffic, tinfo = measured_traffic(wl, ecn, B, kernel_ms)
        slot_bytes = code.N * code.q * 4 + code.E * (code.q * 4 if ecn == "syndrome" else (5 * n_m + 8 + 15) // 16 * 16)
        leg = {"value": value, "unit": "Mbit/s", "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "frames_per_s": fps,
               "config": config_dict(wl, code, B, "per-step working set %.1f GB and inputs %.0f MB per GPU, both larger than the 126 MB L2 (no explicit flush)"
                                     % (geo["slots"] * slot_bytes / 1e9, noisy.nbytes / 1e6), ecn),
               "geometry": geo,
               "e2e": {"value": e2e_val, "unit": "Mbit/s", "h2d_bytes_per_step": int(noisy.nbytes), "d2h_bytes_per_step": int(sum(o.nbytes for o in out)),
                       "ms_per_step": 1e3 * e2e_s / args.steps},
               "gpu_launches": int(launches),
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                            "traffic_source": tinfo,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                            "kernel": "decode_kernel<%d, closed, %s>" % (code.q, "syndrome_ems" if ecn == "syndrome" else "CheckPassLogEMS"),
                            "kernel_ms": kernel_ms, "bytes_per_frame": bpf, "frames_per_launch": B},
               "clocks": clocks, "simulation": sim,
               "counters": {"frames_per_step": int(counters[0]), "frames_nonzero_syndrome": int(counters[1]), "sum_iterations": int(counters[2]),
                            "slow_path_selects": dec.slow_selects()}}
        if shard is not None:
            leg["sharding_check"] = shard
        leg["outputs"] = {"decide": d_res, "syndrome": s_res, "iterations": it_res}
    dec.close()
    return leg


def ours(args, rank, local_rank, world):
    import nbldpc
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if nbldpc.device_count() < 1:
        raise RuntimeError("bench.py needs a B200: the product has no CPU fallback")
    wl = args.workload
    matrix, n_m, nb_oper, offset, ebn, dflt_B = WORKLOADS[wl]
    path, matrix_desc = workload_matrix(wl)
    code = nbldpc.Code(path)
    synd_ok = n_m in SYND and code.dc_min == code.dc_max and 4 <= code.dc_max <= 8
    B_of = {"bubble": args.frames or dflt_B, "syndrome": args.frames or SYND_FRAMES.get(wl, dflt_B)}
    # the headline leg is the check node asked for; the default run carries the other one of the workload as a second, complete leg
    legs = [args.ecn]
    if not args.no_also and synd_ok and wl in BASELINE_CONFIG:
        legs.append("syndrome" if args.ecn == "bubble" else "bubble")
    Bmax = max(B_of[e] for e in legs)
    noisy, bits, sigma = synth_frames(code, Bmax, ebn, rank)
    nbldpc.pin(noisy)
    out = (nbldpc.pin(np.zeros((Bmax, code.N), np.int32)), nbldpc.pin(np.zeros(Bmax, np.int32)), nbldpc.pin(np.zeros(Bmax, np.int32)))
    res = {}
    for i, ecn in enumerate(legs):
        res[ecn] = measure_leg(nbldpc, code, wl, ecn, B_of[ecn], args, rank, local_rank, world, dist, noisy, bits, sigma, out, with_sim=(i == 0 and not args.no_also))
    if rank == 0:
        passes = NB_ITER_MAX - 1
        head = res[legs[0]]
        line = {"metric": "decoded info Mbit/s at fixed iterations (%d passes)" % passes, "value": head["value"], "unit": "Mbit/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic (encoder codewords + numpy Gaussian noise at the reference's sigma)",
                "git": git_head(), "source_id": source_id(), "matrix": matrix_desc}
        for k in ("frames_per_s", "config", "geometry", "e2e", "gpu_launches", "roofline", "clocks", "simulation", "counters", "sharding_check"):
            if k in head:
                line[k] = head[k]
        if world == 1 and not args.no_cpu and wl not in NO_REFERENCE:
            cores = host_cores()
            for ecn in legs:
                rate, kind, sample, wall, nfr = run_reference_cpu(wl, cpu_sample_size(wl, ecn), cores, ecn=ecn)
                res[ecn]["cpu_baseline"] = {"value": rate * code.info_bits / 1e6, "unit": "Mbit/s", "cores": cores, "kind": kind, "sample": sample,
                                            "frames_per_s": rate, "wall_s": wall}
            line["cpu_baseline"] = head["cpu_baseline"]
        if len(legs) > 1:
            other = res[legs[1]]
            other["note"] = "the same workload and frames through the reference's other check node (NB_LDPC.c:%s instead of :%s), measured like the " \
                            "headline leg (same steps and warm-up); `bench.py --ecn %s` makes it the headline" % (
                                ("388", "392", "syndrome") if legs[1] == "syndrome" else ("392", "388", "bubble"))
            other.pop("outputs")
            line["config5_as_written" if (legs[1] == "syndrome" and BASELINE_CONFIG.get(wl) == 5) else "other_check_node"] = other
        outputs = head.pop("outputs")
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    nbldpc.unpin(noisy)
    for o in out:
        nbldpc.unpin(o)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(d, outputs, limit=48 << 20):
    """The arrays the decode call returns (decisions [B, N], syndromes [B], iteration counts [B]) as float32 .npy files.  When the
    decisions exceed `limit` bytes, a fixed seeded sample of frames is written and decide_frames.npy names them."""
    os.makedirs(d, exist_ok=True)
    dec = outputs["decide"]
    B, N = dec.shape
    keep = np.arange(B)
    if B * N * 4 > limit:
        keep = np.sort(np.random.default_rng(0).choice(B, limit // (N * 4), replace=False))
    np.save(os.path.join(d, "decide.npy"), dec[keep].astype(np.float32))
    np.save(os.path.join(d, "decide_frames.npy"), keep.astype(np.float64))
    np.save(os.path.join(d, "syndrome.npy"), outputs["syndrome"].astype(np.float32))
    np.save(os.path.join(d, "iterations.npy"), outputs["iterations"].astype(np.float32))


def code_bits(code, syms):
    b = code.tables()[0]
    return b[syms]


_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries loaded later write there too (NCCL prints its version banner on stdout
    when NCCL_DEBUG is VERSION or WARN): from here on file descriptor 1 is stderr for everybody, and emit() alone writes to the
    real stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="AD_64800_R12_GF256", choices=sorted(WORKLOADS))
    ap.add_argument("--ecn", default="bubble", choices=["bubble", "syndrome"],
                    help="check node: bubble = CheckPassLogEMS (the reference's shipped hot path), syndrome = syndrome_ems")
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU per step (0 = workload default)")
    ap.add_argument("--frames-per-cta", type=int, default=0)
    ap.add_argument("--cns-per-step", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-also", action="store_true", help="skip the short syndrome_ems leg of the default run")
    ap.add_argument("--count-errors", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not (args.impl == "ours" and world == 1 and args.gpus > 1):           # (the torchrun relaunch below keeps its children's stdout)
        claim_stdout()
    if args.impl == "reference":
        if args.workload in NO_REFERENCE:
            if rank == 0:
                emit({"impl": "reference", "unavailable": "the reference's LoadCode cannot read the full-alist file of workload %s" % args.workload})
            return
        reference_arm(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000)] + sys.argv
        sys.exit(subprocess.call(cmd))
    ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
