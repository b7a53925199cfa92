"""Frame sharding over the GPUs of one node (one process per GPU, torch.distributed) -- host logic only.

Frames of a Monte-Carlo run are independent (SURVEY.md section 8e): frame f consumes the drand48 draws
[f*D, (f+1)*D) with D = (K + 2N) * log2(q) (K*log2(q) information bits, tools.c:124-136, then two draws per
transmitted bit, channel.c:56-57; D = K*log2(q) + 4N for a code sent one symbol per constellation point, 64-APSK or any
mapped table, two draws for each of the I and Q samples of a symbol, channel.c:234-263; D = K*log2(q) + 5N or + 6N under
symbol or component Rayleigh fading, one or two amplitude draws more per symbol; D = K*log2(q) + 4NP for the split channel,
P points per symbol).  Under a puncturing pattern of p variables only the N - p transmitted symbols draw: N becomes N - p in
the second term.  So every rank can generate its own frames by LCG jump-ahead.  There is no
collective on the decode path.  Results meet in ONE collective:

  * `allreduce_counters` -- sum of the int64 counters (throughput runs: frames, non-zero syndromes, iterations, ...);
  * `monte_carlo` -- gathers (bit errors, syndrome, iterations) per frame on rank 0, which applies the reference's
    sequential rule "stop after the 40th erroneous frame" (NB_LDPC.c:506) in frame order, so the statistics are
    the single-process ones whatever the number of ranks.

torch is used for the process group only (NCCL on GPUs, gloo in the CPU tests).
"""
import numpy as np


FADINGS = {"symbol": 1, "component": 2}                    # FADING_SYMBOL, FADING_COMPONENT of the library


def _extra(channel, fading, points):
    """the channel's own parameter: fading=None | "symbol" | "component" -> 0, 1, 2 for "mapped"; points P for "split" (required);
    0 otherwise.  fading belongs to the mapped channel only, points to the split channel only."""
    if points is not None and channel != "split":
        raise ValueError("points=%r needs channel='split', not %r" % (points, channel))
    if fading is not None and channel != "mapped":
        raise ValueError("fading=%r needs channel='mapped', not %r" % (fading, channel))
    if channel == "split":
        if points is None:
            raise ValueError("channel='split' needs points=P")
        return int(points)
    if fading is None:
        return 0
    if fading not in FADINGS:
        raise ValueError("fading must be 'symbol' or 'component', not %r" % (fading,))
    return FADINGS[fading]


def _sigma_apsk64(code, ebn, punctured=None):
    from . import sigma_apsk64
    return sigma_apsk64(ebn)


# per channel, with x = the channel's own parameter (_extra: fading of "mapped", points of "split") and pv = the puncturing
# pattern (None = none): drand48 draws per symbol after the K*log2(q) information bits (code, x), sigma(code, ebn, pv), the host
# noise of one frame (code, nbin, ebn, mod, x, pv) and the device source of a batch (decoder, frame0, B, ebn, x)
_CHANNELS = {
    "bpsk": (lambda code, x: 2 * code.logq, lambda code, ebn, pv: code.sigma(ebn, punctured=pv),
             lambda code, nbin, ebn, mod, x, pv: code.noise(nbin, ebn, punctured=pv),
             lambda d, frame0, B, ebn, x: d.source_frames(frame0, B, ebn)),
    "apsk64": (lambda code, x: 4, _sigma_apsk64,
               lambda code, nbin, ebn, mod, x, pv: code.noise_apsk64(nbin, ebn, punctured=pv),
               lambda d, frame0, B, ebn, x: d.source_frames_apsk64(frame0, B, ebn)),
    "mapped": (lambda code, x: 4 + x, _sigma_apsk64,
               lambda code, nbin, ebn, mod, x, pv: (code.noise_faded(nbin, mod, ebn, x, punctured=pv) if x
                                                    else code.noise_mapped(nbin, mod, ebn, punctured=pv)),
               lambda d, frame0, B, ebn, x: d.source_frames_faded(frame0, B, ebn, x) if x else d.source_frames_mapped(frame0, B, ebn)),
    "split": (lambda code, x: 4 * x, _sigma_apsk64,
              lambda code, nbin, ebn, mod, x, pv: code.noise_split(nbin, mod, x, ebn, punctured=pv),
              lambda d, frame0, B, ebn, x: d.source_frames_split(frame0, B, ebn)),
}


def _channel(channel):
    if channel not in _CHANNELS:
        raise ValueError("channel must be 'bpsk', 'apsk64', 'mapped' or 'split', not %r" % (channel,))
    return _CHANNELS[channel]


def _npunct(code, punctured):
    """p of a puncturing pattern (None = 0); a pattern the library would refuse is a ValueError here too"""
    if punctured is None:
        return 0
    v = np.asarray(punctured).reshape(-1)
    if v.size and (not np.issubdtype(v.dtype, np.integer) or v.min() < 0 or v.max() >= code.N or np.unique(v).size != v.size
                   or v.size >= code.N):
        raise ValueError("puncturing pattern must be p < N = %d distinct variable indices in [0, N)" % code.N)
    return v.size


def draws_per_frame(code, channel="bpsk", fading=None, points=None, punctured=None):
    """drand48 draws one frame of the reference's main loop consumes: tools.c:124-136, then channel.c:56-57 ("bpsk",
    ModelChannel_AWGN_BPSK) or channel.c:234-263 ("apsk64", ModelChannel_AWGN_64; "mapped", the same on any q-point table;
    "split", the same over points=P points per symbol); fading="symbol" / "component" (mapped only): one / two Rayleigh
    amplitude draws more per symbol; punctured = variable indices never sent: those symbols draw nothing"""
    x = _extra(channel, fading, points)
    return code.K * code.logq + _channel(channel)[0](code, x) * (code.N - _npunct(code, punctured))


def frame_range(total, rank, world):
    """Contiguous block of frame indices [lo, hi) of `rank` (SURVEY.md 8e: [g*F/G, (g+1)*F/G))"""
    return (rank * total) // world, ((rank + 1) * total) // world


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def allreduce_counters(counters, device=None):
    """Sum an int64 counter vector over all ranks (the only collective of a throughput run)."""
    c = np.ascontiguousarray(counters, np.int64)
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return c.copy()
    import torch
    t = torch.from_numpy(c.copy())
    if device is not None:
        t = t.to(device)
    dist.all_reduce(t)
    return t.cpu().numpy()


def gather_rows(rows):
    """Concatenate per-rank int64 [n_r, k] arrays on rank 0 in rank order (None elsewhere)."""
    rows = np.ascontiguousarray(rows, np.int64)
    dist = _dist()
    if dist is None or dist.get_world_size() == 1:
        return rows
    out = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
    dist.gather_object(rows, out, dst=0)
    return np.concatenate(out, axis=0) if out is not None else None


def monte_carlo(code, frames, ebn, decode=None, batch=256, rank=0, world=1, max_err_frames=40, decoder=None, channel="bpsk",
                constellation=None, fading=None, points=None, punctured=None):
    """The reference's Monte-Carlo loop (NB_LDPC.c:250-511) sharded by frame block over `world` ranks.

    Either decode(noisy, sigma) -> (decide[B, N], synd[B], iters[B]) with frames made by the host source, or
    decoder=<Decoder>: frames are generated, decoded and scored on the rank's GPU (nbgpu_source_frames / nbgpu_run /
    nbgpu_source_results) and only 12 bytes per frame reach the host.
    channel="bpsk" (ModelChannel_AWGN_BPSK): noisy[B, N, logq], e.g. Decoder.decode_noisy; "apsk64" (ModelChannel_AWGN_64,
    GF(64) codes): noisy[B, N, 2] with sigma_apsk64, e.g. Decoder.decode_apsk64, and Decoder.source_frames_apsk64; "mapped":
    the same on constellation=mod[q][2] (any field), e.g. Decoder.decode_mapped on a decoder with mod bound, and
    Decoder.source_frames_mapped (the decoder gets mod bound here).  fading="symbol" | "component" (channel="mapped" only):
    the same under Rayleigh fading, frames rx[B, N, 4], e.g. Decoder.decode_faded, and Decoder.source_frames_faded.
    channel="split", points=P: every symbol sent as P points of constellation=mod[M][2] (e.g. split_qam(q, P)), frames
    noisy[B, N, P, 2], e.g. Decoder.decode_split on a decoder with the table bound, and Decoder.source_frames_split (the decoder
    gets the table bound here).
    punctured = variable indices never sent (any channel): frames hold the N - p transmitted symbols, [B, N - p, ...], and the
    decoder gets the pattern bound here; BPSK sigma is taken at the rate of the transmitted word (Code.sigma).
    Returns on rank 0 the dict of the reference's statistics, None on the other ranks."""
    lo, hi = frame_range(frames, rank, world)
    D = draws_per_frame(code, channel, fading, points, punctured)
    x = _extra(channel, fading, points)
    _, sigma_of, noise, source = _channel(channel)
    if channel in ("mapped", "split") and constellation is None:
        raise ValueError("channel=%r needs constellation=mod" % (channel,))
    if channel == "mapped" and decoder is not None:
        decoder.set_constellation(constellation)
    if channel == "split" and decoder is not None:
        decoder.set_split_constellation(constellation, x)
    if decoder is not None and (punctured is not None or decoder.nt != code.N):
        decoder.set_puncturing(() if punctured is None else punctured)
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(lo * D)
    sigma = sigma_of(code, ebn, punctured)
    bing = code.tables()[0]
    rows = np.zeros((hi - lo, 3), np.int64)
    for b0 in range(lo, hi, batch):
        b1 = min(hi, b0 + batch)
        if decoder is not None:
            source(decoder, b0, b1 - b0, ebn, x)
            decoder.run()
            rows[b0 - lo:b1 - lo] = np.stack(decoder.source_results(), axis=1)
            continue
        bits, noisy = [], []
        for _ in range(b0, b1):
            _, nbin = code.random_codeword()
            bits.append(nbin)
            noisy.append(noise(code, nbin, ebn, constellation, x, punctured))
        dec, synd, it = decode(np.stack(noisy), sigma)
        for i in range(b1 - b0):
            err = int((bing[dec[i, :code.K]] != bits[i][:code.K]).sum())                    # NB_LDPC.c:479-485
            rows[b0 - lo + i] = (err, int(synd[i]), int(it[i]))
    allrows = gather_rows(rows)
    if allrows is None:
        return None
    stats = dict(frames=0, err_frames=0, undetected=0, bit_errors=0, sum_it=0, stopped=False)
    for err, synd, it in allrows:                                                          # NB_LDPC.c:474-507, frame order
        stats["frames"] += 1
        stats["sum_it"] += int(it)
        stats["bit_errors"] += int(err)
        if err:
            stats["err_frames"] += 1
            if synd == 0:
                stats["undetected"] += 1
        if stats["err_frames"] == max_err_frames:
            stats["stopped"] = True
            break
    stats["frames_in_results_file"] = stats["frames"] if stats["stopped"] else frames + 1    # 'nb' after the loop, :576
    return stats
