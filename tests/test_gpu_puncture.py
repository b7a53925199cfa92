"""Puncturing: variables of the code that are never sent (nbgpu_set_puncturing, nbgpu_awgn_punctured_noise,
nbgpu_sigma_punctured).  The host stream is pinned to a Python restatement on the oracle's drand48, and a punctured decode to
nbgpu_decode_llr on the expanded rows (zero rows at punctured variables) and to the oracle fed with those rows, for every input
kind."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import CONSOLE, EXE, ESN, PI, field_code, matrix_path, multigpu, run_driver, soft, waves

gpu = pytest.mark.gpu

SPLIT_P = {16: 2, 64: 3, 256: 4}                               # QPSK points per symbol of the split kind
FADING = {"faded_symbol": nbldpc.FADING_SYMBOL, "faded_component": nbldpc.FADING_COMPONENT}
S_FADED = {nbldpc.FADING_SYMBOL: 5, nbldpc.FADING_COMPONENT: 6}


def kinds(q, with_llr=True):
    return (["bpsk"] + (["llr"] if with_llr else []) + (["apsk64"] if q == 64 else []) +
            ["mapped", "faded_symbol", "faded_component", "split"])


def table(code, kind):
    if kind == "apsk64":
        return nbldpc.apsk64_table()
    if kind == "split":
        return nbldpc.split_qam(code.q, SPLIT_P[code.q])
    if kind in ("mapped", "faded_symbol", "faded_component"):
        return nbldpc.constellation(nbldpc.MAP_QAM, code.q)
    return None


def ebn_of(code, kind):
    return {"bpsk": 2.5, "llr": 2.5, "split": 4.0, "faded_symbol": ESN[code.q] + 6, "faded_component": ESN[code.q] + 6}.get(kind, ESN[code.q])


def sigma_of(code, kind, ebn, pv=None):
    return code.sigma(ebn, punctured=pv) if kind in ("bpsk", "llr") else nbldpc.sigma_apsk64(ebn)


def noise(code, kind, nbin, ebn, pv):
    mod = table(code, kind)
    if kind in ("bpsk", "llr"):
        return code.noise(nbin, ebn, punctured=pv)
    if kind == "apsk64":
        return code.noise_apsk64(nbin, ebn, punctured=pv)
    if kind == "mapped":
        return code.noise_mapped(nbin, mod, ebn, punctured=pv)
    if kind in FADING:
        return code.noise_faded(nbin, mod, ebn, FADING[kind], punctured=pv)
    return code.noise_split(nbin, mod, SPLIT_P[code.q], ebn, punctured=pv)


def draws(code, kind, pv=None):
    if kind in FADING:
        return multigpu.draws_per_frame(code, "mapped", fading=kind[6:], punctured=pv)
    if kind == "split":
        return multigpu.draws_per_frame(code, "split", points=SPLIT_P[code.q], punctured=pv)
    return multigpu.draws_per_frame(code, "bpsk" if kind == "llr" else kind, punctured=pv)


def host_frames(code, kind, frame0, B, ebn, pv=None):
    """frames [frame0, frame0 + B) of the host source: (codewords [B, N], bits [B, N, logq], frames [B, N or N - p, ...])"""
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(frame0 * draws(code, kind, pv))
    cws, bits, frames = [], [], []
    for _ in range(B):
        cw, nbin = code.random_codeword()
        cws.append(cw); bits.append(nbin); frames.append(noise(code, kind, nbin, ebn, pv))
    return np.stack(cws), np.stack(bits), np.stack(frames)


class Calls:
    """the per-kind calls of a Decoder: decode(frames, sigma), upload(frames, sigma), channel(frames, sigma, want_sorted),
    source(frame0, B, ebn); binds the kind's table"""

    def __init__(self, d, code, kind):
        mod = table(code, kind)
        if kind in ("mapped",) + tuple(FADING):
            d.set_constellation(mod)
        if kind == "split":
            d.set_split_constellation(mod, SPLIT_P[code.q])
        f = FADING.get(kind)
        name = {"bpsk": "noisy", "apsk64": "apsk64", "mapped": "mapped", "faded_symbol": "faded", "faded_component": "faded",
                "split": "split"}.get(kind)
        if kind == "llr":
            self.decode = lambda x, s: d.decode_llr(x)
            self.upload = lambda x, s: d.upload_llr(x)
            self.channel = self.source = None
            return
        self.decode = getattr(d, "decode_" + name)
        self.upload = (lambda x, s: d._upload(nbldpc.lib().nbgpu_upload_apsk64, x, 2, s)) if kind == "apsk64" else getattr(d, "upload_" + name)
        self.channel = d.channel if kind == "bpsk" else getattr(d, "channel_" + name)
        src = {"bpsk": d.source_frames}.get(kind) or getattr(d, "source_frames_" + name)
        self.source = (lambda f0, B, e: src(f0, B, e, f)) if f else src


def spread_pattern(code, frac, seed=0):
    """about frac * N variables, no check node with two punctured neighbours, in a shuffled order"""
    rng = np.random.default_rng(seed + code.N)
    checks = [set() for _ in range(code.N)]
    for m in range(code.M):
        for e in range(code.row_ptr[m], code.row_ptr[m + 1]):
            checks[code.col[e]].add(m)
    want = max(1, int(round(frac * code.N)))
    used, out = set(), []
    for n in rng.permutation(code.N):
        if len(out) == want:
            break
        if checks[n] and not (checks[n] & used):
            out.append(int(n)); used |= checks[n]
    return np.array(out, np.int32)


def pattern(code, seed=0):
    """a quarter of the variables, unsorted (checks may have several punctured neighbours)"""
    return np.random.default_rng(seed + 7 * code.N).permutation(code.N)[:max(1, code.N // 4)].astype(np.int32)


def transmitted(code, pv):
    return np.setdiff1d(np.arange(code.N), pv)


def expand(code, rows, pv):
    """llr[B][N][q] with zero rows at the punctured variables"""
    out = np.array(rows, np.float32, copy=True)
    out[:, pv] = 0.0
    return out


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def oracle_noise(o, code, kind, nbin, ebn, tx, sigma):
    """the punctured stream on the oracle's drand48: each transmitted variable, in order, takes its channel's draws"""
    mod = table(code, kind)
    logq = code.logq
    out = []
    for n in tx:
        som = sum(int(nbin[n, b]) << b for b in range(logq))
        if kind in FADING:
            d = [float(np.float32(o.drand48())) for _ in range(S_FADED[FADING[kind]])]
            ri = float(np.float32(math.sqrt(-math.log(d[4]))))
            rq = float(np.float32(math.sqrt(-math.log(d[5])))) if len(d) == 6 else ri
            y = [np.float32(r * float(mod[som, c]) + sigma * math.sqrt(-2.0 * math.log(d[2 * c])) * math.cos(2.0 * PI * d[2 * c + 1]))
                 for c, r in ((0, ri), (1, rq))]
            out.append([y[0], y[1], np.float32(ri), np.float32(rq)])
            continue
        P, dims = (logq, 1) if kind in ("bpsk", "llr") else (SPLIT_P[code.q], 2) if kind == "split" else (1, 2)
        m = logq // P
        row = []
        for j in range(P):
            sub = (som >> (j * m)) & ((1 << m) - 1)
            for c in range(dims):
                point = float(1 - 2 * sub) if dims == 1 else float(mod[sub, c])
                u = float(np.float32(o.drand48())); v = float(np.float32(o.drand48()))
                row.append(np.float32(point + sigma * math.sqrt(-2.0 * math.log(u)) * math.cos(2.0 * PI * v)))
        out.append(row)
    return np.array(out, np.float32)


@pytest.mark.parametrize("q", [16, 64, 256])
def test_host_punctured_noise_equals_the_oracle_stream(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    nbin = np.random.default_rng(q).integers(0, 2, (code.N, code.logq)).astype(np.int32)
    pv = pattern(code)
    tx = transmitted(code, pv)
    for kind in kinds(q, with_llr=False):
        ebn = ebn_of(code, kind)
        code.rng_default(); code.rng_skip(999)
        got = noise(code, kind, nbin, ebn, pv)
        assert got.shape[0] == len(tx)
        o.rng_default(); o.rng_skip(999)
        ref = oracle_noise(o, code, kind, nbin, ebn, tx, sigma_of(code, kind, ebn, pv))
        assert got.reshape(len(tx), -1).tobytes() == ref.tobytes(), kind
        o.rng_default(); o.rng_skip(999 + (draws(code, kind, pv) - code.K * code.logq))    # exactly S * Nt draws
        assert code.drand48() == o.drand48(), kind
    o.close()


@pytest.mark.parametrize("q", [16, 64, 256])
def test_empty_pattern_is_todays_stream_and_sigma(q):
    code, _ = field_code(q)
    nbin = np.random.default_rng(q + 1).integers(0, 2, (code.N, code.logq)).astype(np.int32)
    for kind in kinds(q, with_llr=False):
        ebn = ebn_of(code, kind)
        code.rng_default(); a = noise(code, kind, nbin, ebn, None); xa = code.rng.x
        code.rng_default(); b = noise(code, kind, nbin, ebn, [])
        assert a.tobytes() == b.tobytes() and code.rng.x == xa, kind
        assert draws(code, kind, []) == draws(code, kind), kind
    for ebn in (-1.0, 0.5, 2.5, 7.25):
        assert code.sigma(ebn, punctured=[]) == code.sigma(ebn)


@pytest.mark.parametrize("q", [16, 64, 256])
def test_punctured_rate_and_sigma(q):
    code, _ = field_code(q)
    for p in (1, 2, code.N // 3, code.N - 1):
        pv = np.arange(p)[::-1]
        rate_p = np.float32(code.N - code.M) / np.float32(code.N - p)
        for ebn in (0.5, 2.5, 6.0):
            e = float(np.float32(ebn))
            ref = np.float32(math.sqrt(1.0 / (2.0 * float(rate_p) * math.pow(10, e / 10.0))))
            assert code.sigma(ebn, punctured=pv) == float(ref), (p, ebn)
        assert code.sigma(2.0, punctured=pv) < code.sigma(2.0)     # a higher rate: less noise per bit at the same Eb/N0
    L = nbldpc.lib()
    for p in (-1, code.N, code.N + 5):
        assert math.isnan(L.nbgpu_sigma_punctured(code.h, p, C.c_float(2.0)))


@pytest.mark.parametrize("q", [16, 64, 256])
def test_draws_per_frame_punctured_skips_whole_frames(q):
    code, _ = field_code(q)
    pv = pattern(code)
    for kind in kinds(q, with_llr=False):
        D = draws(code, kind, pv)
        assert D == draws(code, kind) - len(pv) * (draws(code, kind) - code.K * code.logq) // code.N, kind
        ebn = ebn_of(code, kind)
        _, _, frames = host_frames(code, kind, 0, 5, ebn, pv)
        for f in (1, 4):
            code.rng_default(); code.rng_skip(f * D)
            _, nb = code.random_codeword()
            assert noise(code, kind, nb, ebn, pv).tobytes() == frames[f].tobytes(), (kind, f)


def test_punctured_noise_refusals():
    code, _ = field_code(64)
    L = nbldpc.lib()
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 64)
    out = np.zeros((code.N, 6), np.float32)
    fm, fo = mod.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float))
    ip = C.POINTER(C.c_int)

    def call(p, vars, channel=nbldpc.CHANNEL_BPSK, arg=0, m=fm, o=fo):
        v = None if vars is None else np.ascontiguousarray(vars, np.int32)
        return L.nbgpu_awgn_punctured_noise(code.h, C.byref(code.rng), None, channel, arg, m, C.c_float(2.0), p,
                                            v.ctypes.data_as(ip) if v is not None else None, o)
    code.rng_default()
    x0 = code.rng.x
    for p, vars in ((1, None), (-1, [0]), (code.N, list(range(code.N))), (2, [0, code.N]), (2, [3, -1]), (3, [1, 5, 1])):
        assert call(p, vars) == nbldpc.EINVAL, (p, vars)
        assert "puncturing pattern" in L.nbgpu_last_error(None).decode()
    for channel, arg, m in ((4, 0, fm), (-1, 0, fm), (nbldpc.CHANNEL_FADED, 3, fm), (nbldpc.CHANNEL_SPLIT, 4, fm),
                            (nbldpc.CHANNEL_MAPPED, 0, None)):
        assert call(1, [2], channel, arg, m) == nbldpc.EINVAL, channel
    assert call(1, [2], o=None) == nbldpc.EINVAL
    assert code.rng.x == x0 and not out.any()                 # a refused call draws and writes nothing
    for bad in ([1.5], [2 ** 32 + 1], ["a"]):
        with pytest.raises(ValueError):
            code.noise(None, 2.0, punctured=bad)
    for bad in ([1, 1], [code.N], [-1], list(range(code.N))):
        with pytest.raises(nbldpc.NbgpuError):
            code.noise(None, 2.0, punctured=bad)
        with pytest.raises(ValueError):
            multigpu.draws_per_frame(code, "bpsk", punctured=bad)
        with pytest.raises(ValueError):
            multigpu.monte_carlo(code, 4, 2.0, decode=lambda *a: None, punctured=bad)
    with pytest.raises(ValueError):
        field_code(256)[0].noise_apsk64(None, 2.0, punctured=[1])


def test_c_driver_refuses_a_bad_pattern_before_any_device(tmp_path):
    assert os.path.exists(EXE)
    g64 = matrix_path("matrices/N96_K48_GF64")                 # N = 16 symbols
    files = {"dup": "3 5 3", "range": "2 16", "negative": "-1", "word": "2 x 4", "all": " ".join(map(str, range(16)))}
    for name, text in files.items():
        (tmp_path / name).write_text(text)
    for arg in [str(tmp_path / n) for n in files] + [str(tmp_path / "missing")]:
        r = subprocess.run([EXE, "10", "10", g64, "3.0", "20", "0.3", "25", "8", "0", "0", "1", "0", "0", "0", "1", arg],
                           cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode != 0 and "puncturing pattern" in r.stdout, (arg, r.stdout[-2000:])
        assert "AllocateDecoder" not in r.stdout and "LDPC code parameters" not in r.stdout, arg


def test_puncturing_abi_without_a_gpu():
    L = C.CDLL(nbldpc.LIB_PATH)
    for name in ("nbgpu_set_puncturing", "nbgpu_sigma_punctured", "nbgpu_awgn_punctured_noise"):
        assert hasattr(L, name), name
    lib = nbldpc.lib()
    assert lib.nbgpu_set_puncturing(None, 0, None) == nbldpc.EINVAL
    assert (nbldpc.CHANNEL_BPSK, nbldpc.CHANNEL_MAPPED, nbldpc.CHANNEL_FADED, nbldpc.CHANNEL_SPLIT) == (0, 1, 2, 3)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_channel_rows_are_the_unpunctured_rows_and_zero_rows(q):
    code, _ = field_code(q)
    pv = pattern(code)
    tx = transmitted(code, pv)
    B = 6
    d0 = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    d1 = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    d1.set_puncturing(pv)
    for kind in kinds(q, with_llr=False):
        c0, c1 = Calls(d0, code, kind), Calls(d1, code, kind)
        ebn = ebn_of(code, kind)
        _, _, full = host_frames(code, kind, 3, B, ebn)
        sigma = sigma_of(code, kind, ebn)
        llr, il, ig = c0.channel(full, sigma, want_sorted=True)
        pl, pil, pig = c1.channel(full[:, tx], sigma, want_sorted=True)
        assert pl.shape == (B, code.N, q)
        assert pl[:, tx].tobytes() == llr[:, tx].tobytes(), kind
        assert pil[:, tx].tobytes() == il[:, tx].tobytes() and (pig[:, tx] == ig[:, tx]).all(), kind
        assert not pl[:, pv].any() and not pil[:, pv].any() and (pig[:, pv] == np.arange(q)).all(), kind
        with pytest.raises(ValueError):
            c1.channel(full, sigma)                            # [B, N, ...] is not [B, N - p, ...]
    d0.close(); d1.close()


DECODE_CASES = [(q, k, early, ecn) for q in (16, 64, 256) for i, k in enumerate(kinds(q))
                for early, ecn in [((True, 0), (False, 0), (True, 1))[i % 3]]]


@gpu
@pytest.mark.parametrize("q,kind,early,ecn", DECODE_CASES)
def test_punctured_decode_equals_decode_llr_on_expanded_rows_and_the_oracle(q, kind, early, ecn):
    """decode_* (streamed: more than two waves) and upload_* + run against decode_llr on the expanded rows and the oracle fed
    with them; LIST and BITS soft output against decode_llr"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    n_m = 16 if q == 16 else 20
    kw = dict(ecn_kind=1, d1=n_m - 1, d2=min(15, n_m - 1), d3=5, cfg_trunc=1000, n_cv=25) if ecn else {}
    cfg = o.build_config_table(int(code.row_deg[0]), n_m - 1, min(15, n_m - 1), 5, 1000) if ecn else None
    B = waves(code, n_m, early, **kw)
    pv = pattern(code, seed=q)
    tx = transmitted(code, pv)
    d0 = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    d1 = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    d1.set_puncturing(pv)
    ebn = ebn_of(code, kind)
    src = "bpsk" if kind == "llr" else kind
    c0, c1 = Calls(d0, code, src), Calls(d1, code, kind)
    _, _, full = host_frames(code, src, 40, B, ebn)
    sigma = sigma_of(code, src, ebn)
    rows = c0.channel(full, sigma)
    llr = expand(code, rows, pv)
    frames = rows[:, tx] if kind == "llr" else full[:, tx]
    ref = d0.decode_llr(llr)
    got = c1.decode(frames, sigma)
    assert all((x == y).all() for x, y in zip(got, ref))
    c1.upload(frames, sigma); d1.run()
    assert all((x == y).all() for x, y in zip(d1.download(), ref))
    dec, synd, it = got
    for f in range(0, B, 7):
        r = o.decode_frame(llr[f], n_m, 25, 10, 0.3, force=not early, ecn=ecn, cfg=cfg, n_cv=25 if ecn else 0)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    for kind_, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d0.set_soft_output(kind_, k); d1.set_soft_output(kind_, k)
        d0.decode_llr(llr); rsoft = soft(d0, kind_)
        assert rsoft[0].shape[1] == code.N
        c1.decode(frames, sigma)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d1, kind_), rsoft)), kind_
        c1.upload(frames, sigma); d1.run()
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d1, kind_), rsoft)), kind_
    d0.close(); d1.close(); o.close()


def _far(code, kind, pv):
    D = draws(code, kind, pv)
    far = (1 << 32) // D + 1000
    assert far * D > 1 << 32
    return far


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_generated_punctured_frames_equal_the_host_stream_and_score_alike(q):
    code, _ = field_code(q)
    B = 160
    pv = pattern(code, seed=1)
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    d.set_puncturing(pv)
    bing = code.tables()[0]
    for kind in kinds(q, with_llr=False):
        c = Calls(d, code, kind)
        ebn = ebn_of(code, kind)
        for frame0 in (0, 12345, _far(code, kind, pv)):
            c.source(frame0, B, ebn)
            cw, _, frames = host_frames(code, kind, frame0, B, ebn, pv)
            gcw, gframes = d.source_download()
            assert gframes.shape == frames.shape and gframes.shape[1] == code.N - len(pv), kind
            assert (gcw == cw).all() and gframes.tobytes() == frames.tobytes(), (kind, frame0)
        d.run()
        errs, synd, it = d.source_results()
        _, bits, frames = host_frames(code, kind, _far(code, kind, pv), B, ebn, pv)
        dec, hsynd, hit = c.decode(frames, sigma_of(code, kind, ebn, pv))
        herr = np.array([(bing[dec[f, :code.K]] != bits[f, :code.K]).sum() for f in range(B)])
        assert (errs == herr).all() and (synd == hsynd).all() and (it == hit).all(), kind
        # the widest margin flags most samples: the host fix-up works on compact indices
        d.source_set_margin(2.0 ** -20)
        c.source(7, 64, ebn)
        assert d.source_fixups() > 0
        cw, _, frames = host_frames(code, kind, 7, 64, ebn, pv)
        gcw, gframes = d.source_download()
        assert (gcw == cw).all() and gframes.tobytes() == frames.tobytes(), kind
        d.source_set_margin(2.0 ** -46)
    d.close()


@gpu
def test_puncturing_state_rules():
    code, _ = field_code(64)
    B = 32
    pv = pattern(code)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    L = nbldpc.lib()
    # refusals leave the context unchanged (no pattern)
    for p, vars in ((1, None), (-1, [0]), (code.N, list(range(code.N))), (2, [0, code.N]), (2, [-3, 1]), (3, [1, 5, 1])):
        v = None if vars is None else np.ascontiguousarray(vars, np.int32)
        assert L.nbgpu_set_puncturing(d.h, p, v.ctypes.data_as(C.POINTER(C.c_int)) if v is not None else None) == nbldpc.EINVAL
        assert "nbgpu_set_puncturing" in L.nbgpu_last_error(d.h).decode()
    d.source_frames(3, B, 2.0)
    assert d.source_download()[1].shape == (B, code.N, code.logq)
    d.run(); d.source_results()
    # bound: a refused re-binding keeps the pattern and the batch
    d.set_puncturing(pv)
    d.source_frames(3, B, 2.0); d.run(); ref = d.source_results()
    for bad in ([1, 1], [code.N]):
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.set_puncturing(bad)
        assert e.value.code == nbldpc.EINVAL
    d.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    assert d.source_download()[1].shape == (B, code.N - len(pv), code.logq)
    # frames of the unpunctured layout are refused
    for call in (lambda: d.decode_noisy(np.zeros((B, code.N, 6), np.float32), 0.5),
                 lambda: d.upload_llr(np.zeros((B, code.N, 64), np.float32)),
                 lambda: d.decode_noisy(np.zeros((B * (code.N - len(pv)) * 6,), np.float32), 0.5)):
        with pytest.raises(ValueError):
            call()
    # re-binding (the same pattern) drops the batch: run names the reason; soft output, results and download are gone
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.source_frames(3, B, 2.0); d.run(); d.soft_bits()
    d.set_puncturing(pv[::-1])
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.run()
    assert e.value.code == nbldpc.ESTATE and "nbgpu_set_puncturing" in str(e.value)
    for call in (d.soft_bits, d.source_results, d.source_download):
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE, call
    # constellation bindings are independent of the pattern, both ways
    qam = nbldpc.constellation(nbldpc.MAP_QAM, 64)
    d.set_constellation(qam)
    d.source_frames_mapped(5, B, 15.0); d.run(); ref = d.source_results()
    d.set_constellation(qam)                                     # drops the mapped batch, keeps the pattern
    d.source_frames_mapped(5, B, 15.0); d.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    assert d.source_download()[1].shape == (B, code.N - len(pv), 2)
    d.set_puncturing([])                                         # unbinding keeps the table
    d.source_frames_mapped(5, B, 15.0)
    assert d.source_download()[1].shape == (B, code.N, 2)
    d.set_soft_output(nbldpc.SOFT_NONE)
    # a context that bound and unbound a pattern decodes as one that never bound
    d0 = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d0.set_constellation(qam)
    _, _, noisy = host_frames(code, "bpsk", 9, B, 1.5)
    _, _, mapped = host_frames(code, "mapped", 9, B, 12.0)
    assert all((x == y).all() for x, y in zip(d.decode_noisy(noisy, 0.7), d0.decode_noisy(noisy, 0.7)))
    assert all((x == y).all() for x, y in zip(d.decode_mapped(mapped, 0.3), d0.decode_mapped(mapped, 0.3)))
    assert d.channel(noisy, 0.7).tobytes() == d0.channel(noisy, 0.7).tobytes()
    for x in (d, d0):
        x.source_frames(11, B, 1.5); x.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), d0.source_results()))
    assert all(x.tobytes() == y.tobytes() for x, y in zip(d.source_download(), d0.source_download()))
    d.close(); d0.close()


@gpu
@pytest.mark.parametrize("q,kind", [(64, "bpsk"), (256, "mapped")])
def test_c_driver_punctured_sources_and_monte_carlo_agree(tmp_path, q, kind):
    code, path = field_code(q)
    pv = spread_pattern(code, 0.1)
    pfile = tmp_path / "pattern.txt"
    pfile.write_text(" ".join(map(str, pv)) + "\n")
    channel = 0 if kind == "bpsk" else 2
    esn = 3.0 if kind == "bpsk" else ESN[q] + 1
    ebn = "%.1f" % esn
    tail = ("0", "0", "1", str(pfile))
    out1, file1 = run_driver(tmp_path, "device", path, ebn, 16, 1, channel, *tail)
    out0, file0 = run_driver(tmp_path, "host", path, ebn, 16, 0, channel, *tail)
    assert "punctured" in out1 and "%d of %d" % (len(pv), code.N) in out1
    last = [re.findall(CONSOLE, o)[-1] for o in (out1, out0)]
    assert last[0] == last[1], last
    assert file1 == file0 and len(file1) == 1, (file1, file0)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q) if kind == "mapped" else None
    mc = multigpu.monte_carlo
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=128)
    d.set_puncturing(pv)
    if mod is not None:
        d.set_constellation(mod)
    dec = d.decode_noisy if kind == "bpsk" else d.decode_mapped
    for st in (mc(code, 2000, esn, decode=dec, batch=128, channel=kind, constellation=mod, punctured=pv),
               mc(code, 2000, esn, batch=128, decoder=d, channel=kind, constellation=mod, punctured=pv)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0][0]), int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]), st
    d.close()
    # without the pattern the console has no puncturing line
    outn, _ = run_driver(tmp_path, "none", path, ebn, 16, 1, channel, "0", "0", "1", "-")
    assert "punctured" not in outn
    # an Eb/N0 sweep equals its single points
    lo = esn - 1
    out, lines = run_driver(tmp_path, "sweep", path, "%.1f:%.1f:1" % (lo, lo + 1), 16, 1, channel, *tail)
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 2 and len(lines) == 2
    for i in range(2):
        o1, l1 = run_driver(tmp_path, "single%d" % i, path, "%.1f" % (lo + i), 16, 1, channel, *tail)
        assert re.findall(CONSOLE, o1)[-1] == re.findall(CONSOLE, blocks[i])[-1] and l1 == [lines[i]], (i, l1, lines[i])


@gpu
@pytest.mark.parametrize("rel", ["matrices/N96_K48_GF64", "matrices/KN/N96_K48_GF256.txt"])
def test_punctured_symbols_are_recovered_by_the_graph(rel):
    """about 10 % of the variables punctured, no check node with two of them: at an Es/N0 where the unpunctured code decodes
    every frame of the fixed stream, every punctured symbol of every frame is decided as sent, although no sample of it
    reached the decoder"""
    code = nbldpc.Code(matrix_path(rel))
    pv = spread_pattern(code, 0.1)
    assert len(pv) >= 1
    B, esn = 384, ESN[code.q] + 6
    mod = nbldpc.constellation(nbldpc.MAP_QAM, code.q)
    d0 = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d1 = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d1.set_puncturing(pv)
    for d in (d0, d1):
        d.set_constellation(mod)
        d.source_frames_mapped(0, B, esn); d.run()
    cw0, _ = d0.source_download(want_noisy=False)
    assert (d0.download()[0] == cw0).all()                      # the unpunctured code decodes every frame
    cw1, _ = d1.source_download(want_noisy=False)
    dec1 = d1.download()[0]
    assert (dec1[:, pv] == cw1[:, pv]).all()
    assert (d1.source_results()[0] == 0).all()
    d0.close(); d1.close()
