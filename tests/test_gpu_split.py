"""The split channel: one GF(q) symbol sent as P points of an M-point constellation mod[M][2], M = 2^(log2(q)/P)
(nbgpu_split_qam, nbgpu_set_split_constellation and the *_split calls).  The host stream is pinned to a Python restatement on
the oracle's drand48, the device intake to a numpy restatement of the header's definition, and decoding to nbgpu_decode_llr
and the oracle fed with those LLRs."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import CONSOLE, EXE, PI, field_code, matrix_path, multigpu, run_driver, seeded_table, soft, waves

gpu = pytest.mark.gpu

POINTS = {16: (2, 4), 64: (2, 3, 6), 256: (2, 4, 8)}
PAIRS = [(q, p) for q in POINTS for p in POINTS[q]]
QAM_PAIRS = [(16, 2), (64, 3), (256, 2), (256, 4)]
ESN = {2: 1.0, 4: 4.0, 8: 7.0, 16: 10.0}                     # Es/N0 per point (dB) by points of the table M


def size(q, P):
    return 1 << ((q.bit_length() - 1) // P)


def table(q, P, seed=5):
    """a seeded table of M points, two of them coincident when M >= 4"""
    M = size(q, P)
    if M >= 4:
        return seeded_table(M, seed)
    return np.random.default_rng(seed).normal(0, 1.7, (M, 2)).astype(np.float32)


def tables(q, P):
    return ([nbldpc.split_qam(q, P)] if (q, P) in QAM_PAIRS else []) + [table(q, P)]


def images(code):
    bingf = code.tables()[0].astype(np.int64)
    return (bingf << np.arange(bingf.shape[1])).sum(1)


def split_llr(noisy, mod, img, P, sigma):
    """the header's definition: t_j[x] in f64 from f32 differences and squares, LLR[k] = f32(sum_j t_j[sub_j(img[k])])"""
    m = (len(img).bit_length() - 1) // P
    M = 1 << m
    assert mod.shape == (M, 2)
    den = 2.0 * float(np.float32(sigma) * np.float32(sigma))
    y = np.asarray(noisy, np.float32).reshape(-1, P, 2)
    dI = (y[:, :, None, 0] - mod[None, None, :, 0]).astype(np.float32)
    dQ = (y[:, :, None, 1] - mod[None, None, :, 1]).astype(np.float32)
    t = (dI * dI).astype(np.float64) / den + (dQ * dQ).astype(np.float64) / den            # [N, P, M]
    sub = (img[:, None] >> (np.arange(P) * m)[None, :]) & (M - 1)                           # [q, P]
    s = t[:, 0, sub[:, 0]]
    for j in range(1, P):
        s = s + t[:, j, sub[:, j]]
    return s.astype(np.float32)


def oracle_noise_split(o, nbin, mod, P, ebn):
    """the split stream on the oracle's drand48: per point u, v for I then u, v for Q"""
    sigma = o.sigma_apsk64(ebn)
    N, logq = nbin.shape
    m = logq // P
    out = np.zeros((N, P, 2), np.float32)
    for n in range(N):
        som = sum(int(nbin[n, b]) << b for b in range(logq))
        for j in range(P):
            sub = (som >> (j * m)) & ((1 << m) - 1)
            for c in range(2):
                u = float(np.float32(o.drand48())); v = float(np.float32(o.drand48()))
                out[n, j, c] = np.float32(float(mod[sub, c]) + sigma * math.sqrt(-2.0 * math.log(u)) * math.cos(2.0 * PI * v))
    return out


def host_split(code, frame0, B, ebn, mod, P):
    """frames [frame0, frame0 + B) of the host source: (codewords, bits, noisy [B, N, P, 2])"""
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(frame0 * multigpu.draws_per_frame(code, "split", points=P))
    cws, bits, noisy = [], [], []
    for _ in range(B):
        cw, nbin = code.random_codeword()
        cws.append(cw); bits.append(nbin); noisy.append(code.noise_split(nbin, mod, P, ebn))
    return np.stack(cws), np.stack(bits), np.stack(noisy)


def same_split_stream(d, code, frame0, B, ebn, mod, P):
    cw, _, noisy = host_split(code, frame0, B, ebn, mod, P)
    gcw, gnoisy = d.source_download()
    assert gnoisy.shape == (B, code.N, P, 2)
    return (gcw == cw).all() and gnoisy.tobytes() == noisy.tobytes()


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_split_qam_tables_are_gray_unit_power_and_refuse_other_pairs():
    for q, P in QAM_PAIRS:
        mod = nbldpc.split_qam(q, P)
        M = size(q, P)
        assert mod.shape == (M, 2)
        assert abs(float((mod.astype(np.float64) ** 2).sum(1).mean()) - 1.0) < 1e-6
        L = int(round(math.sqrt(M)))
        for c in range(2):                                     # nearest neighbours on each axis differ in one bit
            other = mod[:, 1 - c]
            for x in range(M):
                line = np.flatnonzero(other == other[x])
                assert len(line) == L
                order = line[np.argsort(mod[line, c])]
                assert all(bin(int(a) ^ int(b)).count("1") == 1 for a, b in zip(order[:-1], order[1:]))
        if M == 4:
            assert sorted(map(tuple, mod.tolist())) == sorted((np.float32(a / math.sqrt(2)), np.float32(b / math.sqrt(2)))
                                                              for a in (-1, 1) for b in (-1, 1))
    assert nbldpc.split_qam(256, 2).tobytes() == nbldpc.constellation(nbldpc.MAP_QAM, 16).tobytes()
    L = nbldpc.lib()
    buf = np.zeros((16, 2), np.float32)
    fp = buf.ctypes.data_as(C.POINTER(C.c_float))
    for q, P in [(16, 4), (64, 2), (64, 6), (256, 8), (256, 3), (256, 1), (16, 1), (32, 5), (128, 7), (256, 0), (64, -3), (4, 1)]:
        assert L.nbgpu_split_qam(q, P, fp) == nbldpc.EINVAL, (q, P)
        assert L.nbgpu_last_error(None)
    assert L.nbgpu_split_qam(256, 2, None) == nbldpc.EINVAL
    assert not buf.any()


@pytest.mark.parametrize("q,P", PAIRS)
def test_host_split_noise_equals_the_oracle_stream(q, P):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    nbin = np.random.default_rng(q + P).integers(0, 2, (code.N, code.logq)).astype(np.int32)
    for mod in tables(q, P):
        for ebn in (ESN[size(q, P)] - 3, ESN[size(q, P)] + 2):
            code.rng_default(); code.rng_skip(4321)
            got = code.noise_split(nbin, mod, P, ebn)
            o.rng_default(); o.rng_skip(4321)
            assert got.shape == (code.N, P, 2)
            assert got.tobytes() == oracle_noise_split(o, nbin, mod, P, ebn).tobytes(), ebn
            o.rng_default(); o.rng_skip(4321 + 4 * code.N * P)    # exactly 4NP draws
            assert code.drand48() == o.drand48()
    code.rng_default()
    z = code.noise_split(None, tables(q, P)[0], P, 5.0)
    o.rng_default()
    assert z.tobytes() == oracle_noise_split(o, np.zeros((code.N, code.logq), np.int32), tables(q, P)[0], P, 5.0).tobytes()
    o.close()


def test_split_noise_refusals():
    code, _ = field_code(256)
    L = nbldpc.lib()
    mod = np.zeros((16, 2), np.float32)
    out = np.zeros((code.N, 8, 2), np.float32)
    fm, fo = mod.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float))
    for P in (0, 1, 3, 5, 16):
        assert L.nbgpu_awgn_split_noise(code.h, C.byref(code.rng), None, P, fm, C.c_float(5.0), fo) == nbldpc.EINVAL, P
    assert L.nbgpu_awgn_split_noise(code.h, C.byref(code.rng), None, 2, None, C.c_float(5.0), fo) == nbldpc.EINVAL
    assert L.nbgpu_awgn_split_noise(None, C.byref(code.rng), None, 2, fm, C.c_float(5.0), fo) == nbldpc.EINVAL
    assert L.nbgpu_awgn_split_noise(code.h, C.byref(code.rng), None, 2, fm, C.c_float(5.0), None) == nbldpc.EINVAL
    assert not out.any()


def test_split_table_of_another_size_is_refused():
    """the library reads 2M floats of the table, M = 2^(log2 q / P): the bindings refuse a table of another size instead of
    handing it a short buffer (e.g. the QPSK table of P = 4 passed with P = 2)"""
    code, _ = field_code(256)
    for mod, P in ((nbldpc.split_qam(256, 4), 2), (nbldpc.split_qam(256, 2), 4), (np.zeros((4, 2), np.float32), 8)):
        with pytest.raises(ValueError):
            code.noise_split(None, mod, P, 5.0)
        with pytest.raises(ValueError):
            multigpu.monte_carlo(code, 4, 5.0, decode=lambda *a: None, channel="split", constellation=mod, points=P)
    code.rng_default()
    x0 = code.rng.x
    with pytest.raises(ValueError):
        code.noise_split(None, nbldpc.split_qam(256, 4), 2, 5.0)
    assert code.rng.x == x0                                    # a refused call draws nothing


@pytest.mark.parametrize("P", [2, 4, 8])
def test_draws_per_frame_split_skips_whole_frames(P):
    code, _ = field_code(256)
    mod = tables(256, P)[0]
    D = multigpu.draws_per_frame(code, "split", points=P)
    assert D == code.K * 8 + 4 * code.N * P
    _, _, noisy = host_split(code, 0, 6, 5.0, mod, P)
    for f in (1, 4, 5):
        code.rng_default(); code.rng_skip(f * D)
        _, nb = code.random_codeword()
        assert code.noise_split(nb, mod, P, 5.0).tobytes() == noisy[f].tobytes()


def test_points_and_fading_belong_to_their_channels():
    code, _ = field_code(64)
    for ch in ("bpsk", "apsk64", "mapped"):
        with pytest.raises(ValueError):
            multigpu.draws_per_frame(code, ch, points=2)
        with pytest.raises(ValueError):
            multigpu.monte_carlo(code, 10, 5.0, decode=lambda *a: None, channel=ch, constellation=np.zeros((64, 2)), points=3)
    with pytest.raises(ValueError):
        multigpu.draws_per_frame(code, "split", fading="symbol", points=3)
    with pytest.raises(ValueError):
        multigpu.monte_carlo(code, 10, 5.0, decode=lambda *a: None, channel="split", constellation=nbldpc.split_qam(64, 3),
                             points=3, fading="symbol")
    with pytest.raises(ValueError):
        multigpu.draws_per_frame(code, "split")
    with pytest.raises(ValueError):
        multigpu.monte_carlo(code, 10, 5.0, decode=lambda *a: None, channel="split", points=3)


def test_c_driver_refuses_split_misuse_before_any_device(tmp_path):
    assert os.path.exists(EXE)
    g256, g64 = matrix_path("matrices/KN/N96_K48_GF256.txt"), matrix_path("matrices/N96_K48_GF64")
    for path, tail, msg in ((g256, ["0", "0", "0", "2"], "channel 2 only"), (g256, ["1", "0", "0", "4"], "channel 2 only"),
                            (g256, ["2", "1", "0", "2"], "neither fading nor degrees"),
                            (g256, ["2", "0", "3.5", "2"], "neither fading nor degrees"),
                            (g256, ["2", "0", "0", "3"], "nbgpu_split_qam"), (g256, ["2", "0", "0", "8"], "nbgpu_split_qam"),
                            (g64, ["2", "0", "0", "2"], "nbgpu_split_qam"), (g256, ["2", "0", "0", "0"], "must be >= 1")):
        r = subprocess.run([EXE, "10", "10", path, "3.0", "20", "0.3", "25", "8", "0", "0", "1", *tail],
                           cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode != 0 and msg in r.stdout, (tail, r.stdout[-2000:])
        assert "AllocateDecoder" not in r.stdout and "LDPC code parameters" not in r.stdout, tail


def test_split_abi_without_a_gpu():
    L = C.CDLL(nbldpc.LIB_PATH)
    for name in ("nbgpu_split_qam", "nbgpu_awgn_split_noise", "nbgpu_set_split_constellation", "nbgpu_channel_split",
                 "nbgpu_decode_split", "nbgpu_upload_split", "nbgpu_source_frames_split"):
        assert hasattr(L, name), name
    lib = nbldpc.lib()
    assert lib.nbgpu_set_split_constellation(None, 2, None) == nbldpc.EINVAL
    assert lib.nbgpu_decode_split(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    assert lib.nbgpu_upload_split(None, None, C.c_float(1.0), 1) == nbldpc.EINVAL
    assert lib.nbgpu_channel_split(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    assert lib.nbgpu_source_frames_split(None, None, None, 0, 1, C.c_float(1.0)) == nbldpc.EINVAL


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_channel_split_equals_the_definition(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    img = images(code)
    B = 5
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    for P in POINTS[q]:
        for mod in tables(q, P):
            d.set_split_constellation(mod, P)
            ebn = ESN[size(q, P)]
            _, _, noisy = host_split(code, 3, B, ebn, mod, P)
            sigma = nbldpc.sigma_apsk64(ebn)
            llr, il, ig = d.channel_split(noisy, sigma, want_sorted=True)
            for f in range(B):
                ref = split_llr(noisy[f], mod, img, P, sigma)
                assert llr[f].tobytes() == ref.tobytes(), (P, f)
                ril, rig = o.sort_intrinsic(ref)
                assert il[f].tobytes() == ril.tobytes() and (ig[f] == rig).all(), (P, f)
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("q,P,early,ecn", [(16, 2, True, 0), (16, 4, False, 0), (64, 3, True, 0), (64, 2, False, 0),
                                           (256, 2, True, 0), (256, 4, False, 0), (256, 8, True, 0), (16, 2, True, 1),
                                           (256, 4, True, 1)])
def test_decode_split_equals_decode_llr_and_the_oracle(q, P, early, ecn):
    """decode_split (streamed) and upload_split + run (resident) on batches of more than two waves, frame for frame against
    decode_llr on the defined LLRs and the oracle's decode loop fed with them; LIST and BITS soft output against decode_llr"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    n_m = 16 if q == 16 else 20
    kw = dict(ecn_kind=1, d1=n_m - 1, d2=min(15, n_m - 1), d3=5, cfg_trunc=1000, n_cv=25) if ecn else {}
    cfg = o.build_config_table(int(code.row_deg[0]), n_m - 1, min(15, n_m - 1), 5, 1000) if ecn else None
    B = waves(code, n_m, early, **kw)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    mod = tables(q, P)[0]
    d.set_split_constellation(mod, P)
    ebn = ESN[size(q, P)]
    _, _, noisy = host_split(code, 40, B, ebn, mod, P)
    sigma = nbldpc.sigma_apsk64(ebn)
    img = images(code)
    llr = np.stack([split_llr(noisy[f], mod, img, P, sigma) for f in range(B)])
    ref = d.decode_llr(llr)
    got = d.decode_split(noisy, sigma)
    assert all((x == y).all() for x, y in zip(got, ref))
    d.upload_split(noisy, sigma); d.run()
    assert all((x == y).all() for x, y in zip(d.download(), ref))
    dec, synd, it = got
    for f in range(B):
        r = o.decode_frame(llr[f], n_m, 25, 10, 0.3, force=not early, ecn=ecn, cfg=cfg, n_cv=25 if ecn else 0)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        d.decode_llr(llr); rsoft = soft(d, kind)
        d.decode_split(noisy, sigma)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), rsoft)), kind
        d.upload_split(noisy, sigma); d.run()
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), rsoft)), kind
    d.close(); o.close()


def _far(code, P):
    D = multigpu.draws_per_frame(code, "split", points=P)
    far = (1 << 32) // D + 1000
    assert far * D > 1 << 32
    return far


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_generated_split_frames_equal_the_host_stream_and_score_alike(q):
    code, _ = field_code(q)
    B = 160
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    bing = code.tables()[0]
    for P in POINTS[q]:
        mod = tables(q, P)[0]
        d.set_split_constellation(mod, P)
        ebn = ESN[size(q, P)]
        for frame0 in (0, 12345, _far(code, P)):
            d.source_frames_split(frame0, B, ebn)
            assert same_split_stream(d, code, frame0, B, ebn, mod, P), (P, frame0)
        d.run()
        errs, synd, it = d.source_results()
        _, bits, noisy = host_split(code, _far(code, P), B, ebn, mod, P)
        dec, hsynd, hit = d.decode_split(noisy, nbldpc.sigma_apsk64(ebn))
        herr = np.array([(bing[dec[f, :code.K]] != bits[f, :code.K]).sum() for f in range(B)])
        assert (errs == herr).all() and (synd == hsynd).all() and (it == hit).all(), P
    d.close()


@gpu
def test_flagged_split_samples_are_recomputed_from_the_split_table():
    code, _ = field_code(256)
    B = 64
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    for P in (2, 4):
        mod = tables(256, P)[0]
        d.set_split_constellation(mod, P)
        ebn = ESN[size(256, P)]
        d.source_set_margin(2.0 ** -46)
        d.source_frames_split(7, B, ebn)
        base = d.source_fixups()
        assert same_split_stream(d, code, 7, B, ebn, mod, P)
        d.source_set_margin(2.0 ** -20)
        d.source_frames_split(7, B, ebn)
        n = d.source_fixups()
        assert n > max(100, 50 * base) and n > 0.6 * B * code.N * 2 * P, (n, base)
        assert same_split_stream(d, code, 7, B, ebn, mod, P)
    d.close()


@gpu
def test_split_state_rules():
    code, _ = field_code(256)
    B = 32
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    qpsk, qam16 = nbldpc.split_qam(256, 4), nbldpc.split_qam(256, 2)
    noisy = np.zeros((B, code.N, 4, 2), np.float32)
    # no split table bound (a mapped table does not count): every split call is refused
    d.set_constellation(nbldpc.constellation(nbldpc.MAP_QAM, 256))
    calls = (lambda: d.decode_split(noisy, 0.5), lambda: d.upload_split(noisy, 0.5), lambda: d.channel_split(noisy, 0.5),
             lambda: d.source_frames_split(0, B, 4.0))
    for call in calls:
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE and "nbgpu_set_split_constellation" in str(e.value)
    # refusals leave the context unchanged: still no split table
    L = nbldpc.lib()
    for P, mod in ((3, qpsk), (1, qpsk), (0, qpsk), (16, qpsk), (4, np.full((4, 2), np.nan, np.float32)),
                   (2, np.where(np.arange(32).reshape(16, 2) == 21, np.inf, qam16).astype(np.float32))):
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.set_split_constellation(mod, P)
        assert e.value.code == nbldpc.EINVAL, P
    assert L.nbgpu_set_split_constellation(d.h, 4, None) == nbldpc.EINVAL
    for call in calls:
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE
    # a table of another size than 2^(log2 q / P) points is refused before the library sees it
    for mod, P in ((qpsk, 2), (qam16, 4)):
        with pytest.raises(ValueError):
            d.set_split_constellation(mod, P)
    for call in calls:
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE
    # bound; a refused re-binding keeps the table
    d.set_split_constellation(qpsk, 4)
    for call in (lambda: d.decode_split(noisy[:, :, :2], 0.5), lambda: d.upload_split(noisy.reshape(B, code.N, 8), 0.5),
                 lambda: d.channel_split(noisy[:, :, :2], 0.5)):   # frames of another P are not reinterpreted as more frames
        with pytest.raises(ValueError):
            call()
    with pytest.raises(nbldpc.NbgpuError):
        d.set_split_constellation(np.full((4, 2), -np.inf, np.float32), 4)
    d.source_frames_split(3, B, 4.0)
    assert same_split_stream(d, code, 3, B, 4.0, qpsk, 4)
    d.run(); ref = d.source_results()
    # nbgpu_set_constellation does not drop a split batch
    d.set_constellation(nbldpc.constellation(nbldpc.MAP_QAM, 256))
    d.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    # re-binding the split table drops it; its samples stay downloadable
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.source_frames_split(3, B, 4.0); d.run(); d.soft_bits()
    d.set_split_constellation(qam16, 2)
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.run()
    assert e.value.code == nbldpc.ESTATE and "split" in str(e.value)
    for call in (d.soft_bits, d.source_results):
        with pytest.raises(nbldpc.NbgpuError):
            call()
    assert same_split_stream(d, code, 3, B, 4.0, qpsk, 4)
    # ... and does not drop a mapped or a BPSK batch
    for gen in (lambda: d.source_frames_mapped(5, B, 20.0), lambda: d.source_frames(5, B, 3.0)):
        gen(); d.run(); ref = d.source_results()
        d.set_split_constellation(qpsk, 4)
        d.run()
        assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    # split batches of another P after re-binding, alternating with mapped ones
    d.set_split_constellation(qam16, 2)
    for _ in range(2):
        d.source_frames_split(11, B, 10.0)
        assert same_split_stream(d, code, 11, B, 10.0, qam16, 2)
        d.source_frames_mapped(11, B, 20.0)
        assert d.source_download()[1].shape == (B, code.N, 2)
    d.close()


@gpu
@pytest.mark.parametrize("q,P", [(16, 2), (256, 4)])
def test_c_driver_split_sources_contexts_and_monte_carlo_agree(tmp_path, q, P):
    code, path = field_code(q)
    esn = ESN[size(q, P)] + 1
    ebn = "%.1f" % esn
    out1, file1 = run_driver(tmp_path, "device", path, ebn, 16, 1, 2, "0", "0", str(P))
    out0, file0 = run_driver(tmp_path, "host", path, ebn, 16, 0, 2, "0", "0", str(P))
    out2, file2 = run_driver(tmp_path, "two_contexts", path, ebn, 16, 1, 2, "0", "0", str(P), devices="0,0")
    last = [re.findall(CONSOLE, o)[-1] for o in (out1, out0, out2)]
    assert last[0] == last[1] == last[2], last
    assert file1 == file0 == file2 and len(file1) == 1, (file1, file0, file2)
    mod = nbldpc.split_qam(q, P)
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=128)
    d.set_split_constellation(mod, P)
    for st in (multigpu.monte_carlo(code, 2000, esn, decode=d.decode_split, batch=128, channel="split", constellation=mod, points=P),
               multigpu.monte_carlo(code, 2000, esn, batch=128, decoder=d, channel="split", constellation=mod, points=P)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0][0]), int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]), st
    d.close()
    # an Es/N0 sweep equals its single points
    lo = esn - 1
    out, lines = run_driver(tmp_path, "sweep", path, "%.1f:%.1f:1" % (lo, lo + 1), 16, 1, 2, "0", "0", str(P))
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 2 and len(lines) == 2
    for i in range(2):
        o1, l1 = run_driver(tmp_path, "single%d" % i, path, "%.1f" % (lo + i), 16, 1, 2, "0", "0", str(P))
        assert re.findall(CONSOLE, o1)[-1] == re.findall(CONSOLE, blocks[i])[-1] and l1 == [lines[i]], (i, l1, lines[i])
