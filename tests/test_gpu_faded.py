"""The faded mapped channel: one GF(q) symbol per point of a q-point constellation, received through a real Rayleigh
amplitude known at the receiver, y_c = rho_c * m_c + sigma * n_c (NBGPU_FADING_SYMBOL: rho_I = rho_Q; NBGPU_FADING_COMPONENT:
independent, for rotated constellations), frames rx[N][4] = (y_I, y_Q, rho_I, rho_Q).  The header of the library defines
the channel; `oracle_noise_faded` and `oracle_llr_faded` below restate that definition on the oracle's drand48 and on numpy,
and the decoder is checked against the oracle's decode loop fed with `oracle_llr_faded`.  With rho = 1 the faded intake is
the mapped intake bit for bit."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import (CONSOLE, ESN, EXE, FADING_NAMES, PI, field_code, host_frames, matrix_path, multigpu, run_driver, same_stream,
                    seeded_table, soft, waves)

gpu = pytest.mark.gpu
KINDS = {"symbol": nbldpc.FADING_SYMBOL, "component": nbldpc.FADING_COMPONENT}
S = {nbldpc.FADING_SYMBOL: 5, nbldpc.FADING_COMPONENT: 6}       # draws per symbol
FADE_ESN = {16: 16.0, 64: 22.0, 256: 29.0}                       # average Es/N0 (dB) at which faded frames mix easy and hard ones
SSD_DEGREES = math.degrees(math.atan(1.0 / 16.0))               # 3.576 degrees: a rotation for 256-QAM under component fading


# ---- the channel as the header defines it ------------------------------------------------------------------------------
def oracle_noise_faded(o, nbin, mod, ebn, fading):
    """per symbol u_I, v_I, u_Q, v_Q, w_I (, w_Q) from the oracle's drand48 stream; rho = (float)sqrt(-log(w)),
    y_c = (float)((double)rho_c * m_c + sigma * sqrt(-2 ln u_c) * cos(2 PI v_c))"""
    sigma = o.sigma_apsk64(ebn)
    logq = nbin.shape[1]
    rx = np.zeros((nbin.shape[0], 4), np.float32)
    for n in range(nbin.shape[0]):
        som = sum(int(nbin[n, b]) << b for b in range(logq))
        d = [float(np.float32(o.drand48())) for _ in range(S[fading])]
        rho = [np.float32(math.sqrt(-math.log(d[4])))]
        rho.append(np.float32(math.sqrt(-math.log(d[5]))) if fading == nbldpc.FADING_COMPONENT else rho[0])
        for c in range(2):
            u, v = d[2 * c], d[2 * c + 1]
            rx[n, c] = np.float32(float(rho[c]) * float(mod[som, c]) + sigma * math.sqrt(-2.0 * math.log(u)) * math.cos(2.0 * PI * v))
        rx[n, 2:] = rho
    return rx


def oracle_llr_faded(o, rx, mod, sigma):
    """f32 products rho * m, differences and squares; f64 divisions by 2 (float)(sigma^2) and sum, rounded to f32"""
    img = (o.bingf.astype(np.int64) << np.arange(o.bingf.shape[1])).sum(1)
    den = 2.0 * float(np.float32(sigma) * np.float32(sigma))
    rx = rx.astype(np.float32)
    p0 = (rx[:, 2:3] * mod[img, 0][None, :]).astype(np.float32)
    p1 = (rx[:, 3:4] * mod[img, 1][None, :]).astype(np.float32)
    d0 = (rx[:, 0:1] - p0).astype(np.float32)
    d1 = (rx[:, 1:2] - p1).astype(np.float32)
    a = (d0 * d0).astype(np.float64) / den
    b = (d1 * d1).astype(np.float64) / den
    return (a + b).astype(np.float32)


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("q", [16, 64, 256])
def test_host_faded_noise_equals_the_oracle(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    nbin = np.random.default_rng(q + 1).integers(0, 2, (code.N, code.logq)).astype(np.int32)
    for mod in (nbldpc.constellation(nbldpc.MAP_QAM, q), seeded_table(q)):
        for fading in (nbldpc.FADING_SYMBOL, nbldpc.FADING_COMPONENT):
            for ebn in (FADE_ESN[q] - 6, FADE_ESN[q]):
                code.rng_default(); code.rng_skip(4321)
                got = code.noise_faded(nbin, mod, ebn, fading)
                o.rng_default(); o.rng_skip(4321)
                assert got.tobytes() == oracle_noise_faded(o, nbin, mod, ebn, fading).tobytes(), (fading, ebn)
                # exactly S*N draws: the next draw is draw S*N of the stream
                o.rng_default(); o.rng_skip(4321 + S[fading] * code.N)
                assert code.drand48() == o.drand48()
                if fading == nbldpc.FADING_SYMBOL:
                    assert (got[:, 2] == got[:, 3]).all()
                else:
                    assert (got[:, 2] != got[:, 3]).mean() > 0.9
                assert (got[:, 2:] >= 0).all()
    # the all-zero word, a bad fading value and the NULL refusals
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    code.rng_default()
    z = code.noise_faded(None, mod, 12.0, nbldpc.FADING_COMPONENT)
    o.rng_default()
    assert z.tobytes() == oracle_noise_faded(o, np.zeros((code.N, code.logq), np.int32), mod, 12.0, nbldpc.FADING_COMPONENT).tobytes()
    for bad in (0, 3, -1):
        with pytest.raises(nbldpc.NbgpuError) as e:
            code.noise_faded(None, mod, 12.0, bad)
        assert e.value.code == nbldpc.EINVAL
    L, fp = nbldpc.lib(), z.ctypes.data_as(C.POINTER(C.c_float))
    mp = mod.ctypes.data_as(C.POINTER(C.c_float))
    assert L.nbgpu_awgn_faded_noise(code.h, C.byref(code.rng), None, None, C.c_float(5.0), 1, fp) == nbldpc.EINVAL
    assert L.nbgpu_awgn_faded_noise(None, C.byref(code.rng), None, mp, C.c_float(5.0), 1, fp) == nbldpc.EINVAL
    assert L.nbgpu_awgn_faded_noise(code.h, C.byref(code.rng), None, mp, C.c_float(5.0), 1, None) == nbldpc.EINVAL
    o.close()


def test_rayleigh_amplitudes_have_unit_mean_power():
    code, _ = field_code(256)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 256)
    code.rng_default()
    rho = np.concatenate([code.noise_faded(None, mod, 20.0, nbldpc.FADING_COMPONENT)[:, 2:].ravel() for _ in range(4200)])
    assert rho.size >= 10 ** 5
    assert abs(float((rho.astype(np.float64) ** 2).mean()) - 1.0) < 0.02
    # Rayleigh: P(rho^2 < x) = 1 - exp(-x)
    for x in (0.1, 1.0, 3.0):
        assert abs(float((rho.astype(np.float64) ** 2 < x).mean()) - (1 - math.exp(-x))) < 0.01, x


@pytest.mark.parametrize("fading", ["symbol", "component"])
def test_draws_per_frame_faded_skips_whole_frames(fading):
    code, _ = field_code(256)
    fd = KINDS[fading]
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 256)
    D = multigpu.draws_per_frame(code, "mapped", fading=fading)
    assert D == code.K * 8 + S[fd] * code.N
    _, _, rx = host_frames(code, 0, 7, 25.0, "mapped", mod, fd)
    for f in (1, 3, 6):
        code.rng_default(); code.rng_skip(f * D)
        _, nb = code.random_codeword()
        assert code.noise_faded(nb, mod, 25.0, fd).tobytes() == rx[f].tobytes()


def test_fading_is_a_property_of_the_mapped_channel_only():
    code, _ = field_code(64)
    for ch in ("bpsk", "apsk64"):
        with pytest.raises(ValueError):
            multigpu.draws_per_frame(code, ch, fading="symbol")
        with pytest.raises(ValueError):
            multigpu.monte_carlo(code, 10, 5.0, decode=lambda *a: None, channel=ch, fading="symbol")
    for bad in ("rayleigh", 1):
        with pytest.raises(ValueError):
            multigpu.draws_per_frame(code, "mapped", fading=bad)
    for ch in ("qam16", "faded"):
        with pytest.raises(ValueError):
            multigpu.draws_per_frame(code, ch)
    assert multigpu.draws_per_frame(code, "mapped", fading=None) == multigpu.draws_per_frame(code, "mapped")


@pytest.mark.parametrize("q", [16, 64, 256])
def test_rotate_constellation(q):
    qam = nbldpc.constellation(nbldpc.MAP_QAM, q)
    for mod in (qam, seeded_table(q)):
        assert nbldpc.rotate_constellation(mod, 0.0).tobytes() == mod.tobytes()
        for deg in (SSD_DEGREES, -31.7, 90.0, 400.0):
            got = nbldpc.rotate_constellation(mod, deg)
            t = math.radians(deg)
            c, s = math.cos(t), math.sin(t)
            ref = np.array([[np.float32(float(i) * c - float(k) * s), np.float32(float(i) * s + float(k) * c)] for i, k in mod], np.float32)
            assert got.tobytes() == ref.tobytes(), deg
    p = (nbldpc.rotate_constellation(qam, SSD_DEGREES).astype(np.float64) ** 2).sum(1).mean()
    assert abs(p - 1.0) < 1e-6
    # in place
    L = nbldpc.lib()
    buf = qam.copy()
    fp = buf.ctypes.data_as(C.POINTER(C.c_float))
    assert L.nbgpu_rotate_constellation(q, C.c_double(SSD_DEGREES), fp, fp) == nbldpc.OK
    assert buf.tobytes() == nbldpc.rotate_constellation(qam, SSD_DEGREES).tobytes()


def test_rotate_constellation_refusals():
    L = nbldpc.lib()
    src = np.ones((256, 2), np.float32)
    out = np.zeros((256, 2), np.float32)
    sp, op = src.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float))
    for q, deg, a, b in ((32, 1.0, sp, op), (4, 1.0, sp, op), (0, 1.0, sp, op), (16, 1.0, None, op), (16, 1.0, sp, None),
                         (16, math.nan, sp, op), (16, math.inf, sp, op), (16, -math.inf, sp, op)):
        assert L.nbgpu_rotate_constellation(q, C.c_double(deg), a, b) == nbldpc.EINVAL, (q, deg)
        assert L.nbgpu_last_error(None)
    assert not out.any()
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.rotate_constellation(np.ones((32, 2), np.float32), 1.0)


def test_faded_abi_without_a_gpu():
    assert (nbldpc.FADING_SYMBOL, nbldpc.FADING_COMPONENT) == (1, 2)
    L = nbldpc.lib()
    for name in ("nbgpu_rotate_constellation", "nbgpu_awgn_faded_noise", "nbgpu_channel_faded", "nbgpu_decode_faded",
                 "nbgpu_upload_faded", "nbgpu_source_frames_faded"):
        assert hasattr(C.CDLL(nbldpc.LIB_PATH), name), name
    assert L.nbgpu_decode_faded(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    assert L.nbgpu_upload_faded(None, None, C.c_float(1.0), 1) == nbldpc.EINVAL
    assert L.nbgpu_channel_faded(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    for fading in (1, 2, 0, 3):
        assert L.nbgpu_source_frames_faded(None, None, None, 0, 1, C.c_float(1.0), fading) == nbldpc.EINVAL


def test_c_driver_refuses_fading_without_a_constellation_before_any_device(tmp_path):
    assert os.path.exists(EXE)
    path = matrix_path("matrices/KN/N96_K48_GF256.txt")
    for tail, msg in ((["0", "1"], "not to BPSK"), (["0", "0", "10"], "not to BPSK"), (["2", "3"], "fading must be 0"),
                      (["2", "-1"], "fading must be 0"), (["3", "1"], "channel must be 0")):
        r = subprocess.run([EXE, "10", "10", path, "3.0", "20", "0.3", "25", "8", "0", "0", "1"] + tail,
                           cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode != 0 and msg in r.stdout, (tail, r.stdout[-2000:])
        assert "AllocateDecoder" not in r.stdout and "LDPC code parameters" not in r.stdout


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_channel_faded_equals_the_oracle(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    B = 6
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    rng = np.random.default_rng(q)
    for mod in (nbldpc.rotate_constellation(nbldpc.constellation(nbldpc.MAP_QAM, q), 11.0), seeded_table(q)):
        d.set_constellation(mod)
        for fading in (nbldpc.FADING_SYMBOL, nbldpc.FADING_COMPONENT):
            _, _, rx = host_frames(code, 5, B, FADE_ESN[q] - 4, "mapped", mod, fading)
            # channel state the stream never makes: erased (0), negative, large, and -0
            n = rx.shape[0] * rx.shape[1]
            flat = rx.reshape(n, 4)
            pick = rng.permutation(n)
            flat[pick[:n // 10], 2:] = 0.0
            flat[pick[n // 10:n // 5], 2] = -0.75
            flat[pick[n // 5:n // 4], 3] = 1.0e3
            flat[pick[n // 4:n // 4 + 5], 2:] = -0.0
            sigma = nbldpc.sigma_apsk64(FADE_ESN[q] - 4)
            llr, il, ig = d.channel_faded(rx, sigma, want_sorted=True)
            for f in range(B):
                ref = oracle_llr_faded(o, rx[f], mod, sigma)
                assert llr[f].tobytes() == ref.tobytes(), (fading, f)
                ril, rig = o.sort_intrinsic(ref)
                assert il[f].tobytes() == ril.tobytes() and (ig[f] == rig).all(), (fading, f)
            erased = (rx[..., 2] == 0) & (rx[..., 3] == 0)
            assert erased.any() and (llr[erased] == llr[erased][:, :1]).all()        # an erased symbol's row is constant
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("q", [16, 256])
def test_faded_intake_with_unit_amplitudes_is_the_mapped_intake(q):
    """rho = 1: decode_faded equals decode_mapped bit for bit (decisions, syndromes, iterations, LIST and BITS soft output),
    streamed and through upload_faded + run; channel_faded equals channel_mapped"""
    code, _ = field_code(q)
    n_m = 16 if q == 16 else 20
    B = waves(code, n_m)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B, frames_per_cta=1)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    d.set_constellation(mod)
    _, _, noisy = host_frames(code, 0, B, ESN[q], "mapped", mod)
    rx = np.concatenate([noisy, np.ones_like(noisy)], axis=2)
    sigma = nbldpc.sigma_apsk64(ESN[q])
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        ref = d.decode_mapped(noisy, sigma); rsoft = soft(d, kind)
        got = d.decode_faded(rx, sigma); gsoft = soft(d, kind)
        assert all((x == y).all() for x, y in zip(got, ref)) and all(x.tobytes() == y.tobytes() for x, y in zip(gsoft, rsoft))
        d.upload_faded(rx, sigma); d.run()
        assert all((x == y).all() for x, y in zip(d.download(), ref)) and all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), rsoft))
    assert len(set(ref[2].tolist())) > 1
    a = d.channel_mapped(noisy[:3], sigma, want_sorted=True)
    b = d.channel_faded(rx[:3], sigma, want_sorted=True)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    d.close()


@gpu
@pytest.mark.parametrize("q,early,ecn,fading,erase", [(16, True, 0, 1, False), (16, False, 0, 2, False), (256, True, 0, 2, False),
                                                      (256, False, 0, 1, False), (16, True, 1, 2, False), (256, True, 1, 1, False),
                                                      (256, True, 0, 1, True)])
def test_decode_faded_equals_the_oracle(q, early, ecn, fading, erase):
    """decode_faded (streamed) and upload_faded + run on batches of more than two waves, frame for frame against the oracle's
    decode loop on oracle_llr_faded; L-Bubble and the syndrome-based check node; one case with ~10 % erased symbols"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    n_m = 16 if q == 16 else 20
    kw = dict(ecn_kind=1, d1=n_m - 1, d2=min(15, n_m - 1), d3=5, cfg_trunc=1000, n_cv=25) if ecn else {}
    cfg = o.build_config_table(int(code.row_deg[0]), n_m - 1, min(15, n_m - 1), 5, 1000) if ecn else None
    B = waves(code, n_m, early, **kw)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    if fading == nbldpc.FADING_COMPONENT:
        mod = nbldpc.rotate_constellation(mod, SSD_DEGREES)
    d.set_constellation(mod)
    ebn = FADE_ESN[q]
    _, _, rx = host_frames(code, 60, B, ebn, "mapped", mod, fading)
    if erase:
        er = np.random.default_rng(3).random(rx.shape[:2]) < 0.1
        rx[er, 2:] = 0.0
    sigma = nbldpc.sigma_apsk64(ebn)
    dec, synd, it = d.decode_faded(rx, sigma)
    d.upload_faded(rx, sigma); d.run()
    dec2, synd2, it2 = d.download()
    assert (dec2 == dec).all() and (synd2 == synd).all() and (it2 == it).all()
    for f in range(B):
        r = o.decode_frame(oracle_llr_faded(o, rx[f], mod, sigma), n_m, 25, 10, 0.3, force=not early,
                           ecn=ecn, cfg=cfg, n_cv=25 if ecn else 0)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_generated_faded_frames_equal_the_host_stream(q):
    code, _ = field_code(q)
    B = 200
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    d.set_constellation(mod)
    for fading in (nbldpc.FADING_SYMBOL, nbldpc.FADING_COMPONENT):
        D = multigpu.draws_per_frame(code, "mapped", fading=FADING_NAMES[fading])
        far = (1 << 32) // D + 1000
        for frame0 in (0, 12345, far):
            d.source_frames_faded(frame0, B, FADE_ESN[q], fading)
            assert same_stream(d, code, frame0, B, FADE_ESN[q], "mapped", mod, fading), (fading, frame0)
        # the widest margin flags many symbols; each is recomputed whole and the stream is unchanged
        base = d.source_fixups()
        d.source_set_margin(2.0 ** -20)
        d.source_frames_faded(7, B, FADE_ESN[q] - 5, fading)
        n = d.source_fixups()
        assert n > max(100, 50 * base) and n > 0.5 * B * code.N, (n, base)
        assert same_stream(d, code, 7, B, FADE_ESN[q] - 5, "mapped", mod, fading)
        d.source_set_margin(2.0 ** -46)
    d.close()


@gpu
def test_faded_state_rules():
    code, _ = field_code(64)
    B = 32
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    qam, apsk = nbldpc.constellation(nbldpc.MAP_QAM, 64), nbldpc.apsk64_table()
    rx = np.zeros((B, code.N, 4), np.float32)
    # no table bound: every faded call is refused
    for call in (lambda: d.decode_faded(rx, 0.5), lambda: d.upload_faded(rx, 0.5), lambda: d.channel_faded(rx, 0.5),
                 lambda: d.source_frames_faded(0, B, 10.0, nbldpc.FADING_SYMBOL)):
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE and "nbgpu_set_constellation" in str(e.value)
    d.set_constellation(qam)
    # a bad fading value is refused and leaves the resident batch alone
    d.source_frames_faded(3, B, 20.0, nbldpc.FADING_SYMBOL)
    for bad in (0, 3, -2):
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.source_frames_faded(3, B, 20.0, bad)
        assert e.value.code == nbldpc.EINVAL
    assert same_stream(d, code, 3, B, 20.0, "mapped", qam, nbldpc.FADING_SYMBOL)
    d.run()
    d.source_results()
    # re-binding drops the resident faded batch, generated or uploaded ...
    d.set_soft_output(nbldpc.SOFT_BITS)
    for make in (lambda: d.source_frames_faded(3, B, 20.0, nbldpc.FADING_COMPONENT),
                 lambda: d.upload_faded(host_frames(code, 3, B, 20.0, "mapped", qam, nbldpc.FADING_SYMBOL)[2], 0.1)):
        make(); d.run(); d.soft_bits()
        d.set_constellation(qam)
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.run()
        assert e.value.code == nbldpc.ESTATE and "faded" in str(e.value)
        for call in (d.soft_bits, d.source_results):
            with pytest.raises(nbldpc.NbgpuError):
                call()
    # ... but not a BPSK or a 64-APSK one
    d.source_frames(5, B, 3.0); d.run(); ref = d.source_results()
    d.set_constellation(qam)
    d.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    d.source_frames_apsk64(5, B, 8.0); d.run(); ref = d.source_results()
    d.set_constellation(apsk)
    d.run()
    assert all((x == y).all() for x, y in zip(d.source_results(), ref))
    # BPSK, LLR, 64-APSK, mapped and faded batches alternate on one context
    d.set_constellation(qam)
    _, _, mn = host_frames(code, 11, B, 14.0, "mapped", qam)
    llr = d.channel_mapped(mn, nbldpc.sigma_apsk64(14.0))
    rm = d.decode_mapped(mn, nbldpc.sigma_apsk64(14.0))
    for _ in range(2):
        d.source_frames(900, B, 2.5)
        assert d.source_download()[1].shape == (B, code.N, 6)
        assert all((x == y).all() for x, y in zip(d.decode_llr(llr), rm))
        d.source_frames_apsk64(11, B, 8.5)
        assert d.source_download()[1].shape == (B, code.N, 2)
        d.source_frames_mapped(11, B, 14.0)
        d.run()
        assert (d.download()[0] == rm[0]).all()
        for fading in (nbldpc.FADING_SYMBOL, nbldpc.FADING_COMPONENT):
            d.source_frames_faded(11, B, 20.0, fading)
            assert same_stream(d, code, 11, B, 20.0, "mapped", qam, fading)
            d.run()
            d.source_results()
    d.close()


@gpu
@pytest.mark.parametrize("q,fading", [(16, nbldpc.FADING_SYMBOL), (256, nbldpc.FADING_COMPONENT)])
def test_soft_output_of_generated_faded_batch_equals_host_frames(q, fading):
    code, _ = field_code(q)
    B, ebn = 48, FADE_ESN[q]
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    _, _, rx = host_frames(code, 20, B, ebn, "mapped", mod, fading)
    sigma = nbldpc.sigma_apsk64(ebn)
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=B)
    d.set_constellation(mod)
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        d.decode_faded(rx, sigma)
        ref = soft(d, kind)
        d.source_frames_faded(20, B, ebn, fading)
        d.run()
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), ref)), kind
    d.close()


@gpu
@pytest.mark.parametrize("q,fading,degrees", [(16, 1, "0"), (256, 2, "3.576")])
def test_c_driver_faded_sources_contexts_and_monte_carlo_agree(tmp_path, q, fading, degrees):
    code, path = field_code(q)
    esn, n_m = FADE_ESN[q], (16 if q == 16 else 20)
    out1, file1 = run_driver(tmp_path, "device", path, "%.1f" % esn, n_m, 1, 2, str(fading), degrees)
    out0, file0 = run_driver(tmp_path, "host", path, "%.1f" % esn, n_m, 0, 2, str(fading), degrees)
    out2, file2 = run_driver(tmp_path, "two_contexts", path, "%.1f" % esn, n_m, 1, 2, str(fading), degrees, devices="0,0")
    last = [re.findall(CONSOLE, o)[-1] for o in (out1, out0, out2)]
    assert last[0] == last[1] == last[2], last
    assert file1 == file0 == file2 and len(file1) == 1, (file1, file0, file2)
    mod = nbldpc.rotate_constellation(nbldpc.constellation(nbldpc.MAP_QAM, q), float(degrees))
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=128)
    d.set_constellation(mod)
    kw = dict(batch=128, channel="mapped", constellation=mod, fading=FADING_NAMES[fading])
    for st in (multigpu.monte_carlo(code, 2000, esn, decode=d.decode_faded, **kw), multigpu.monte_carlo(code, 2000, esn, decoder=d, **kw)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0][0]), int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]), st
    d.close()
    # a two-point sweep equals its single points
    lo = esn - 2
    out, lines = run_driver(tmp_path, "sweep", path, "%.1f:%.1f:2" % (lo, lo + 2), n_m, 1, 2, str(fading), degrees)
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 2 and len(lines) == 2
    for i in range(2):
        o1, l1 = run_driver(tmp_path, "single%d" % i, path, "%.1f" % (lo + 2 * i), n_m, 1, 2, str(fading), degrees)
        assert re.findall(CONSOLE, o1)[-1] == re.findall(CONSOLE, blocks[i])[-1] and l1 == [lines[i]], (i, l1, lines[i])


@gpu
def test_rayleigh_fading_costs_frames_that_awgn_does_not():
    """on the fixed stream: at the lowest Es/N0 of a 1 dB grid where 256-QAM over AWGN decodes every one of 384 frames, symbol
    fading loses many (on this short code both channels are error-free a few dB higher, so the point is found from below)"""
    code, _ = field_code(256)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 256)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=128)
    first = 16.0
    for esn in np.arange(first, 31.0):
        awgn = multigpu.monte_carlo(code, 384, esn, batch=128, decoder=d, channel="mapped", constellation=mod)
        if awgn["err_frames"] == 0:
            break
    assert awgn["err_frames"] == 0 and esn > first, (esn, awgn)           # found, and AWGN lost frames 1 dB lower
    faded = multigpu.monte_carlo(code, 384, esn, batch=128, decoder=d, channel="mapped", constellation=mod, fading="symbol")
    assert faded["err_frames"] >= 10, (esn, faded)
    d.close()
