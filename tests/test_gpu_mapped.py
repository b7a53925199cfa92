"""The mapped channel: one GF(q) symbol sent as one point of a q-point constellation mod[q][2] (nbgpu_constellation,
nbgpu_set_constellation and the *_mapped calls), for GF(16), GF(64) and GF(256).  64-APSK is the mapped channel on the
64-APSK table, so with that table every mapped call reproduces its *_apsk64 counterpart bit for bit; with Gray square QAM
and other tables the results are checked against `oracle_noise_mapped` below and `common.oracle_llr_mapped`, the table-taking
forms of the oracle's 64-APSK noise and LLR, which the CPU tests pin to the oracle's own 64-APSK functions on the APSK table."""
import ctypes as C
import math
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import (CONSOLE, ESN, EXE, PI, field_code, host_frames, matrix_path, multigpu, oracle_llr_mapped, run_driver,
                    same_stream, seeded_table, soft, waves)

gpu = pytest.mark.gpu


# ---- the oracle's mapped channel (the 64-APSK functions of oracle/nbldpc_oracle.c with the table as an argument) ----------
def qam_closed_form(q):
    L = int(round(math.sqrt(q))); m = L.bit_length() - 1
    mod = np.zeros((q, 2), np.float32)
    for x in range(q):
        for c in range(2):
            g = (x >> (c * m)) & (L - 1)
            level = 0
            while g:                                           # inverse binary-reflected Gray code
                level ^= g; g >>= 1
            mod[x, c] = np.float32((2 * level - (L - 1)) / math.sqrt(2 * (q - 1) / 3))
    return mod


def oracle_noise_mapped(o, nbin, mod, ebn):
    """channel.c:234-263 on mod: per symbol u, v for I then u, v for Q from the oracle's drand48 stream"""
    sigma = o.sigma_apsk64(ebn)
    logq = nbin.shape[1]
    noisy = np.zeros((nbin.shape[0], 2), np.float32)
    for n in range(nbin.shape[0]):
        som = sum(int(nbin[n, b]) << b for b in range(logq))
        for c in range(2):
            u = float(np.float32(o.drand48())); v = float(np.float32(o.drand48()))
            noisy[n, c] = np.float32(float(mod[som, c]) + sigma * math.sqrt(-2.0 * math.log(u)) * math.cos(2.0 * PI * v))
    return noisy


# ---- CPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("q", [16, 64, 256])
def test_qam_table_is_the_closed_form_gray_labelled_and_unit_power(q):
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    assert mod.shape == (q, 2) and mod.tobytes() == qam_closed_form(q).tobytes()
    assert abs(float((mod.astype(np.float64) ** 2).sum(1).mean()) - 1.0) < 1e-6
    L = int(round(math.sqrt(q)))
    for c in range(2):                                         # nearest neighbours on each axis differ in one bit
        other = mod[:, 1 - c]
        for x in range(q):
            same_line = np.flatnonzero(other == other[x])
            assert len(same_line) == L
            order = same_line[np.argsort(mod[same_line, c])]
            for a, b in zip(order[:-1], order[1:]):
                assert bin(int(a) ^ int(b)).count("1") == 1, (c, a, b)


def test_constellation_kinds_and_refusals():
    assert nbldpc.constellation(nbldpc.MAP_APSK64, 64).tobytes() == nbldpc.apsk64_table().tobytes()
    lib = nbldpc.lib()
    buf = np.zeros((256, 2), np.float32)
    fp = buf.ctypes.data_as(C.POINTER(C.c_float))
    for kind, q in ((nbldpc.MAP_APSK64, 16), (nbldpc.MAP_APSK64, 256), (nbldpc.MAP_QAM, 32), (nbldpc.MAP_QAM, 4), (0, 64), (3, 64)):
        assert lib.nbgpu_constellation(kind, q, fp) == nbldpc.EINVAL, (kind, q)
        assert lib.nbgpu_last_error(None)
    assert lib.nbgpu_constellation(nbldpc.MAP_QAM, 16, None) == nbldpc.EINVAL
    assert not buf.any()


def test_oracle_mapped_forms_are_the_oracle_apsk64_functions():
    """on the APSK table the Python mapped forms reproduce nbo_channel_noise_apsk64 / nbo_channel_llr_apsk64 bit for bit"""
    path = matrix_path("matrices/N96_K48_GF64")
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    mod = o.apsk64_table()
    assert mod.tobytes() == nbldpc.apsk64_table().tobytes()
    nbin = np.random.default_rng(1).integers(0, 2, (code.N, 6)).astype(np.int32)
    for ebn in (4.0, 9.0):
        o.rng_default(); o.rng_skip(777)
        ref = o.channel_noise_apsk64(nbin, ebn)
        o.rng_default(); o.rng_skip(777)
        got = oracle_noise_mapped(o, nbin, mod, ebn)
        assert got.tobytes() == ref.tobytes()
        sigma = o.sigma_apsk64(ebn)
        assert oracle_llr_mapped(o, ref, mod, sigma).tobytes() == o.channel_llr_apsk64(ref, sigma).tobytes()
    o.close()


@pytest.mark.parametrize("q", [16, 64, 256])
def test_host_mapped_noise_equals_apsk64_and_the_oracle(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    nbin = np.random.default_rng(q).integers(0, 2, (code.N, code.logq)).astype(np.int32)
    tables = [nbldpc.constellation(nbldpc.MAP_QAM, q), seeded_table(q)]
    if q == 64:                                                # the APSK table through the generic path = the 64-APSK stream
        code.rng_default(); code.rng_skip(99)
        ref = code.noise_apsk64(nbin, 8.0)
        code.rng_default(); code.rng_skip(99)
        assert code.noise_mapped(nbin, nbldpc.apsk64_table(), 8.0).tobytes() == ref.tobytes()
    for mod in tables:
        for ebn in (ESN[q] - 4, ESN[q]):
            code.rng_default(); code.rng_skip(1234)
            got = code.noise_mapped(nbin, mod, ebn)
            o.rng_default(); o.rng_skip(1234)
            assert got.tobytes() == oracle_noise_mapped(o, nbin, mod, ebn).tobytes(), ebn
            # exactly 4N draws: the next draw is draw 4N of the stream
            o.rng_default(); o.rng_skip(1234 + 4 * code.N)
            assert code.drand48() == o.drand48()
    # the all-zero word, and the NULL refusals
    code.rng_default()
    z = code.noise_mapped(None, tables[0], 5.0)
    o.rng_default()
    assert z.tobytes() == oracle_noise_mapped(o, np.zeros((code.N, code.logq), np.int32), tables[0], 5.0).tobytes()
    fp = z.ctypes.data_as(C.POINTER(C.c_float))
    assert nbldpc.lib().nbgpu_awgn_mapped_noise(code.h, C.byref(code.rng), None, None, C.c_float(5.0), fp) == nbldpc.EINVAL
    assert nbldpc.lib().nbgpu_awgn_mapped_noise(None, C.byref(code.rng), None, tables[0].ctypes.data_as(C.POINTER(C.c_float)),
                                                C.c_float(5.0), fp) == nbldpc.EINVAL
    o.close()


def test_draws_per_frame_mapped_skips_whole_frames():
    code, _ = field_code(256)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 256)
    D = multigpu.draws_per_frame(code, "mapped")
    assert D == code.K * 8 + 4 * code.N
    _, _, noisy = host_frames(code, 0, 7, 20.0, "mapped", mod)
    for f in (1, 3, 6):
        code.rng_default(); code.rng_skip(f * D)
        _, nb = code.random_codeword()
        assert code.noise_mapped(nb, mod, 20.0).tobytes() == noisy[f].tobytes()


def test_c_driver_refuses_channel_3_before_any_device(tmp_path):
    assert os.path.exists(EXE)
    r = subprocess.run([EXE, "10", "10", matrix_path("matrices/KN/N96_K48_GF256.txt"), "3.0", "20", "0.3", "25", "8", "0", "0", "1", "3"],
                       cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode != 0 and "channel must be 0" in r.stdout, r.stdout[-2000:]
    assert "AllocateDecoder" not in r.stdout and "LDPC code parameters" not in r.stdout


def test_mapped_abi_without_a_gpu():
    L = C.CDLL(nbldpc.LIB_PATH)
    for name in ("nbgpu_constellation", "nbgpu_awgn_mapped_noise", "nbgpu_set_constellation", "nbgpu_channel_awgn_mapped",
                 "nbgpu_decode_mapped", "nbgpu_upload_mapped", "nbgpu_source_frames_mapped"):
        assert hasattr(L, name), name
    assert (nbldpc.MAP_APSK64, nbldpc.MAP_QAM) == (1, 2)
    lib = nbldpc.lib()
    assert lib.nbgpu_set_constellation(None, None) == nbldpc.EINVAL
    assert lib.nbgpu_decode_mapped(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    assert lib.nbgpu_upload_mapped(None, None, C.c_float(1.0), 1) == nbldpc.EINVAL
    assert lib.nbgpu_channel_awgn_mapped(None, None, C.c_float(1.0), 1, None, None, None) == nbldpc.EINVAL
    assert lib.nbgpu_source_frames_mapped(None, None, None, 0, 1, C.c_float(1.0)) == nbldpc.EINVAL


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_channel_mapped_equals_the_oracle(q):
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    B = 6
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    tables = [nbldpc.constellation(nbldpc.MAP_QAM, q), seeded_table(q)] + ([nbldpc.apsk64_table()] if q == 64 else [])
    for mod in tables:
        d.set_constellation(mod)
        _, _, noisy = host_frames(code, 3, B, ESN[q] - 3, "mapped", mod)
        sigma = nbldpc.sigma_apsk64(ESN[q] - 3)
        llr, il, ig = d.channel_mapped(noisy, sigma, want_sorted=True)
        for f in range(B):
            ref = oracle_llr_mapped(o, noisy[f], mod, sigma)
            assert llr[f].tobytes() == ref.tobytes(), f
            ril, rig = o.sort_intrinsic(ref)
            assert il[f].tobytes() == ril.tobytes() and (ig[f] == rig).all(), f
    if q == 64:                                                # the last table was the APSK one
        a = d.channel_apsk64(noisy, sigma, want_sorted=True)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(a, (llr, il, ig)))
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("early", [True, False])
def test_decode_mapped_with_the_apsk_table_equals_decode_apsk64(early):
    code, _ = field_code(64)
    mod = nbldpc.apsk64_table()
    B = waves(code, 20, early)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1)
    d.set_constellation(mod)
    _, _, noisy = host_frames(code, 0, B, 8.0, "mapped", mod)
    sigma = nbldpc.sigma_apsk64(8.0)
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        ref = d.decode_apsk64(noisy, sigma); rsoft = soft(d, kind)
        got = d.decode_mapped(noisy, sigma); gsoft = soft(d, kind)
        assert all((x == y).all() for x, y in zip(got, ref)) and all(x.tobytes() == y.tobytes() for x, y in zip(gsoft, rsoft))
        d.upload_mapped(noisy, sigma); d.run()
        assert all((x == y).all() for x, y in zip(d.download(), ref)) and all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), rsoft))
    if early:
        assert len(set(ref[2].tolist())) > 1
    d.close()


@gpu
@pytest.mark.parametrize("q,early,ecn", [(16, True, 0), (16, False, 0), (256, True, 0), (256, False, 0), (16, True, 1), (256, True, 1)])
def test_decode_mapped_qam_equals_the_oracle(q, early, ecn):
    """decode_mapped (streamed) and upload_mapped + run (resident) on batches of more than two waves, frame for frame
    against the oracle's decode loop on the oracle's mapped LLRs; L-Bubble and the syndrome-based check node"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    n_m = 16 if q == 16 else 20
    kw = dict(ecn_kind=1, d1=n_m - 1, d2=min(15, n_m - 1), d3=5, cfg_trunc=1000, n_cv=25) if ecn else {}
    cfg = o.build_config_table(int(code.row_deg[0]), n_m - 1, min(15, n_m - 1), 5, 1000) if ecn else None
    B = waves(code, n_m, early, **kw)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    d.set_constellation(mod)
    ebn = ESN[q]
    _, _, noisy = host_frames(code, 40, B, ebn, "mapped", mod)
    sigma = nbldpc.sigma_apsk64(ebn)
    dec, synd, it = d.decode_mapped(noisy, sigma)
    d.upload_mapped(noisy, sigma); d.run()
    dec2, synd2, it2 = d.download()
    assert (dec2 == dec).all() and (synd2 == synd).all() and (it2 == it).all()
    for f in range(B):
        r = o.decode_frame(oracle_llr_mapped(o, noisy[f], mod, sigma), n_m, 25, 10, 0.3, force=not early,
                           ecn=ecn, cfg=cfg, n_cv=25 if ecn else 0)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    d.close(); o.close()


def _far(code):
    D = multigpu.draws_per_frame(code, "mapped")
    far = (1 << 32) // D + 1000
    assert far * D > 1 << 32
    return far


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_generated_mapped_frames_equal_the_host_stream(q):
    code, _ = field_code(q)
    B = 200
    d = nbldpc.Decoder(code, min(20, q), 25, 10, 0.3, max_batch=B)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    d.set_constellation(mod)
    for frame0 in (0, 12345, _far(code)):
        for ebn in (ESN[q] - 3, ESN[q]):
            d.source_frames_mapped(frame0, B, ebn)
            assert same_stream(d, code, frame0, B, ebn, "mapped", mod), (frame0, ebn)
    if q == 64:                                                # the APSK table bound: the 64-APSK stream
        d.set_constellation(nbldpc.apsk64_table())
        for frame0 in (0, _far(code)):
            d.source_frames_mapped(frame0, B, 8.0)
            _, a = d.source_download()
            d.source_frames_apsk64(frame0, B, 8.0)
            _, b = d.source_download()
            assert a.tobytes() == b.tobytes()
    d.close()


@gpu
def test_flagged_mapped_samples_are_recomputed_with_the_batch_table():
    code, _ = field_code(256)
    B, ebn = 64, 20.0
    mod = nbldpc.constellation(nbldpc.MAP_QAM, 256)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d.set_constellation(mod)
    d.source_frames_mapped(7, B, ebn)
    base = d.source_fixups()
    assert same_stream(d, code, 7, B, ebn, "mapped", mod)
    d.source_set_margin(2.0 ** -20)
    d.source_frames_mapped(7, B, ebn)
    n = d.source_fixups()
    assert n > max(100, 50 * base) and n > 0.6 * B * code.N * 2, (n, base)
    assert same_stream(d, code, 7, B, ebn, "mapped", mod)
    d.close()


@gpu
def test_mapped_state_rules():
    code, _ = field_code(64)
    B = 32
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    qam, apsk = nbldpc.constellation(nbldpc.MAP_QAM, 64), nbldpc.apsk64_table()
    noisy = np.zeros((B, code.N, 2), np.float32)
    # no table bound: every mapped call is refused
    for call in (lambda: d.decode_mapped(noisy, 0.5), lambda: d.upload_mapped(noisy, 0.5), lambda: d.channel_mapped(noisy, 0.5),
                 lambda: d.source_frames_mapped(0, B, 10.0)):
        with pytest.raises(nbldpc.NbgpuError) as e:
            call()
        assert e.value.code == nbldpc.ESTATE and "nbgpu_set_constellation" in str(e.value)
    # refusals leave the context unchanged (still no table, then still the bound one)
    for bad in (np.full((64, 2), np.nan, np.float32), np.where(np.arange(128).reshape(64, 2) == 77, np.inf, qam).astype(np.float32)):
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.set_constellation(bad)
        assert e.value.code == nbldpc.EINVAL
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.source_frames_mapped(0, B, 10.0)
    assert e.value.code == nbldpc.ESTATE
    d.set_constellation(qam)
    d.source_frames_mapped(3, B, 14.0)
    with pytest.raises(nbldpc.NbgpuError):
        d.set_constellation(np.full((64, 2), -np.inf, np.float32))
    assert same_stream(d, code, 3, B, 14.0, "mapped", qam)
    d.run()
    d.source_results()
    # re-binding drops the resident mapped batch ...
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.source_frames_mapped(3, B, 14.0); d.run(); d.soft_bits()
    d.set_constellation(qam)
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.run()
    assert e.value.code == nbldpc.ESTATE
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
    # BPSK, 64-APSK and mapped batches alternate on one context
    d.set_constellation(qam)
    for _ in range(2):
        d.source_frames(900, B, 2.5)
        assert d.source_download()[1].shape == (B, code.N, 6)
        d.source_frames_apsk64(11, B, 8.5)
        _, a = d.source_download()
        assert a.shape == (B, code.N, 2)
        d.source_frames_mapped(11, B, 14.0)
        assert same_stream(d, code, 11, B, 14.0, "mapped", qam)
    # with QAM bound, decode_apsk64 still uses the APSK table
    _, _, an = host_frames(code, 0, B, 8.0, "mapped", apsk)
    sigma = nbldpc.sigma_apsk64(8.0)
    r1 = d.decode_apsk64(an, sigma)
    d.set_constellation(apsk)
    r2 = d.decode_mapped(an, sigma)
    assert all((x == y).all() for x, y in zip(r1, r2))
    d.set_constellation(qam)
    r3 = d.decode_mapped(an, sigma)
    assert not all((x == y).all() for x, y in zip(r1, r3))
    d.close()


@gpu
def test_source_download_refuses_a_generated_batch_an_upload_replaced():
    """an upload or a decode overwrites the generated samples: nbgpu_source_download refuses (NBGPU_ESTATE) instead of returning
    the old codewords beside the new samples; a batch that nbgpu_set_constellation dropped keeps its samples"""
    code, _ = field_code(64)
    B = 16
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    qam = nbldpc.constellation(nbldpc.MAP_QAM, 64)
    d.set_constellation(qam)
    for replace in (lambda: d.upload_noisy(np.zeros((B, code.N, code.logq), np.float32), 0.5),
                    lambda: d.decode_mapped(np.zeros((B, code.N, 2), np.float32), 0.5),
                    lambda: d.decode_llr(np.zeros((B, code.N, code.q), np.float32))):
        d.source_frames(3, B, 3.0)
        replace()
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.source_download()
        assert e.value.code == nbldpc.ESTATE
    d.source_frames_mapped(3, B, 14.0)
    d.set_constellation(qam)
    assert same_stream(d, code, 3, B, 14.0, "mapped", qam)
    d.close()


@gpu
@pytest.mark.parametrize("q", [16, 256])
def test_soft_output_of_generated_mapped_batch_equals_host_frames(q):
    code, _ = field_code(q)
    B, ebn = 48, ESN[q]
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    _, _, noisy = host_frames(code, 20, B, ebn, "mapped", mod)
    sigma = nbldpc.sigma_apsk64(ebn)
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=B)
    d.set_constellation(mod)
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        d.decode_mapped(noisy, sigma)
        ref = soft(d, kind)
        d.source_frames_mapped(20, B, ebn)
        d.run()
        assert all(x.tobytes() == y.tobytes() for x, y in zip(soft(d, kind), ref)), kind
    d.close()


@gpu
@pytest.mark.parametrize("q", [16, 256])
def test_c_driver_qam_sources_contexts_and_monte_carlo_agree(tmp_path, q):
    code, path = field_code(q)
    ebn = "%.1f" % ESN[q]
    out1, file1 = run_driver(tmp_path, "device", path, ebn, 16, 1, 2)
    out0, file0 = run_driver(tmp_path, "host", path, ebn, 16, 0, 2)
    out2, file2 = run_driver(tmp_path, "two_contexts", path, ebn, 16, 1, 2, devices="0,0")
    last = [re.findall(CONSOLE, o)[-1] for o in (out1, out0, out2)]
    assert last[0] == last[1] == last[2], last
    assert file1 == file0 == file2 and len(file1) == 1, (file1, file0, file2)
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=128)
    d.set_constellation(mod)
    for st in (multigpu.monte_carlo(code, 2000, ESN[q], decode=d.decode_mapped, batch=128, channel="mapped", constellation=mod),
               multigpu.monte_carlo(code, 2000, ESN[q], batch=128, decoder=d, channel="mapped", constellation=mod)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0][0]), int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]), st
    d.close()
    # an Es/N0 sweep equals its single points
    lo = ESN[q] - 1
    out, lines = run_driver(tmp_path, "sweep", path, "%.1f:%.1f:1" % (lo, lo + 1), 16, 1, 2)
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 2 and len(lines) == 2
    for i in range(2):
        o1, l1 = run_driver(tmp_path, "single%d" % i, path, "%.1f" % (lo + i), 16, 1, 2)
        assert re.findall(CONSOLE, o1)[-1] == re.findall(CONSOLE, blocks[i])[-1] and l1 == [lines[i]], (i, l1, lines[i])
