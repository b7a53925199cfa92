"""64-APSK frames generated on the device (nbgpu_source_frames_apsk64, ModelChannel_AWGN_64) against the host source
(nbgpu_random_codeword + nbgpu_awgn_apsk64_noise), which the CPU tests pin against the oracle and the reference: same
codeword and noisy samples, bit for bit, anywhere in the drand48 stream; the same decoder results, soft output and
Monte-Carlo statistics as host frames through nbgpu_decode_apsk64."""
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import CONSOLE, EXE, code_path, host_frames, matrix_path, multigpu, run_driver, same_stream

gpu = pytest.mark.gpu


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_draws_per_frame_apsk64_skips_whole_frames():
    """frame f of a sequential host run = skip f*(6K + 4N) draws, then one frame (random_codeword + noise_apsk64)"""
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    D = multigpu.draws_per_frame(code, "apsk64")
    assert D == 6 * code.K + 4 * code.N
    ebn = 7.0
    cw, _, noisy = host_frames(code, 0, 9, ebn, "apsk64")
    for f in (1, 4, 8):
        code.rng_default()
        code.rng_skip(f * D)
        c1, nb = code.random_codeword()
        assert (c1 == cw[f]).all()
        assert code.noise_apsk64(nb, ebn).tobytes() == noisy[f].tobytes()
    with pytest.raises(ValueError):
        multigpu.draws_per_frame(code, "qam16")


def test_c_driver_apsk64_refuses_other_fields_before_any_device(tmp_path):
    """channel 1 on a GF(256) code fails after loading the code, naming q, before it creates a context"""
    assert os.path.exists(EXE)
    r = subprocess.run([EXE, "10", "10", matrix_path("matrices/KN/N96_K48_GF256.txt"), "3.0", "20", "0.3", "25", "8", "0", "0", "1", "1"],
                       cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode != 0 and "q = 256" in r.stdout, r.stdout[-2000:]
    assert "no CPU fallback" not in r.stdout and "AllocateDecoder" not in r.stdout


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("rel", ["matrices/N96_K48_GF64", "matrices/Mat24_N480_M240", "matrices/MatDeclercq_R12_GF64"])
def test_generated_apsk64_frames_equal_the_host_stream(rel):
    code = nbldpc.Code(code_path(rel))
    B = 6 if code.N > 5000 else 200
    D = multigpu.draws_per_frame(code, "apsk64")
    far = (1 << 32) // D + 1000                              # frame0 * D > 2^32: 64-bit draw offsets
    assert far * D > 1 << 32
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    for frame0 in (0, 12345, far):
        for ebn in (6.0, 9.5):
            d.source_frames_apsk64(frame0, B, ebn)
            assert same_stream(d, code, frame0, B, ebn, "apsk64"), (frame0, ebn)
    d.close()


@gpu
def test_flagged_apsk64_samples_are_recomputed_by_the_host():
    """with the widest margin nearly every sample (I and Q, all symbol images) takes the host path; the stream must not change"""
    code = nbldpc.Code(code_path("matrices/Mat24_N480_M240"))
    B, ebn = 64, 5.0
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=B)
    d.source_frames_apsk64(7, B, ebn)
    base = d.source_fixups()
    assert same_stream(d, code, 7, B, ebn, "apsk64")
    d.source_set_margin(2.0 ** -20)
    d.source_frames_apsk64(7, B, ebn)
    n = d.source_fixups()
    assert n > max(100, 50 * base) and n > 0.6 * B * code.N * 2, (n, base)   # > 60 %: both I and Q samples were flagged
    assert same_stream(d, code, 7, B, ebn, "apsk64")
    d.close()


@gpu
def test_default_margin_flags_about_one_apsk64_sample_in_a_million():
    code = nbldpc.Code(code_path("matrices/MatDeclercq_R12_GF64"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=768)
    d.source_frames_apsk64(100, 768, 8.0)                    # 16.6 M samples
    n = d.source_fixups()
    assert n < 200, n
    d.close()


@gpu
@pytest.mark.parametrize("rel,ebn", [("matrices/N96_K48_GF64", 8.0), ("matrices/Mat24_N480_M240", 10.3)])
def test_apsk64_results_equal_the_host_driven_run(rel, ebn):
    """source -> run -> results reproduces (bit errors, syndrome, iterations) and the decisions of host frames through
    decode_apsk64; the first frames also against the oracle's 64-APSK LLR + decode loop"""
    path = code_path(rel)
    code = nbldpc.Code(path)
    frames, batch, n_m = 2000, 512, 16
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=batch)
    bing = code.tables()[0]
    sigma = nbldpc.sigma_apsk64(ebn)
    iters = set()
    for f0 in range(0, frames, batch):
        B = min(batch, frames - f0)
        cw, bits, noisy = host_frames(code, f0, B, ebn, "apsk64")
        dec, synd, it = d.decode_apsk64(noisy, sigma)
        err = np.array([(bing[dec[i, :code.K]] != bits[i][:code.K]).sum() for i in range(B)])
        d.source_frames_apsk64(f0, B, ebn)
        d.run()
        e2, s2, it2 = d.source_results()
        assert (e2 == err).all() and (s2 == synd).all() and (it2 == it).all(), f0
        dec2, _, _ = d.download()
        assert (dec2 == dec).all(), f0
        iters |= set(it.tolist())
        if f0 == 0:
            o = ol.Oracle(path, code.dialect)
            for f in range(32):
                r = o.decode_frame(o.channel_llr_apsk64(noisy[f], sigma), n_m, 25, 10, 0.3)
                assert (dec2[f] == r["decide"]).all() and s2[f] == r["synd"] and it2[f] == r["iters"], f
            o.close()
    assert len(iters) > 1, "pick an Eb/N0 at which the frames differ in iterations"
    d.close()


@gpu
def test_bpsk_and_apsk64_batches_alternate_on_one_context():
    code = nbldpc.Code(code_path("matrices/N96_K48_GF64"))
    B = 64
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d.source_frames(5, B, 3.0)
    assert same_stream(d, code, 5, B, 3.0, "bpsk")
    d.source_frames_apsk64(5, B, 8.0)
    assert same_stream(d, code, 5, B, 8.0, "apsk64")
    d.source_frames(900, B, 2.5)
    assert same_stream(d, code, 900, B, 2.5, "bpsk")
    # a later upload replaces the generated batch
    d.source_frames_apsk64(70, B, 8.0)
    d.run()
    d.source_results()
    d.upload_noisy(np.zeros((B, code.N, code.logq), np.float32), 0.5)
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.source_results()
    assert e.value.code == nbldpc.ESTATE
    # B beyond max_batch: refused, the context still generates
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.source_frames_apsk64(0, B + 1, 8.0)
    assert e.value.code == nbldpc.EINVAL
    d.source_frames_apsk64(11, B, 8.5)
    assert same_stream(d, code, 11, B, 8.5, "apsk64")
    d.close()
    # another field than GF(64): refused with the intake's wording, the context still generates BPSK frames
    c256 = nbldpc.Code(matrix_path("matrices/KN/N96_K48_GF256.txt"))
    d = nbldpc.Decoder(c256, 20, 25, 10, 0.3, max_batch=8)
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.source_frames_apsk64(0, 8, 8.0)
    assert e.value.code == nbldpc.EINVAL and "q = 256" in str(e.value)
    d.source_frames(3, 8, 3.0)
    assert same_stream(d, c256, 3, 8, 3.0, "bpsk")
    d.close()


@gpu
def test_soft_output_of_generated_apsk64_batch_equals_host_frames():
    code = nbldpc.Code(code_path("matrices/N96_K48_GF64"))
    B, ebn, n_m = 48, 8.0, 16
    _, _, noisy = host_frames(code, 20, B, ebn, "apsk64")
    sigma = nbldpc.sigma_apsk64(ebn)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B)
    for kind, k in ((nbldpc.SOFT_LIST, 4), (nbldpc.SOFT_BITS, 0)):
        d.set_soft_output(kind, k)
        d.decode_apsk64(noisy, sigma)
        ref = d.soft_list() if kind == nbldpc.SOFT_LIST else (d.soft_bits(),)
        d.source_frames_apsk64(20, B, ebn)
        d.run()
        got = d.soft_list() if kind == nbldpc.SOFT_LIST else (d.soft_bits(),)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(got, ref)), kind
    d.close()


def _driver(tmp_path, sub, ebn, source, devices="0"):
    return run_driver(tmp_path, sub, code_path("matrices/N96_K48_GF64"), ebn, 20, source, 1, devices=devices)


@gpu
def test_c_driver_apsk64_device_and_host_sources_agree_with_monte_carlo(tmp_path):
    out1, file1 = _driver(tmp_path, "device", "8.0", 1)
    out0, file0 = _driver(tmp_path, "host", "8.0", 0)
    out2, file2 = _driver(tmp_path, "two_contexts", "8.0", 1, "0,0")
    last = [re.findall(CONSOLE, o)[-1] for o in (out1, out0, out2)]
    assert last[0] == last[1] == last[2], last
    assert file1 == file0 == file2 and len(file1) == 1, (file1, file0, file2)
    code = nbldpc.Code(code_path("matrices/N96_K48_GF64"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=128)
    for st in (multigpu.monte_carlo(code, 2000, 8.0, decode=d.decode_apsk64, batch=128, channel="apsk64"),
               multigpu.monte_carlo(code, 2000, 8.0, batch=128, decoder=d, channel="apsk64")):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0][0]), int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]), st
        mf = re.search(r"FER=\s*(\d+)\s*/\s*(\d+)", file1[0])
        assert (int(mf.group(1)), int(mf.group(2))) == (st["err_frames"], st["frames_in_results_file"]), file1
    d.close()


@gpu
def test_c_driver_apsk64_ebn_sweep_equals_single_points(tmp_path):
    out, lines = _driver(tmp_path, "sweep", "7.5:8.5:0.5", 1)
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 3 and len(lines) == 3
    for i, ebn in enumerate(["7.5", "8.0", "8.5"]):
        o1, l1 = _driver(tmp_path, "single%d" % i, ebn, 1)
        assert re.findall(CONSOLE, o1)[-1] == re.findall(CONSOLE, blocks[i])[-1] and l1 == [lines[i]], (ebn, l1, lines[i])
