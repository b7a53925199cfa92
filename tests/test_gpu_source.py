"""Frame source on the device (SURVEY.md 8f.1) against the host frame source, which the CPU tests pin against the
reference binary: same information bits, codeword and noisy samples, bit for bit, anywhere in the drand48 stream."""
import numpy as np
import pytest

import nbldpc
from common import code_path

multigpu = __import__("importlib").import_module("ems-decoder-of-nb-ldpc-codes_b200.multigpu")

pytestmark = pytest.mark.gpu

CODES = [("matrices/N96_K48_GF64", 20), ("matrices/Mat24_N480_M240", 16), ("matrices/KN/N96_K48_GF256.txt", 20),
         ("matrices/MatDeclercq_R12_GF64", 20), ("matrices/Ahmed_64800_R34_GF16", 16), ("matrices/AD_64800_R12_GF256", 20)]


def _host_frames(code, frame0, B, ebn):
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(frame0 * multigpu.draws_per_frame(code))
    cws, bits, noisy = [], [], []
    for _ in range(B):
        cw, nbin = code.random_codeword()
        cws.append(cw); bits.append(nbin); noisy.append(code.noise(nbin, ebn))
    return np.stack(cws), np.stack(bits), np.stack(noisy)


@pytest.mark.parametrize("rel,n_m", CODES)
def test_generated_frames_equal_the_host_stream(rel, n_m):
    code = nbldpc.Code(code_path(rel))
    big = code.N > 5000
    B = 6 if big else 200
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B)
    for frame0, ebn in ((0, 2.0), (12345, 3.5)):
        cw, _, noisy = _host_frames(code, frame0, B, ebn)
        d.source_frames(frame0, B, ebn)
        gcw, gnoisy = d.source_download()
        assert (gcw == cw).all()
        assert gnoisy.tobytes() == noisy.reshape(gnoisy.shape).tobytes()
    d.close()


def test_flagged_samples_are_recomputed_by_the_host():
    """with the widest margin a large share of the samples takes the host path; the stream must not change"""
    code = nbldpc.Code(code_path("matrices/Mat24_N480_M240"))
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=64)
    cw, _, noisy = _host_frames(code, 7, 64, 1.5)
    d.source_frames(7, 64, 1.5)
    base = d.source_fixups()
    d.source_set_margin(2.0 ** -20)
    d.source_frames(7, 64, 1.5)
    assert d.source_fixups() > max(100, 50 * base)
    gcw, gnoisy = d.source_download()
    assert (gcw == cw).all() and gnoisy.tobytes() == noisy.reshape(gnoisy.shape).tobytes()
    with pytest.raises(nbldpc.NbgpuError):
        d.source_set_margin(1.0)
    d.close()


def test_default_margin_flags_about_one_sample_in_a_million():
    code = nbldpc.Code(code_path("matrices/AD_64800_R12_GF256"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=256)
    d.source_frames(100, 256, 2.0)                       # 16.6 M samples
    n = d.source_fixups()
    assert n < 200, n
    d.close()


@pytest.mark.parametrize("rel,n_m,ebn,frames,batch", [("matrices/N96_K48_GF64", 20, 3.0, 2000, 512),
                                                     ("matrices/Mat24_N480_M240", 16, 1.5, 200, 64)])
def test_results_equal_the_host_driven_run(rel, n_m, ebn, frames, batch):
    """source -> run -> results reproduces (bit errors, syndrome, iterations) of host frames through decode_noisy"""
    code = nbldpc.Code(code_path(rel))
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=batch)
    bing = code.tables()[0]
    sigma = code.sigma(ebn)
    for f0 in range(0, frames, batch):
        B = min(batch, frames - f0)
        cw, bits, noisy = _host_frames(code, f0, B, ebn)
        dec, synd, it = d.decode_noisy(noisy, sigma)
        err = np.array([(bing[dec[i, :code.K]] != bits[i].reshape(code.N, code.logq)[:code.K]).sum() for i in range(B)])
        d.source_frames(f0, B, ebn)
        d.run()
        e2, s2, it2 = d.source_results()
        assert (e2 == err).all() and (s2 == synd).all() and (it2 == it).all()
        dec2, _, _ = d.download()
        assert (dec2 == dec).all()
    d.close()


def test_source_argument_errors():
    c1 = nbldpc.Code(code_path("matrices/N96_K48_GF64")); c2 = nbldpc.Code(code_path("matrices/Mat24_N480_M240"))
    d = nbldpc.Decoder(c1, 20, 25, 10, 0.3, max_batch=8)
    with pytest.raises(nbldpc.NbgpuError):
        d.source_results()                               # nothing generated
    with pytest.raises(nbldpc.NbgpuError):
        d.source_frames(0, 9, 3.0)                       # beyond max_batch
    d.code = c2
    with pytest.raises(nbldpc.NbgpuError):
        d.source_frames(0, 4, 3.0)                       # another code
    d.code = c1
    d.source_frames(0, 4, 3.0)
    d.close()
