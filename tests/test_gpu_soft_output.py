"""Soft output of whole batches (nbgpu_set_soft_output): the k most likely symbols (SOFT_LIST) or the bit reliabilities
(SOFT_BITS) of every decoded variable, computed by the decode kernel from the final APP of each frame.  Compared bit for bit
with the oracle's final APP (decode_frame(want_state=True)) for every frame of batches whose slots were reused."""
import ctypes as C
import functools
import os

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import code_path, matrix_path, product_frames, random_regular_code, write_alist_ubs
from test_gpu_parity import mpath

gpu = pytest.mark.gpu
SENT = np.float32(1e5)


def ref_list(app, k):
    """nbo_select_nm (NB_LDPC.c:354-374) on every row of app[..., q] with n_m = k: ascending, ties -> lowest symbol, values
    >= 1e5 never selected (the slot keeps (1e5, symbol 0)), then llr[i] -= llr[0], llr[0] = 0"""
    order = np.argsort(app, axis=-1, kind="stable")[..., :k]
    val = np.take_along_axis(app, order, -1)
    bad = ~(val < SENT)
    val = np.where(bad, SENT, val).astype(np.float32)
    sym = np.where(bad, 0, order).astype(np.int32)
    llr = (val - val[..., :1]).astype(np.float32)
    llr[..., 0] = 0.0
    return llr, sym


def ref_bits(app, bingf):
    """b[l] = min{APP[s] : bingf[s][l] = 1} - min{APP[s] : bingf[s][l] = 0}, one f32 subtraction"""
    out = np.empty(app.shape[:-1] + (bingf.shape[1],), np.float32)
    for l in range(bingf.shape[1]):
        one = bingf[:, l] == 1
        out[..., l] = app[..., one].min(-1) - app[..., ~one].min(-1)
    return out


def ks_for(q, n_m):
    return sorted({1, 5, n_m, min(q, 32)})


def check_ref_list_is_the_oracle(o, rows, k):
    """the vectorised rule above IS the oracle's truncation (checked row by row on a sample)"""
    gl, gs = ref_list(rows, k)
    for r in range(rows.shape[0]):
        l, s = o.select_nm(rows[r], k)
        assert gl[r].tobytes() == l.tobytes() and (gs[r] == s).all(), r


def wave_of(code, n_m, fpc=1, **kw):
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=1 << 14, frames_per_cta=fpc, **kw)
    g = d.geometry()
    d.close()
    return g["grid"] * g["frames_per_cta"]


# (code, n_m, Eb/N0): the GF(16) two-edges-per-warp path, the GF(64) and GF(256) bubble paths, a 480-symbol GF(64) code
CASES = [("synthetic/GF16_N32_M8_dc8", 16, 4.0), ("matrices/N96_K48_GF64", 20, 2.5), ("matrices/KN/N96_K48_GF256.txt", 20, 2.5),
         ("matrices/Mat24_N480_M240", 16, 1.5)]


@functools.lru_cache(maxsize=None)
def multi_wave_case(rel, n_m, ebn, early):
    """a batch of more than two waves of the persistent grid (one frame per CTA group), its hard output without soft output,
    and the oracle's final APP of every frame"""
    code = nbldpc.Code(mpath(rel))
    o = ol.Oracle(mpath(rel), code.dialect)
    wave = wave_of(code, n_m)
    B = 2 * wave + 37
    fr, sigma = product_frames(code, B, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    app = np.empty((B, code.N, code.q), np.float32)
    for f in range(B):
        app[f] = o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3, force=not early, want_state=True)["app"]
    return code, o, wave, noisy, sigma, app


@gpu
@pytest.mark.parametrize("early", [True, False])
@pytest.mark.parametrize("rel,n_m,ebn", CASES)
def test_list_equals_oracle_every_frame(rel, n_m, ebn, early):
    code, o, wave, noisy, sigma, app = multi_wave_case(rel, n_m, ebn, early)
    B = noisy.shape[0]
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1)
    assert d.geometry()["grid"] * d.geometry()["frames_per_cta"] == wave and B > 2 * wave
    for k in ks_for(code.q, n_m):
        check_ref_list_is_the_oracle(o, app[[0, wave, B - 1]].reshape(-1, code.q), k)
        d.set_soft_output(nbldpc.SOFT_LIST, k)
        dec, _, it = d.decode_noisy(noisy, sigma)
        llr, sym = d.soft_list()
        assert llr.shape == (B, code.N, k) and sym.shape == (B, code.N, k)
        rl, rs = ref_list(app, k)
        for f in range(B):
            assert llr[f].tobytes() == rl[f].tobytes() and (sym[f] == rs[f]).all(), (k, f)
        assert (sym[..., 0] == dec).all()
    if early:
        assert len(set(it.tolist())) > 1, "the batch should mix frames that stop early and frames that do not"
    d.close()


@gpu
@pytest.mark.parametrize("early", [True, False])
@pytest.mark.parametrize("rel,n_m,ebn", CASES)
def test_bits_equal_numpy_from_oracle_app(rel, n_m, ebn, early):
    code, o, wave, noisy, sigma, app = multi_wave_case(rel, n_m, ebn, early)
    B = noisy.shape[0]
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=B, frames_per_cta=1)
    d.set_soft_output(nbldpc.SOFT_BITS)
    dec, _, _ = d.decode_noisy(noisy, sigma)
    b = d.soft_bits()
    assert b.shape == (B, code.N, code.logq)
    ref = ref_bits(app, o.bingf)
    for f in range(B):
        assert b[f].tobytes() == ref[f].tobytes(), f
    # sign rule: the decided symbol's bit 0 <=> b >= 0, bit 1 <=> b <= 0 (rows with a selectable minimum)
    bits = o.bingf[dec]
    live = (app.min(-1) < SENT)[..., None]
    assert ((bits == 0) <= (b >= 0) | ~live).all() and ((bits == 1) <= (b <= 0) | ~live).all()
    d.close()


@gpu
@pytest.mark.parametrize("rel,n_m,dd,ebn,frames", [("matrices/N96_K48_GF64", 20, (19, 15, 5), 2.0, 96),
                                                    ("synthetic/GF256_N24_M12_dc4", 20, (19, 15, 5), 3.0, 40)])
def test_syndrome_check_node_soft_output_equals_oracle(rel, n_m, dd, ebn, frames):
    code = nbldpc.Code(mpath(rel))
    o = ol.Oracle(mpath(rel), code.dialect)
    cfg = o.build_config_table(int(code.row_deg[0]), *dd, 1000)
    fr, sigma = product_frames(code, frames, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=frames, ecn_kind=1, d1=dd[0], d2=dd[1], d3=dd[2], cfg_trunc=1000, n_cv=25)
    app = np.stack([o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3, want_state=True, ecn=1, cfg=cfg, n_cv=25)["app"]
                    for f in range(frames)])
    d.set_soft_output(nbldpc.SOFT_LIST, n_m)
    dec, _, _ = d.decode_noisy(noisy, sigma)
    llr, sym = d.soft_list()
    rl, rs = ref_list(app, n_m)
    assert llr.tobytes() == rl.tobytes() and (sym == rs).all() and (sym[..., 0] == dec).all()
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.decode_noisy(noisy, sigma)
    assert d.soft_bits().tobytes() == ref_bits(app, o.bingf).tobytes()
    o.close(); d.close()


@gpu
def test_every_input_path_gives_the_same_soft_output():
    rel, n_m = "matrices/N96_K48_GF64", 20
    code = nbldpc.Code(matrix_path(rel))
    wave = wave_of(code, n_m)
    B = 2 * wave + 37
    fr, sigma = product_frames(code, B, 2.5)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B, frames_per_cta=1)
    for kind, k, get in ((nbldpc.SOFT_LIST, n_m, d.soft_list), (nbldpc.SOFT_BITS, 0, lambda: (d.soft_bits(),))):
        d.set_soft_output(kind, k)
        l0 = d.launch_count()
        hard = d.decode_noisy(noisy, sigma)                       # >= 2 waves: the streamed end-to-end path
        streamed = get()
        os.environ["NBGPU_NO_CHUNKS"] = "1"
        try:
            hard2 = d.decode_noisy(noisy, sigma)                  # upload + run + download
            plain = get()
        finally:
            del os.environ["NBGPU_NO_CHUNKS"]
        assert d.launch_count() - l0 == 2
        assert all((x == y).all() for x, y in zip(hard, hard2))
        assert all(x.tobytes() == y.tobytes() for x, y in zip(streamed, plain))
        d.decode_llr(d.channel(noisy, sigma))                     # dense-LLR intake
        assert all(x.tobytes() == y.tobytes() for x, y in zip(streamed, get()))
    # device frame source + run == the same frames generated on the host
    d.set_soft_output(nbldpc.SOFT_LIST, n_m)
    d.source_frames(0, B, 2.5)
    d.run()
    dev = d.soft_list()
    d.decode_noisy(noisy, sigma)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(dev, d.soft_list()))
    d.close()


@gpu
def test_apsk64_soft_output_equals_oracle():
    path = code_path("matrices/N96_K48_GF64")
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    code.prepare_encoder(); code.rng_default()
    ebn, B, n_m = 8.0, 48, 16
    sigma = nbldpc.sigma_apsk64(ebn)
    noisy = np.stack([code.noise_apsk64(code.random_codeword()[1], ebn) for _ in range(B)])
    app = np.stack([o.decode_frame(o.channel_llr_apsk64(noisy[f], sigma), n_m, 25, 10, 0.3, want_state=True)["app"] for f in range(B)])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B)
    d.set_soft_output(nbldpc.SOFT_LIST, 8)
    d.decode_apsk64(noisy, sigma)
    llr, sym = d.soft_list()
    rl, rs = ref_list(app, 8)
    assert llr.tobytes() == rl.tobytes() and (sym == rs).all()
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.decode_apsk64(noisy, sigma)
    assert d.soft_bits().tobytes() == ref_bits(app, o.bingf).tobytes()
    o.close(); d.close()


@gpu
@pytest.mark.parametrize("rel,n_m,ebn", [("synthetic/GF16_N32_M8_dc8", 16, 4.0), ("matrices/N96_K48_GF64", 20, 2.5)])
def test_soft_output_does_not_change_hard_output(rel, n_m, ebn):
    code = nbldpc.Code(mpath(rel))
    B = 2 * wave_of(code, n_m) + 5
    fr, sigma = product_frames(code, B, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B, frames_per_cta=1)
    ref = d.decode_noisy(noisy, sigma)
    for kind, k in ((nbldpc.SOFT_LIST, 1), (nbldpc.SOFT_LIST, n_m), (nbldpc.SOFT_BITS, 0), (nbldpc.SOFT_NONE, 0)):
        d.set_soft_output(kind, k)
        out = d.decode_noisy(noisy, sigma)
        assert all((x == y).all() for x, y in zip(ref, out)), (kind, k)
        if kind == nbldpc.SOFT_LIST:
            assert (d.soft_list()[1][..., 0] == ref[0]).all()
    d.close()


@gpu
def test_irregular_code_and_isolated_variable(tmp_path):
    """the graph of test_irregular_and_isolated_variables: variable 29 is in no check, its soft output is that of its intake row"""
    rng = np.random.default_rng(11)
    random_regular_code(rng, 30, 15, 64, 4)                         # advances rng exactly as that test does: the same graph
    deg = np.array([5, 4, 4, 3, 4, 4, 3, 5, 4, 2, 4, 4, 3, 4, 4], np.int32)
    col = np.concatenate([rng.permutation(29)[:k] for k in deg]).astype(np.int32)      # variable 29 stays isolated
    val = rng.integers(1, 64, col.size).astype(np.int32)
    arr = dict(N=30, M=15, q=64, row_deg=deg, col=col, val=val)
    write_alist_ubs(str(tmp_path / "irr"), arr)
    code = nbldpc.Code(arrays=arr)
    o = ol.Oracle(str(tmp_path / "irr"))
    B = 40
    llr = (rng.random((B, 30, 64)) * 12).astype(np.float32)
    cw = rng.integers(0, 64, (B, 30))
    np.put_along_axis(llr, cw[:, :, None], 0.0, axis=2)
    app = np.stack([o.decode_frame(llr[f], 12, 20, 6, 0.3, want_state=True)["app"] for f in range(B)])
    d = nbldpc.Decoder(code, 12, 20, 6, 0.3, max_batch=B)
    d.set_soft_output(nbldpc.SOFT_LIST, 12)
    d.decode_llr(llr)
    sl, ss = d.soft_list()
    rl, rs = ref_list(app, 12)
    assert sl.tobytes() == rl.tobytes() and (ss == rs).all()
    il, is_ = ref_list(llr[:, 29], 12)
    assert sl[:, 29].tobytes() == il.tobytes() and (ss[:, 29] == is_).all()
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.decode_llr(llr)
    b = d.soft_bits()
    assert b.tobytes() == ref_bits(app, o.bingf).tobytes()
    assert b[:, 29].tobytes() == ref_bits(llr[:, 29], o.bingf).tobytes()
    o.close(); d.close()


@gpu
def test_full_size_multi_wave_list_spot_checked_against_oracle():
    """config 5 (AD_64800_R12_GF256, n_m = 20) at the bench's Eb/N0: a batch of more than two waves, LIST k = 20; frames of the
    FIRST wave, whose slots were reused long ago (nbgpu_get_state cannot reach them), are checked too"""
    rel, n_m = "matrices/AD_64800_R12_GF256", 20
    code = nbldpc.Code(code_path(rel))
    wave = wave_of(code, n_m)
    B = 2 * wave + 13
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B, frames_per_cta=1)
    fr, sigma = product_frames(code, 6, 2.0)
    rng = np.random.default_rng(7)
    noisy = np.stack([f["noisy"] for f in fr])[rng.integers(0, 6, B)]
    noisy = noisy + (rng.standard_normal(noisy.shape) * 0.02).astype(np.float32)       # every frame differs
    d.set_soft_output(nbldpc.SOFT_LIST, n_m)
    dec, _, _ = d.decode_noisy(noisy, sigma)
    llr, sym = d.soft_list()
    assert (sym[..., 0] == dec).all()
    o = ol.Oracle(code_path(rel), code.dialect)
    for f in [0, 1, wave // 2, B // 2, B - 1]:
        app = o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3, want_state=True)["app"]
        rl, rs = ref_list(app, n_m)
        assert llr[f].tobytes() == rl.tobytes() and (sym[f] == rs).all(), f
    o.close(); d.close()


def _code_of(err):
    return err.value.code


@gpu
def test_errors_and_state():
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    fr, sigma = product_frames(code, 8, 2.5)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=8)
    for kind, k in ((3, 0), (-1, 0), (nbldpc.SOFT_LIST, 0), (nbldpc.SOFT_LIST, 33), (nbldpc.SOFT_BITS, 1), (nbldpc.SOFT_NONE, 2)):
        with pytest.raises(nbldpc.NbgpuError) as e:
            d.set_soft_output(kind, k)
        assert _code_of(e) == nbldpc.EINVAL, (kind, k)
    d.set_soft_output(nbldpc.SOFT_LIST, 32)                         # min(q, 32) for GF(64)
    with pytest.raises(nbldpc.NbgpuError) as e:                    # nothing decoded yet
        d.soft_list()
    assert _code_of(e) == nbldpc.EINVAL
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.soft_bits()
    assert _code_of(e) == nbldpc.EINVAL
    d.set_soft_output(nbldpc.SOFT_LIST, 6)
    ref = d.decode_noisy(noisy, sigma)
    first = d.soft_list()
    with pytest.raises(nbldpc.NbgpuError) as e:                    # the other kind
        d.soft_bits()
    assert _code_of(e) == nbldpc.ESTATE
    d.select_nm(np.zeros((4, code.q), np.float32))                 # unit-boundary calls leave the soft output alone
    assert all(x.tobytes() == y.tobytes() for x, y in zip(first, d.soft_list()))
    d.set_soft_output(nbldpc.SOFT_LIST, 6)                          # re-arming invalidates the last batch
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.soft_list()
    assert _code_of(e) == nbldpc.ESTATE
    d.upload_noisy(noisy, sigma); d.run(); d.sync()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(first, d.soft_list()))
    d.upload_noisy(noisy[:4], sigma)                                # a new batch, not yet decoded
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.soft_list()
    assert _code_of(e) == nbldpc.ESTATE
    d.set_soft_output(nbldpc.SOFT_NONE)
    out = d.decode_noisy(noisy, sigma)
    with pytest.raises(nbldpc.NbgpuError) as e:
        d.soft_list()
    assert _code_of(e) == nbldpc.ESTATE
    fresh = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=8)
    assert all((x == y).all() for x, y in zip(out, fresh.decode_noisy(noisy, sigma)))
    assert all((x == y).all() for x, y in zip(out, ref))
    fresh.close(); d.close()


def test_soft_output_abi_without_a_gpu():
    """the entry points are exported and validate their context before touching a device"""
    L = C.CDLL(nbldpc.LIB_PATH)
    for name in ("nbgpu_set_soft_output", "nbgpu_download_soft_list", "nbgpu_download_soft_bits"):
        assert hasattr(L, name)
    assert (nbldpc.SOFT_NONE, nbldpc.SOFT_LIST, nbldpc.SOFT_BITS) == (0, 1, 2)
    lib = nbldpc.lib()
    assert lib.nbgpu_set_soft_output(None, nbldpc.SOFT_LIST, 4) == nbldpc.EINVAL
    assert lib.nbgpu_download_soft_list(None, None, None) == nbldpc.EINVAL
    assert lib.nbgpu_download_soft_bits(None, None) == nbldpc.EINVAL
