"""Codes over fields labelled otherwise than the reference labels them, against the oracle with the same tables.

Every other test builds its codes with the reference's tables: exponent labelling (symbol k >= 1 is alpha^(k-1)) over the
polynomials 0x13, 0x43 and 0x11D.  nbgpu_create runs the closed-form kernels when MULGF/DIVGF have the exponent form and the
table-driven kernels (rotations through the q x q rotin/rotout tables) otherwise.  Here each field gets three more labellings
(common.labelled_tables): `reciprocal` keeps the closed form but changes every binary image, `polynomial` (symbol = image)
and `shuffled` (a random bijection) take the table-driven kernels.  The oracle reads nothing but its tables, so with the
same tables copied in (common.oracle_with_tables) it is the reference for all of them, bit for bit."""
import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import (ESN, LABELLINGS, code_arrays, is_closed, labelled_tables, oracle_frames, oracle_llr_mapped, oracle_with_tables,
                    product_frames)
from test_gpu_parity import _lists, mpath
from test_gpu_soft_output import ref_bits, ref_list, wave_of
from test_gpu_source import _host_frames

gpu = pytest.mark.gpu

CODES = {16: "synthetic/GF16_N24_M12_dc4", 64: "matrices/N96_K48_GF64", 256: "matrices/KN/N96_K48_GF256.txt"}
EBN = {16: 3.0, 64: 2.5, 256: 2.5}                   # Eb/N0 at which the frames mix early stops and failures
OTHER = ("reciprocal", "polynomial", "shuffled")
# syndrome check node: (n_m, d1, d2, d3, trunc, n_cv), inside the regime of test_gpu_fuzz (at most 4 passes, Eb/N0 <= 3)
SYND = {16: (12, 11, 5, 3, 0, 10), 64: (20, 19, 15, 5, 300, 25), 256: (20, 19, 15, 5, 1000, 25)}
N_M = {16: 16, 64: 20, 256: 20}


def labelled(q, labelling):
    """(product code, relabelled oracle, tables) of the field's test code"""
    path = mpath(CODES[q])
    base = nbldpc.Code(path)
    t = labelled_tables(q, labelling)
    return nbldpc.Code(arrays=code_arrays(base, t)), oracle_with_tables(path, base.dialect, t), t


def _decoder_kw(q, ecn):
    """(n_m, nb_iter_max, Decoder keywords, oracle keywords) of one check node"""
    if not ecn:
        return N_M[q], 10, {}, {}
    n_m, d1, d2, d3, trunc, n_cv = SYND[q]
    return n_m, 4, dict(ecn_kind=1, d1=d1, d2=d2, d3=d3, cfg_trunc=trunc, n_cv=n_cv), (d1, d2, d3, trunc, n_cv)


def _oracle_kw(o, dc, okw):
    if not okw:
        return {}
    d1, d2, d3, trunc, n_cv = okw
    return dict(ecn=1, cfg=o.build_config_table(dc, d1, d2, d3, trunc), n_cv=n_cv)


# ---- CPU: the helpers and the host layer -------------------------------------------------------------------------------
@pytest.mark.parametrize("q", [16, 64, 256])
def test_labellings_select_the_intended_kernel_family(q):
    """reference/reciprocal keep the exponent closed form, polynomial/shuffled do not; the reference labelling IS the
    default tables of the product and of the oracle"""
    code = nbldpc.Code(mpath(CODES[q]))
    o = ol.Oracle(mpath(CODES[q]), code.dialect)
    t = {lab: labelled_tables(q, lab) for lab in LABELLINGS}
    for got, want in zip(t["reference"], code.tables()):
        assert (got == want).all()
    for got, want in zip(t["reference"], (o.bingf, o.addgf, o.mulgf, o.divgf)):
        assert (got == want).all()
    assert [is_closed(t[lab][2], t[lab][3]) for lab in LABELLINGS] == [True, True, False, False]
    assert not (t["reciprocal"][0] == t["reference"][0]).all()                  # other binary images, same MUL/DIV
    assert (t["reciprocal"][2] == t["reference"][2]).all() and (t["reciprocal"][3] == t["reference"][3]).all()
    o.close()


def test_oracle_with_reference_tables_decodes_as_before():
    """copying the default tables into the oracle changes nothing it computes (APP and CtoV bytes)"""
    q = 64
    path = mpath(CODES[q])
    o0 = ol.Oracle(path)
    o1 = oracle_with_tables(path, 1, labelled_tables(q, "reference"))
    fr, sigma = oracle_frames(o0, 3, 2.0)
    for f in fr:
        a = o0.decode_frame(f["llr"], 20, 25, 10, 0.3, want_state=True)
        b = o1.decode_frame(f["llr"], 20, 25, 10, 0.3, want_state=True)
        assert a["app"].tobytes() == b["app"].tobytes() and a["ctov"].tobytes() == b["ctov"].tobytes()
        assert (a["decide"] == b["decide"]).all() and a["iters"] == b["iters"]
    o0.close(); o1.close()


@pytest.mark.parametrize("labelling", OTHER)
@pytest.mark.parametrize("q", [16, 64, 256])
def test_host_layer_with_labelled_tables_equals_the_oracle(q, labelling):
    """nbgpu_code_from_arrays keeps the tables; the host frame source (encoder, binary images, BPSK noise) equals the
    relabelled oracle's stream, and every codeword has syndrome 0 under the new tables"""
    code, o, t = labelled(q, labelling)
    for got, want in zip(code.tables(), t):
        assert (got == want).all()
    fr, _ = product_frames(code, 20, EBN[q])
    ofr, _ = oracle_frames(o, 20, EBN[q], want_llr=False)
    _, addgf, mulgf, _ = t
    r0 = np.repeat(np.arange(code.M), code.row_deg)
    for a, b in zip(fr, ofr):
        assert (a["cw"] == b["cw"]).all() and (a["nbin"] == b["nbin"]).all()
        assert a["noisy"].tobytes() == b["noisy"].tobytes()
        assert o.syndrome(a["cw"]) == 0
        prod = mulgf[code.val, a["cw"][code.col]]                              # h_e * x_col(e) per edge
        synd = np.zeros(code.M, np.int64)
        for e in range(code.E):
            synd[r0[e]] = addgf[synd[r0[e]], prod[e]]
        assert (synd == 0).all()
    assert len({a["cw"].tobytes() for a in fr}) == len(fr)
    o.close()


# ---- GPU: kernels at the unit boundary ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("labelling", OTHER)
@pytest.mark.parametrize("q", [16, 64, 256])
def test_unit_kernels_equal_the_relabelled_oracle(q, labelling):
    """check_node (both check nodes), decision_syndrome and the BPSK channel with its intrinsic sort"""
    code, o, _ = labelled(q, labelling)
    rng = np.random.default_rng(q + len(labelling))
    nodes = (0, code.M // 2, code.M - 1)
    for ecn in (0, 1):
        n_m, nb_iter_max, kw, okw = _decoder_kw(q, ecn)
        d = nbldpc.Decoder(code, n_m, 25, nb_iter_max, 0.3, max_batch=8, **kw)
        B = 64
        for node in nodes:
            dc = int(code.row_deg[node])
            ok = _oracle_kw(o, dc, okw)
            vl = np.zeros((B, dc, n_m), np.float32); vg = np.zeros((B, dc, n_m), np.int32)
            for b in range(B):
                vl[b], vg[b] = _lists(rng, dc, n_m, q, short_frac=0.0)           # full lists: M_VtoC_GF never holds -1
            cl, cg = d.check_node(node, vl, vg)
            for b in range(B):
                if ecn:
                    rl, rg = o.check_node_syndrome(node, vl[b], vg[b], n_m, ok["cfg"], 0.3, ok["n_cv"])
                else:
                    rl, rg = o.check_node(node, vl[b], vg[b], n_m, 25, 0.3)
                assert cl[b].tobytes() == rl.tobytes() and (cg[b] == rg).all(), (ecn, node, b)
        d.close()
    d = nbldpc.Decoder(code, N_M[q], 25, 10, 0.3, max_batch=8)
    fr, sigma = oracle_frames(o, 5, EBN[q])
    noisy = np.stack([f["noisy"] for f in fr])
    llr, il, ig = d.channel(noisy, sigma, want_sorted=True)
    for f in range(5):
        assert llr[f].tobytes() == fr[f]["llr"].tobytes(), f
        rl, rg = o.sort_intrinsic(fr[f]["llr"])
        assert il[f].tobytes() == rl.tobytes() and (ig[f] == rg).all(), f
    app = (rng.random((6, code.N, q)) * 30).astype(np.float32)
    app[1] = np.round(app[1])                                                   # ties -> lowest symbol
    app[2] = 1e5                                                                # nothing selectable -> symbol 0
    app[3] = llr[0]
    one_hot = np.full((5, code.N, q), 9.0, np.float32)                         # the codewords: syndrome 0
    np.put_along_axis(one_hot, np.stack([f["cw"] for f in fr])[:, :, None].astype(np.int64), 0.0, axis=2)
    app = np.concatenate([app, one_hot])
    dec, synd = d.decision_syndrome(app)
    for b in range(app.shape[0]):
        r = o.decision(app[b])
        assert (dec[b] == r).all() and synd[b] == o.syndrome(r), b
    assert (synd[6:] == 0).all()
    d.close(); o.close()


# ---- GPU: whole decode, multi-wave batches, soft output ----------------------------------------------------------------
def _multi_wave(code, o, q, ecn, early):
    """a batch of more than two waves of the grid at one frame per CTA group (the kernels reuse slots), real codewords of
    the labelled host source; the oracle's results and final APP of every frame"""
    n_m, nb_iter_max, kw, okw = _decoder_kw(q, ecn)
    wave = wave_of(code, n_m, **kw)
    B = 2 * wave + 37
    fr, sigma = product_frames(code, B, EBN[q])
    noisy = np.stack([f["noisy"] for f in fr])
    ok = _oracle_kw(o, int(code.row_deg[0]), okw)
    ref = [o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, nb_iter_max, 0.3, force=not early, want_state=True, **ok)
           for f in range(B)]
    d = nbldpc.Decoder(code, n_m, 25, nb_iter_max, 0.3, early_stop=early, max_batch=B, frames_per_cta=1, **kw)
    assert d.geometry()["grid"] * d.geometry()["frames_per_cta"] == wave and B > 2 * wave
    return d, noisy, sigma, ref, wave


def _check_decode(d, noisy, sigma, ref, wave):
    B = noisy.shape[0]
    dec, synd, it = d.decode_noisy(noisy, sigma)
    for f in range(B):
        assert (dec[f] == ref[f]["decide"]).all() and synd[f] == ref[f]["synd"] and it[f] == ref[f]["iters"], f
    checked = 0
    for f in (0, 1, wave - 1, B - 2, B - 1):
        try:
            app, ctov = d.get_state(f)
        except nbldpc.NbgpuError as e:                      # slot reused by a later frame
            assert e.code == nbldpc.ESTATE and f < B - 2
            continue
        assert app.tobytes() == ref[f]["app"].tobytes() and ctov.tobytes() == ref[f]["ctov"].tobytes(), f
        checked += 1
    assert checked >= 2
    return dec, synd, it


@gpu
@pytest.mark.parametrize("ecn", [0, 1], ids=["bubble", "syndrome"])
@pytest.mark.parametrize("early", [True, False], ids=["early", "fixed"])
@pytest.mark.parametrize("labelling", OTHER)
@pytest.mark.parametrize("q", [16, 64, 256])
def test_decode_and_soft_output_equal_the_relabelled_oracle(q, labelling, early, ecn):
    """decisions, syndromes and iterations of every frame, APP/CtoV bytes of the frames whose slots still hold them, and
    SOFT_LIST / SOFT_BITS of every frame (ref_bits with the labelling's BINGF)"""
    code, o, t = labelled(q, labelling)
    d, noisy, sigma, ref, wave = _multi_wave(code, o, q, ecn, early)
    dec, synd, it = _check_decode(d, noisy, sigma, ref, wave)
    if early and not ecn:
        assert len(set(it.tolist())) > 1, "the batch should mix frames that stop early and frames that do not"
    app = np.stack([r["app"] for r in ref])
    k = min(q, 32) - 3
    d.set_soft_output(nbldpc.SOFT_LIST, k)
    dec2, _, _ = d.decode_noisy(noisy, sigma)
    llr, sym = d.soft_list()
    rl, rs = ref_list(app, k)
    assert llr.tobytes() == rl.tobytes() and (sym == rs).all() and (dec2 == dec).all()
    d.set_soft_output(nbldpc.SOFT_BITS)
    d.decode_noisy(noisy, sigma)
    assert d.soft_bits().tobytes() == ref_bits(app, t[0]).tobytes()
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("ecn", [0, 1], ids=["bubble", "syndrome"])
@pytest.mark.parametrize("q", [16, 64, 256])
def test_forced_table_kernels_equal_the_closed_kernels(q, ecn, monkeypatch):
    """NBGPU_GF_TABLES=1 runs the table-driven kernels on the reference's tables: every output must be the closed kernels'"""
    code = nbldpc.Code(mpath(CODES[q]))
    n_m, nb_iter_max, kw, _ = _decoder_kw(q, ecn)
    wave = wave_of(code, n_m, **kw)
    B = 2 * wave + 37
    fr, sigma = product_frames(code, B, EBN[q])
    noisy = np.stack([f["noisy"] for f in fr])
    monkeypatch.delenv("NBGPU_GF_TABLES", raising=False)
    closed = nbldpc.Decoder(code, n_m, 25, nb_iter_max, 0.3, max_batch=B, frames_per_cta=1, **kw)
    monkeypatch.setenv("NBGPU_GF_TABLES", "1")
    table = nbldpc.Decoder(code, n_m, 25, nb_iter_max, 0.3, max_batch=B, frames_per_cta=1, **kw)
    outs = []
    for d in (closed, table):
        r = list(d.decode_noisy(noisy, sigma)) + list(d.get_state(B - 1)) + list(d.get_state(B - 2))
        d.set_soft_output(nbldpc.SOFT_LIST, min(q, 32))
        d.decode_noisy(noisy, sigma)
        r += list(d.soft_list())
        d.set_soft_output(nbldpc.SOFT_BITS)
        d.decode_noisy(noisy, sigma)
        r.append(d.soft_bits())
        outs.append(r)
    for a, b in zip(*outs):
        assert a.tobytes() == b.tobytes()
    closed.close(); table.close()


# ---- GPU: device frame source, refusal of another code, mapped channel ------------------------------------------------
@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_device_source_with_shuffled_tables(q):
    """source_frames equals the labelled host stream; source_results counts bit errors with the labelling's BINGF"""
    code, o, t = labelled(q, "shuffled")
    B = 200
    d = nbldpc.Decoder(code, N_M[q], 25, 10, 0.3, max_batch=B)
    ebn = EBN[q] - 1.0                                                           # enough frames with bit errors
    for frame0 in (0, 777):
        cw, bits, noisy = _host_frames(code, frame0, B, ebn)
        d.source_frames(frame0, B, ebn)
        gcw, gnoisy = d.source_download()
        assert (gcw == cw).all() and gnoisy.tobytes() == noisy.reshape(gnoisy.shape).tobytes()
        d.run()
        err, synd, it = d.source_results()
        dec, synd2, it2 = d.download()
        want = (t[0][dec[:, :code.K]] != bits.reshape(B, code.N, code.logq)[:, :code.K]).sum((1, 2))
        assert (err == want).all() and (synd == synd2).all() and (it == it2).all()
        assert (want > 0).any() and (want == 0).any()
    d.close(); o.close()


@gpu
def test_source_refuses_a_code_with_other_tables():
    """same graph, other field labelling: all three source calls refuse it and leave the context as it was; a second handle
    on the context's own tables is accepted"""
    q = 64
    code, o, t = labelled(q, "shuffled")
    other = nbldpc.Code(mpath(CODES[q]))                                     # reference tables, same graph and coefficients
    twin = nbldpc.Code(arrays=code_arrays(other, t))
    assert (other.col == code.col).all() and (other.val == code.val).all()
    B = 64
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=B)
    d.set_constellation(nbldpc.constellation(nbldpc.MAP_QAM, q))
    d.source_frames(3, B, 2.0)
    d.run()
    before = d.source_results()
    for fn in (d.source_frames, d.source_frames_apsk64, d.source_frames_mapped):
        d.code = other
        with pytest.raises(nbldpc.NbgpuError) as e:
            fn(0, B, 3.0)
        assert e.value.code == nbldpc.EINVAL and "not the one" in str(e.value), fn
        d.code = code
        for a, b in zip(before, d.source_results()):                          # the decoded batch is still there
            assert (a == b).all()
    d.code = twin
    d.source_frames(3, B, 2.0)
    d.run()
    for a, b in zip(before, d.source_results()):
        assert (a == b).all()
    d.code = code
    cw, _, noisy = _host_frames(code, 11, B, 2.0)
    d.source_frames(11, B, 2.0)
    gcw, gnoisy = d.source_download()
    assert (gcw == cw).all() and gnoisy.tobytes() == noisy.reshape(gnoisy.shape).tobytes()
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
def test_mapped_qam_with_shuffled_tables_equals_the_oracle(q):
    """Gray QAM indexed by the shuffled binary images: decode_mapped against the oracle's mapped LLR (it reads o.bingf)"""
    code, o, _ = labelled(q, "shuffled")
    mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
    code.prepare_encoder(); code.rng_default()
    B = 32
    d = nbldpc.Decoder(code, N_M[q], 25, 10, 0.3, max_batch=B)
    d.set_constellation(mod)
    iters = set()
    for esn in (ESN[q] - 4.0, ESN[q] - 2.0, ESN[q]):                        # at one Es/N0 every frame may stop after one pass
        noisy = np.stack([code.noise_mapped(code.random_codeword()[1], mod, esn) for _ in range(B)])
        sigma = nbldpc.sigma_apsk64(esn)
        dec, synd, it = d.decode_mapped(noisy, sigma)
        iters |= set(it.tolist())
        for f in range(B):
            r = o.decode_frame(oracle_llr_mapped(o, noisy[f], mod, sigma), N_M[q], 25, 10, 0.3)
            assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], (esn, f)
    assert len(iters) > 1, "the frames should differ in iterations"
    d.close(); o.close()
