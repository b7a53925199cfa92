"""Parity of the CUDA path (through the C ABI) against the oracle and the golden fixtures.  Integer outputs
(decisions, syndromes, iteration counts, symbols) and all float32 LLRs are required to be BIT-exact -- stricter
than the 1e-5 relative tolerance BASELINE.json allows for message LLRs."""
import os

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import (Golden, code_path, golden_names, matrix_path, mpath, oracle_frames, product_frames, random_regular_code, sha,
                    write_alist_ubs)

pytestmark = pytest.mark.gpu

Q_CODES = {16: "synthetic/GF16_N32_M8_dc8", 64: "matrices/N96_K48_GF64", 256: "matrices/KN/N96_K48_GF256.txt"}


def _dec(rel, n_m, nb_oper=25, nb_iter_max=10, offset=0.3, **kw):
    code = nbldpc.Code(mpath(rel))
    return code, nbldpc.Decoder(code, n_m, nb_oper, nb_iter_max, offset, **kw)


def _rows(rng, B, q):
    """APP-Mvc like rows with the awkward cases mixed in: exact ties, values >= 1e5, negatives, all-sentinel."""
    r = (rng.random((B, q)) * 40).astype(np.float32)
    for b in range(B):
        k = b % 8
        if k == 1:
            r[b] = np.round(r[b])                                   # many exact ties
        elif k == 2:
            r[b, rng.integers(0, q, q // 2)] = 1e5                  # sentinels inside
        elif k == 3:
            r[b] = r[b] - 20                                        # negative values
        elif k == 4:
            r[b] = 1e5 + rng.random(q).astype(np.float32)          # nothing selectable: (1e5, symbol 0)
        elif k == 5:
            r[b] = np.float32(3.25)                                  # everything tied
        elif k == 6:
            r[b, : q - 3] = 2e5                                      # fewer than n_m selectable
        elif k == 7:
            base = np.float32(7.0)
            r[b] = base + (rng.integers(0, 4, q) * np.float32(np.spacing(base))).astype(np.float32)   # 1-ulp neighbours
    return r


@pytest.mark.parametrize("q,n_m", [(16, 16), (16, 6), (64, 20), (64, 32), (256, 20), (256, 5), (256, 32)])
def test_select_nm(q, n_m):
    code, d = _dec(Q_CODES[q], n_m)
    o = ol.Oracle(mpath(Q_CODES[q]), code.dialect)
    rng = np.random.default_rng(q * 100 + n_m)
    rows = _rows(rng, 4000, q)
    gl, gg = d.select_nm(rows)
    for b in range(rows.shape[0]):
        l, g = o.select_nm(rows[b], n_m)
        assert gl[b].tobytes() == l.tobytes() and (gg[b] == g).all(), (b, b % 8)
    o.close(); d.close()


def _lists(rng, B, n_m, GF, short_frac=0.3):
    llr = np.zeros((B, n_m), np.float32); gf = np.zeros((B, n_m), np.int32)
    for b in range(B):
        v = np.cumsum(rng.random(n_m).astype(np.float32) * 2)
        if b % 3 == 0:
            v = np.round(v * 2) / 2
        v = np.sort(v - v[0]).astype(np.float32)
        llr[b] = v
        gf[b] = rng.permutation(GF)[:n_m] if GF >= n_m else rng.integers(0, GF, n_m)
        if rng.random() < short_frac:
            L = int(rng.integers(1, n_m))
            llr[b, L:] = 1e5; gf[b, L:] = -1
    return llr, gf


@pytest.mark.parametrize("q,n_m,nb_oper", [(16, 16, 25), (64, 20, 25), (64, 8, 6), (64, 5, 60), (256, 20, 25), (256, 32, 80)])
def test_elementary_step(q, n_m, nb_oper):
    code, d = _dec(Q_CODES[q], n_m, nb_oper)
    o = ol.Oracle(mpath(Q_CODES[q]), code.dialect)
    rng = np.random.default_rng(7 + q + n_m)
    B = 3000
    a, ia = _lists(rng, B, n_m, q); b, ib = _lists(rng, B, n_m, q)
    out, io = d.elementary_step(a, b, ia, ib)
    for k in range(B):
        l, g = o.elementary_step(a[k], b[k], ia[k], ib[k], n_m, nb_oper)
        assert out[k].tobytes() == l.tobytes() and (io[k] == g).all(), k
    o.close(); d.close()


@pytest.mark.parametrize("rel,n_m,nb_oper,offset", [("matrices/N96_K48_GF64", 20, 25, 0.3), ("matrices/Mat28_N72_M18", 12, 25, 1.0),
                                                    ("matrices/Mat212_N96_M16", 16, 20, 0.0), ("matrices/Mat26_N48_M16", 16, 25, 0.3),
                                                    ("synthetic/GF16_N32_M8_dc8", 16, 25, 0.3), ("synthetic/GF16_N24_M12_dc4", 9, 25, 0.3),
                                                    ("matrices/KN/N96_K48_GF256.txt", 20, 25, 0.3),
                                                    ("matrices/KN/N576_K480_GF64.txt", 10, 14, 0.5)])
def test_check_node_random(rel, n_m, nb_oper, offset):
    code, d = _dec(rel, n_m, nb_oper, 10, offset)
    o = ol.Oracle(mpath(rel), code.dialect)
    rng = np.random.default_rng(3)
    for node in sorted(set(rng.integers(0, code.M, 6).tolist())):
        dc = int(code.row_deg[node])
        B = 150
        vl = np.zeros((B, dc, n_m), np.float32); vg = np.zeros((B, dc, n_m), np.int32)
        for b in range(B):
            vl[b], vg[b] = _lists(rng, dc, n_m, code.q, short_frac=0.0)
        cl, cg = d.check_node(node, vl, vg)
        for b in range(B):
            l, g = o.check_node(node, vl[b], vg[b], n_m, nb_oper, offset)
            assert cl[b].tobytes() == l.tobytes() and (cg[b] == g).all(), (node, b)
    o.close(); d.close()


def _synd_kw(g):
    """Decoder keyword arguments of a fixture recorded with the reference's syndrome_ems as check node"""
    if not g.synd_params:
        return {}
    d1, d2, d3, trunc, n_cv = g.synd_params
    return dict(ecn_kind=1, d1=d1, d2=d2, d3=d3, cfg_trunc=trunc, n_cv=n_cv)


@pytest.mark.parametrize("name", [n for n in golden_names() if "cn_node" in Golden(n).z])
def test_check_node_on_reference_messages(name):
    g = Golden(name)
    code = nbldpc.Code(matrix_path(g.matrix))                 # messages recorded on the reference's own code: no stand-in
    d = nbldpc.Decoder(code, g.n_m, g.nb_oper, g.nb_iter_max, g.offset, **_synd_kw(g))
    z = g.z
    nodes = z["cn_node"]
    for node in np.unique(nodes):
        sel = np.nonzero(nodes == node)[0]
        cl, cg = d.check_node(int(node), z["cn_in_llr"][sel], z["cn_in_gf"][sel].astype(np.int32))
        assert cl.tobytes() == z["cn_out_llr"][sel].tobytes()
        if g.synd_params:
            assert (cg == z["cn_out_gf"][sel]).all()
        else:
            assert (cg == np.arange(g.GF)[None, None, :]).all()
    d.close()


@pytest.mark.parametrize("rel,n_m,dd,trunc,n_cv", [("matrices/Mat24_N480_M240", 16, (15, 10, 5), 0, 20),
                                                   ("matrices/KN/N96_K48_GF256.txt", 20, (19, 15, 5), 1000, 25),
                                                   ("matrices/N96_K48_GF64", 20, (19, 15, 5), 300, 25),
                                                   ("synthetic/GF16_N24_M12_dc4", 12, (11, 5, 3), 0, 10),
                                                   ("synthetic/GF64_N48_M16_dc6", 10, (9, 3, 2), 0, 8)])
def test_syndrome_check_node_random(rel, n_m, dd, trunc, n_cv):
    """syndrome_ems (presorting, syndromes, stable sort, decorrelation, bayes, saturation) on random lists incl. exact ties"""
    code = nbldpc.Code(mpath(rel))
    o = ol.Oracle(mpath(rel), code.dialect)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, ecn_kind=1, d1=dd[0], d2=dd[1], d3=dd[2], cfg_trunc=trunc, n_cv=n_cv)
    dc = int(code.row_deg[0])
    cfg = o.build_config_table(dc, *dd, trunc)
    assert (nbldpc.config_table(dc, *dd, trunc) == cfg).all()
    rng = np.random.default_rng(5)
    B = 96
    vl = np.sort(rng.random((B, dc, n_m)).astype(np.float32) * rng.choice([1, 5, 20], (B, 1, 1)).astype(np.float32), axis=2)
    vl[1::3] = np.round(vl[1::3] * 4) / 4                              # exact ties between syndromes
    vl[:, :, 0] = 0
    vl = np.sort(vl, axis=2).astype(np.float32)
    vg = np.stack([np.stack([rng.permutation(code.q)[:n_m] for _ in range(dc)]) for _ in range(B)]).astype(np.int32)
    for node in (0, code.M - 1):
        cl, cg = d.check_node(node, vl, vg)
        for b in range(B):
            rl, rg = o.check_node_syndrome(node, vl[b], vg[b], n_m, cfg, 0.3, n_cv)
            assert cl[b].tobytes() == rl.tobytes(), (node, b)
            assert (cg[b] == rg).all(), (node, b)
    o.close(); d.close()


@pytest.mark.parametrize("q", [16, 64, 256])
def test_channel_and_decision(q):
    code, d = _dec(Q_CODES[q], min(q, 16))
    o = ol.Oracle(mpath(Q_CODES[q]), code.dialect)
    fr, sigma = oracle_frames(o, 5, 2.0)
    noisy = np.stack([f["noisy"] for f in fr])
    llr, il, ig = d.channel(noisy, sigma, want_sorted=True)
    for f in range(5):
        assert llr[f].tobytes() == fr[f]["llr"].tobytes()
        ol_, og_ = o.sort_intrinsic(fr[f]["llr"])
        assert il[f].tobytes() == ol_.tobytes() and (ig[f] == og_).all()
    rng = np.random.default_rng(1)
    app = (rng.random((6, code.N, q)) * 30).astype(np.float32)
    app[1] = np.round(app[1])                       # ties -> lowest symbol
    app[2, :, :] = 1e5                              # nothing below the sentinel -> symbol 0 (tools.c:317-329)
    app[3] = llr[0]
    dec, synd = d.decision_syndrome(app)
    for b in range(6):
        r = o.decision(app[b])
        assert (dec[b] == r).all() and synd[b] == o.syndrome(r)
    cw = np.stack([f["cw"] for f in fr])
    one_hot = np.full((5, code.N, q), 9.0, np.float32)
    np.put_along_axis(one_hot, cw[:, :, None].astype(np.int64), 0.0, axis=2)
    dec, synd = d.decision_syndrome(one_hot)
    assert (dec == cw).all() and (synd == 0).all()
    o.close(); d.close()


# ---------------------------------------------------------------------------------------------------
# whole decode loop
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_names())
def test_decode_equals_reference_run(name):
    """Product frame source -> nbgpu_decode_noisy -> decisions / syndrome / iterations / APP bits of the reference run."""
    g = Golden(name)
    code = nbldpc.Code(matrix_path(g.matrix))
    fr, sigma = product_frames(code, g.nf, g.ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    for nb_iter_max in sorted({g.nb_iter_max, 2, 4}):
        d = nbldpc.Decoder(code, g.n_m, g.nb_oper, nb_iter_max, g.offset, max_batch=g.nf, **_synd_kw(g))
        dec, synd, it = d.decode_noisy(noisy, sigma)
        for f in range(g.nf):
            rd, rs, ri, p = g.final(f, nb_iter_max)
            assert (dec[f] == rd).all(), (f, nb_iter_max)
            assert synd[f] == rs and it[f] == ri, (f, nb_iter_max, synd[f], rs, it[f], ri)
            if g.app_sha[f, p - 1]:
                app, _ = d.get_state(f)
                assert sha(app) == g.app_sha[f, p - 1], "APP not bit-identical (frame %d after %d passes)" % (f, p)
        d.close()


@pytest.mark.parametrize("rel,n_m,nb_oper,ebn,frames,early", [
    ("matrices/N96_K48_GF64", 20, 25, 2.0, 300, True), ("matrices/N96_K48_GF64", 30, 45, 3.0, 100, True),
    ("matrices/N96_K48_GF64", 20, 25, 3.0, 64, False), ("matrices/Mat24_N480_M240", 16, 25, 1.5, 24, True),
    ("matrices/Mat26_N48_M16", 16, 25, 2.5, 200, True), ("matrices/Mat26_N48_M16", 6, 8, 2.5, 50, True),
    ("matrices/Mat212_N480_M80", 12, 18, 3.5, 12, True), ("matrices/KN/N128_K64_GF256.txt", 20, 25, 2.5, 60, True),
    ("matrices/KN/N576_K480_GF64.txt", 16, 25, 4.0, 12, True),
    ("synthetic/GF16_N32_M8_dc8", 16, 25, 4.0, 200, True), ("synthetic/GF16_N24_M12_dc4", 12, 25, 3.0, 200, True),
    ("synthetic/GF256_N24_M12_dc4", 24, 30, 3.0, 40, True), ("synthetic/GF64_N60_M12_dc10", 14, 25, 5.0, 40, True)])
def test_decode_batches_equal_oracle(rel, n_m, nb_oper, ebn, frames, early):
    code = nbldpc.Code(mpath(rel))
    o = ol.Oracle(mpath(rel), code.dialect)
    fr, sigma = product_frames(code, frames, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, nb_oper, 10, 0.3, early_stop=early, max_batch=frames)
    dec, synd, it = d.decode_noisy(noisy, sigma)
    llr = d.channel(noisy, sigma)
    dec2, synd2, it2 = d.decode_llr(llr)                      # the dense-LLR intake gives the same result
    assert (dec == dec2).all() and (synd == synd2).all() and (it == it2).all()
    for f in range(frames):
        r = o.decode_frame(llr[f], n_m, nb_oper, 10, 0.3, force=not early, want_state=(f < 4 or f == frames - 1))
        assert (dec[f] == r["decide"]).all(), f
        assert synd[f] == r["synd"], f
        assert it[f] == r["iters"], f
        if "app" in r:
            try:
                app, ctov = d.get_state(f)
            except nbldpc.NbgpuError as e:
                assert e.code == nbldpc.ESTATE
                continue
            assert app.tobytes() == r["app"].tobytes(), f
            assert ctov.tobytes() == r["ctov"].tobytes(), f
    o.close(); d.close()


@pytest.mark.parametrize("rel,n_m,dd,trunc,n_cv,ebn,frames", [("matrices/N96_K48_GF64", 20, (19, 15, 5), 1000, 25, 2.0, 96),
                                                              ("matrices/Mat24_N480_M240", 16, (15, 6, 3), 200, 12, 1.5, 16),
                                                              ("synthetic/GF256_N24_M12_dc4", 20, (19, 15, 5), 1000, 25, 3.0, 24),
                                                              ("synthetic/GF16_N24_M12_dc4", 12, (11, 5, 3), 0, 10, 3.0, 64)])
def test_syndrome_decode_batches_equal_oracle(rel, n_m, dd, trunc, n_cv, ebn, frames):
    """the whole decode loop with the syndrome-based check node (NB_LDPC.c:388 instead of :392)"""
    code = nbldpc.Code(mpath(rel))
    o = ol.Oracle(mpath(rel), code.dialect)
    cfg = o.build_config_table(int(code.row_deg[0]), *dd, trunc)
    fr, sigma = product_frames(code, frames, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=frames, ecn_kind=1, d1=dd[0], d2=dd[1], d3=dd[2], cfg_trunc=trunc, n_cv=n_cv)
    dec, synd, it = d.decode_noisy(noisy, sigma)
    llr = d.channel(noisy, sigma)
    for f in range(frames):
        r = o.decode_frame(llr[f], n_m, 25, 10, 0.3, want_state=(f < 3), ecn=1, cfg=cfg, n_cv=n_cv)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
        if "app" in r:
            try:
                app, ctov = d.get_state(f)
            except nbldpc.NbgpuError as e:
                assert e.code == nbldpc.ESTATE
                continue
            assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), f
    o.close(); d.close()


def test_syndrome_parameter_errors():
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    for kw in (dict(d1=40), dict(n_cv=600), dict(border=3), dict(cfg_trunc=5000, d2=19, d3=19)):
        with pytest.raises(nbldpc.NbgpuError) as e:
            nbldpc.Decoder(code, 20, 25, 10, 0.3, ecn_kind=1, **kw)
        assert e.value.code == nbldpc.EINVAL
    code8 = nbldpc.Code(mpath("synthetic/GF16_N32_M8_dc8"))
    d = nbldpc.Decoder(code8, 16, 25, 10, 0.3, ecn_kind=1, d1=15, d2=3, d3=2, n_cv=4)      # dc = 8 is accepted
    d.close()
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.Decoder(nbldpc.Code(mpath("synthetic/GF64_N60_M12_dc10")), 14, 25, 10, 0.3, ecn_kind=1)


def test_streamed_end_to_end_path_equals_resident_launch():
    """nbgpu_decode_noisy starts ONE launch while the batch is still being copied in (the CTAs wait for their frames, see
    decode_host); the results must equal the plain upload / run / download path (NBGPU_NO_CHUNKS=1)"""
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=1 << 17)
    geo = d.geometry()
    B = 5 * geo["grid"] * geo["frames_per_cta"] + 37                    # >= 2 waves: the streamed path; ragged tail
    assert B <= 1 << 17
    fr, sigma = product_frames(code, 64, 2.5)
    rng = np.random.default_rng(3)
    noisy = np.stack([f["noisy"] for f in fr])[rng.integers(0, 64, B)]
    noisy += (rng.standard_normal(noisy.shape) * 0.05).astype(np.float32)
    l0 = d.launch_count()
    a = d.decode_noisy(noisy, sigma)
    assert d.launch_count() - l0 == 1
    os.environ["NBGPU_NO_CHUNKS"] = "1"
    try:
        l0 = d.launch_count()
        b = d.decode_noisy(noisy, sigma)
        assert d.launch_count() - l0 == 1
    finally:
        del os.environ["NBGPU_NO_CHUNKS"]
    for x, y in zip(a, b):
        assert (x == y).all()
    o = ol.Oracle(matrix_path("matrices/N96_K48_GF64"))
    for f in (0, B // 2, B - 1):
        r = o.decode_frame(o.channel_llr(noisy[f], sigma), 20, 25, 10, 0.3)
        assert (a[0][f] == r["decide"]).all() and a[1][f] == r["synd"] and a[2][f] == r["iters"]
    o.close(); d.close()


def test_full_alist_dvb_size_code_equals_oracle(tmp_path):
    """matrices/KN/N64800_K48600_GF256.txt (full alist, rate 3/4 over GF(256), check degree 8): the reference cannot load it;
    the oracle port gets the same graph through a UBS copy"""
    code = nbldpc.Code(code_path("matrices/KN/N64800_K48600_GF256.txt"))
    a = dict(N=code.N, M=code.M, q=code.q, row_deg=code.row_deg, col=code.col, val=code.val)
    p = str(tmp_path / "ubs")
    write_alist_ubs(p, a)
    o = ol.Oracle(p)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=6)
    d.source_frames(0, 6, 3.6)
    _, noisy = d.source_download()
    d.run()
    dec, synd, it = d.download()
    sigma = code.sigma(3.6)
    for f in (0, 5):
        r = o.decode_frame(o.channel_llr(noisy[f], sigma), 20, 25, 10, 0.3)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"]
    o.close(); d.close()


def test_contexts_with_different_geometries_coexist():
    """two decoders of the same kernel (GF(64), closed form) but different shared-memory plans, used alternately"""
    c1 = nbldpc.Code(matrix_path("matrices/N96_K48_GF64")); c2 = nbldpc.Code(code_path("matrices/Mat24_N480_M240"))
    d1 = nbldpc.Decoder(c1, 20, 25, 10, 0.3, max_batch=64)
    d2 = nbldpc.Decoder(c2, 8, 25, 10, 0.3, max_batch=8, cns_per_step=12)
    assert d1.geometry()["smem_bytes"] != d2.geometry()["smem_bytes"]
    f1, s1 = product_frames(c1, 64, 2.5); f2, s2 = product_frames(c2, 8, 2.0)
    n1 = np.stack([f["noisy"] for f in f1]); n2 = np.stack([f["noisy"] for f in f2])
    a = d1.decode_noisy(n1, s1); b = d2.decode_noisy(n2, s2); a2 = d1.decode_noisy(n1, s1); b2 = d2.decode_noisy(n2, s2)
    for x, y in zip(a + b, a2 + b2):
        assert (x == y).all()
    d1.close(); d2.close()


def test_batch_shapes_and_errors():
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    fr, sigma = product_frames(code, 37, 2.5)
    noisy = np.stack([f["noisy"] for f in fr])
    ref = None
    for fpc, mb in [(0, 37), (1, 37), (3, 40), (8, 64)]:
        d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=mb, frames_per_cta=fpc)
        out = d.decode_noisy(noisy, sigma)
        one = d.decode_noisy(noisy[5:6], sigma)                # B = 1
        assert (one[0][0] == out[0][5]).all() and one[1][0] == out[1][5] and one[2][0] == out[2][5]
        perm = np.random.default_rng(0).permutation(37)
        outp = d.decode_noisy(noisy[perm], sigma)              # frames are independent
        assert (outp[0] == out[0][perm]).all() and (outp[2] == out[2][perm]).all()
        if ref is not None:
            assert all((a == b).all() for a, b in zip(ref, out))
        ref = out
        with pytest.raises(nbldpc.NbgpuError):
            d.decode_noisy(np.zeros((mb + 1, code.N, code.logq), np.float32), sigma)
        d.close()
    for bad in (dict(n_m=4), dict(n_m=33), dict(n_m=65), dict(nb_iter_max=1), dict(nb_oper=0)):
        kw = dict(n_m=20, nb_oper=25, nb_iter_max=10, offset=0.3)
        kw.update(bad)
        with pytest.raises(nbldpc.NbgpuError) as e:
            nbldpc.Decoder(code, **kw)
        assert e.value.code == nbldpc.EINVAL


def test_irregular_and_isolated_variables(tmp_path):
    """Check degrees that differ per row (the reference sizes its scratch by row 0, init.c:320, and is only safe when
    row 0 has the largest degree) and a variable that no check touches."""
    rng = np.random.default_rng(11)
    a = random_regular_code(rng, 30, 15, 64, 4)
    # rows 0..4 keep degree 4... build an irregular graph: degrees 5,4,4,3,... with distinct columns per row
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
    d = nbldpc.Decoder(code, 12, 20, 6, 0.3, max_batch=B)
    dec, synd, it = d.decode_llr(llr)
    for f in range(B):
        r = o.decode_frame(llr[f], 12, 20, 6, 0.3)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    o.close(); d.close()


# ---------------------------------------------------------------------------------------------------
# BASELINE.json sizes: size-independent properties (the oracle needs seconds per frame here)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rel,n_m,ebn_hi", [("matrices/AD_64800_R12_GF256", 20, 3.2), ("matrices/Ahmed_64800_R34_GF16", 16, 4.5),
                                            ("matrices/MatDeclercq_R12_GF64", 20, 2.6)])
def test_full_size_round_trip_and_invariances(rel, n_m, ebn_hi):
    code = nbldpc.Code(code_path(rel))
    B = 24
    fr, sigma = product_frames(code, B, ebn_hi)
    noisy = np.stack([f["noisy"] for f in fr]); cw = np.stack([f["cw"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B)
    dec, synd, it = d.decode_noisy(noisy, sigma)
    # encode -> AWGN at a comfortable SNR -> decode returns the transmitted codewords, syndrome 0, early stop
    assert (synd == 0).all() and (dec == cw).all() and (it < 10).all()
    # idempotent and order independent
    dec2, synd2, it2 = d.decode_noisy(noisy, sigma)
    assert (dec2 == dec).all() and (it2 == it).all()
    perm = np.random.default_rng(2).permutation(B)
    dec3, synd3, it3 = d.decode_noisy(noisy[perm], sigma)
    assert (dec3 == dec[perm]).all() and (it3 == it[perm]).all()
    # a syndrome of 0 really is a codeword of H (checked with the product's own Decision+Syndrom kernel on one-hot APPs)
    d.close()
    # fixed-iteration mode runs all passes and still ends on the codeword
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=False, max_batch=B)
    dec4, synd4, it4 = d.decode_noisy(noisy[:8], sigma)
    assert (dec4 == cw[:8]).all() and (synd4 == 0).all() and (it4 == 10).all()
    d.close()


@pytest.mark.parametrize("rel,n_m,ebn,ecn", [("matrices/N96_K48_GF64", 20, 2.5, 0), ("matrices/Mat24_N480_M240", 16, 1.5, 0),
                                              ("matrices/KN/N96_K48_GF256.txt", 20, 2.5, 0), ("matrices/Mat24_N480_M240", 20, 1.2, 1)])
def test_fixed_iteration_mode_equals_oracle_with_forced_passes(rel, n_m, ebn, ecn):
    """The metric's mode (early termination off, NbIterMax-1 passes for every frame): Decision and Syndrom run only after the
    last pass on the GPU; decisions, syndrome, iteration count and every APP / CtoV bit must equal the oracle run with the
    break of NB_LDPC.c:470 disabled -- for frames that would have converged early and for frames that never do."""
    path = code_path(rel)
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    kw, okw = {}, {}
    if ecn:
        cfg = o.build_config_table(int(code.row_deg[0]), n_m - 1, 15, 5, 1000)
        kw = dict(ecn_kind=1, d1=n_m - 1, d2=15, d3=5, cfg_trunc=1000, n_cv=25)
        okw = dict(ecn=1, cfg=cfg, n_cv=25)
    B = 24 if code.N > 100 else 64
    fr, sigma = product_frames(code, B, ebn)
    noisy = np.stack([f["noisy"] for f in fr])
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=False, max_batch=B, **kw)
    dec, synd, it = d.decode_noisy(noisy, sigma)
    assert (it == 10).all()
    nconv = 0
    for f in range(B):
        llr = o.channel_llr(fr[f]["noisy"], sigma)
        r = o.decode_frame(llr, n_m, 25, 10, 0.3, force=True, want_state=(f % 6 == 0), **okw)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"], f
        nconv += int(r["synd"] == 0)
        if f % 6 == 0:
            app, ctov = d.get_state(f)
            assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), f
    assert nconv > 0 and (nconv < B or ecn == 1), "the batch should mix frames that converge and frames that do not"
    o.close(); d.close()


def test_full_size_multi_wave_batch_spot_checked_against_oracle():
    """BASELINE config 5 at the operating point of the bench (Eb/N0 2.0 dB, some frames never converge): a batch larger than
    the persistent grid (several frames per CTA, streamed end-to-end path), six frames spot-checked against the oracle"""
    rel, n_m = "matrices/AD_64800_R12_GF256", 20
    code = nbldpc.Code(code_path(rel))
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=1400)
    geo = d.geometry()
    B = min(1400, 4 * geo["grid"] * geo["frames_per_cta"] + 13)
    fr, sigma = product_frames(code, 6, 2.0)
    rng = np.random.default_rng(7)
    pick = rng.integers(0, 6, B)
    noisy = np.stack([f["noisy"] for f in fr])[pick]
    noisy = noisy + (rng.standard_normal(noisy.shape) * 0.02).astype(np.float32)       # every frame differs
    dec, synd, it = d.decode_noisy(noisy, sigma)
    assert len(set(it.tolist())) > 1, "the batch should mix converging and non-converging frames"
    o = ol.Oracle(code_path(rel), code.dialect)
    for f in [0, 1, B // 3, B // 2, B - 2, B - 1]:
        r = o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    o.close(); d.close()


def _multi_wave_case(rel, n_m, ebn, ecn, frames_checked, state_frames=2, fpc=1):
    """A batch of at least four waves of the persistent grid through the streamed end-to-end path at a benched operating
    point; `frames_checked` frames compared with the oracle (decisions, syndrome, iterations), the last `state_frames` of
    them -- they sit in the last wave, so their slots still hold their state -- also on every APP and CtoV bit."""
    code = nbldpc.Code(code_path(rel))
    o = ol.Oracle(code_path(rel), code.dialect)
    kw, okw = {}, {}
    if ecn:
        cfg = o.build_config_table(int(code.row_deg[0]), min(19, n_m - 1), 15, 5, 1000)
        kw = dict(ecn_kind=1, d1=min(19, n_m - 1), d2=15, d3=5, cfg_trunc=1000, n_cv=25)
        okw = dict(ecn=1, cfg=cfg, n_cv=25)
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=4096, frames_per_cta=fpc, **kw)     # enough groups to fill the persistent grid
    geo = d.geometry()
    d.close()
    wave = geo["grid"] * geo["frames_per_cta"]
    B = 4 * wave + 17
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=B, frames_per_cta=fpc, **kw)
    assert d.geometry()["grid"] * d.geometry()["frames_per_cta"] == wave and B > 4 * wave, "the batch must span more than four waves of the grid"
    fr, sigma = product_frames(code, 6, ebn)
    rng = np.random.default_rng(11 + ecn)
    pick = rng.integers(0, 6, B)
    noisy = np.stack([f["noisy"] for f in fr])[pick]
    noisy = noisy + (rng.standard_normal(noisy.shape) * 0.02).astype(np.float32)       # every frame differs
    dec, synd, it = d.decode_noisy(noisy, sigma)
    frames = [0, wave, B // 2] + list(range(B - max(frames_checked - 3, state_frames), B))
    for f in frames:
        want_state = f >= B - state_frames
        r = o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3, want_state=want_state, **okw)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], (rel, f)
        if want_state:
            app, ctov = d.get_state(f)
            assert app.tobytes() == r["app"].tobytes(), "APP bits of frame %d differ" % f
            assert ctov.tobytes() == r["ctov"].tobytes(), "CtoV bits of frame %d differ" % f
    o.close(); d.close()
    return it


def test_config5_syndrome_multi_wave_against_oracle():
    """BASELINE config 5 as written (syndrome_decoder path) at the bench's operating point, Eb/N0 2.0 dB"""
    _multi_wave_case("matrices/AD_64800_R12_GF256", 20, 2.0, 1, frames_checked=5, state_frames=1)


def test_config3_multi_wave_against_oracle_never_converges():
    """BASELINE config 3 at 1.2 dB: no frame converges, every check node of every pass is compared through the final state"""
    it = _multi_wave_case("matrices/MatDeclercq_R12_GF64", 20, 1.2, 0, frames_checked=6, state_frames=2, fpc=2)
    assert (it == 10).mean() > 0.9


def test_config4_multi_wave_against_oracle_short_lists():
    """BASELINE config 4 (GF(16), dc = 8) at 3.0 dB: 12.5 % of the check-to-variable rows carry fewer than n_m - 1 pairs"""
    _multi_wave_case("matrices/Ahmed_64800_R34_GF16", 16, 3.0, 0, frames_checked=6, state_frames=2)


# ---------------------------------------------------------------------------------------------------
# 64-APSK channel (ModelChannel_AWGN_64, channel.c:112-312): SURVEY 8f row 2
# ---------------------------------------------------------------------------------------------------
def test_apsk64_intake_kernel_equals_oracle_and_reference_vectors():
    """LLR part of ModelChannel_AWGN_64 on the GPU: dense LLR bit-equal to the oracle, the sorted intrinsic_LLR / intrinsic_GF
    bit-equal to the vectors recorded from the reference (tests/golden/channels/apsk64_n96_gf64.npz)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "channels", "apsk64_n96_gf64.npz"))
    path = matrix_path(str(z["matrix"]))
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    code.prepare_encoder(); code.rng_default()
    ebn = float(z["ebn"]); sigma = nbldpc.sigma_apsk64(ebn)
    noisy = []
    for f in range(z["nbin"].shape[0]):
        _, nb = code.random_codeword()
        assert (nb == z["nbin"][f]).all()
        noisy.append(code.noise_apsk64(nb, ebn))
    noisy = np.stack(noisy)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=len(noisy))
    llr, il, ig = d.channel_apsk64(noisy, sigma, want_sorted=True)
    for f in range(len(noisy)):
        assert llr[f].tobytes() == o.channel_llr_apsk64(noisy[f], sigma).tobytes(), f
        assert il[f].tobytes() == z["illr"][f].tobytes() and (ig[f] == z["igf"][f]).all(), f
    o.close(); d.close()


@pytest.mark.parametrize("rel,ebn", [("matrices/N96_K48_GF64", 8.0), ("matrices/Mat24_N480_M240", 10.3)])
def test_apsk64_decode_equals_oracle(rel, ebn):
    """nbgpu_decode_apsk64 (intake fused into the decoder) against the oracle's 64-APSK LLR + decode loop, frames that converge
    and frames that do not."""
    path = code_path(rel)
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    code.prepare_encoder(); code.rng_default()
    sigma = nbldpc.sigma_apsk64(ebn)
    B = 48
    noisy = np.stack([code.noise_apsk64(code.random_codeword()[1], ebn) for _ in range(B)])
    d = nbldpc.Decoder(code, 16, 25, 10, 0.3, max_batch=B)
    dec, synd, it = d.decode_apsk64(noisy, sigma)
    assert len(set(it.tolist())) > 1, "pick an Eb/N0 at which the frames differ in iterations"
    for f in range(B):
        r = o.decode_frame(o.channel_llr_apsk64(noisy[f], sigma), 16, 25, 10, 0.3)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f
    o.close(); d.close()


def test_apsk64_needs_gf64():
    code = nbldpc.Code(matrix_path("matrices/KN/N96_K48_GF256.txt"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=2)
    with pytest.raises(nbldpc.NbgpuError):
        d.decode_apsk64(np.zeros((2, code.N, 2), np.float32), 0.3)
    d.close()


# ---------------------------------------------------------------------------------------------------
# Monte-Carlo statistics: the C driver (csrc/nbldpc_mc.c) and the sharded loop (multigpu.py) against the stock binary
# ---------------------------------------------------------------------------------------------------
KNOWN = [  # args of the reference binary, console (undetected, err frames, frames, bit errors, avr_it), frames in the results file
    (["2000", "10", "matrices/N96_K48_GF64", "3.0", "20", "0.3", "25"], 0, (24, 2000, 153, "1.56"), 2001),
    (["200", "10", "matrices/Mat24_N480_M240", "1.5", "16", "0.3", "25"], 0, (11, 200, 165, "6.23"), 201),
    (["200", "10", "matrices/Mat24_N480_M240", "1.5", "20", "0.3", "25"], 1, (1, 200, 3, "5.30"), 201),      # syndrome_ems, SURVEY 8c
]


@pytest.mark.parametrize("source", [1, 0], ids=["device_source", "host_source"])
@pytest.mark.parametrize("args,ecn,console,nfile", KNOWN)
def test_c_driver_reproduces_reference_console_and_results_file(args, ecn, console, nfile, source, tmp_path):
    import re
    import subprocess
    exe = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
    assert os.path.exists(exe), "build the C driver with make -C <package>/csrc"
    os.makedirs(tmp_path / "data")
    a = list(args)
    a[2] = matrix_path(a[2])
    r = subprocess.run([exe] + a + ["128", "0", str(ecn), str(source)], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
    m = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)", r.stdout)
    assert m, r.stdout[-2000:]
    last = m[-1]
    assert (int(last[1]), int(last[2]), int(last[3]), last[4]) == console
    files = list((tmp_path / "data").glob("results_*.txt"))
    assert len(files) == 1
    line = files[0].read_text()
    mf = re.search(r"FER=\s*(\d+)\s*/\s*(\d+)", line)
    assert (int(mf.group(1)), int(mf.group(2))) == (console[0], nfile), line


@pytest.mark.parametrize("devices", ["0,0", "0-1", "all"])
@pytest.mark.parametrize("args,ecn,console,nfile", KNOWN[:2])
def test_c_driver_on_several_devices(args, ecn, console, nfile, devices, tmp_path):
    """nbldpc_mc with one host thread + one context per device: frame blocks by drand48 jump-ahead, per-frame rows merged in
    frame order (40-erroneous-frames rule), one ncclAllReduce of the counters.  "0,0" runs the threaded rounds with two
    contexts on one GPU (no NCCL: a device cannot be two ranks); "0-1" and "all" need two or more GPUs."""
    import re
    import subprocess
    ndev = nbldpc.device_count()
    if devices != "0,0" and ndev < 2:
        pytest.skip("needs two or more GPUs (run under gpurun --gpus 2 / 8)")
    exe = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
    os.makedirs(tmp_path / "data")
    a = list(args)
    a[2] = matrix_path(a[2])
    r = subprocess.run([exe] + a + ["96", devices, str(ecn), "1"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    m = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)", r.stdout)
    assert m, r.stdout[-2000:]
    last = m[-1]
    assert (int(last[1]), int(last[2]), int(last[3]), last[4]) == console
    if devices != "0,0":
        assert "one ncclAllReduce" in r.stdout and ("devices: %d" % (2 if devices == "0-1" else ndev)) in r.stdout
    line = list((tmp_path / "data").glob("results_*.txt"))[0].read_text()
    mf = re.search(r"FER=\s*(\d+)\s*/\s*(\d+)", line)
    assert (int(mf.group(1)), int(mf.group(2))) == (console[0], nfile), line


def test_c_driver_stops_at_the_40th_erroneous_frame_in_frame_order(tmp_path):
    """NB_LDPC.c:506: at a low SNR the run ends with the frame of the 40th error, whatever the batch size and the number of
    contexts (frames decoded beyond it are dropped); one and two contexts must print the same last line."""
    import re
    import subprocess
    exe = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
    outs = []
    for devices, batch in (("0", "64"), ("0,0", "24"), ("0,0", "100")):
        d = tmp_path / ("run_%s_%s" % (devices.replace(",", "_"), batch))
        os.makedirs(d / "data")
        r = subprocess.run([exe, "2000", "10", matrix_path("matrices/N96_K48_GF64"), "2.0", "20", "0.3", "25", batch, devices, "0", "1"], cwd=d,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:]
        m = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)", r.stdout)
        outs.append(m[-1])
        assert int(m[-1][1]) == 40 and int(m[-1][2]) < 2000
        line = list((d / "data").glob("results_*.txt"))[0].read_text()
        mf = re.search(r"FER=\s*(\d+)\s*/\s*(\d+)", line)
        assert (int(mf.group(1)), int(mf.group(2))) == (40, int(m[-1][2])), line            # results file: nb = frame of the 40th error
    assert outs[0] == outs[1] == outs[2], outs


def test_c_driver_ebn_sweep_reuses_one_context(tmp_path):
    """BASELINE config 2 is an Eb/N0 sweep (start.sh:14-23: one process per point).  `nbldpc_mc ... first:last:step` runs the
    points one after the other on ONE context; every point must print and log what its own process would."""
    import re
    import subprocess
    exe = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
    pat = r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)"
    mat = matrix_path("matrices/Mat24_N480_M240")

    def run(ebn, sub):
        d = tmp_path / sub
        os.makedirs(d / "data")
        r = subprocess.run([exe, "200", "10", mat, ebn, "16", "0.3", "25", "100", "0"], cwd=d, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:]
        lines = list((d / "data").glob("results_*.txt"))[0].read_text().splitlines()
        return r.stdout, [ln.split("time:")[0] for ln in lines]

    out, lines = run("1.5:2.0:0.25", "sweep")
    blocks = out.split("---- Eb/No = ")[1:]
    assert len(blocks) == 3 and len(lines) == 3
    last = [re.findall(pat, b)[-1] for b in blocks]
    assert (int(last[0][1]), int(last[0][2]), int(last[0][3]), last[0][4]) == (11, 200, 165, "6.23")      # SURVEY 8c known answer at 1.5 dB
    for i, ebn in enumerate(["1.5", "1.75", "2.0"]):
        o1, l1 = run(ebn, "single%d" % i)
        assert re.findall(pat, o1)[-1] == last[i] and l1 == [lines[i]], (ebn, l1, lines[i])


def test_reference_main_with_gpu_check_node(tmp_path):
    """The compiled drop-in (boundary 1, include/bubble_decoder.h:17): oracle/_ref/essai_gpucn is the reference's unmodified
    main() built with -DCheckPassLogEMS=nbgpu_CheckPassLogEMS and linked against libnbldpc_b200.so through the maintainer-side
    binding csrc/nbgpu_bind.c (nbgpu_bind_code on the reference's own code_t / table_t).  Its console must equal the stock
    binary's on the reference's own small case."""
    import re
    import subprocess
    gpucn, stock = os.path.join(ol.REF_DIR, "essai_gpucn"), os.path.join(ol.REF_DIR, "essai_ubs")
    if not (os.path.exists(gpucn) and os.path.exists(stock)):
        pytest.skip("oracle/_ref/essai_gpucn not available (build oracle/_ref where /root/reference exists)")
    args = ["2000", "10", "matrices/N96_K48_GF64", "3.0", "20", "0.3", "25"]
    outs = []
    for exe in (gpucn, stock):
        d = tmp_path / os.path.basename(exe)
        os.makedirs(d / "data")
        os.symlink(os.path.join(ol.REF_DIR, "matrices"), d / "matrices")
        r = subprocess.run([exe] + args, cwd=d, stdin=subprocess.DEVNULL, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:]
        m = re.findall(r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)", r.stdout)
        assert m, r.stdout[-2000:]
        outs.append(m[-1])
        res = list((d / "data").glob("results_*.txt"))[0].read_text().split("time:")[0]
        outs.append(res)
    assert outs[0] == outs[2] == ("0", "24", "2000", "153", "1.56"), outs
    assert outs[1] == outs[3], outs                       # the results-file line up to the time stamp


def test_sharded_monte_carlo_on_the_gpu():
    multigpu = __import__("importlib").import_module("ems-decoder-of-nb-ldpc-codes_b200.multigpu")
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, max_batch=256)
    st = multigpu.monte_carlo(code, 2000, 3.0, d.decode_noisy, batch=256)
    assert (st["err_frames"], st["frames"], st["bit_errors"], st["frames_in_results_file"]) == (24, 2000, 153, 2001)
    assert "%.2f" % (st["sum_it"] / st["frames"]) == "1.56"
    st2 = multigpu.monte_carlo(code, 2000, 3.0, batch=200, decoder=d)                      # frames made on the device
    assert st2 == st
    # the two halves of a 2-rank run, computed one after the other, give the same per-frame rows
    lo = multigpu.monte_carlo(code, 2000, 3.0, d.decode_noisy, batch=256, rank=0, world=1)
    assert lo == st
    d.close()
