"""The Min-Max check node (ecn_kind = 4, include/nbldpc_b200.h).  On the CPU: the oracle's node against a numpy brute force over
every configuration, byte for byte, and the refusal of unknown kinds.  On a B200: the decoder bit for bit against the oracle on
every path, channel and geometry, the dense unit boundary, the C driver against monte_carlo, and the error count on a fixed
frame stream against the oracle's."""
import os
import re
import subprocess

import numpy as np
import pytest

import minmax_oracle as mo
import nbldpc
import oracle_lib as ol
from common import (CONSOLE, ESN, EXE, code_path, field_code, labelled_tables, matrix_path, multigpu, oracle_with_tables,
                    code_arrays, is_closed, random_regular_code, waves, write_alist_ubs)
from test_gpu_soft_output import ref_bits, ref_list
from test_gpu_spa import _encodable, _random_frames, bpsk_frames, images, one_check_code

gpu = pytest.mark.gpu

N_M, NB_OPER, OFFSET = 20, 25, 0.3  # validated, not used by the node
MINMAX = 4


def brute_force(o, node, mvc):
    """the Min-Max node by enumeration of every configuration of the other edges, in float32: t_e[z] is the least, over the
    configurations (y_j), j != e, with XOR y_j = z, of max_j u_j[y_j]"""
    q, e0 = o.GF, int(o.row_ptr[node])
    dc = int(o.row_deg[node])
    h = o.val[e0:e0 + dc]
    img = images(o)
    rot = [img[o.mulgf[np.arange(q), h[e]]] for e in range(dc)]
    u = []
    for e in range(dc):
        m = np.asarray(mvc[e], np.float32)
        ue = np.empty(q, np.float32)
        ue[rot[e]] = m - m.min()
        u.append(ue)
    out = np.empty((dc, q), np.float32)
    for e in range(dc):
        others = [j for j in range(dc) if j != e]
        val, syn = np.zeros([q] * len(others), np.float32), np.zeros([q] * len(others), np.int64)
        for a, j in enumerate(others):
            shape = [1] * len(others); shape[a] = q
            val = np.maximum(val, u[j].reshape(shape))
            syn = syn ^ np.arange(q).reshape(shape)
        t = np.full(q, np.inf, np.float32)
        np.minimum.at(t, syn.ravel(), val.ravel())
        out[e] = t[rot[e]]
    return out


def node_inputs(rng, q, dc, kind):
    """Mvc rows of one node: random, peaked (one small value per row, one value above 1e5), exact ties, or with all-zero rows
    (punctured variables)"""
    if kind == "random":
        return (rng.exponential(rng.choice([0.5, 3.0, 10.0, 30.0]), (dc, q)) - rng.uniform(0, 5)).astype(np.float32)
    if kind == "peaked":
        m = rng.uniform(20.0, 100.0, (dc, q)).astype(np.float32)
        m[np.arange(dc), rng.integers(0, q, dc)] = rng.uniform(0.0, 2.0, dc)
        m[0, rng.integers(0, q)] = 1e5 + 3.0
        return m
    if kind == "ties":
        return rng.integers(0, 4, (dc, q)).astype(np.float32) * np.float32(0.75)
    m = rng.exponential(4.0, (dc, q)).astype(np.float32)
    m[rng.choice(dc, max(1, dc - 1), replace=False)] = 0.0
    return m


KINDS = ("random", "peaked", "ties", "zero")


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("q,dc", [(16, 2), (16, 3), (16, 4), (64, 2), (64, 3), (256, 2), (256, 3)])
@pytest.mark.parametrize("kind", KINDS)
def test_oracle_check_node_equals_brute_force(tmp_path, q, dc, kind):
    for seed in range(3):
        o = one_check_code(q, dc, seed, str(tmp_path))
        mvc = node_inputs(np.random.default_rng(100 * seed + q + dc), q, dc, kind)
        got = mo.minmax_check_node(o, 0, mvc)
        assert got.tobytes() == brute_force(o, 0, mvc).tobytes(), (seed, kind)
        assert (got.min(1) == 0).all()
        o.close()


@pytest.mark.parametrize("kind", [5, -1])
def test_unknown_check_node_kinds_are_refused(kind):
    code, _ = field_code(64)
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Decoder(code, N_M, NB_OPER, 10, OFFSET, ecn_kind=kind)
    msg = str(e.value)
    assert "ecn_kind %d" % kind in msg
    assert all(s in msg for s in ("0 = CheckPassLogEMS", "1 = syndrome_ems", "2 = sum-product", "4 = Min-Max"))
    code.close()


# ---------------------------------------------------------------------------------------------------------------- GPU
def oracle_decode(o, llr, nb_iter_max, early, want_state=False):
    return mo.decode_frame(o, llr, nb_iter_max, force=not early, want_state=want_state)


def assert_frames(o, llrs, res, nb_iter_max, early, frames=None):
    dec, synd, it = res
    for f in (range(len(llrs)) if frames is None else frames):
        r = oracle_decode(o, llrs[f], nb_iter_max, early)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], f


def assert_state(d, o, llrs, nb_iter_max, early, nframes=2):
    for f in range(nframes):
        r = oracle_decode(o, llrs[f], nb_iter_max, early, want_state=True)
        app, ctov = d.get_state(f)
        assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), f


EBN = {16: 3.0, 64: 2.5, 256: 2.5}


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
@pytest.mark.parametrize("early", [True, False])
def test_decoder_paths_equal_oracle(q, early):
    """decode_noisy (streamed), decode_llr, upload + run and a device-source batch, against the oracle; APP and CtoV too"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    B, it_max = 24, 8
    d = nbldpc.Decoder(code, N_M if q > 16 else 16, NB_OPER, it_max, OFFSET, early_stop=early, ecn_kind=MINMAX, max_batch=B)
    noisy, sigma = bpsk_frames(code, B, EBN[q])
    llrs = d.channel(noisy, sigma)
    res = d.decode_noisy(noisy, sigma)
    assert_frames(o, llrs, res, it_max, early)
    assert_state(d, o, llrs, it_max, early)
    assert all((x == y).all() for x, y in zip(res, d.decode_llr(llrs)))
    d.upload_noisy(noisy, sigma); d.run()
    assert all((x == y).all() for x, y in zip(res, d.download()))
    d.source_frames(0, B, EBN[q]); d.run()
    _, s2, i2 = d.source_results()
    assert (s2 == res[1]).all() and (i2 == res[2]).all()
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("rel,q,ebn", [("matrices/Ahmed_64800_R34_GF16", 16, 3.4), ("matrices/MatDeclercq_R12_GF64", 64, 1.4)])
@pytest.mark.parametrize("early", [True, False])
def test_multi_wave_full_size(rel, q, ebn, early):
    """config 4 (a GF(16) code of 16200 symbols, dc = 8) and config 3 (GF(64)); seeded stand-ins of those shapes when the
    matrices are absent.  More than two waves of one frame per CTA: every path equal, frames of the first, second and last
    wave equal to the oracle"""
    code = nbldpc.Code(code_path(rel))
    assert code.q == q
    o = ol.Oracle(code_path(rel), code.dialect)
    B = waves(code, 16, early, ecn_kind=MINMAX)
    it_max = 6
    d = nbldpc.Decoder(code, 16, NB_OPER, it_max, OFFSET, early_stop=early, ecn_kind=MINMAX, max_batch=B, frames_per_cta=1)
    g = d.geometry()
    noisy, sigma = bpsk_frames(code, B, ebn)
    res = d.decode_noisy(noisy, sigma)
    d.upload_noisy(noisy, sigma); d.run()
    assert all((x == y).all() for x, y in zip(res, d.download()))
    d.source_frames(0, B, ebn); d.run()
    _, s2, i2 = d.source_results()
    assert (s2 == res[1]).all() and (i2 == res[2]).all()
    frames = [0, g["grid"] + 1, B - 1]
    llrs = {f: o.channel_llr(noisy[f], sigma) for f in frames}
    assert_frames(o, llrs, res, it_max, early, frames)
    d.close(); o.close()


@gpu
def test_other_channels_punctured_and_soft_output():
    """64-APSK, mapped, faded, split and a punctured BPSK batch decode as the oracle does on the channel's LLR rows; soft output
    of both kinds comes from the final APP"""
    for q in (16, 64, 256):
        code, path = field_code(q)
        o = ol.Oracle(path, code.dialect)
        B, it_max = 12, 8
        d = nbldpc.Decoder(code, 16, NB_OPER, it_max, OFFSET, ecn_kind=MINMAX, max_batch=B)
        code.prepare_encoder(); code.rng_default()
        bits = [code.random_codeword()[1] for _ in range(B)]
        mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
        d.set_constellation(mod)
        esn = ESN[q] - 3
        cases = [(np.stack([code.noise_mapped(b, mod, esn) for b in bits]), d.channel_mapped, d.decode_mapped, nbldpc.sigma_apsk64(esn)),
                 (np.stack([code.noise_faded(b, mod, esn + 4, nbldpc.FADING_SYMBOL) for b in bits]), d.channel_faded, d.decode_faded,
                  nbldpc.sigma_apsk64(esn + 4))]
        if q == 64:
            cases.append((np.stack([code.noise_apsk64(b, esn) for b in bits]), d.channel_apsk64, d.decode_apsk64, nbldpc.sigma_apsk64(esn)))
        P = {16: 2, 64: 3, 256: 4}[q]
        split = nbldpc.split_qam(q, P)
        d.set_split_constellation(split, P)
        cases.append((np.stack([code.noise_split(b, split, P, 3.0) for b in bits]), d.channel_split, d.decode_split, nbldpc.sigma_apsk64(3.0)))
        for noisy, chan, dec, sigma in cases:
            assert_frames(o, chan(noisy, sigma), dec(noisy, sigma), it_max, True)
        noisy = np.stack([code.noise(b, 3.0) for b in bits])
        sigma = code.sigma(3.0)
        llrs = d.channel(noisy, sigma)
        for kind, k in ((nbldpc.SOFT_LIST, 5), (nbldpc.SOFT_BITS, 0)):
            d.set_soft_output(kind, k)
            d.decode_noisy(noisy, sigma)
            got = d.soft_list() if kind == nbldpc.SOFT_LIST else d.soft_bits()
            for f in range(3):
                app = oracle_decode(o, llrs[f], it_max, True, want_state=True)["app"]
                if kind == nbldpc.SOFT_LIST:
                    rl, rs = ref_list(app, k)
                    assert got[0][f].tobytes() == rl.tobytes() and (got[1][f] == rs).all(), f
                else:
                    assert got[f].tobytes() == ref_bits(app, o.bingf).tobytes(), f
        d.set_soft_output(nbldpc.SOFT_NONE)
        pv = np.arange(1, code.N, 7, dtype=np.int32)
        d.set_puncturing(pv)
        noisy = np.stack([code.noise(b, 3.0, punctured=pv) for b in bits])
        sigma = code.sigma(3.0, punctured=pv)
        llrs = d.channel(noisy, sigma)
        assert (llrs[:, pv] == 0).all()
        assert_frames(o, llrs, d.decode_noisy(noisy, sigma), it_max, True)
        d.close(); o.close(); code.close()


@gpu
def test_gf_labelling_irregular_and_degree_16_codes(tmp_path):
    """a non-closed field labelling (table-driven rotation), an irregular code with degrees 2 ... 6 and a dc = 16 GF(256) code,
    bit for bit against the oracle, with two launch geometries each"""
    rng = np.random.default_rng(11)
    cases = []
    base, path = field_code(64)
    tables = labelled_tables(64, "shuffled", seed=2)
    assert not is_closed(tables[2], tables[3])
    cases.append((nbldpc.Code(arrays=code_arrays(base, tables)), oracle_with_tables(path, base.dialect, tables), 2.5))
    rd = np.array([2, 3, 4, 5, 6, 4, 3, 5], np.int32)
    N = 20
    col = np.concatenate([rng.choice(N, k, replace=False) for k in rd]).astype(np.int32)
    a = dict(N=N, M=len(rd), q=16, row_deg=rd, col=col, val=rng.integers(1, 16, len(col)).astype(np.int32))
    p_irr = os.path.join(str(tmp_path), "irregular_gf16")
    write_alist_ubs(p_irr, a)
    cases.append((nbldpc.Code(p_irr), ol.Oracle(p_irr, 1), 4.0))
    a = random_regular_code(rng, 64, 8, 256, 16)
    p16 = os.path.join(str(tmp_path), "dc16_gf256")
    write_alist_ubs(p16, a)
    cases.append((nbldpc.Code(p16), ol.Oracle(p16, 1), 6.0))
    for code, o, ebn in cases:
        noisy, sigma = bpsk_frames(code, 16, ebn) if code.K > 0 and _encodable(code) else _random_frames(code, 16)
        for geo in (dict(), dict(frames_per_cta=2, cns_per_step=8)):
            d = nbldpc.Decoder(code, 16, NB_OPER, 6, OFFSET, ecn_kind=MINMAX, max_batch=16, **geo)
            llrs = d.channel(noisy, sigma)
            assert_frames(o, llrs, d.decode_noisy(noisy, sigma), 6, True)
            assert_state(d, o, llrs, 6, True, 1)
            d.close()
        code.close(); o.close()
    base.close()


@gpu
def test_check_node_dense_against_oracle_and_brute_force(tmp_path):
    for q, dc in ((16, 4), (64, 3), (256, 3), (256, 2), (256, 5)):
        o = one_check_code(q, dc, 7, str(tmp_path))
        code = nbldpc.Code(os.path.join(str(tmp_path), "cn_%d_%d_%d" % (q, dc, 7)))
        d = nbldpc.Decoder(code, 16, NB_OPER, 4, OFFSET, ecn_kind=MINMAX, max_batch=4)
        rng = np.random.default_rng(q + dc)
        mvc = np.stack([node_inputs(rng, q, dc, KINDS[b % 4]) for b in range(40)])
        got = d.check_node_dense(0, mvc)
        for b in range(len(mvc)):
            assert got[b].tobytes() == mo.minmax_check_node(o, 0, mvc[b]).tobytes(), (q, dc, b)
            if b < 8 and dc <= 3:
                assert got[b].tobytes() == brute_force(o, 0, mvc[b]).tobytes(), (q, dc, b)
        with pytest.raises(nbldpc.NbgpuError, match="nbgpu_check_node_dense"):
            d.check_node(0, np.zeros((1, dc, 16), np.float32), np.zeros((1, dc, 16), np.int32))
        d.close()
        e = nbldpc.Decoder(code, 16, NB_OPER, 4, OFFSET, ecn_kind=0, max_batch=4)
        with pytest.raises(nbldpc.NbgpuError, match="ecn_kind = 4"):
            e.check_node_dense(0, mvc[:1])
        e.close(); code.close(); o.close()


@gpu
def test_c_driver_ecn4_equals_monte_carlo(tmp_path):
    path = matrix_path("matrices/N96_K48_GF64")
    os.makedirs(tmp_path / "data")
    r = subprocess.run([EXE, "2000", "10", path, "3.0", "20", "0.3", "25", "128", "0", "4", "1"], cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    last = re.findall(CONSOLE, r.stdout)[-1]
    code = nbldpc.Code(path)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, ecn_kind=MINMAX, max_batch=128)
    for st in (multigpu.monte_carlo(code, 2000, 3.0, decoder=d, batch=128), multigpu.monte_carlo(code, 2000, 3.0, decode=d.decode_noisy, batch=128)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0]), int(last[1]), int(last[2]), int(last[3]), last[4]), st
    d.close(); code.close()


@gpu
def test_error_count_on_the_fixed_stream_equals_oracle():
    """frames 0 ... 1999 of the reference stream at 3.0 dB, 10 iterations, N96_K48_GF64: the Min-Max erroneous-frame count of
    the GPU equals the oracle's on the same frames; L-Bubble stays at 24"""
    path = matrix_path("matrices/N96_K48_GF64")
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)

    def oracle_batch(noisy, sigma):
        rs = [oracle_decode(o, o.channel_llr(x, sigma), 10, True) for x in noisy]
        return np.stack([r["decide"] for r in rs]), np.array([r["synd"] for r in rs]), np.array([r["iters"] for r in rs])

    counts = {}
    for name, kind in (("Min-Max", MINMAX), ("L-Bubble n_m=20", 0)):
        d = nbldpc.Decoder(code, 20, 25, 10, 0.3, ecn_kind=kind, max_batch=500)
        counts[name] = multigpu.monte_carlo(code, 2000, 3.0, decoder=d, batch=500, max_err_frames=10 ** 9)
        d.close()
    ref = multigpu.monte_carlo(code, 2000, 3.0, decode=oracle_batch, batch=500, max_err_frames=10 ** 9)
    print("erroneous frames of 2000 at 3.0 dB:", {k: v["err_frames"] for k, v in counts.items()}, "oracle Min-Max:", ref["err_frames"])
    assert counts["L-Bubble n_m=20"]["err_frames"] == 24
    assert {k: counts["Min-Max"][k] for k in ("err_frames", "undetected", "bit_errors", "sum_it")} == \
        {k: ref[k] for k in ("err_frames", "undetected", "bit_errors", "sum_it")}
    code.close(); o.close()
