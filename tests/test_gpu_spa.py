"""The sum-product check node (ecn_kind = 2, include/nbldpc_b200.h).  On the CPU: the oracle's E and L against float64, its
dense check node against a float64 brute force over every configuration, exact symbol marginals on a cycle-free code, and the
refusal of unknown kinds.  On a B200: the decoder bit for bit against the oracle on every path, channel and geometry, the
dense unit boundary, the C driver against monte_carlo, and the node against L-Bubble on a fixed frame stream."""
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
import spa_oracle as so
from common import (CONSOLE, ESN, EXE, code_path, field_code, labelled_tables, matrix_path, multigpu, mpath, oracle_with_tables,
                    code_arrays, is_closed, random_regular_code, waves, write_alist_ubs)
from test_gpu_soft_output import ref_bits, ref_list

gpu = pytest.mark.gpu

LN_TAU = 20 * np.log(2.0)          # -ln tau: the largest CtoV value
N_M, NB_OPER, OFFSET = 20, 25, 0.3  # validated, not used by the node


def tol(exact):
    """|CtoV - exact| allowed where exact < -ln tau: an absolute error of 2^-21 c_max in c (a few ulp of c_max, the f32
    round-off of the two transforms) seen through the log, plus 1e-4 for E, L and the products"""
    return 1e-4 + 2.0 ** -21 * np.exp(np.minimum(exact, LN_TAU))


def one_check_code(q, dc, seed, tmp):
    """an oracle on a code of one check node of degree dc with random coefficients"""
    rng = np.random.default_rng(seed)
    a = dict(N=dc, M=1, q=q, row_deg=np.array([dc], np.int32), col=np.arange(dc, dtype=np.int32),
             val=rng.integers(1, q, size=dc).astype(np.int32))
    path = os.path.join(tmp, "cn_%d_%d_%d" % (q, dc, seed))
    write_alist_ubs(path, a)
    return ol.Oracle(path, 1)


def images(o):
    return (o.bingf.astype(np.int64) << np.arange(o.logGF)).sum(1)


def brute_force(o, node, mvc):
    """float64 sum-product check node by enumeration of every configuration of the other edges: -ln(P_e(x) / max P_e)"""
    q, e0 = o.GF, int(o.row_ptr[node])
    dc = int(o.row_deg[node])
    h = o.val[e0:e0 + dc]
    img = images(o)
    rot = [img[o.mulgf[np.arange(q), h[e]]] for e in range(dc)]
    p = []
    for e in range(dc):
        m = mvc[e].astype(np.float64)
        p.append(np.where((m >= 1e5) & (m > m.min()), 0.0, np.exp(m.min() - m)))
    out = np.zeros((dc, q))
    for e in range(dc):
        others = [j for j in range(dc) if j != e]
        prob, syn = np.ones([q] * len(others)), np.zeros([q] * len(others), np.int64)
        for a, j in enumerate(others):
            shape = [1] * len(others); shape[a] = q
            prob = prob * p[j].reshape(shape)
            syn = syn ^ rot[j].reshape(shape)
        pe = np.bincount(syn.ravel(), weights=prob.ravel(), minlength=q)[rot[e]]
        with np.errstate(divide="ignore"):
            out[e] = np.log(pe.max()) - np.log(pe)
    return out


def node_inputs(rng, q, dc, peaked):
    if not peaked:
        return rng.exponential(rng.choice([0.5, 3.0, 10.0, 30.0]), (dc, q)).astype(np.float32)
    m = rng.uniform(20.0, 100.0, (dc, q)).astype(np.float32)
    m[np.arange(dc), rng.integers(0, q, dc)] = rng.uniform(0.0, 2.0, dc)
    m[0, rng.integers(0, q)] = 1e5 + 3.0                                      # one absent value
    return m


def check_against_brute(ctov, exact):
    inside = exact < LN_TAU
    assert (np.abs(ctov - exact)[inside] <= tol(exact)[inside]).all(), np.abs(ctov - exact)[inside].max()
    assert ((ctov >= 0) & (ctov <= LN_TAU + 1e-5)).all()
    assert (ctov[~inside] >= LN_TAU - 0.05).all()                           # at the cap


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_exp_and_log_against_float64():
    """E and L on a dense sample of their domains, within the bounds stated in the header (1.22 and 1.97 ulp)"""
    o = ol.Oracle(matrix_path("matrices/N96_K48_GF64"), 1)
    rng = np.random.default_rng(1)
    d = np.concatenate([-rng.uniform(0, 87, 40000), -rng.exponential(1e-3, 10000), [0.0, -87.0, -1e-30]]).astype(np.float32)
    e = so.spa_exp(d)
    ref = np.exp(d.astype(np.float64))
    ulp = np.spacing(ref.astype(np.float32)).astype(np.float64)
    assert (np.abs(e - ref) <= 1.22 * ulp).all(), (np.abs(e - ref) / ulp).max()
    assert so.spa_exp(np.float32([-87.01, -200.0, -np.inf])).tolist() == [0.0, 0.0, 0.0]
    x = np.concatenate([2.0 ** rng.uniform(-24, 9, 40000), 1 + rng.uniform(-1e-3, 1e-3, 10000), [1.0, 2.0 ** -20, 256.0]]).astype(np.float32)
    lg = so.spa_log(x)
    ref = np.log(x.astype(np.float64))
    ulp = np.where(ref == 0, 0.0, np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64))
    assert (np.abs(lg - ref) <= 1.97 * ulp).all(), (np.abs(lg - ref) / np.maximum(ulp, 1e-300)).max()
    o.close()


@pytest.mark.parametrize("q,dc", [(16, 2), (16, 3), (16, 4), (64, 2), (64, 3), (256, 2), (256, 3)])
@pytest.mark.parametrize("peaked", [False, True])
def test_oracle_check_node_against_brute_force(tmp_path, q, dc, peaked):
    for seed in range(4):
        o = one_check_code(q, dc, seed, str(tmp_path))
        mvc = node_inputs(np.random.default_rng(100 * seed + q + dc), q, dc, peaked)
        check_against_brute(so.check_node(o, 0, mvc), brute_force(o, 0, mvc))
        o.close()


def tree_code(tmp):
    """a cycle-free GF(16) code: checks {0, 1, 2}, {2, 3, 4} and {4, 5, 6} share variables 2 and 4"""
    a = dict(N=7, M=3, q=16, row_deg=np.array([3, 3, 3], np.int32), col=np.array([0, 1, 2, 2, 3, 4, 4, 5, 6], np.int32),
             val=np.array([3, 7, 1, 12, 5, 9, 2, 14, 6], np.int32))
    path = os.path.join(tmp, "tree_gf16")
    write_alist_ubs(path, a)
    return a, path


def exact_marginals(o, llr):
    """-ln(P(x_n = x) / max) over every codeword, P(c) proportional to exp(-sum_n llr[n][c_n])"""
    q, N = o.GF, o.N
    img = images(o)
    words = np.indices([q] * N).reshape(N, -1).T
    ok = np.ones(len(words), bool)
    for m in range(o.M):
        s = np.zeros(len(words), np.int64)
        for e in range(o.row_ptr[m], o.row_ptr[m + 1]):
            s ^= img[o.mulgf[words[:, o.col[e]], o.val[e]]]
        ok &= s == 0
    cw = words[ok]
    w = np.exp(-llr.astype(np.float64)[np.arange(N), cw].sum(1))
    out = np.zeros((N, q))
    for n in range(N):
        p = np.bincount(cw[:, n], weights=w, minlength=q)
        out[n] = np.log(p.max()) - np.log(p)
    return out


def test_oracle_decodes_cycle_free_code_to_exact_marginals(tmp_path):
    a, path = tree_code(str(tmp_path))
    arrays = dict(a, **dict(zip(("bingf", "addgf", "mulgf", "divgf"), nbldpc.Code(path).tables())))
    code = nbldpc.Code(arrays=arrays)                                    # nbgpu_code_from_arrays takes the same graph
    assert code.N == 7 and code.M == 3 and list(code.row_deg) == [3, 3, 3]
    o = ol.Oracle(path, 1)
    rng = np.random.default_rng(3)
    for _ in range(5):
        llr = rng.uniform(0.0, 3.0, (7, 16)).astype(np.float32)
        r = so.decode_frame(o, llr, 5, force=True, want_state=True)
        app = r["app"].astype(np.float64)
        got = app - app.min(1, keepdims=True)
        exact = exact_marginals(o, llr)
        assert np.abs(got - exact).max() < 1e-3, np.abs(got - exact).max()
    code.close(); o.close()


def test_unknown_check_node_kind_is_refused():
    code, _ = field_code(64)
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Decoder(code, N_M, NB_OPER, 10, OFFSET, ecn_kind=3)
    msg = str(e.value)
    assert "ecn_kind 3" in msg and "0 = CheckPassLogEMS" in msg and "1 = syndrome_ems" in msg and "2 = sum-product" in msg
    code.close()


def test_check_node_dense_is_exported():
    lib = nbldpc.lib()
    assert lib.nbgpu_check_node_dense(None, 0, None, None, 1) == nbldpc.EINVAL


# ---------------------------------------------------------------------------------------------------------------- GPU
def oracle_decode(o, llr, nb_iter_max, early, want_state=False):
    return so.decode_frame(o, llr, nb_iter_max, force=not early, want_state=want_state)


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


def bpsk_frames(code, B, ebn, frame0=0):
    code.prepare_encoder(); code.rng_default()
    code.rng_skip(frame0 * multigpu.draws_per_frame(code, "bpsk"))
    noisy = np.stack([code.noise(code.random_codeword()[1], ebn) for _ in range(B)])
    return noisy, code.sigma(ebn)


EBN = {16: 3.0, 64: 2.5, 256: 2.5}


@gpu
@pytest.mark.parametrize("q", [16, 64, 256])
@pytest.mark.parametrize("early", [True, False])
def test_decoder_paths_equal_oracle(q, early):
    """decode_noisy (streamed), decode_llr, upload + run and a device-source batch, against the oracle; APP and CtoV too"""
    code, path = field_code(q)
    o = ol.Oracle(path, code.dialect)
    B, it_max = 24, 8
    d = nbldpc.Decoder(code, N_M if q > 16 else 16, NB_OPER, it_max, OFFSET, early_stop=early, ecn_kind=2, max_batch=B)
    noisy, sigma = bpsk_frames(code, B, EBN[q])
    llrs = d.channel(noisy, sigma)
    res = d.decode_noisy(noisy, sigma)
    assert_frames(o, llrs, res, it_max, early)
    assert_state(d, o, llrs, it_max, early)
    for r2 in (d.decode_llr(llrs),):
        assert all((x == y).all() for x, y in zip(res, r2))
    d.upload_noisy(noisy, sigma); d.run()
    assert all((x == y).all() for x, y in zip(res, d.download()))
    d.source_frames(0, B, EBN[q]); d.run()
    _, s2, i2 = d.source_results()
    assert (s2 == res[1]).all() and (i2 == res[2]).all()
    d.close(); o.close()


@gpu
@pytest.mark.parametrize("early", [True, False])
def test_multi_wave_full_size(early):
    """config 4 (a GF(16) code of 16200 symbols, dc = 8; a seeded stand-in of that shape when the matrix is absent), more than
    two waves of one frame per CTA: every path equal, frames of the first, second and last wave equal to the oracle"""
    rel = "matrices/Ahmed_64800_R34_GF16"
    code = nbldpc.Code(code_path(rel))
    o = ol.Oracle(code_path(rel), code.dialect)
    B = waves(code, 16, early, ecn_kind=2)
    it_max = 6
    d = nbldpc.Decoder(code, 16, NB_OPER, it_max, OFFSET, early_stop=early, ecn_kind=2, max_batch=B, frames_per_cta=1)
    g = d.geometry()
    noisy, sigma = bpsk_frames(code, B, 3.4)
    res = d.decode_noisy(noisy, sigma)
    d.upload_noisy(noisy, sigma); d.run()
    assert all((x == y).all() for x, y in zip(res, d.download()))
    d.source_frames(0, B, 3.4); d.run()
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
        d = nbldpc.Decoder(code, 16, NB_OPER, it_max, OFFSET, ecn_kind=2, max_batch=B)
        code.prepare_encoder(); code.rng_default()
        bits = [code.random_codeword()[1] for _ in range(B)]
        mod = nbldpc.constellation(nbldpc.MAP_QAM, q)
        d.set_constellation(mod)
        esn = ESN[q] - 3
        cases = [("mapped", np.stack([code.noise_mapped(b, mod, esn) for b in bits]), d.channel_mapped, d.decode_mapped, nbldpc.sigma_apsk64(esn)),
                 ("faded", np.stack([code.noise_faded(b, mod, esn + 4, nbldpc.FADING_SYMBOL) for b in bits]), d.channel_faded, d.decode_faded,
                  nbldpc.sigma_apsk64(esn + 4))]
        if q == 64:
            cases.append(("apsk64", np.stack([code.noise_apsk64(b, esn) for b in bits]), d.channel_apsk64, d.decode_apsk64, nbldpc.sigma_apsk64(esn)))
        P = {16: 2, 64: 3, 256: 4}[q]
        split = nbldpc.split_qam(q, P)
        d.set_split_constellation(split, P)
        cases.append(("split", np.stack([code.noise_split(b, split, P, 3.0) for b in bits]), d.channel_split, d.decode_split, nbldpc.sigma_apsk64(3.0)))
        for name, noisy, chan, dec, sigma in cases:
            llrs = chan(noisy, sigma)
            assert_frames(o, llrs, dec(noisy, sigma), it_max, True)
        # soft output of both kinds, from the APP the oracle ends with
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
        # punctured: decode = the oracle on the expanded rows (zero rows at punctured variables)
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
    # non-closed labelling on the GF(64) code
    base, path = field_code(64)
    tables = labelled_tables(64, "shuffled", seed=2)
    assert not is_closed(tables[2], tables[3])
    cases.append((nbldpc.Code(arrays=code_arrays(base, tables)), oracle_with_tables(path, base.dialect, tables), 2.5))
    # irregular GF(16) code
    rd = np.array([2, 3, 4, 5, 6, 4, 3, 5], np.int32)
    N = 20
    col = np.concatenate([rng.choice(N, k, replace=False) for k in rd]).astype(np.int32)
    a = dict(N=N, M=len(rd), q=16, row_deg=rd, col=col, val=rng.integers(1, 16, len(col)).astype(np.int32))
    p_irr = os.path.join(str(tmp_path), "irregular_gf16")
    write_alist_ubs(p_irr, a)
    cases.append((nbldpc.Code(p_irr), ol.Oracle(p_irr, 1), 4.0))
    # dc = 16 GF(256) code
    a = random_regular_code(rng, 64, 8, 256, 16)
    p16 = os.path.join(str(tmp_path), "dc16_gf256")
    write_alist_ubs(p16, a)
    cases.append((nbldpc.Code(p16), ol.Oracle(p16, 1), 6.0))
    for code, o, ebn in cases:
        noisy, sigma = bpsk_frames(code, 16, ebn) if code.K > 0 and _encodable(code) else _random_frames(code, 16)
        for geo in (dict(), dict(frames_per_cta=2, cns_per_step=8)):
            d = nbldpc.Decoder(code, 16, NB_OPER, 6, OFFSET, ecn_kind=2, max_batch=16, **geo)
            llrs = d.channel(noisy, sigma)
            assert_frames(o, llrs, d.decode_noisy(noisy, sigma), 6, True)
            assert_state(d, o, llrs, 6, True, 1)
            d.close()
        code.close(); o.close()
    base.close()


def _encodable(code):
    try:
        code.prepare_encoder()
        return True
    except Exception:
        return False


def _random_frames(code, B):
    """BPSK samples of random words (not codewords): the decoder's arithmetic does not care"""
    rng = np.random.default_rng(code.N)
    return (1.0 - 2.0 * rng.integers(0, 2, (B, code.N, code.logq)) + 0.8 * rng.normal(size=(B, code.N, code.logq))).astype(np.float32), 0.8


@gpu
def test_check_node_dense_against_oracle_and_brute_force(tmp_path):
    for q, dc in ((16, 4), (64, 3), (256, 3), (256, 2)):
        o = one_check_code(q, dc, 7, str(tmp_path))
        code = nbldpc.Code(os.path.join(str(tmp_path), "cn_%d_%d_%d" % (q, dc, 7)))
        d = nbldpc.Decoder(code, 16, NB_OPER, 4, OFFSET, ecn_kind=2, max_batch=4)
        rng = np.random.default_rng(q + dc)
        mvc = np.stack([node_inputs(rng, q, dc, b % 2 == 1) for b in range(40)])
        got = d.check_node_dense(0, mvc)
        for b in range(len(mvc)):
            ref = so.check_node(o, 0, mvc[b])
            assert got[b].tobytes() == ref.tobytes(), (q, dc, b)
            if b < 6:
                check_against_brute(got[b], brute_force(o, 0, mvc[b]))
        with pytest.raises(nbldpc.NbgpuError, match="nbgpu_check_node_dense"):
            d.check_node(0, np.zeros((1, dc, 16), np.float32), np.zeros((1, dc, 16), np.int32))
        d.close()
        e = nbldpc.Decoder(code, 16, NB_OPER, 4, OFFSET, ecn_kind=0, max_batch=4)
        with pytest.raises(nbldpc.NbgpuError, match="ecn_kind = 2"):
            e.check_node_dense(0, mvc[:1])
        e.close(); code.close(); o.close()


@gpu
def test_cycle_free_code_on_the_device(tmp_path):
    a, path = tree_code(str(tmp_path))
    code = nbldpc.Code(path)
    o = ol.Oracle(path, 1)
    d = nbldpc.Decoder(code, 16, NB_OPER, 5, OFFSET, early_stop=False, ecn_kind=2, max_batch=8)
    llr = np.random.default_rng(5).uniform(0.0, 3.0, (8, 7, 16)).astype(np.float32)
    res = d.decode_llr(llr)
    assert_frames(o, llr, res, 5, False)
    app, _ = d.get_state(0)
    exact = exact_marginals(o, llr[0])
    assert np.abs(app - app.min(1, keepdims=True) - exact).max() < 1e-3
    d.close(); code.close(); o.close()


@gpu
def test_c_driver_ecn2_equals_monte_carlo(tmp_path):
    path = matrix_path("matrices/N96_K48_GF64")
    os.makedirs(tmp_path / "data")
    r = subprocess.run([EXE, "2000", "10", path, "3.0", "20", "0.3", "25", "128", "0", "2", "1"], cwd=tmp_path,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    last = re.findall(CONSOLE, r.stdout)[-1]
    code = nbldpc.Code(path)
    d = nbldpc.Decoder(code, 20, 25, 10, 0.3, ecn_kind=2, max_batch=128)
    for st in (multigpu.monte_carlo(code, 2000, 3.0, decoder=d, batch=128), multigpu.monte_carlo(code, 2000, 3.0, decode=d.decode_noisy, batch=128)):
        assert (st["undetected"], st["err_frames"], st["frames"], st["bit_errors"], "%.2f" % (st["sum_it"] / st["frames"])) == \
            (int(last[0]), int(last[1]), int(last[2]), int(last[3]), last[4]), st
    d.close(); code.close()


@gpu
def test_sum_product_is_not_worse_than_l_bubble_on_the_fixed_stream():
    """frames 0 ... 1999 of the reference stream at 3.0 dB, 10 iterations, N96_K48_GF64: erroneous frames of both nodes"""
    path = matrix_path("matrices/N96_K48_GF64")
    code = nbldpc.Code(path)
    counts = {}
    for name, kind in (("sum-product", 2), ("L-Bubble n_m=20", 0)):
        d = nbldpc.Decoder(code, 20, 25, 10, 0.3, ecn_kind=kind, max_batch=500)
        counts[name] = multigpu.monte_carlo(code, 2000, 3.0, decoder=d, batch=500, max_err_frames=10 ** 9)["err_frames"]
        d.close()
    print("erroneous frames of 2000 at 3.0 dB:", counts)
    assert counts["L-Bubble n_m=20"] == 24
    assert counts["sum-product"] <= counts["L-Bubble n_m=20"]
    code.close()
