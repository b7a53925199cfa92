"""Host side of the product (plain C, no GPU needed): alist loader, GF tables, frame source, statistics,
pass schedule, and the C-ABI surface itself."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import Golden, code_path, golden_names, matrix_path, oracle_frames, product_frames, random_regular_code, write_alist_full, write_alist_kn, write_alist_ubs, ROOT


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "nbldpc_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = sorted(set(re.findall(r"\b(nbgpu_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 30
    L = C.CDLL(nbldpc.LIB_PATH)
    missing = [s for s in declared if not hasattr(L, s)]
    assert not missing, missing
    out = subprocess.run(["nm", "-D", "--defined-only", nbldpc.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (nbgpu_[a-z0-9_]+)", out))
    assert set(declared) <= exported


def test_no_gpu_means_error_not_fallback():
    if nbldpc.device_count() > 0:
        pytest.skip("a GPU is present")
    code = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Decoder(code, 20, 25, 10, 0.3)
    assert e.value.code == nbldpc.ECUDA and "no CPU fallback" in str(e.value)


@pytest.mark.parametrize("rel,dialect", [("matrices/N96_K48_GF64", 1), ("matrices/KN/N96_K48_GF64.txt", 2),
                                         ("matrices/KN/N96_K48_GF256.txt", 2), ("matrices/Ahmed_64800_R34_GF16", 1),
                                         ("matrices/AD_64800_R12_GF256", 1), ("matrices/MatDeclercq_R12_GF64", 1),
                                         ("matrices/KN/N576_K480_GF64.txt", 2), ("matrices/Mat212_N480_M80", 1)])
def test_loader_and_tables_equal_oracle(rel, dialect):
    p = code_path(rel)
    o = ol.Oracle(p, dialect)
    for d in (dialect, nbldpc.ALIST_AUTO):
        c = nbldpc.Code(p, d)
        assert c.dialect == dialect
        assert (c.N, c.M, c.K, c.q, c.logq, c.E, c.dc_max) == (o.N, o.M, o.K, o.GF, o.logGF, o.E, o.dc_max)
        assert np.float32(c.rate) == np.float32(o.rate)
        assert (c.row_deg == o.row_deg).all() and (c.col == o.col).all() and (c.val == o.val).all()
        b, a, m, dv = c.tables()
        assert (b == o.bingf).all() and (a == o.addgf).all() and (m == o.mulgf).all() and (dv == o.divgf).all()
        c.close()
    o.close()


def test_same_code_in_both_dialects():
    a = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    b = nbldpc.Code(matrix_path("matrices/KN/N96_K48_GF64.txt"))
    assert a.dialect == 1 and b.dialect == 2
    assert (a.col == b.col).all() and (a.val == b.val).all()


def _irregular_code(rng, q):
    dcs = [int(x) for x in rng.choice([2, 3, 4, 6], 9)]
    N = 20
    cols, vals = [], []
    for dc in dcs:
        cols += [int(x) for x in rng.choice(N, dc, replace=False)]
        vals += [int(x) for x in rng.integers(1, q, dc)]
    return dict(N=N, M=len(dcs), q=q, row_deg=np.array(dcs, np.int32), col=np.array(cols, np.int32), val=np.array(vals, np.int32))


@pytest.mark.parametrize("pad", [False, True])
def test_full_alist_layout(tmp_path, pad):
    """SURVEY.md 8f.4: the layout of matrices/KN/N64800_* (LoadCode of the reference cannot read it), exact and zero-padded"""
    a = _irregular_code(np.random.default_rng(11), 64)
    p = str(tmp_path / "full")
    write_alist_full(p, a, pad=pad)
    for dialect in (nbldpc.ALIST_AUTO, nbldpc.ALIST_FULL):
        c = nbldpc.Code(p, dialect=dialect)
        assert c.dialect == nbldpc.ALIST_FULL and (c.row_deg == a["row_deg"]).all() and (c.col == a["col"]).all() and (c.val == a["val"]).all()
        assert (c.dc_min, c.dc_max) == (2, 6)
    # a column list that contradicts the row lists is not accepted as this layout
    txt = open(p).read().split("\n")
    li = next(i for i in range(4, 4 + a["N"]) if len(txt[i].split()) >= 2 and txt[i].split()[0] != "0")
    first = txt[li].split()
    first[1] = str((int(first[1]) + 1) % 63)
    txt[li] = " ".join(first)
    open(p, "w").write("\n".join(txt))
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.Code(p, dialect=nbldpc.ALIST_FULL)
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.Code(p)


@pytest.mark.parametrize("seed", range(6))
def test_three_layouts_of_one_random_code_load_identically(tmp_path, seed):
    rng = np.random.default_rng(100 + seed)
    a = _irregular_code(rng, int(rng.choice([16, 64, 256])))
    codes = []
    for name, writer, dialect in (("u", write_alist_ubs, nbldpc.ALIST_UBS), ("k", write_alist_kn, nbldpc.ALIST_KN),
                                  ("f", write_alist_full, nbldpc.ALIST_FULL), ("p", lambda p, x: write_alist_full(p, x, pad=True), nbldpc.ALIST_FULL)):
        p = str(tmp_path / name)
        writer(p, a)
        c = nbldpc.Code(p)                               # dialect detected from the file
        assert c.dialect == dialect, name
        codes.append(c)
    for c in codes:
        assert (c.row_deg == a["row_deg"]).all() and (c.col == a["col"]).all() and (c.val == a["val"]).all()
        assert (c.tables()[1] == codes[0].tables()[1]).all()


def test_shipped_full_alist_matrix_loads_and_encodes():
    c = nbldpc.Code(code_path("matrices/KN/N64800_K48600_GF256.txt"))
    assert (c.dialect, c.N, c.M, c.q, c.dc_min, c.dc_max) == (nbldpc.ALIST_FULL, 8100, 2025, 256, 8, 8)
    c.prepare_encoder()
    cw, _ = c.random_codeword()
    _, add, mul, _ = c.tables()
    prod = mul[c.val, cw[c.col]]                              # every check sums to zero (GF addition through the table)
    for m in range(0, c.M, 7):
        s = 0
        for x in prod[c.row_ptr[m]:c.row_ptr[m + 1]]:
            s = add[s, x]
        assert s == 0


def test_loader_errors(tmp_path):
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Code(str(tmp_path / "missing"))
    assert e.value.code == nbldpc.EIO
    p = tmp_path / "bad_gf"
    p.write_text("4 2 32\n1 1 1 1\n2 2\n0 1\n2 3\n1 1\n1 1\n")
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Code(str(p))
    assert e.value.code == nbldpc.EINVAL                       # init.c:431-435 exits; we return an error
    p = tmp_path / "short"
    p.write_text("4 2 16\n1 1 1 1\n2 2\n0 1\n2\n")
    with pytest.raises(nbldpc.NbgpuError) as e:
        nbldpc.Code(str(p))
    assert e.value.code == nbldpc.EIO
    rng = np.random.default_rng(0)
    a = random_regular_code(rng, 12, 6, 16, 4)
    a["col"][3] = 99
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.Code(arrays=a)


def test_from_arrays_roundtrip(tmp_path):
    rng = np.random.default_rng(5)
    a = random_regular_code(rng, 24, 12, 64, 4)
    c1 = nbldpc.Code(arrays=a)
    write_alist_ubs(str(tmp_path / "m"), a)
    c2 = nbldpc.Code(str(tmp_path / "m"))
    assert c2.dialect == 1 and (c1.col == c2.col).all() and (c1.val == c2.val).all()
    o = ol.Oracle(str(tmp_path / "m"))
    b, ad, m, dv = c1.tables()
    assert (ad == o.addgf).all() and (m == o.mulgf).all() and (dv == o.divgf).all()
    # reference tables handed in explicitly (the INTEGRATION.md route) are accepted, broken ones are not
    a2 = dict(a, bingf=o.bingf, addgf=o.addgf, mulgf=o.mulgf, divgf=o.divgf)
    nbldpc.Code(arrays=a2).close()
    bad = o.addgf.copy(); bad[3, 5] ^= 1
    with pytest.raises(nbldpc.NbgpuError):
        nbldpc.Code(arrays=dict(a2, addgf=bad))


@pytest.mark.parametrize("name", ["n96_gf64_nm20", "n96_gf256_kn_nm20", "mat24_n480_nm16", "mat28_n72_nm12", "ahmed_r34_gf16_nm16"])
def test_frame_source_equals_reference_stream(name):
    g = Golden(name)
    c = nbldpc.Code(matrix_path(g.matrix))
    o = ol.Oracle(matrix_path(g.matrix), g.dialect)
    nf = min(g.nf, 3)
    pf, sigma = product_frames(c, nf, g.ebn)
    of, osig = oracle_frames(o, nf, g.ebn, want_llr=False)
    assert np.float32(sigma) == np.float32(osig)
    for f in range(nf):
        assert (pf[f]["nbin"] == g.z["nbin"][f]).all()
        assert (pf[f]["cw"] == of[f]["cw"]).all()
        assert pf[f]["noisy"].tobytes() == of[f]["noisy"].tobytes()
        assert o.syndrome(pf[f]["cw"]) == 0
    o.close()


def test_rng_jump_ahead_gives_independent_frames():
    c = nbldpc.Code(matrix_path("matrices/N96_K48_GF64"))
    c.prepare_encoder()
    pf, _ = product_frames(c, 4, 3.0)
    D = (c.K + 2 * c.N) * c.logq                      # drand48 draws per frame (SURVEY.md 8d)
    c.rng_default(); c.rng_skip(3 * D)
    cw, nbin = c.random_codeword()
    assert (cw == pf[3]["cw"]).all()
    assert c.noise(nbin, 3.0).tobytes() == pf[3]["noisy"].tobytes()


def test_rank_deficient_matrix_is_an_error():
    a = dict(N=4, M=2, q=16, row_deg=np.array([2, 2], np.int32), col=np.array([0, 1, 0, 1], np.int32),
             val=np.array([1, 1, 1, 1], np.int32))
    c = nbldpc.Code(arrays=a)
    with pytest.raises(nbldpc.NbgpuError) as e:
        c.prepare_encoder()
    assert e.value.code == nbldpc.ERANK                 # tools.c:181-185 exits


def test_statistics_follow_reference_rules():
    """NB_LDPC.c:474-507 incl. the stop at the 40th erroneous frame, against the oracle's Monte-Carlo loop."""
    p = matrix_path("matrices/N96_K48_GF64")
    o = ol.Oracle(p)
    c = nbldpc.Code(p)
    frames = 400
    ebn = 1.0                                           # many frame errors -> the 40-error stop triggers
    ref = o.monte_carlo(frames, ebn, 20, 25, 10, 0.3)
    of, sigma = oracle_frames(o, frames, ebn)
    dec = np.zeros((frames, o.N), np.int32); synd = np.zeros(frames, np.int32); it = np.zeros(frames, np.int32)
    for f, fr in enumerate(of):
        r = o.decode_frame(fr["llr"], 20, 25, 10, 0.3)
        dec[f], synd[f], it[f] = r["decide"], r["synd"], r["iters"]
    bits = np.stack([fr["nbin"] for fr in of])
    stats = np.zeros(6, np.int64)
    for lo in range(0, frames, 64):                      # batches, as the GPU driver feeds them
        c.accumulate_stats(bits[lo:lo + 64], dec[lo:lo + 64], synd[lo:lo + 64], it[lo:lo + 64], stats)
    assert ref[1] == 40 and stats[5] == 1
    assert [int(x) for x in stats[:5]] == [ref[0], ref[1], ref[2], ref[3], ref[4]]
    # the same rule fed with per-frame error counts (what nbgpu_source_results delivers), other batch size
    bing = c.tables()[0]
    err = np.array([(bing[dec[f, :c.K]] != bits[f].reshape(c.N, c.logq)[:c.K]).sum() for f in range(frames)], np.int32)
    stats2 = np.zeros(6, np.int64)
    for lo in range(0, frames, 50):
        e, sy, itr = (np.ascontiguousarray(x[lo:lo + 50], np.int32) for x in (err, synd, it))
        assert nbldpc.lib().nbgpu_accumulate_results(e.ctypes.data_as(C.POINTER(C.c_int)), sy.ctypes.data_as(C.POINTER(C.c_int)),
                                                     itr.ctypes.data_as(C.POINTER(C.c_int)), len(e), stats2.ctypes.data_as(C.POINTER(C.c_long))) == 0
    assert (stats2 == stats).all()
    o.close()


# ---- pass schedule -------------------------------------------------------------------------------
class _Sched(C.Structure):
    _fields_ = [("nsteps", C.c_int), ("step_ptr", C.POINTER(C.c_int)), ("order", C.POINTER(C.c_int)), ("depth", C.c_int)]


@pytest.mark.parametrize("rel,cap,depth", [("matrices/N96_K48_GF64", 64, 4), ("matrices/Mat24_N480_M240", 16, 6),
                                           ("matrices/MatDeclercq_R12_GF64", 64, 474), ("matrices/Ahmed_64800_R34_GF16", 8, 21),
                                           ("matrices/AD_64800_R12_GF256", 64, 15), ("matrices/AD_64800_R12_GF256", 1, 15)])
def test_schedule_preserves_reference_order(rel, cap, depth):
    c = nbldpc.Code(matrix_path(rel))
    L = nbldpc.lib()
    s = _Sched()
    L.nbgpu_build_schedule.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Sched)]
    assert L.nbgpu_build_schedule(c.h, cap, C.byref(s)) == 0
    assert s.depth == depth                              # SURVEY.md section 2.1 catalogue
    sp = np.ctypeslib.as_array(s.step_ptr, (s.nsteps + 1,)).copy()
    order = np.ctypeslib.as_array(s.order, (c.M,)).copy()
    assert sorted(order.tolist()) == list(range(c.M)) and sp[0] == 0 and sp[-1] == c.M
    assert (np.diff(sp) <= cap).all() and (np.diff(sp) >= 1).all()
    step_of = np.zeros(c.M, np.int64)
    for st in range(s.nsteps):
        step_of[order[sp[st]:sp[st + 1]]] = st
    last = np.full(c.N, -1, np.int64)                   # step of the latest (file order) check touching each variable
    for m in range(c.M):
        cols = c.col[c.row_ptr[m]:c.row_ptr[m + 1]]
        assert (last[cols] < step_of[m]).all(), "check %d would run before/with an earlier check sharing a variable" % m
        last[cols] = step_of[m]


def test_c_driver_is_built_and_fails_loudly_without_a_gpu(tmp_path):
    """csrc/nbldpc_mc.c: the plain-C Monte-Carlo driver links against the C ABI only; without a GPU it reports the error of
    nbgpu_create instead of decoding on the CPU"""
    import subprocess
    exe = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
    assert os.path.exists(exe)
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode != 0 and "NbMonteCarlo" in r.stdout
    if nbldpc.device_count() == 0:
        r = subprocess.run([exe, "4", "10", matrix_path("matrices/N96_K48_GF64"), "3.0", "20", "0.3", "25"], cwd=tmp_path,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode != 0 and "no CPU fallback" in r.stdout


def test_apsk64_host_side_equals_oracle():
    """Host side of the 64-APSK channel (nbgpu_apsk64_table, nbgpu_sigma_apsk64, nbgpu_awgn_apsk64_noise): constellation, sigma
    and the noisy samples on the reference's drand48 stream equal the oracle's, bit for bit; other fields are refused."""
    path = matrix_path("matrices/N96_K48_GF64")
    code = nbldpc.Code(path)
    o = ol.Oracle(path)
    assert nbldpc.apsk64_table().tobytes() == o.apsk64_table().tobytes()
    code.prepare_encoder(); code.rng_default(); o.prepare_encoder(); o.rng_default()
    for ebn in (4.0, 9.0):
        assert nbldpc.sigma_apsk64(ebn) == o.sigma_apsk64(ebn)
        for _ in range(5):
            _, nb = code.random_codeword()
            _, nb_o = o.random_codeword()
            assert (nb == nb_o).all()
            assert code.noise_apsk64(nb, ebn).tobytes() == o.channel_noise_apsk64(nb_o, ebn).tobytes()
    o.close()
    c256 = nbldpc.Code(matrix_path("matrices/KN/N96_K48_GF256.txt"))
    with pytest.raises(nbldpc.NbgpuError):
        c256.noise_apsk64(None, 9.0)
