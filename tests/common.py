"""Shared helpers of the test-suite: fixture loading, matrix lookup, seeded frame generation, the channels' host frames and
the Monte-Carlo driver."""
import glob
import hashlib
import importlib
import os
import subprocess

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol

multigpu = importlib.import_module("ems-decoder-of-nb-ldpc-codes_b200.multigpu")

ROOT = ol.ROOT
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
MATRIX_DIRS = [ROOT, ol.REF_DIR]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def matrix_path(rel):
    """rel = 'matrices/...' as in the reference tree: the repository's matrices/, then the copies oracle/Makefile makes."""
    for d in MATRIX_DIRS:
        p = os.path.join(d, rel)
        if os.path.exists(p):
            return p
    pytest.skip("matrix %s not available (neither in matrices/ nor in oracle/_ref)" % rel)


# (N, M, GF, check degree) of the reference's matrices that matrices/ lacks; every one has column degree 2
SHAPES = {"matrices/AD_64800_R12_GF256": (8100, 4050, 256, 4), "matrices/Ahmed_64800_R34_GF16": (16200, 4050, 16, 8),
          "matrices/MatDeclercq_R12_GF64": (10800, 5400, 64, 4), "matrices/Mat24_N480_M240": (480, 240, 64, 4),
          "matrices/Mat26_N48_M16": (48, 16, 64, 6),
          "matrices/Mat212_N96_M16": (96, 16, 64, 12), "matrices/Mat212_N480_M80": (480, 80, 64, 12),
          "matrices/KN/N576_K480_GF64.txt": (96, 16, 64, 12), "matrices/KN/N128_K64_GF256.txt": (16, 8, 256, 4),
          "matrices/KN/N64800_K48600_GF256.txt": (8100, 2025, 256, 8)}
_STANDIN = {}


def code_path(rel):
    """matrix_path(rel) when the file is here; otherwise a seeded random code of the same shape, written in the same layout
    (UBS, KN, or full alist for N64800_*).  For tests that compare the product with the oracle on a code of that size and
    field: they need such a code, not that particular one.  Tests against recorded reference runs use matrix_path."""
    for d in MATRIX_DIRS:
        if os.path.exists(os.path.join(d, rel)):
            return os.path.join(d, rel)
    if rel not in _STANDIN:
        import tempfile
        N, M, q, dc = SHAPES[rel]
        a = random_regular_code(np.random.default_rng(N + M + q + dc), N, M, q, dc)
        path = os.path.join(tempfile.mkdtemp(prefix="nbldpc_standin_"), os.path.basename(rel))
        if "N64800" in rel:
            write_alist_full(path, a)
        elif rel.startswith("matrices/KN/"):
            write_alist_kn(path, a)
        else:
            write_alist_ubs(path, a)
        _STANDIN[rel] = path
    return _STANDIN[rel]


_SYN = {}


def mpath(rel):
    """reference matrices, plus small synthetic GF(16) codes (the only GF(16) matrix of the reference is the 64800-bit one)"""
    if not rel.startswith("synthetic/"):
        return code_path(rel)
    if rel not in _SYN:
        import re
        import tempfile
        q, N, M, dc = [int(x) for x in re.match(r"synthetic/GF(\d+)_N(\d+)_M(\d+)_dc(\d+)", rel).groups()]
        a = random_regular_code(np.random.default_rng(q + N + dc), N, M, q, dc)
        path = os.path.join(tempfile.mkdtemp(prefix="nbldpc_syn_"), rel.split("/")[1])
        write_alist_ubs(path, a)
        _SYN[rel] = path
    return _SYN[rel]


def golden_names():
    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Golden:
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
        self.z = z
        self.name = name
        self.frames, self.nb_iter_max, self.n_m, self.nb_oper = [int(x) for x in z["args"]]
        self.ebn = float(z["ebn"]); self.offset = float(z["offset"])
        self.matrix = str(z["matrix"]); self.dialect = 2 if str(z["dialect"]) == "kn" else 1
        self.N, self.M, self.GF, self.logGF, self.E = [int(x) for x in z["header"]]
        self.nf = z["nbin"].shape[0]
        self.npasses = z["npasses"]
        self.decide = z["decide"].astype(np.int32)
        self.synd = z["synd"]
        self.app_sha = z["app_sha"]
        self.llr_sha = z["llr_sha"]
        # (d1, d2, d3, trunc, n_cv) when the fixture was produced with the reference's syndrome_ems as check node
        self.synd_params = tuple(int(x) for x in z["synd_params"]) if "synd_params" in z else None

    def final(self, f, nb_iter_max=None):
        """(decide, synd, iters) the reference reports for frame f when run with nb_iter_max (<= the fixture's)."""
        P = (nb_iter_max or self.nb_iter_max) - 1
        p = min(int(self.npasses[f]), P)
        synd = int(self.synd[f, p - 1])
        iters = p if synd == 0 else P + 1          # sum_it += iter+1 (NB_LDPC.c:474): iter == P when never converged
        return self.decide[f, p - 1], synd, iters, p


def oracle_frames(o, nframes, ebn, want_llr=True):
    """The reference's frame stream (NB_LDPC.c:250-262) from the oracle port: per frame codeword, bits, noisy, llr."""
    o.prepare_encoder()
    o.rng_default()
    sigma = o.sigma(ebn)
    out = []
    for _ in range(nframes):
        cw, nbin = o.random_codeword()
        noisy = o.channel_noise(nbin, ebn)
        llr = o.channel_llr(noisy, sigma) if want_llr else None
        out.append(dict(cw=cw, nbin=nbin, noisy=noisy, llr=llr))
    return out, sigma


def product_frames(code, nframes, ebn):
    """Same stream from the product's host layer (nbgpu_random_codeword / nbgpu_awgn_bpsk_noise)."""
    code.prepare_encoder()
    code.rng_default()
    out = []
    for _ in range(nframes):
        cw, nbin = code.random_codeword()
        noisy = code.noise(nbin, ebn)
        out.append(dict(cw=cw, nbin=nbin, noisy=noisy))
    return out, code.sigma(ebn)


# ---- labelled fields: GF(2)[x]/poly with any bijection from symbols to binary images --------------------------------
REFERENCE_POLY = {16: 0x13, 64: 0x43, 256: 0x11D}           # struct.h:117/145/217
RECIPROCAL_POLY = {16: 0x19, 64: 0x61, 256: 0x171}          # the same polynomials with their coefficients reversed
LABELLINGS = ("reference", "reciprocal", "polynomial", "shuffled")


def _gf_mul(a, b, poly, q):
    """carry-less product of binary images a, b (numpy int arrays) reduced modulo poly"""
    a = np.asarray(a, np.int64); b = np.asarray(b, np.int64)
    r = np.zeros(np.broadcast(a, b).shape, np.int64)
    for l in range(q.bit_length() - 1):
        r ^= np.where((b >> l) & 1, a, 0)
        a = a << 1
        a = np.where(a & q, a ^ poly, a)
    return r


def exponent_images(q, poly):
    """img[0] = 0, img[k] = x^(k-1) mod poly: the reference's labelling (symbol k >= 1 is alpha^(k-1))"""
    img = np.zeros(q, np.int64)
    x = 1
    for k in range(1, q):
        img[k] = x
        x <<= 1
        if x & q:
            x ^= poly
    return img


def field_tables(q, poly, img):
    """(bingf, addgf, mulgf, divgf) of GF(2)[x]/poly where symbol s has the binary image img[s] (img[0] = 0), in the layout of
    nbgpu_code_from_arrays and the oracle (DIVGF[a][0] = -1 as in Table_Div_GF)"""
    lg = q.bit_length() - 1
    img = np.asarray(img, np.int64)
    assert img.shape == (q,) and img[0] == 0 and sorted(img.tolist()) == list(range(q)), "img must be a bijection with img[0] = 0"
    assert poly >> lg == 1, "poly must have degree log2 q"
    x, order = 2, 1
    while x != 1:
        x = int(_gf_mul(x, 2, poly, q)); order += 1
    assert order == q - 1, "poly 0x%x is not primitive: x has order %d" % (poly, order)
    inv = np.zeros(q, np.int64); inv[img] = np.arange(q)
    bingf = ((img[:, None] >> np.arange(lg)) & 1).astype(np.int32)
    addgf = inv[img[:, None] ^ img[None, :]].astype(np.int32)
    mulgf = inv[_gf_mul(img[:, None], img[None, :], poly, q)].astype(np.int32)
    # a^-1 = a^(q-2) in the multiplicative group
    recip = np.ones(q, np.int64)
    for _ in range(q - 2):
        recip = _gf_mul(recip, img, poly, q)
    divgf = np.full((q, q), -1, np.int32)
    divgf[:, 1:] = inv[_gf_mul(img[:, None], recip[None, 1:], poly, q)]
    # field axioms on the symbol tables, all q^3 triples
    M = mulgf.astype(np.uint8); A = addgf.astype(np.uint8)
    a, b, c = np.ix_(np.arange(q), np.arange(q), np.arange(q))
    assert (M == M.T).all(), "MUL is not commutative"
    assert (M[M[a, b], c] == M[a, M[b, c]]).all(), "MUL is not associative"
    assert (M[a, A[b, c]] == A[M[a, b], M[a, c]]).all(), "MUL does not distribute over ADD"
    one = inv[1]
    assert (M[one] == np.arange(q)).all() and (M[:, 0] == 0).all()
    assert (mulgf[divgf[:, 1:], np.arange(1, q)[None, :]] == np.arange(q)[:, None]).all(), "DIV does not invert MUL"
    return bingf, addgf, mulgf, divgf


def labelled_tables(q, labelling, seed=0):
    """the GF(q) tables of one labelling:
    reference  -- exponent labelling over the reference's polynomial (the default tables);
    reciprocal -- exponent labelling over the reciprocal polynomial: the closed-form kernels with other binary images;
    polynomial -- symbol = binary image over the reference's polynomial: the table-driven kernels;
    shuffled   -- a seeded random bijection of the non-zero symbols onto the non-zero images: table-driven kernels, and
                  the images are an arbitrary permutation (the multiplicative identity is not symbol 1)"""
    if labelling == "reference":
        return field_tables(q, REFERENCE_POLY[q], exponent_images(q, REFERENCE_POLY[q]))
    if labelling == "reciprocal":
        return field_tables(q, RECIPROCAL_POLY[q], exponent_images(q, RECIPROCAL_POLY[q]))
    if labelling == "polynomial":
        return field_tables(q, REFERENCE_POLY[q], np.arange(q))
    assert labelling == "shuffled", labelling
    img = np.concatenate([[0], 1 + np.random.default_rng(1000 * q + seed).permutation(q - 1)])
    return field_tables(q, REFERENCE_POLY[q], img)


def is_closed(mulgf, divgf):
    """the predicate of nbgpu_create: MULGF and DIVGF have the exponent closed form, so the kernels compute the rotations
    instead of reading the q x q tables"""
    q = mulgf.shape[0]
    a = np.arange(q)[:, None]; b = np.arange(1, q)[None, :]
    mul = np.where(a > 0, (a + b - 2) % (q - 1) + 1, 0)
    dv = np.where(a > 0, (a - b + (q - 1)) % (q - 1) + 1, 0)
    return bool((mulgf[:, 1:] == mul).all() and (divgf[:, 1:] == dv).all())


def code_arrays(code, tables):
    """nbgpu_code_from_arrays arguments: the graph of `code` (an nbldpc.Code) with the given GF tables"""
    bingf, addgf, mulgf, divgf = tables
    return dict(N=code.N, M=code.M, q=code.q, row_deg=code.row_deg, col=code.col, val=code.val,
                bingf=bingf, addgf=addgf, mulgf=mulgf, divgf=divgf)


def oracle_with_tables(path, dialect, tables):
    """the oracle on the code at `path` with its GF tables overwritten in place (before any encoder is prepared): every
    oracle function reads only these tables once they are built"""
    import ctypes as C
    o = ol.Oracle(path, dialect)
    c = o.h.contents
    for name, t in zip(("bingf", "addgf", "mulgf", "divgf"), tables):
        t = np.ascontiguousarray(t, np.int32)
        assert t.shape == getattr(o, name).shape
        C.memmove(getattr(c, name), t.ctypes.data, t.nbytes)
        setattr(o, name, t.copy())
    return o


def random_regular_code(rng, N, M, q, dc, dv=2):
    """A random check-regular Tanner graph without repeated columns in a row (arrays for nbgpu_code_from_arrays)."""
    assert N * dv == M * dc
    for _ in range(200):
        slots = np.repeat(np.arange(N), dv)
        rng.shuffle(slots)
        rows = slots.reshape(M, dc)
        if all(len(set(r)) == dc for r in rows):
            break
    else:
        for _ in range(1000):                    # dense rows: repair repeated columns by swapping a slot with a random one
            bad = [m for m in range(M) if len(set(rows[m])) < dc]
            if not bad:
                break
            for m in bad:
                k, m2, k2 = rng.integers(dc), rng.integers(M), rng.integers(dc)
                rows[m, k], rows[m2, k2] = rows[m2, k2], rows[m, k]
        else:
            raise RuntimeError("could not build a simple graph")
    col = rows.reshape(-1).astype(np.int32)
    val = rng.integers(1, q, size=M * dc).astype(np.int32)
    return dict(N=N, M=M, q=q, row_deg=np.full(M, dc, np.int32), col=col, val=val)


def write_alist_ubs(path, a):
    with open(path, "w") as f:
        N, M, q = a["N"], a["M"], a["q"]
        f.write("%d %d %d\n" % (N, M, q))
        cd = np.bincount(a["col"], minlength=N)
        f.write(" ".join(str(x) for x in cd) + "\n")
        f.write(" ".join(str(x) for x in a["row_deg"]) + "\n")
        e = 0
        for m in range(M):
            f.write(" ".join(str(x) for x in a["col"][e:e + a["row_deg"][m]]) + "\n"); e += a["row_deg"][m]
        e = 0
        for m in range(M):
            f.write(" ".join(str(x) for x in a["val"][e:e + a["row_deg"][m]]) + "\n"); e += a["row_deg"][m]


def write_alist_full(path, a, pad=False):
    """full alist: max-degree line, column lists then row lists of (index 1-based, exponent) pairs (matrices/KN/N64800_*);
    pad=True fills every list with '0 0' pairs up to the maximum degree, as MacKay's tools do for irregular codes"""
    N, M, q = a["N"], a["M"], a["q"]
    rd = np.asarray(a["row_deg"]); col = np.asarray(a["col"]); val = np.asarray(a["val"])
    rp = np.concatenate([[0], np.cumsum(rd)])
    cols = [[] for _ in range(N)]
    for m in range(M):
        for e in range(rp[m], rp[m + 1]):
            cols[col[e]].append((m + 1, val[e] - 1))
    cd = [len(c) for c in cols]
    dv, dc = max(cd), int(rd.max())
    with open(path, "w") as f:
        f.write("%d %d %d\n%d %d\n" % (N, M, q, dv, dc))
        f.write(" ".join(map(str, cd)) + "\n" + " ".join(map(str, rd)) + "\n")
        for c in cols:
            items = c + ([(0, 0)] * (dv - len(c)) if pad else [])
            f.write("   ".join("%d %d" % it for it in items) + "\n")
        for m in range(M):
            items = [(col[e] + 1, val[e] - 1) for e in range(rp[m], rp[m + 1])]
            items += [(0, 0)] * (dc - len(items)) if pad else []
            f.write("   ".join("%d %d" % it for it in items) + "\n")


def write_alist_kn(path, a):
    """KN dialect (init.c:211-227): degrees, then per row (column 1-based, exponent) pairs"""
    N, M, q = a["N"], a["M"], a["q"]
    rd = np.asarray(a["row_deg"]); col = np.asarray(a["col"]); val = np.asarray(a["val"])
    rp = np.concatenate([[0], np.cumsum(rd)])
    with open(path, "w") as f:
        f.write("%d %d %d\n\n" % (N, M, q))
        f.write(" ".join(map(str, np.bincount(col, minlength=N))) + "\n" + " ".join(map(str, rd)) + "\n\n")
        for m in range(M):
            f.write("   ".join("%d %d" % (col[e] + 1, val[e] - 1) for e in range(rp[m], rp[m + 1])) + "\n")


# ---- channels: host frames, device-source checks, the Monte-Carlo driver ------------------------------------------------
EXE = os.path.join(os.path.dirname(nbldpc.LIB_PATH), "nbldpc_mc")
CONSOLE = r"<(\d+)> FER=\s*(\d+)\s*/\s*(\d+)\s*=\s*[\d.]+\s*BER=\s*(\d+)\s*/\s*x\s*=\s*[\d.eE+-]+\s*avr_it=([\d.]+)"
PI = 3.1415926536                                              # channel.c:18
# one code per field; GF(16) has no matrix file, so a seeded random code stands in (mpath)
CODES = {16: "synthetic/GF16_N24_M12_dc4", 64: "matrices/N96_K48_GF64", 256: "matrices/KN/N96_K48_GF256.txt"}
ESN = {16: 10.0, 64: 15.0, 256: 23.0}                          # Es/N0 (dB) at which the QAM frames mix easy and hard ones
FADING_NAMES = {nbldpc.FADING_SYMBOL: "symbol", nbldpc.FADING_COMPONENT: "component"}


def field_code(q):
    path = mpath(CODES[q])
    return nbldpc.Code(path), path


def seeded_table(q, seed=5):
    """a table that is neither normalised nor symmetric, with two coincident points"""
    mod = np.random.default_rng(seed).normal(0, 1.7, (q, 2)).astype(np.float32)
    mod[3] = mod[1]
    return mod


def oracle_llr_mapped(o, noisy, mod, sigma):
    """channel.c:266-291 on mod: f32 differences and squares, f64 divisions by 2 (float)(sigma^2) and sum, rounded to f32"""
    img = (o.bingf.astype(np.int64) << np.arange(o.bingf.shape[1])).sum(1)
    den = 2.0 * float(np.float32(sigma) * np.float32(sigma))
    d0 = (noisy[:, 0:1].astype(np.float32) - mod[img, 0][None, :]).astype(np.float32)
    d1 = (noisy[:, 1:2].astype(np.float32) - mod[img, 1][None, :]).astype(np.float32)
    a = (d0 * d0).astype(np.float64) / den
    b = (d1 * d1).astype(np.float64) / den
    return (a + b).astype(np.float32)


def host_frames(code, frame0, B, ebn, channel, mod=None, fading=None):
    """frames [frame0, frame0 + B) of the host source: (codewords [B, N], bits [B, N, logq], frames) on channel "bpsk"
    (noisy [B, N, logq]), "apsk64" (noisy [B, N, 2]) or "mapped" on mod (noisy [B, N, 2]; with fading = FADING_SYMBOL or
    FADING_COMPONENT, rx [B, N, 4])"""
    code.prepare_encoder()
    code.rng_default()
    code.rng_skip(frame0 * multigpu.draws_per_frame(code, channel, fading=FADING_NAMES.get(fading)))
    cws, bits, noisy = [], [], []
    for _ in range(B):
        cw, nbin = code.random_codeword()
        cws.append(cw); bits.append(nbin)
        if fading:
            noisy.append(code.noise_faded(nbin, mod, ebn, fading))
        elif channel == "mapped":
            noisy.append(code.noise_mapped(nbin, mod, ebn))
        else:
            noisy.append(code.noise_apsk64(nbin, ebn) if channel == "apsk64" else code.noise(nbin, ebn))
    return np.stack(cws), np.stack(bits), np.stack(noisy)


def same_stream(d, code, frame0, B, ebn, channel, mod=None, fading=None):
    """the batch d generated equals host_frames, codewords and frames bit for bit"""
    cw, _, noisy = host_frames(code, frame0, B, ebn, channel, mod, fading)
    gcw, gnoisy = d.source_download()
    assert gnoisy.shape == noisy.shape
    return (gcw == cw).all() and gnoisy.tobytes() == noisy.tobytes()


def soft(d, kind):
    return d.soft_list() if kind == nbldpc.SOFT_LIST else (d.soft_bits(),)


def waves(code, n_m, early=True, **kw):
    """a batch of more than two waves of the decoder's geometry (one frame per CTA): streamed path and slot reuse"""
    d = nbldpc.Decoder(code, n_m, 25, 10, 0.3, early_stop=early, max_batch=1 << 14, frames_per_cta=1, **kw)
    g = d.geometry()
    d.close()
    return 2 * g["grid"] * g["frames_per_cta"] + 37


def run_driver(tmp_path, sub, path, ebn, n_m, source, channel, *tail, devices="0"):
    """nbldpc_mc on 2000 frames of `path` in tmp_path/sub (channel, then the fading and degrees arguments in tail):
    (console output, results-file lines without their time stamps)"""
    d = tmp_path / sub
    os.makedirs(d / "data")
    r = subprocess.run([EXE, "2000", "10", path, ebn, str(n_m), "0.3", "25", "128", devices, "0", str(source), str(channel), *tail],
                       cwd=d, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:]
    lines = list((d / "data").glob("results_*.txt"))[0].read_text().splitlines()
    return r.stdout, [ln.split("time:")[0] for ln in lines]
