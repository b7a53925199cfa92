"""Seeded random configurations of the decode path against the oracle: field, check degrees (regular and irregular), list
length, pop budget, offset, iteration limit, early termination on/off, both check nodes.  Everything is bit-exact."""
import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import code_arrays, labelled_tables, oracle_with_tables, write_alist_ubs

pytestmark = pytest.mark.gpu


def _random_code(rng, q, N, dcs):
    """Tanner graph with the given check degrees, no repeated column inside a row, every variable used when possible"""
    M = len(dcs)
    cols, vals = [], []
    pool = list(rng.permutation(N))
    for dc in dcs:
        row = []
        while len(row) < dc:
            if not pool:
                pool = list(rng.permutation(N))
            v = pool.pop()
            if v not in row:
                row.append(v)
        cols += row
        vals += list(rng.integers(1, q, dc))
    return dict(N=N, M=M, q=q, row_deg=np.array(dcs, np.int32), col=np.array(cols, np.int32), val=np.array(vals, np.int32))


CASES = list(range(160))


@pytest.mark.parametrize("seed", CASES)
def test_random_configuration_equals_oracle(seed, tmp_path):
    _random_configuration(seed, tmp_path, None)


@pytest.mark.parametrize("seed", list(range(0, 48, 3)) + [3, 7, 11, 15])
def test_random_configuration_with_negative_offset_equals_oracle(seed, tmp_path):
    """offset < 0 (the command line accepts it): the saturation fill value is below the last list entry, so the record
    expansion cannot use its min() form (expand_record, minform = false)"""
    _random_configuration(seed, tmp_path, -0.4 if seed % 2 else -1.5)


@pytest.mark.parametrize("labelling", ["polynomial", "shuffled"])
@pytest.mark.parametrize("seed", list(range(8)) + [11, 15, 19, 23])
def test_random_configuration_with_relabelled_field_equals_oracle(seed, labelling, tmp_path):
    """the same configurations over fields whose MULGF/DIVGF lack the exponent form: the table-driven kernels, against the
    oracle with the same tables"""
    _random_configuration(seed, tmp_path, None, labelling)


def _random_configuration(seed, tmp_path, offset_override, labelling="reference"):
    rng = np.random.default_rng(1000 + seed)
    q = int(rng.choice([16, 64, 256]))
    syndrome = seed % 4 == 3
    if syndrome:
        dc = int(rng.choice([4, 5, 6, 8]))
        dcs = [dc] * int(rng.integers(3, 9))
    elif seed % 3 == 0:
        dcs = [int(x) for x in rng.choice([2, 3, 4, 5, 7], int(rng.integers(4, 12)))]          # irregular
    else:
        dc = int(rng.choice([2, 3, 4, 6, 8, 10, 16]))
        dcs = [dc] * int(rng.integers(3, 10))
    N = max(max(dcs) + 2, len(dcs) + 2, int(sum(dcs) / rng.choice([1.5, 2.0, 3.0])))      # N > M: the rate (and sigma) must be finite
    a = _random_code(rng, q, N, dcs)
    path = str(tmp_path / "code.alist")
    write_alist_ubs(path, a)
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    if labelling != "reference":
        t = labelled_tables(q, labelling, seed)
        o.close()
        o = oracle_with_tables(path, code.dialect, t)
        code = nbldpc.Code(arrays=code_arrays(code, t))
    n_m = int(rng.integers(5, min(q, 32) + 1))
    nb_oper = int(rng.integers(1, 61))
    offset = float(rng.choice([0.0, 0.3, 1.0, 2.5]))
    if offset_override is not None:
        offset = offset_override
    nb_iter_max = int(rng.integers(2, 9))
    early = bool(rng.integers(0, 2))
    frames = int(rng.integers(1, 40))
    ebn = float(rng.choice([1.0, 3.0, 6.0]))
    kw, okw = {}, {}
    if syndrome:
        # presorting_mvc only works while the 2nd/3rd best LLRs stay below its 10000 sentinel (syndrome_decoder.c:325): keep the
        # messages in that regime (moderate SNR, few passes); beyond it the reference reads an uninitialised index
        ebn = min(ebn, 3.0)
        nb_iter_max = min(nb_iter_max, 4)
        d1 = int(rng.integers(1, n_m))
        d2 = int(rng.integers(1, min(n_m, 7)))
        d3 = int(rng.integers(1, min(n_m, 4)))
        trunc = int(rng.choice([0, 200, 1000]))
        size = nbldpc.config_table(dcs[0], d1, d2, d3, trunc).shape[0]
        if size > 1024:
            trunc = 1000
        cfg = o.build_config_table(dcs[0], d1, d2, d3, trunc)
        kept = min(int((cfg[:, d] == 0).sum()) - 3 * d for d in range(dcs[0]))
        n_cv = int(rng.integers(1, max(2, min(kept, 30))))
        if n_cv - 1 >= kept:
            pytest.skip("no admissible n_cv for this table")
        kw = dict(ecn_kind=1, d1=d1, d2=d2, d3=d3, cfg_trunc=trunc, n_cv=n_cv)
        okw = dict(ecn=1, cfg=cfg, n_cv=n_cv)
    code.rng_default()
    code.rng_skip(seed * 1000003)
    sigma = code.sigma(ebn)
    noisy = np.stack([code.noise(None, ebn) for _ in range(frames)])        # all-zero codeword: random graphs need not be full rank
    d = nbldpc.Decoder(code, n_m, nb_oper, nb_iter_max, offset, early_stop=early, max_batch=frames, **kw)
    dec, synd, it = d.decode_noisy(noisy, sigma)
    llr = d.channel(noisy, sigma)
    for f in range(frames):
        r = o.decode_frame(llr[f], n_m, nb_oper, nb_iter_max, offset, force=not early, want_state=(f == 0), **okw)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], (seed, f)
        if f == 0:
            app, ctov = d.get_state(0)
            assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), seed
    o.close(); d.close()


@pytest.mark.parametrize("seed", list(range(24)))
def test_adversarial_llr_inputs_equal_oracle(seed, tmp_path):
    """Dense-LLR intake with values the channel never produces: small integers (exact ties everywhere -> lowest-symbol /
    lowest-bubble rules), negative values, entries at or above the 1e5 sentinel, one-hot rows."""
    rng = np.random.default_rng(5000 + seed)
    q = int(rng.choice([16, 64, 256]))
    dc = int(rng.choice([3, 4, 4, 6]))
    dcs = [dc] * int(rng.integers(3, 8))
    N = max(dc + 2, len(dcs) + 2, sum(dcs) // 2)
    a = _random_code(rng, q, N, dcs)
    path = str(tmp_path / "code.alist")
    write_alist_ubs(path, a)
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    n_m = int(rng.integers(5, min(q, 32) + 1))
    nb_oper = int(rng.integers(4, 40))
    frames = 12
    kind = seed % 4
    if kind == 0:
        llr = rng.integers(0, 6, (frames, N, q)).astype(np.float32)                       # ties everywhere
    elif kind == 1:
        llr = (rng.integers(-8, 24, (frames, N, q)) * 0.5).astype(np.float32)             # negative values too
    elif kind == 2:
        llr = (rng.random((frames, N, q)) * 30).astype(np.float32)
        llr[rng.random(llr.shape) < 0.9] = 1e5                                            # fewer than n_m selectable symbols
        llr[rng.random(llr.shape) < 0.05] = 2.5e5
    else:
        llr = np.full((frames, N, q), 40.0, np.float32)                                   # one-hot rows + a few flips
        np.put_along_axis(llr, rng.integers(0, q, (frames, N, 1)), 0.0, axis=2)
    d = nbldpc.Decoder(code, n_m, nb_oper, 5, 0.3, max_batch=frames)
    dec, synd, it = d.decode_llr(llr)
    for f in range(frames):
        r = o.decode_frame(llr[f], n_m, nb_oper, 5, 0.3, want_state=(f < 2))
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], (seed, f)
        if f < 2:
            app, ctov = d.get_state(f)
            assert np.array_equal(app, r["app"], equal_nan=True) and np.array_equal(ctov, r["ctov"], equal_nan=True), (seed, f)
    o.close(); d.close()


@pytest.mark.parametrize("seed", list(range(12)))
def test_syndrome_node_with_tiny_and_tied_llrs_equals_oracle(seed, tmp_path):
    """The syndrome check node drops the small-operand guard of bayes() only when it can prove that no operand falls below 2^-96
    (synd_prepare): LLRs scaled down to 2^-40 .. 2^-110 (and exact ties, which make long symbol groups) must take the guarded walk
    and still equal the reference bit for bit."""
    rng = np.random.default_rng(7000 + seed)
    q = int(rng.choice([16, 64, 256]))
    dc = int(rng.choice([4, 4, 5]))
    dcs = [dc] * int(rng.integers(3, 7))
    N = max(dc + 2, len(dcs) + 2, sum(dcs) // 2)
    a = _random_code(rng, q, N, dcs)
    path = str(tmp_path / "code.alist")
    write_alist_ubs(path, a)
    code = nbldpc.Code(path)
    o = ol.Oracle(path, code.dialect)
    n_m = int(rng.integers(6, min(q, 20) + 1))
    d1, d2, d3 = int(rng.integers(2, n_m)), int(rng.integers(1, min(n_m, 6))), int(rng.integers(1, min(n_m, 4)))
    trunc = 1000 if nbldpc.config_table(dc, d1, d2, d3, 0).shape[0] > 1024 else 0
    cfg = o.build_config_table(dc, d1, d2, d3, trunc)
    kept = min(int((cfg[:, d] == 0).sum()) - 3 * d for d in range(dc))
    if kept < 2:
        pytest.skip("no admissible n_cv for this table")
    n_cv = int(rng.integers(1, max(2, min(kept, 20))))
    frames = 6
    kind = seed % 3
    if kind == 0:
        llr = (rng.random((frames, N, q)) * 30).astype(np.float32) * np.float32(2.0 ** -int(rng.integers(40, 111)))
    elif kind == 1:
        llr = rng.integers(0, 4, (frames, N, q)).astype(np.float32)                        # ties everywhere
    else:
        llr = (rng.random((frames, N, q)) * 30).astype(np.float32)
        llr[rng.random(llr.shape) < 0.3] *= np.float32(2.0 ** -100)                         # a mix of ordinary and tiny values
    d = nbldpc.Decoder(code, n_m, 20, 4, 0.3, max_batch=frames, ecn_kind=1, d1=d1, d2=d2, d3=d3, cfg_trunc=trunc, n_cv=n_cv)
    dec, synd, it = d.decode_llr(llr)
    for f in range(frames):
        r = o.decode_frame(llr[f], n_m, 20, 4, 0.3, want_state=(f < 2), ecn=1, cfg=cfg, n_cv=n_cv)
        assert (dec[f] == r["decide"]).all() and synd[f] == r["synd"] and it[f] == r["iters"], (seed, f)
        if f < 2:
            app, ctov = d.get_state(f)
            assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), (seed, f)
    o.close(); d.close()
