"""Launch geometry must not change what the decoder computes.

The planner picks warps per CTA, check nodes per warp, frames per CTA group and CTAs per SM; tuning runs override them
(NBGPU_WARPS, NBGPU_CPW, NBGPU_SMEM_KB, NBGPU_CTAS_PER_SM) and callers pass frames_per_cta / cns_per_step.  Some tile paths
are only reached away from the planner's choice: the cb loop of tile_elementary_steps with more than 8 nodes per warp,
one-warp CTAs, the shrink loop under a small shared-memory budget, cns_per_step caps.  Every geometry below is compared with
the oracle, bit for bit; the environment is set with monkeypatch, so no geometry leaks into another test."""
import functools

import numpy as np
import pytest

import nbldpc
import oracle_lib as ol
from common import product_frames, random_regular_code, write_alist_ubs
from test_gpu_fuzz import _random_code
from test_gpu_parity import _lists, mpath
from test_gpu_soft_output import ref_bits

pytestmark = pytest.mark.gpu

B = 40                                                      # frames the oracle decodes per code
BATCH = 1500                                                # decoded batch: frame f is oracle frame f % B; several waves of the grid
# name -> (code, n_m, Eb/N0, syndrome check node)
CODES = {"gf16_dc8": ("synthetic/GF16_N32_M8_dc8", 16, 4.0, False),         # two edges per warp lane group
         "gf64_n96": ("matrices/N96_K48_GF64", 20, 2.5, False),
         "gf256_n96_kn": ("matrices/KN/N96_K48_GF256.txt", 20, 2.5, False),
         "gf64_irregular": ("irregular", 16, 3.0, False),                     # check degrees 2 ... 7
         "gf64_dc16": ("dc16", 20, 5.0, False),
         "gf64_n96_syndrome": ("matrices/N96_K48_GF64", 20, 2.0, True)}
SYND_KW = dict(ecn_kind=1, d1=19, d2=15, d3=5, cfg_trunc=1000, n_cv=25)
GEOMETRIES = {"default": ({}, {}),
              **{"fpc%d" % f: ({}, dict(frames_per_cta=f)) for f in (1, 2, 3, 8)},
              **{"cns%d" % c: ({}, dict(cns_per_step=c)) for c in (1, 2, 5, 12)},
              **{"w%d_cpw%d" % wc: (dict(NBGPU_WARPS=wc[0], NBGPU_CPW=wc[1]), {}) for wc in ((1, 1), (3, 2), (4, 12), (2, 32), (12, 8))},
              "smem_shrink": (dict(NBGPU_WARPS=12, NBGPU_CPW=8, NBGPU_SMEM_KB=24), {}),
              "one_cta_per_sm": (dict(NBGPU_CTAS_PER_SM=1), {})}
ENV = ("NBGPU_WARPS", "NBGPU_CPW", "NBGPU_SMEM_KB", "NBGPU_CTAS_PER_SM", "NBGPU_GF_TABLES", "NBGPU_NO_CHUNKS")


@functools.lru_cache(maxsize=None)
def _path(name):
    rel = CODES[name][0]
    if rel not in ("irregular", "dc16"):
        return mpath(rel)
    import tempfile
    rng = np.random.default_rng(len(rel))
    a = _random_code(rng, 64, 60, [2, 3, 4, 5, 6, 7] * 4) if rel == "irregular" else random_regular_code(rng, 64, 8, 64, 16)
    path = tempfile.mkdtemp(prefix="nbldpc_geo_") + "/" + rel
    write_alist_ubs(path, a)
    return path


@functools.lru_cache(maxsize=None)
def _case(name):
    """the code, B noisy frames of its host source, and the oracle's result and final state of every frame"""
    rel, n_m, ebn, synd = CODES[name]
    code = nbldpc.Code(_path(name))
    o = ol.Oracle(_path(name), code.dialect)
    okw = dict(ecn=1, cfg=o.build_config_table(int(code.row_deg[0]), 19, 15, 5, 1000), n_cv=25) if synd else {}
    code.rng_default()
    if rel in ("irregular", "dc16"):                    # random graphs need not be full rank: the all-zero codeword
        noisy = np.stack([code.noise(None, ebn) for _ in range(B)])
        sigma = code.sigma(ebn)
    else:
        fr, sigma = product_frames(code, B, ebn)
        noisy = np.stack([f["noisy"] for f in fr])
    ref = [o.decode_frame(o.channel_llr(noisy[f], sigma), n_m, 25, 10, 0.3, want_state=True, **okw) for f in range(B)]
    o.close()
    bits = ref_bits(np.stack([r["app"] for r in ref]), code.tables()[0])
    return code, noisy, sigma, ref, bits


def _decoder(monkeypatch, name, geometry, max_batch=BATCH):
    env, kw = GEOMETRIES[geometry]
    for k in ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))
    rel, n_m, ebn, synd = CODES[name]
    code = nbldpc.Code(_path(name))
    return nbldpc.Decoder(code, n_m, 25, 10, 0.3, max_batch=max_batch, **kw, **(SYND_KW if synd else {}))


@pytest.mark.parametrize("geometry", list(GEOMETRIES))
@pytest.mark.parametrize("name", list(CODES))
def test_every_geometry_equals_the_oracle(name, geometry, monkeypatch):
    """every frame of a multi-wave batch: decisions, syndrome, iterations and SOFT_BITS; APP/CtoV of the last two frames"""
    code, noisy, sigma, ref, bits = _case(name)
    d = _decoder(monkeypatch, name, geometry)
    g = d.geometry()
    d.set_soft_output(nbldpc.SOFT_BITS)
    idx = np.arange(BATCH) % B
    dec, synd, it = d.decode_noisy(noisy[idx], sigma)
    assert (dec == np.stack([r["decide"] for r in ref])[idx]).all(), g
    assert (synd == np.array([r["synd"] for r in ref])[idx]).all() and (it == np.array([r["iters"] for r in ref])[idx]).all(), g
    assert d.soft_bits().tobytes() == bits[idx].tobytes(), g
    for f in (BATCH - 2, BATCH - 1):
        app, ctov = d.get_state(f)
        r = ref[f % B]
        assert app.tobytes() == r["app"].tobytes() and ctov.tobytes() == r["ctov"].tobytes(), (f, g)
    if name in ("gf64_n96", "gf256_n96_kn"):
        assert len(set(it.tolist())) > 1, "the batch should mix frames that stop early and frames that do not"
    d.close()


@pytest.mark.parametrize("name", ["gf16_dc8", "gf64_n96", "gf256_n96_kn"])
def test_check_node_with_more_than_eight_nodes_per_warp(name, monkeypatch):
    """nbgpu_check_node runs the decoder's tile code: under 4 warps x 12 nodes the cb loop of tile_elementary_steps runs"""
    d = _decoder(monkeypatch, name, "w4_cpw12")
    assert d.geometry()["cns_per_warp"] > 8, d.geometry()
    code = d.code
    o = ol.Oracle(_path(name), code.dialect)
    n_m = d.p.n_m
    rng = np.random.default_rng(17)
    for node in sorted({0, code.M // 2, code.M - 1}):
        dc = int(code.row_deg[node])
        vl = np.zeros((96, dc, n_m), np.float32); vg = np.zeros((96, dc, n_m), np.int32)
        for b in range(96):
            vl[b], vg[b] = _lists(rng, dc, n_m, code.q, short_frac=0.0)          # full lists: M_VtoC_GF never holds -1
        cl, cg = d.check_node(node, vl, vg)
        for b in range(96):
            rl, rg = o.check_node(node, vl[b], vg[b], n_m, 25, 0.3)
            assert cl[b].tobytes() == rl.tobytes() and (cg[b] == rg).all(), (node, b)
    o.close(); d.close()


def test_the_geometries_reach_the_paths_they_are_here_for(monkeypatch):
    """the geometries as realised (nbgpu_geometry), not as requested: a silently clamped request covers nothing"""
    seen = []
    for name in CODES:
        for geometry in GEOMETRIES:
            d = _decoder(monkeypatch, name, geometry)
            seen.append((name, geometry, d.geometry()))
            d.close()
    real = [g for _, _, g in seen]
    assert any(g["cns_per_warp"] > 8 for g in real), "no geometry with more than 8 check nodes per warp"
    assert any(g["warps_per_cta"] == 1 for g in real), "no one-warp CTA"
    assert any(g["frames_per_cta"] > 1 for g in real), "no CTA group of several frames (early stop is on in every case)"
    default = {n: g for n, geo, g in seen if geo == "default"}
    shrunk = [(n, g) for n, geo, g in seen if geo == "smem_shrink"]
    assert all(g["warps_per_cta"] * g["cns_per_warp"] < 12 * 8 for _, g in shrunk), shrunk
    assert all(g["smem_bytes"] <= 24 * 1024 or g["warps_per_cta"] * g["cns_per_warp"] == 1 for _, g in shrunk), shrunk
    one = {n: g for n, geo, g in seen if geo == "one_cta_per_sm"}
    assert all(one[n]["grid"] <= default[n]["grid"] for n in one), one
    assert any(one[n]["grid"] < default[n]["grid"] for n in one), "one CTA per SM should shrink the grid of some code"
