"""ems-decoder-of-nb-ldpc-codes_b200 -- B200-native EMS decoder for non-binary LDPC codes.

The product is ``libnbldpc_b200.so`` (plain-C host layer + hand-written sm_100a CUDA kernels behind the
C ABI declared in ``include/nbldpc_b200.h``).  This Python module is only a thin ctypes binding of that
ABI for the tests and ``bench.py``; it contains no decoding logic and no CPU fallback: when the shared
library is missing it raises, and every compute entry point fails with NBGPU_ECUDA without a B200.

Import with ``importlib.import_module("ems-decoder-of-nb-ldpc-codes_b200")`` (the directory name is the
repository's, hyphens included) or through ``nbldpc.py`` at the repo root.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NBLDPC_B200_LIB") or os.path.join(HERE, "libnbldpc_b200.so")   # override: tuning builds only

OK, EINVAL, EIO, ENOMEM, ECUDA, ESTATE, ERANK = 0, -1, -2, -3, -4, -5, -6
ALIST_AUTO, ALIST_UBS, ALIST_KN, ALIST_FULL = 0, 1, 2, 3
SOFT_NONE, SOFT_LIST, SOFT_BITS = 0, 1, 2
MAP_APSK64, MAP_QAM = 1, 2
FADING_SYMBOL, FADING_COMPONENT = 1, 2
CHANNEL_BPSK, CHANNEL_MAPPED, CHANNEL_FADED, CHANNEL_SPLIT = 0, 1, 2, 3      # nbgpu_awgn_punctured_noise

_ip = C.POINTER(C.c_int)
_fp = C.POINTER(C.c_float)
_lp = C.POINTER(C.c_long)


class NbgpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("nbgpu error %d: %s" % (code, msg))
        self.code = code


class Params(C.Structure):
    """nbgpu_params (include/nbldpc_b200.h)."""
    _fields_ = [("n_m", C.c_int), ("nb_oper", C.c_int), ("nb_iter_max", C.c_int), ("offset", C.c_float),
                ("ecn_kind", C.c_int), ("early_stop", C.c_int),
                ("d1", C.c_int), ("d2", C.c_int), ("d3", C.c_int), ("cfg_trunc", C.c_int), ("n_cv", C.c_int),
                ("border", C.c_int), ("frames_per_cta", C.c_int), ("cns_per_step", C.c_int)]


class Rng(C.Structure):
    _fields_ = [("x", C.c_uint64)]


def build(force=False):
    """Compile libnbldpc_b200.so in-tree (gcc + nvcc, sm_100a only)."""
    args = ["make", "-s", "-C", os.path.join(HERE, "csrc")]
    if force:
        args.append("-B")
    subprocess.run(args, check=True)


_lib = None


def apsk64_table():
    """The normalised 64-APSK constellation of ModelChannel_AWGN_64 (channel.c:133-222), [64][2], by binary image."""
    mod = np.zeros((64, 2), np.float32)
    _check(lib().nbgpu_apsk64_table(mod.ctypes.data_as(_fp)))
    return mod


def sigma_apsk64(ebn):
    return float(lib().nbgpu_sigma_apsk64(C.c_float(ebn)))


def constellation(kind, q):
    """nbgpu_constellation: mod[q][2] by binary image; MAP_APSK64 (q = 64) or MAP_QAM (Gray square q-QAM, q = 16, 64, 256)."""
    mod = np.zeros((q, 2), np.float32)
    _check(lib().nbgpu_constellation(kind, q, mod.ctypes.data_as(_fp)))
    return mod


def split_qam(q, points):
    """nbgpu_split_qam: the Gray square QAM table mod[M][2], M = 2^(log2(q)/points), by sub-image, of the split channel: (16, 2),
    (64, 3) and (256, 4) give QPSK, (256, 2) gives 16-QAM; other pairs are refused (bind your own table)."""
    M = 1 << ((q.bit_length() - 1) // points) if points > 0 else 0
    mod = np.zeros((max(M, 1), 2), np.float32)
    _check(lib().nbgpu_split_qam(q, points, mod.ctypes.data_as(_fp)))
    return mod


def _split_table(logq, mod, points):
    """mod as the [M][2] f32 table the split calls read, M = 2^(logq / points): a table of another size is a ValueError (the
    library reads exactly 2M floats).  For a points value the library refuses (NBGPU_EINVAL) it reads none, and mod passes
    through flattened."""
    m = np.ascontiguousarray(mod, np.float32)
    if points < 2 or logq % points:
        return m.reshape(-1, 2)
    M = 1 << (logq // points)
    if m.size != 2 * M:
        raise ValueError("split table for %d points per GF(%d) symbol must be [%d][2], not %s" % (points, 1 << logq, M, m.shape))
    return m.reshape(M, 2)


def _pattern(vars):
    """a puncturing pattern as the int32 array the library reads; the library checks range and duplicates.  Values an int32
    cannot hold, or non-integers, are a ValueError (they must not wrap into a valid index)."""
    v = np.asarray(() if vars is None else vars).reshape(-1)
    if v.size and not np.issubdtype(v.dtype, np.integer):
        raise ValueError("puncturing pattern must hold variable indices (integers), not %s" % v.dtype)
    v = v.astype(np.int64)
    if v.size and (v.min() < -2**31 or v.max() >= 2**31):
        raise ValueError("puncturing pattern: index outside the int32 range")
    return np.ascontiguousarray(v, np.int32)


def rotate_constellation(mod, degrees):
    """nbgpu_rotate_constellation: mod[q][2] rotated by `degrees` (computed in double, rounded once), e.g. for signal-space
    diversity under NBGPU_FADING_COMPONENT."""
    m = np.ascontiguousarray(mod, np.float32).reshape(-1, 2)
    out = np.zeros_like(m)
    _check(lib().nbgpu_rotate_constellation(m.shape[0], C.c_double(degrees), m.ctypes.data_as(_fp), out.ctypes.data_as(_fp)))
    return out


def lib():
    """The loaded C-ABI library.  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    sig = {
        "nbgpu_code_load": (C.c_int, [C.POINTER(vp), C.c_char_p, C.c_int]),
        "nbgpu_code_from_arrays": (C.c_int, [C.POINTER(vp), C.c_int, C.c_int, C.c_int, _ip, _ip, _ip, _ip, _ip, _ip, _ip]),
        "nbgpu_code_free": (None, [vp]),
        "nbgpu_code_info": (None, [vp, _ip]),
        "nbgpu_code_rate": (C.c_float, [vp]),
        "nbgpu_code_graph": (None, [vp, _ip, _ip, _ip]),
        "nbgpu_code_tables": (None, [vp, _ip, _ip, _ip, _ip]),
        "nbgpu_rng_reference_default": (None, [C.POINTER(Rng)]),
        "nbgpu_rng_skip": (None, [C.POINTER(Rng), C.c_uint64]),
        "nbgpu_rng_drand48": (C.c_double, [C.POINTER(Rng)]),
        "nbgpu_code_prepare_encoder": (C.c_int, [vp]),
        "nbgpu_random_codeword": (C.c_int, [vp, C.POINTER(Rng), _ip, _ip]),
        "nbgpu_sigma": (C.c_float, [vp, C.c_float]),
        "nbgpu_awgn_bpsk_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, C.c_float, _fp]),
        "nbgpu_apsk64_table": (C.c_int, [_fp]),
        "nbgpu_sigma_apsk64": (C.c_float, [C.c_float]),
        "nbgpu_awgn_apsk64_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, C.c_float, _fp]),
        "nbgpu_channel_awgn_apsk64": (C.c_int, [vp, _fp, C.c_float, C.c_int, _fp, _fp, _ip]),
        "nbgpu_decode_apsk64": (C.c_int, [vp, _fp, C.c_float, C.c_int, _ip, _ip, _ip]),
        "nbgpu_upload_apsk64": (C.c_int, [vp, _fp, C.c_float, C.c_int]),
        "nbgpu_constellation": (C.c_int, [C.c_int, C.c_int, _fp]),
        "nbgpu_awgn_mapped_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, _fp, C.c_float, _fp]),
        "nbgpu_set_constellation": (C.c_int, [vp, _fp]),
        "nbgpu_channel_awgn_mapped": (C.c_int, [vp, _fp, C.c_float, C.c_int, _fp, _fp, _ip]),
        "nbgpu_decode_mapped": (C.c_int, [vp, _fp, C.c_float, C.c_int, _ip, _ip, _ip]),
        "nbgpu_upload_mapped": (C.c_int, [vp, _fp, C.c_float, C.c_int]),
        "nbgpu_rotate_constellation": (C.c_int, [C.c_int, C.c_double, _fp, _fp]),
        "nbgpu_awgn_faded_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, _fp, C.c_float, C.c_int, _fp]),
        "nbgpu_channel_faded": (C.c_int, [vp, _fp, C.c_float, C.c_int, _fp, _fp, _ip]),
        "nbgpu_decode_faded": (C.c_int, [vp, _fp, C.c_float, C.c_int, _ip, _ip, _ip]),
        "nbgpu_upload_faded": (C.c_int, [vp, _fp, C.c_float, C.c_int]),
        "nbgpu_split_qam": (C.c_int, [C.c_int, C.c_int, _fp]),
        "nbgpu_awgn_split_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, C.c_int, _fp, C.c_float, _fp]),
        "nbgpu_set_split_constellation": (C.c_int, [vp, C.c_int, _fp]),
        "nbgpu_channel_split": (C.c_int, [vp, _fp, C.c_float, C.c_int, _fp, _fp, _ip]),
        "nbgpu_decode_split": (C.c_int, [vp, _fp, C.c_float, C.c_int, _ip, _ip, _ip]),
        "nbgpu_upload_split": (C.c_int, [vp, _fp, C.c_float, C.c_int]),
        "nbgpu_sigma_punctured": (C.c_float, [vp, C.c_int, C.c_float]),
        "nbgpu_awgn_punctured_noise": (C.c_int, [vp, C.POINTER(Rng), _ip, C.c_int, C.c_int, _fp, C.c_float, C.c_int, _ip, _fp]),
        "nbgpu_set_puncturing": (C.c_int, [vp, C.c_int, _ip]),
        "nbgpu_create": (C.c_int, [C.POINTER(vp), vp, C.POINTER(Params), C.c_int, C.c_int]),
        "nbgpu_destroy": (None, [vp]),
        "nbgpu_last_error": (C.c_char_p, [vp]),
        "nbgpu_channel_awgn_bpsk": (C.c_int, [vp, _fp, C.c_float, C.c_int, _fp, _fp, _ip]),
        "nbgpu_decode_noisy": (C.c_int, [vp, _fp, C.c_float, C.c_int, _ip, _ip, _ip]),
        "nbgpu_decode_llr": (C.c_int, [vp, _fp, C.c_int, _ip, _ip, _ip]),
        "nbgpu_upload_noisy": (C.c_int, [vp, _fp, C.c_float, C.c_int]),
        "nbgpu_upload_llr": (C.c_int, [vp, _fp, C.c_int]),
        "nbgpu_run": (C.c_int, [vp]),
        "nbgpu_sync": (C.c_int, [vp]),
        "nbgpu_download": (C.c_int, [vp, _ip, _ip, _ip]),
        "nbgpu_last_kernel_ms": (C.c_int, [vp, _fp]),
        "nbgpu_launch_count": (C.c_long, [vp]),
        "nbgpu_timer_begin": (C.c_int, [vp]),
        "nbgpu_timer_end": (C.c_int, [vp, _fp]),
        "nbgpu_host_register": (C.c_int, [vp, C.c_size_t]),
        "nbgpu_host_unregister": (C.c_int, [vp]),
        "nbgpu_geometry": (C.c_int, [vp, _ip]),
        "nbgpu_slow_selects": (C.c_long, [vp]),
        "nbgpu_get_state": (C.c_int, [vp, C.c_int, _fp, _fp]),
        "nbgpu_set_soft_output": (C.c_int, [vp, C.c_int, C.c_int]),
        "nbgpu_download_soft_list": (C.c_int, [vp, _fp, _ip]),
        "nbgpu_download_soft_bits": (C.c_int, [vp, _fp]),
        "nbgpu_source_frames": (C.c_int, [vp, vp, C.POINTER(Rng), C.c_uint64, C.c_int, C.c_float]),
        "nbgpu_source_frames_apsk64": (C.c_int, [vp, vp, C.POINTER(Rng), C.c_uint64, C.c_int, C.c_float]),
        "nbgpu_source_frames_mapped": (C.c_int, [vp, vp, C.POINTER(Rng), C.c_uint64, C.c_int, C.c_float]),
        "nbgpu_source_frames_faded": (C.c_int, [vp, vp, C.POINTER(Rng), C.c_uint64, C.c_int, C.c_float, C.c_int]),
        "nbgpu_source_frames_split": (C.c_int, [vp, vp, C.POINTER(Rng), C.c_uint64, C.c_int, C.c_float]),
        "nbgpu_source_download": (C.c_int, [vp, _ip, _fp]),
        "nbgpu_source_results": (C.c_int, [vp, _ip, _ip, _ip]),
        "nbgpu_source_fixups": (C.c_long, [vp]),
        "nbgpu_source_set_margin": (C.c_int, [vp, C.c_double]),
        "nbgpu_check_node": (C.c_int, [vp, C.c_int, _fp, _ip, _fp, _ip, C.c_int]),
        "nbgpu_check_node_dense": (C.c_int, [vp, C.c_int, _fp, _fp, C.c_int]),
        "nbgpu_elementary_step": (C.c_int, [vp, _fp, _fp, _ip, _ip, _fp, _ip, C.c_int]),
        "nbgpu_select_nm": (C.c_int, [vp, _fp, _fp, _ip, C.c_int]),
        "nbgpu_decision_syndrome": (C.c_int, [vp, _fp, _ip, _ip, C.c_int]),
        "nbgpu_accumulate_stats": (C.c_int, [vp, _ip, _ip, _ip, _ip, C.c_int, _lp]),
        "nbgpu_accumulate_results": (C.c_int, [_ip, _ip, _ip, C.c_int, _lp]),
        "nbgpu_config_table": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, C.c_int]),
        "nbgpu_version": (C.c_char_p, []),
        "nbgpu_device_count": (C.c_int, []),
    }
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args
    _lib = L
    return L


def _i(a):
    return a.ctypes.data_as(_ip) if a is not None else None


def _f(a):
    return a.ctypes.data_as(_fp) if a is not None else None


def _check(rc, ctx=None):
    if rc != OK:
        msg = lib().nbgpu_last_error(ctx)
        raise NbgpuError(rc, msg.decode(errors="replace") if msg else "")


class Code:
    """nbgpu_code: alist matrix + GF(q) tables (reference: code_t + table_t, LoadCode/LoadTables)."""

    def __init__(self, path=None, dialect=ALIST_AUTO, arrays=None):
        L = lib()
        self.h = C.c_void_p()
        if arrays is not None:
            a = arrays
            keep = [np.ascontiguousarray(a[k], np.int32) if a.get(k) is not None else None
                    for k in ("row_deg", "col", "val", "bingf", "addgf", "mulgf", "divgf")]
            _check(L.nbgpu_code_from_arrays(C.byref(self.h), int(a["N"]), int(a["M"]), int(a["q"]),
                                            *[_i(x) for x in keep]))
        else:
            _check(L.nbgpu_code_load(C.byref(self.h), os.fsencode(path), dialect))
        info = np.zeros(10, np.int32)
        L.nbgpu_code_info(self.h, _i(info))
        (self.N, self.M, self.K, self.q, self.logq, self.E, self.dc_max, self.dc_min, self.dialect) = [int(x) for x in info[:9]]
        self.rate = float(L.nbgpu_code_rate(self.h))
        self.row_deg = np.zeros(self.M, np.int32)
        self.col = np.zeros(self.E, np.int32)
        self.val = np.zeros(self.E, np.int32)
        L.nbgpu_code_graph(self.h, _i(self.row_deg), _i(self.col), _i(self.val))
        self.row_ptr = np.concatenate([[0], np.cumsum(self.row_deg)]).astype(np.int64)
        self.rng = Rng()
        L.nbgpu_rng_reference_default(C.byref(self.rng))

    def tables(self):
        q, lg = self.q, self.logq
        b = np.zeros((q, lg), np.int32)
        a = np.zeros((q, q), np.int32); m = np.zeros((q, q), np.int32); d = np.zeros((q, q), np.int32)
        lib().nbgpu_code_tables(self.h, _i(b), _i(a), _i(m), _i(d))
        return b, a, m, d

    @property
    def info_bits(self):
        return self.K * self.logq

    # frame source (host side of the reference: tools.c:124-268, channel.c:51-62)
    def rng_default(self):
        lib().nbgpu_rng_reference_default(C.byref(self.rng))

    def rng_skip(self, n):
        lib().nbgpu_rng_skip(C.byref(self.rng), int(n))

    def drand48(self):
        return lib().nbgpu_rng_drand48(C.byref(self.rng))

    def prepare_encoder(self):
        _check(lib().nbgpu_code_prepare_encoder(self.h))

    def random_codeword(self):
        cw = np.zeros(self.N, np.int32)
        nbin = np.zeros((self.N, self.logq), np.int32)
        _check(lib().nbgpu_random_codeword(self.h, C.byref(self.rng), _i(cw), _i(nbin)))
        return cw, nbin

    def sigma(self, ebn, punctured=None):
        """channel.c:51; punctured = variable indices never sent: sigma at the rate (N - M) / (N - p) of the transmitted word."""
        if punctured is None:
            return float(lib().nbgpu_sigma(self.h, C.c_float(ebn)))
        p = _pattern(punctured).size
        s = float(lib().nbgpu_sigma_punctured(self.h, p, C.c_float(ebn)))
        if s != s:
            _check(EINVAL)
        return s

    def _noise(self, fn, nbin, fps, *args):
        out = np.zeros((self.N, fps), np.float32)
        nb = np.ascontiguousarray(nbin, np.int32) if nbin is not None else None
        _check(fn(self.h, C.byref(self.rng), _i(nb), *args, _f(out)))
        return out

    def _punctured_noise(self, punctured, nbin, fps, channel, arg, mod, ebn):
        """nbgpu_awgn_punctured_noise: the compact frame [N - p, fps] of the transmitted symbols"""
        v = _pattern(punctured)
        out = np.zeros((max(self.N - v.size, 0), fps), np.float32)
        nb = np.ascontiguousarray(nbin, np.int32) if nbin is not None else None
        _check(lib().nbgpu_awgn_punctured_noise(self.h, C.byref(self.rng), _i(nb), channel, int(arg), _f(mod), C.c_float(ebn),
                                                v.size, _i(v), _f(out)))
        return out

    def noise(self, nbin, ebn, punctured=None):
        """channel.c:52-62 for one frame; nbin None = all-zero codeword.  punctured = variable indices never sent: the frame is
        then [N - p, logq] (transmitted symbols in variable order) at sigma(ebn, punctured)."""
        if punctured is not None:
            return self._punctured_noise(punctured, nbin, self.logq, CHANNEL_BPSK, 0, None, ebn)
        return self._noise(lib().nbgpu_awgn_bpsk_noise, nbin, self.logq, C.c_float(ebn))

    def noise_apsk64(self, nbin, ebn, punctured=None):
        """channel.c:234-263 for one frame of a GF(64) code sent as 64-APSK symbols: noisy[N][2] ([N - p][2] punctured)."""
        if punctured is not None:
            if self.q != 64:
                raise ValueError("64-APSK maps one GF(64) symbol to one constellation point (q = %d)" % self.q)
            return self.noise_mapped(nbin, apsk64_table(), ebn, punctured)
        return self._noise(lib().nbgpu_awgn_apsk64_noise, nbin, 2, C.c_float(ebn))

    def noise_mapped(self, nbin, mod, ebn, punctured=None):
        """channel.c:234-263 on the constellation mod[q][2] (by binary image) for one frame: noisy[N][2], sigma_apsk64(ebn)
        ([N - p][2] punctured)."""
        m = np.ascontiguousarray(mod, np.float32).reshape(self.q, 2)
        if punctured is not None:
            return self._punctured_noise(punctured, nbin, 2, CHANNEL_MAPPED, 0, m, ebn)
        return self._noise(lib().nbgpu_awgn_mapped_noise, nbin, 2, _f(m), C.c_float(ebn))

    def noise_faded(self, nbin, mod, ebn, fading, punctured=None):
        """nbgpu_awgn_faded_noise: one frame of the faded mapped channel on mod[q][2], rx[N][4] = (y_I, y_Q, rho_I, rho_Q);
        fading = FADING_SYMBOL (5N draws) or FADING_COMPONENT (6N draws) ([N - p][4] punctured)."""
        m = np.ascontiguousarray(mod, np.float32).reshape(self.q, 2)
        if punctured is not None:
            return self._punctured_noise(punctured, nbin, 4, CHANNEL_FADED, int(fading), m, ebn)
        return self._noise(lib().nbgpu_awgn_faded_noise, nbin, 4, _f(m), C.c_float(ebn), int(fading))

    def noise_split(self, nbin, mod, points, ebn, punctured=None):
        """nbgpu_awgn_split_noise: one frame of the split channel, each symbol sent as `points` points of mod[M][2] (by
        sub-image), noisy[N][points][2]; 4*N*points draws, sigma_apsk64(ebn) ([N - p][points][2] punctured)."""
        m = _split_table(self.logq, mod, int(points))
        if punctured is not None:
            out = self._punctured_noise(punctured, nbin, 2 * points, CHANNEL_SPLIT, int(points), m, ebn)
            return out.reshape(-1, points, 2)
        out = self._noise(lib().nbgpu_awgn_split_noise, nbin, 2 * points, C.c_int(points), _f(m), C.c_float(ebn))
        return out.reshape(self.N, points, 2)

    def accumulate_stats(self, codeword_bits, decide, synd, iters, stats):
        cb = np.ascontiguousarray(codeword_bits, np.int32)
        d = np.ascontiguousarray(decide, np.int32)
        s = np.ascontiguousarray(synd, np.int32)
        it = np.ascontiguousarray(iters, np.int32)
        B = d.shape[0]
        assert stats.dtype == np.int64 and stats.shape == (6,)
        _check(lib().nbgpu_accumulate_stats(self.h, _i(cb), _i(d), _i(s), _i(it), B, stats.ctypes.data_as(_lp)))
        return stats

    def close(self):
        if self.h:
            lib().nbgpu_code_free(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Decoder:
    """nbgpu_ctx: the decode path NB_LDPC.c:266-474 for batches of frames on one B200.

    ecn_kind selects the check node: 0 = CheckPassLogEMS (L-Bubble), 1 = syndrome_ems, 2 = sum-product (belief propagation),
    4 = Min-Max; for 2 and 4, n_m, nb_oper and offset are validated but not used (include/nbldpc_b200.h)."""

    def __init__(self, code, n_m, nb_oper, nb_iter_max, offset, early_stop=True, ecn_kind=0, device=0,
                 max_batch=1, d1=0, d2=0, d3=0, cfg_trunc=0, n_cv=0, border=0, frames_per_cta=0, cns_per_step=0):
        self.code = code
        self.p = Params(n_m, nb_oper, nb_iter_max, offset, ecn_kind, int(early_stop), d1, d2, d3, cfg_trunc, n_cv,
                        border, frames_per_cta, cns_per_step)
        self.h = C.c_void_p()
        self.max_batch = max_batch
        _check(lib().nbgpu_create(C.byref(self.h), code.h, C.byref(self.p), device, max_batch))
        self.B = 0
        self.soft_k = 0
        self._source_shape = ()                               # shape of one symbol of the generated batch
        self._source_nt = code.N                              # symbols per frame of the generated batch
        self.split_points = 0                                 # points per symbol of the bound split table
        self.punctured = np.zeros(0, np.int32)                # the bound puncturing pattern (set_puncturing)
        self.nt = code.N                                      # transmitted symbols per frame: N - p

    def set_puncturing(self, vars):
        """nbgpu_set_puncturing: variables `vars` (distinct, in [0, N), any order; empty = none) are never sent.  Every frame
        this context takes or returns is then [B, N - p, ...], transmitted symbols in variable order; decisions, LLR rows and
        soft output still cover all N variables.  Drops the resident batch."""
        v = _pattern(vars)
        _check(lib().nbgpu_set_puncturing(self.h, v.size, _i(v) if v.size else None), self.h)
        self.punctured = v.copy()
        self.nt = self.code.N - v.size

    def _frames(self, frames, fps):
        """frames as [B, nt, fps] f32; while a pattern is bound anything but [B, N - p, ...] of fps floats per symbol is a
        ValueError (another layout would be read as other frames)"""
        x = np.ascontiguousarray(frames, np.float32)
        if self.nt != self.code.N and (x.ndim < 2 or x.shape[1] != self.nt or int(np.prod(x.shape[2:])) != fps):
            raise ValueError("frames must be [B, %d, ...] with %d floats per symbol (%d of %d variables punctured), not %s"
                             % (self.nt, fps, self.code.N - self.nt, self.code.N, x.shape))
        return x.reshape(-1, self.nt, fps)

    def _out(self, B):
        return (np.zeros((B, self.code.N), np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32))

    # the per-channel calls: frames [B, N, fps] f32 with fps floats per symbol; sigma=None for dense LLRs
    def _decode(self, fn, frames, fps, sigma=None):
        x = self._frames(frames, fps)
        B = x.shape[0]
        d, s, it = self._out(B)
        sig = () if sigma is None else (C.c_float(sigma),)
        _check(fn(self.h, _f(x), *sig, B, _i(d), _i(s), _i(it)), self.h)
        self.B = B
        return d, s, it

    def _channel(self, fn, frames, fps, sigma, want_sorted):
        x = self._frames(frames, fps)
        B = x.shape[0]
        llr = np.zeros((B, self.code.N, self.code.q), np.float32)
        il = np.zeros_like(llr) if want_sorted else None
        ig = np.zeros(llr.shape, np.int32) if want_sorted else None
        _check(fn(self.h, _f(x), C.c_float(sigma), B, _f(llr), _f(il), _i(ig)), self.h)
        return (llr, il, ig) if want_sorted else llr

    def _upload(self, fn, frames, fps, sigma=None):
        x = self._frames(frames, fps)
        sig = () if sigma is None else (C.c_float(sigma),)
        _check(fn(self.h, _f(x), *sig, x.shape[0]), self.h)
        self.B = x.shape[0]                                   # only once the batch is resident: it sizes every download

    def decode_noisy(self, noisy, sigma):
        return self._decode(lib().nbgpu_decode_noisy, noisy, self.code.logq, sigma)

    def decode_apsk64(self, noisy, sigma):
        """nbgpu_decode_apsk64: frames of a GF(64) code received as 64-APSK samples [B, N, 2]."""
        return self._decode(lib().nbgpu_decode_apsk64, noisy, 2, sigma)

    def channel_apsk64(self, noisy, sigma, want_sorted=False):
        return self._channel(lib().nbgpu_channel_awgn_apsk64, noisy, 2, sigma, want_sorted)

    def set_constellation(self, mod):
        """nbgpu_set_constellation: bind mod[q][2] (by binary image) to the *_mapped calls of this context."""
        m = np.ascontiguousarray(mod, np.float32).reshape(self.code.q, 2)
        _check(lib().nbgpu_set_constellation(self.h, _f(m)), self.h)

    def decode_mapped(self, noisy, sigma):
        """nbgpu_decode_mapped: frames received as samples [B, N, 2] of the bound constellation."""
        return self._decode(lib().nbgpu_decode_mapped, noisy, 2, sigma)

    def channel_mapped(self, noisy, sigma, want_sorted=False):
        return self._channel(lib().nbgpu_channel_awgn_mapped, noisy, 2, sigma, want_sorted)

    def upload_mapped(self, noisy, sigma):
        self._upload(lib().nbgpu_upload_mapped, noisy, 2, sigma)

    def decode_faded(self, rx, sigma):
        """nbgpu_decode_faded: frames received over the faded mapped channel, rx [B, N, 4] = (y_I, y_Q, rho_I, rho_Q), on the
        bound constellation."""
        return self._decode(lib().nbgpu_decode_faded, rx, 4, sigma)

    def channel_faded(self, rx, sigma, want_sorted=False):
        return self._channel(lib().nbgpu_channel_faded, rx, 4, sigma, want_sorted)

    def upload_faded(self, rx, sigma):
        self._upload(lib().nbgpu_upload_faded, rx, 4, sigma)

    def set_split_constellation(self, mod, points):
        """nbgpu_set_split_constellation: bind mod[M][2] (by sub-image), M = 2^(log2(q)/points), to the *_split calls."""
        m = _split_table(self.code.logq, mod, int(points))
        _check(lib().nbgpu_set_split_constellation(self.h, int(points), _f(m)), self.h)
        self.split_points = int(points)

    def _split_frames(self, noisy):
        """(frames, floats per symbol) of a split call: frames must be [B, N, P, 2] for the bound P.  Nothing bound: the library
        refuses the call (NBGPU_ESTATE)."""
        x = np.asarray(noisy)
        P = self.split_points
        if P and (x.ndim != 4 or x.shape[1:] != (self.nt, P, 2)):
            raise ValueError("split frames must be [B, %d, %d, 2] for the bound table, not %s" % (self.nt, P, x.shape))
        return x, 2 * max(P, 1)

    def decode_split(self, noisy, sigma):
        """nbgpu_decode_split: frames received as samples [B, N, P, 2] of the bound split table."""
        return self._decode(lib().nbgpu_decode_split, *self._split_frames(noisy), sigma)

    def channel_split(self, noisy, sigma, want_sorted=False):
        return self._channel(lib().nbgpu_channel_split, *self._split_frames(noisy), sigma, want_sorted)

    def upload_split(self, noisy, sigma):
        self._upload(lib().nbgpu_upload_split, *self._split_frames(noisy), sigma)

    def decode_noisy_into(self, noisy, sigma, out):
        """nbgpu_decode_noisy on caller-owned (e.g. pinned) buffers, no allocation: noisy [B,N,logq] f32, out = (decide, synd, iters)."""
        B = noisy.shape[0]
        _check(lib().nbgpu_decode_noisy(self.h, _f(noisy), C.c_float(sigma), B, _i(out[0]), _i(out[1]), _i(out[2])), self.h)
        self.B = B
        return out

    def decode_llr(self, llr):
        return self._decode(lib().nbgpu_decode_llr, llr, self.code.q)

    def upload_noisy(self, noisy, sigma):
        self._upload(lib().nbgpu_upload_noisy, noisy, self.code.logq, sigma)

    def upload_llr(self, llr):
        self._upload(lib().nbgpu_upload_llr, llr, self.code.q)

    def run(self):
        _check(lib().nbgpu_run(self.h), self.h)

    def sync(self):
        _check(lib().nbgpu_sync(self.h), self.h)

    def download(self, out=None):
        d, s, it = out if out is not None else self._out(self.B)
        _check(lib().nbgpu_download(self.h, _i(d), _i(s), _i(it)), self.h)
        return d, s, it

    def source_frames(self, frame0, B, ebn, origin=None):
        """nbgpu_source_frames: frames [frame0, frame0+B) of the reference's stream generated on the device and left resident
        (origin: drand48 state before frame 0 as an int, default = the reference's unseeded stream)."""
        self._source(lib().nbgpu_source_frames, (self.code.logq,), frame0, B, ebn, origin)

    def source_frames_apsk64(self, frame0, B, ebn, origin=None):
        """nbgpu_source_frames_apsk64: the same for a GF(64) code sent as 64-APSK symbols (ModelChannel_AWGN_64); the batch is
        resident as after an upload of noisy[B, N, 2] samples."""
        self._source(lib().nbgpu_source_frames_apsk64, (2,), frame0, B, ebn, origin)

    def source_frames_mapped(self, frame0, B, ebn, origin=None):
        """nbgpu_source_frames_mapped: the same for a code sent on the bound constellation; D = K log2(q) + 4N draws per frame."""
        self._source(lib().nbgpu_source_frames_mapped, (2,), frame0, B, ebn, origin)

    def source_frames_faded(self, frame0, B, ebn, fading, origin=None):
        """nbgpu_source_frames_faded: the same for the faded mapped channel on the bound constellation (fading = FADING_SYMBOL
        or FADING_COMPONENT); source_download then returns rx [B, N, 4]."""
        self._source(lib().nbgpu_source_frames_faded, (4,), frame0, B, ebn, origin, int(fading))

    def source_frames_split(self, frame0, B, ebn, origin=None):
        """nbgpu_source_frames_split: the same for the split channel on the bound split table; D = K log2(q) + 4NP draws per
        frame; source_download then returns noisy [B, N, P, 2]."""
        self._source(lib().nbgpu_source_frames_split, (self.split_points, 2), frame0, B, ebn, origin)

    def _source(self, fn, shape, frame0, B, ebn, origin, *extra):
        r = Rng()
        lib().nbgpu_rng_reference_default(C.byref(r))
        if origin is not None:
            r.x = origin
        _check(fn(self.h, self.code.h, C.byref(r), frame0, B, C.c_float(ebn), *extra), self.h)
        self.B = B
        self._source_shape = shape
        self._source_nt = self.nt

    def source_download(self, want_noisy=True):
        """(codeword [B, N], noisy) of the generated batch: noisy is [B, N, logq] for BPSK, [B, N, 2] for 64-APSK and mapped,
        [B, N, 4] for faded, [B, N, P, 2] for split; [B, N - p, ...] under a puncturing pattern"""
        cw = np.zeros((self.B, self.code.N), np.int32)
        noisy = np.zeros((self.B, self._source_nt) + self._source_shape, np.float32) if want_noisy else None
        _check(lib().nbgpu_source_download(self.h, _i(cw), _f(noisy)), self.h)
        return cw, noisy

    def source_results(self):
        """(bit_errors[B], synd[B], iters[B]) of the generated batch after run()"""
        e, s, it = (np.zeros(self.B, np.int32) for _ in range(3))
        _check(lib().nbgpu_source_results(self.h, _i(e), _i(s), _i(it)), self.h)
        return e, s, it

    def source_fixups(self):
        return int(lib().nbgpu_source_fixups(self.h))

    def source_set_margin(self, margin):
        _check(lib().nbgpu_source_set_margin(self.h, C.c_double(margin)), self.h)

    def last_kernel_ms(self):
        ms = C.c_float(0)
        _check(lib().nbgpu_last_kernel_ms(self.h, C.byref(ms)), self.h)
        return ms.value

    def launch_count(self):
        return int(lib().nbgpu_launch_count(self.h))

    def timer_begin(self):
        _check(lib().nbgpu_timer_begin(self.h), self.h)

    def timer_end(self):
        ms = C.c_float(0)
        _check(lib().nbgpu_timer_end(self.h, C.byref(ms)), self.h)
        return ms.value

    def geometry(self):
        g = np.zeros(8, np.int32)
        _check(lib().nbgpu_geometry(self.h, _i(g)), self.h)
        return dict(zip(("grid", "frames_per_cta", "cns_per_step", "steps_per_pass", "smem_bytes", "slots", "warps_per_cta",
                         "cns_per_warp"), [int(x) for x in g]))

    def slow_selects(self):
        return int(lib().nbgpu_slow_selects(self.h))

    def get_state(self, frame):
        app = np.zeros((self.code.N, self.code.q), np.float32)
        ctov = np.zeros((self.code.E, self.code.q), np.float32)
        _check(lib().nbgpu_get_state(self.h, frame, _f(app), _f(ctov)), self.h)
        return app, ctov

    def set_soft_output(self, kind, k=0):
        """nbgpu_set_soft_output: every later decode launch also returns SOFT_LIST (the k most likely symbols per variable)
        or SOFT_BITS (log2 q bit reliabilities per variable); SOFT_NONE turns it off."""
        rc = lib().nbgpu_set_soft_output(self.h, kind, k)
        if rc in (OK, ENOMEM):                                # ENOMEM leaves soft output off
            self.soft_k = k if rc == OK else 0
        _check(rc, self.h)

    def soft_list(self):
        """(llr [B,N,k] f32, sym [B,N,k] i32) of the last decode launch, armed with SOFT_LIST"""
        llr = np.zeros((self.B, self.code.N, self.soft_k), np.float32)
        sym = np.zeros(llr.shape, np.int32)
        _check(lib().nbgpu_download_soft_list(self.h, _f(llr), _i(sym)), self.h)
        return llr, sym

    def soft_bits(self):
        """bit reliabilities [B,N,logq] f32 of the last decode launch, armed with SOFT_BITS (> 0 favours bit 0)"""
        llr = np.zeros((self.B, self.code.N, self.code.logq), np.float32)
        _check(lib().nbgpu_download_soft_bits(self.h, _f(llr)), self.h)
        return llr

    def channel(self, noisy, sigma, want_sorted=False):
        return self._channel(lib().nbgpu_channel_awgn_bpsk, noisy, self.code.logq, sigma, want_sorted)

    def check_node(self, node, vllr, vgf):
        dc = int(self.code.row_deg[node])
        vllr = np.ascontiguousarray(vllr, np.float32).reshape(-1, dc, self.p.n_m)
        vgf = np.ascontiguousarray(vgf, np.int32).reshape(-1, dc, self.p.n_m)
        B = vllr.shape[0]
        cl = np.zeros((B, dc, self.code.q), np.float32)
        cg = np.zeros((B, dc, self.code.q), np.int32)
        _check(lib().nbgpu_check_node(self.h, node, _f(vllr), _i(vgf), _f(cl), _i(cg), B), self.h)
        return cl, cg

    def check_node_dense(self, node, mvc):
        """nbgpu_check_node_dense: the context's dense node, sum-product (ecn_kind=2) or Min-Max (ecn_kind=4), on B sets of dense
        rows, mvc [B, dc, q] -> CtoV [B, dc, q]"""
        dc = int(self.code.row_deg[node])
        mvc = np.ascontiguousarray(mvc, np.float32).reshape(-1, dc, self.code.q)
        ctov = np.zeros(mvc.shape, np.float32)
        _check(lib().nbgpu_check_node_dense(self.h, node, _f(mvc), _f(ctov), mvc.shape[0]), self.h)
        return ctov

    def elementary_step(self, in1, in2, idx1, idx2):
        n_m = self.p.n_m
        in1 = np.ascontiguousarray(in1, np.float32).reshape(-1, n_m)
        in2 = np.ascontiguousarray(in2, np.float32).reshape(-1, n_m)
        idx1 = np.ascontiguousarray(idx1, np.int32).reshape(-1, n_m)
        idx2 = np.ascontiguousarray(idx2, np.int32).reshape(-1, n_m)
        B = in1.shape[0]
        out = np.zeros((B, n_m), np.float32)
        io = np.zeros((B, n_m), np.int32)
        _check(lib().nbgpu_elementary_step(self.h, _f(in1), _f(in2), _i(idx1), _i(idx2), _f(out), _i(io), B), self.h)
        return out, io

    def select_nm(self, rows):
        rows = np.ascontiguousarray(rows, np.float32).reshape(-1, self.code.q)
        B = rows.shape[0]
        ol = np.zeros((B, self.p.n_m), np.float32)
        og = np.zeros((B, self.p.n_m), np.int32)
        _check(lib().nbgpu_select_nm(self.h, _f(rows), _f(ol), _i(og), B), self.h)
        return ol, og

    def decision_syndrome(self, app):
        app = np.ascontiguousarray(app, np.float32).reshape(-1, self.code.N, self.code.q)
        B = app.shape[0]
        d = np.zeros((B, self.code.N), np.int32)
        s = np.zeros(B, np.int32)
        _check(lib().nbgpu_decision_syndrome(self.h, _f(app), _i(d), _i(s), B), self.h)
        return d, s

    def close(self):
        if self.h:
            lib().nbgpu_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def config_table(dc, d1, d2, d3, trunc=0):
    """nbgpu_config_table: the [size, dc] configuration table of the syndrome-based check node."""
    size = lib().nbgpu_config_table(dc, d1, d2, d3, trunc, None, 0)
    if size < 0:
        _check(size)
    t = np.zeros((size, dc), np.int32)
    _check(min(lib().nbgpu_config_table(dc, d1, d2, d3, trunc, _i(t), size), 0))
    return t


def pin(arr):
    """Page-lock a numpy array in place (nbgpu_host_register); returns the array."""
    _check(lib().nbgpu_host_register(C.c_void_p(arr.ctypes.data), arr.nbytes))
    return arr


def unpin(arr):
    _check(lib().nbgpu_host_unregister(C.c_void_p(arr.ctypes.data)))


from . import multigpu  # noqa: E402,F401  (frame sharding over ranks; host logic only)


def device_count():
    return int(lib().nbgpu_device_count())


def version():
    return lib().nbgpu_version().decode()
