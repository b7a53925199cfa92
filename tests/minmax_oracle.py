"""ctypes bindings for the Min-Max oracle (tests/minmax_oracle.c), a checker of its own beside liboracle.so: it is compiled on
first use into a temporary directory (keyed by the source's hash, so a read-only tree is fine) and works on the code of an
``oracle_lib.Oracle``."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib as ol

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "minmax_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read() + open(os.path.join(ol.ORACLE_DIR, "nbldpc_oracle.h"), "rb").read()
        d = os.path.join(tempfile.gettempdir(), "nbldpc_minmax_oracle_%s" % hashlib.sha256(src).hexdigest()[:16])
        path = os.path.join(d, "liboracle_minmax.so")
        if not os.path.exists(path):
            os.makedirs(d, exist_ok=True)
            tmp = path + ".%d" % os.getpid()
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-Wall", "-ffp-contract=off", "-I", ol.ORACLE_DIR, "-o", tmp, SRC],
                           check=True)
            os.replace(tmp, path)
        L = C.CDLL(path)
        L.nbo_check_node_minmax.argtypes = [C.POINTER(ol.NboCode), C.c_int, ol.c_float_p, ol.c_float_p]
        L.nbo_minmax_decode_frame.argtypes = [C.POINTER(ol.NboCode), C.POINTER(ol.NboParams), ol.c_float_p, ol.c_int_p,
                                              C.POINTER(C.c_int), C.POINTER(C.c_int), ol.c_int_p, ol.c_int_p, ol.c_float_p,
                                              ol.c_float_p]
        _lib = L
    return _lib


def minmax_check_node(o, node, mvc):
    """steps 2-5 of the Min-Max node on check node `node` of the oracle's code: mvc [dc, GF] -> CtoV [dc, GF], symbol order"""
    dc = int(o.row_deg[node])
    mvc = np.ascontiguousarray(mvc, np.float32).reshape(dc, o.GF)
    cl = np.zeros((dc, o.GF), np.float32)
    lib().nbo_check_node_minmax(o.h, node, ol._fp(mvc), ol._fp(cl))
    return cl


def decode_frame(o, llr, nb_iter_max, force=False, want_state=False):
    """one frame of the oracle's decode loop with the Min-Max node, as Oracle.decode_frame returns it:
    dict(decide, synd, iters, passes, decide_trace, synd_trace[, app, ctov])"""
    llr = np.ascontiguousarray(llr, np.float32)
    p = ol.NboParams()
    p.nb_iter_max, p.force_passes, p.ecn = nb_iter_max, int(force), 4
    P = max(nb_iter_max - 1, 1)
    decide = np.zeros(o.N, np.int32)
    dtr = np.zeros((P, o.N), np.int32)
    strc = np.full(P, -1, np.int32)
    synd, iters = C.c_int(0), C.c_int(0)
    app = np.zeros((o.N, o.GF), np.float32) if want_state else None
    ctov = np.zeros((o.E, o.GF), np.float32) if want_state else None
    passes = lib().nbo_minmax_decode_frame(o.h, C.byref(p), ol._fp(llr), ol._ip(decide), C.byref(synd), C.byref(iters), ol._ip(dtr),
                                           ol._ip(strc), ol._fp(app) if want_state else None, ol._fp(ctov) if want_state else None)
    r = dict(decide=decide, synd=synd.value, iters=iters.value, passes=passes, decide_trace=dtr[:passes], synd_trace=strc[:passes])
    if want_state:
        r["app"] = app
        r["ctov"] = ctov
    return r
