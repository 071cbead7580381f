"""ctypes loader of tests/forced_oracle.c (TEST INFRASTRUCTURE ONLY): UTTT_SP_FORCED_PLAYOUTS' pruning and the oracle's
throughput-mode search with forced root playouts, under the hash evaluator.  Built with gcc into a temporary directory
on first use (the tree may be read-only)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

SRC = os.path.join(O.ROOT, "tests", "forced_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="uttt_forced_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libforced_oracle.so")
        subprocess.check_call(["gcc", "-O3", "-fPIC", "-std=c11", "-shared", "-o", so, SRC, "-lm"])
        L = C.CDLL(so)
        L.orc_prune_targets.argtypes = [C.c_int, O.i32p, O.f32p, O.f32p, C.c_float, O.i32p]
        L.orc_prune_targets.restype = None
        L.orc_az_search_forced_root_hash.argtypes = [C.POINTER(O.OrcState), C.c_int, C.c_float, O.i32p, O.f32p, O.i32p]
        L.orc_az_search_forced_root_hash.restype = C.c_int
        _lib = L
    return _lib


def prune(n, w, p, k):
    """the policy targets t of root children with visit counts n, summed values w and priors p (legal order)"""
    n = np.ascontiguousarray(n, np.int32)
    t = np.zeros(len(n), np.int32)
    lib().orc_prune_targets(len(n), n, np.ascontiguousarray(w, np.float32), np.ascontiguousarray(p, np.float32), k, t)
    return t


def forced_root(w, sims, k):
    """(n, w, t) of the root children in legal order after the forced search of packed state w"""
    n = np.zeros(81, np.int32)
    ws = np.zeros(81, np.float32)
    t = np.zeros(81, np.int32)
    m = lib().orc_az_search_forced_root_hash(C.byref(O.state_from_packed(w)), sims, k, n, ws, t)
    return n[:m].copy(), ws[:m].copy(), t[:m].copy()
