"""ctypes loader of tests/resign_oracle.c (TEST INFRASTRUCTURE ONLY): the oracle's hash-evaluator searches returning the
root children's (n, w), and the root value UTTT_SP_RESIGN records, computed from them on the host.  Built with gcc into
a temporary directory on first use (the tree may be read-only)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

SRC = os.path.join(O.ROOT, "tests", "resign_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="uttt_resign_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libresign_oracle.so")
        subprocess.check_call(["gcc", "-O3", "-fPIC", "-std=c11", "-shared", "-o", so, SRC, "-lm"])
        L = C.CDLL(so)
        SP = C.POINTER(O.OrcState)
        L.orc_pv_mcts_root_hash.argtypes = [SP, C.c_int, C.c_int, C.c_int, O.i32p, O.f32p]
        L.orc_pv_mcts_root_hash.restype = C.c_int
        L.orc_az_search_root_hash.argtypes = [SP, C.c_int, O.i32p, O.f32p]
        L.orc_az_search_root_hash.restype = C.c_int
        _lib = L
    return _lib


def root_children(w, sims, batch, mode):
    """(n, w) of the root children in legal order after a search of packed state w under the hash evaluator: mode
    "exact" (reference-exact, reference terminal sign), "exact_correct" (the same with the correct sign) or "az" (the
    throughput mode with one leaf per round and no root noise; batch is ignored)"""
    n = np.zeros(81, np.int32)
    ws = np.zeros(81, np.float32)
    s = C.byref(O.state_from_packed(w))
    if mode == "az":
        m = lib().orc_az_search_root_hash(s, sims, n, ws)
    else:
        m = lib().orc_pv_mcts_root_hash(s, sims, batch, 1 if mode == "exact_correct" else 0, n, ws)
    return n[:m].copy(), ws[:m].copy()


def root_value(n, w):
    """-w/n (fp32) of the first root child with the most visits; 0 if it is unvisited"""
    i = int(np.argmax(n))
    return np.float32(-w[i] / np.float32(n[i])) if n[i] > 0 else np.float32(0.0)
