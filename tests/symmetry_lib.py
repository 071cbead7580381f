"""ctypes loader of tests/symmetry_oracle.c (TEST INFRASTRUCTURE ONLY): the board symmetries restated on the oracle's
[9][9] arrays and the hash-evaluator searches with UTTT_SP_RANDOM_SYMMETRY.  Built with gcc together with the unchanged
oracle/uttt_oracle.c into a temporary directory on first use (the tree may be read-only)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle_lib as O

SRC = os.path.join(O.ROOT, "tests", "symmetry_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="uttt_sym_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libsymmetry_oracle.so")
        subprocess.check_call(["gcc", "-O3", "-fPIC", "-std=c11", "-shared", "-o", so, SRC,
                               os.path.join(O.ORACLE_DIR, "uttt_oracle.c"), "-lm"])
        L = C.CDLL(so)
        SP = C.POINTER(O.OrcState)
        L.orc_symmetry.argtypes = [SP, C.c_int, SP]
        L.orc_symmetry_action.argtypes = [C.c_int, C.c_int]
        L.orc_symmetry_action.restype = C.c_int
        L.orc_symmetry_draw.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32]
        L.orc_symmetry_draw.restype = C.c_int
        L.orc_pv_mcts_scores_hash_sym.argtypes = [SP, C.c_uint32, C.c_uint64, C.c_uint32, C.c_float, C.c_int, C.c_int,
                                                  O.f32p, O.i32p]
        L.orc_pv_mcts_scores_hash_sym.restype = C.c_int
        L.orc_py_mcts_counts_hash_sym.argtypes = [SP, C.c_uint32, C.c_uint64, C.c_uint32, C.c_int, C.c_int, O.i32p]
        L.orc_py_mcts_counts_hash_sym.restype = C.c_int
        L.orc_az_search_hash_sym.argtypes = [SP, C.c_uint64, C.c_int, O.i32p]
        L.orc_az_search_hash_sym.restype = C.c_int
        L.orc_selfplay_hash_sym.argtypes = [C.c_uint32, C.c_uint64, C.c_int, C.c_int, O.u32p, O.u16p, O.u8p]
        L.orc_selfplay_hash_sym.restype = C.c_int
        _lib = L
    return _lib


def symmetry(w, g):
    """packed state -> packed image under symmetry g (computed on the [9][9] arrays)"""
    out = O.OrcState()
    lib().orc_symmetry(C.byref(O.state_from_packed(w)), int(g), C.byref(out))
    return O.packed_from_state(out)


def action_map(g):
    """sigma_g as an array: [a] = the action at the image of action a's cell"""
    return np.array([lib().orc_symmetry_action(a, int(g)) for a in range(81)], np.int64)


def draw(seed, game, ply, j):
    return lib().orc_symmetry_draw(seed, game, ply, j)


def cpp_search(w, game, temperature, sims, batch, seed=0, ply=0):
    """C++-semantics search -> (scores, visit counts) in legal order"""
    sc = np.zeros(81, np.float32)
    cn = np.zeros(81, np.int32)
    n = lib().orc_pv_mcts_scores_hash_sym(C.byref(O.state_from_packed(w)), seed, game, ply, temperature, sims, batch, sc, cn)
    return sc[:n].copy(), cn[:n].copy()


def py_search(w, game, sims, batch):
    cn = np.zeros(81, np.int32)
    n = lib().orc_py_mcts_counts_hash_sym(C.byref(O.state_from_packed(w)), 0, game, 0, sims, batch, cn)
    return cn[:n].copy()


def az_search(w, game, sims):
    cn = np.zeros(81, np.int32)
    n = lib().orc_az_search_hash_sym(C.byref(O.state_from_packed(w)), game, sims, cn)
    return cn[:n].copy()


def selfplay(seed, game, sims, batch):
    """-> (plies, states (81,8), counts (81,81), actions (81,))"""
    st = np.zeros((81, 8), np.uint32)
    cn = np.zeros((81, 81), np.uint16)
    ac = np.zeros(81, np.uint8)
    n = lib().orc_selfplay_hash_sym(seed, game, sims, batch, st, cn, ac)
    return n, st, cn, ac
