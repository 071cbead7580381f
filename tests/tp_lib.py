"""ctypes loader of tests/tp_oracle.c (TEST INFRASTRUCTURE ONLY): one move's search of the throughput mode for any number
of leaves per round, under the hash evaluator (optionally with the random symmetry) or fed recorded rows.  Built with
gcc together with tests/symmetry_oracle.c into a temporary directory on first use (the tree may be read-only)."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

import oracle_lib as O

SRC = os.path.join(O.ROOT, "tests", "tp_oracle.c")
SYM_SRC = os.path.join(O.ROOT, "tests", "symmetry_oracle.c")
COVERAGE = ("rounds", "blocked", "terminal_backups", "terminal_guard_stops", "terminal_only_rounds")
_lib = None


def lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="uttt_tp_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libtp_oracle.so")
        subprocess.check_call(["gcc", "-O3", "-fPIC", "-std=c11", "-shared", "-o", so, SRC, SYM_SRC, "-lm"])
        L = C.CDLL(so)
        fp = C.POINTER(C.c_float)
        L.orc_tp_search.argtypes = [C.POINTER(O.OrcState), C.c_int, C.c_int, C.c_float, fp, C.c_float, C.c_int,
                                    C.c_uint32, C.c_uint64, C.c_uint32, C.c_int, fp, fp,
                                    O.i32p, O.f32p, O.f32p, O.i32p, fp, C.c_int, O.u32p, O.i32p, C.POINTER(C.c_int), O.i32p]
        L.orc_tp_search.restype = C.c_int
        _lib = L
    return _lib


@dataclass
class Move:
    """one move's search: root children's n, w, p and policy targets t in legal order, the root value, the queued
    positions (the root first) with the round each was queued in, coverage counters (COVERAGE) and the number of evaluations"""
    n: np.ndarray
    w: np.ndarray
    p: np.ndarray
    t: np.ndarray
    value: np.float32
    leaves: np.ndarray
    rounds: np.ndarray
    cov: dict
    evals: int


def _fptr(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def search(w, sims, m, forced_k=0.0, eta=None, eps=0.0, sym=None, rows=None, leaf_cap=None):
    """the throughput-mode search of packed state w: `sims` simulations, `m` leaves per round, forced playouts with k =
    forced_k (0: off), root noise eta[81] (by action id) mixed with eps; the evaluator is the hash evaluator, under the
    symmetry keyed by sym = (seed, game, ply) if given, or rows = (policy (n,81), value (n,)) consumed in order"""
    eta_a = None if eta is None else np.ascontiguousarray(eta, np.float32).reshape(81)
    if rows is not None:
        pol = np.ascontiguousarray(rows[0], np.float32).reshape(-1, 81)
        val = np.ascontiguousarray(rows[1], np.float32).reshape(-1)
        n_rows = len(val)
    else:
        pol = val = None
        n_rows = -1
    seed, game, ply = sym if sym is not None else (0, 0, 0)
    cap = leaf_cap or (sims + 1)
    n = np.zeros(81, np.int32)
    ws = np.zeros(81, np.float32)
    p = np.zeros(81, np.float32)
    t = np.zeros(81, np.int32)
    v = C.c_float(0.0)
    leaves = np.zeros((cap, 8), np.uint32)
    rnd = np.zeros(cap, np.int32)
    nl = C.c_int(0)
    cov = np.zeros(6, np.int32)
    k = lib().orc_tp_search(C.byref(O.state_from_packed(w)), int(sims), int(m), float(forced_k), _fptr(eta_a), float(eps),
                            1 if sym is not None else 0, seed, game, ply, n_rows, _fptr(pol), _fptr(val),
                            n, ws, p, t, C.byref(v), cap, leaves, rnd, C.byref(nl), cov)
    if k < 0:
        raise RuntimeError({-1: "recorded rows ran out", -2: "leaf capacity too small",
                            -3: "virtual loss outstanding at the decision", -4: "bad arguments"}[k])
    return Move(n[:k].copy(), ws[:k].copy(), p[:k].copy(), t[:k].copy(), np.float32(v.value), leaves[:nl.value].copy(),
                rnd[:nl.value].copy(), dict(zip(COVERAGE, cov[:5].tolist())), int(cov[5]))


def positions(n_games=40, seed=4242, stride=1):
    """roots from every phase of the game: every `stride`-th state of Philox playouts, their last plies (terminal-heavy),
    one-legal-move roots and the finished final states"""
    out = []
    for g in range(n_games):
        sts = O.playout_states(seed, g)[0]
        out.append(sts[::stride])
        out.append(sts[-4:])
    sts = np.unique(np.concatenate(out), axis=0)
    return sts


def hash_rows(leaves):
    """the hash evaluator's rows (policy (n,81), value (n,)) of packed positions, in order"""
    pol = np.zeros((len(leaves), 81), np.float32)
    val = np.zeros(len(leaves), np.float32)
    for j, leaf in enumerate(leaves):
        v = C.c_float(0.0)
        O.oracle().orc_hash_eval(C.byref(O.state_from_packed(leaf)), pol[j], C.byref(v))
        val[j] = v.value
    return pol, val


def search_cases():
    """the (m, sims, roots) groups the GPU search tests compare bit for bit: m in {2, 3, 4, 8, 16}, sims in {1, m - 1, 7,
    50, 200} over roots from every phase of the game (with finished ones), and a few roots at 800 sims and m = 16"""
    sts = positions(n_games=24, seed=4242, stride=3)
    out = []
    for m in (2, 3, 4, 8, 16):
        for sims in sorted({1, m - 1, 7, 50, 200}):
            if sims >= 1:
                out.append((m, sims, sts))
    out.append((16, 800, sts[::25]))
    return out
