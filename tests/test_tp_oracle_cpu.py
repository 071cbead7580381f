"""CPU: tests/tp_oracle.c, the throughput-mode search for any number of leaves per round, against the oracle's one-leaf
searches it generalises, and its own invariants.

1. m = 1 without noise is plain sequential PUCT with an evaluated root: the counts of orc_az_search_hash, the forced
   search and targets of tests/forced_oracle.c, the symmetric search of tests/symmetry_oracle.c and the (n, w) and root
   value of tests/resign_oracle.c, bit for bit.
2. m > 1: the counts sum to the budget, the targets obey the forced-playout invariants, the queued leaves are the rows
   consumed, and feeding the hash evaluator's rows back reproduces the search.
3. The position set the GPU tests use exercises every path of the round: blocked stops, terminal backups, terminal-guard
   stops and terminal-only rounds.
"""
import numpy as np
import pytest

import forced_lib as FL
import oracle_lib as O
import resign_lib as R
import symmetry_lib as S
import tp_lib as TP

SIMS = 50


@pytest.fixture(scope="module")
def roots():
    sts = TP.positions(n_games=40, seed=4242, stride=1)
    live = [w for w in sts if len(O.oracle_probe(w)[1]) > 0]
    return np.stack(live)


def _sample(sts, n, seed=0):
    idx = np.random.default_rng(seed).choice(len(sts), size=min(n, len(sts)), replace=False)
    return sts[np.sort(idx)]


# ------------------------------------------------------------------ 1. m = 1 against the one-leaf searches
def test_m1_equals_orc_az_search_hash_and_resign_root_values(roots):
    for w in _sample(roots, 300):
        for sims in (7, SIMS):
            mv = TP.search(w, sims, 1)
            assert np.array_equal(mv.n, O.oracle_az_search(w, sims))
            n, ws = R.root_children(w, sims, 1, "az")
            assert np.array_equal(mv.n, n) and np.array_equal(mv.w.view(np.uint32), ws.view(np.uint32))
            assert mv.value.view(np.uint32) == R.root_value(n, ws).view(np.uint32)
            assert np.array_equal(mv.t, mv.n)
            assert mv.cov["blocked"] == 0 and mv.evals == len(mv.leaves)


def test_m1_forced_equals_the_forced_oracle(roots):
    pruned = 0
    for w in _sample(roots, 300, seed=1):
        mv = TP.search(w, SIMS, 1, forced_k=2.0)
        n, ws, t = FL.forced_root(w, SIMS, 2.0)
        assert np.array_equal(mv.n, n) and np.array_equal(mv.w.view(np.uint32), ws.view(np.uint32))
        assert np.array_equal(mv.t, t)
        assert np.array_equal(FL.prune(mv.n, mv.w, mv.p, 2.0), mv.t)
        pruned += int((t != n).any())
    assert pruned > 0


def test_m1_symmetric_equals_the_symmetry_oracle(roots):
    for i, w in enumerate(_sample(roots, 300, seed=2)):
        mv = TP.search(w, SIMS, 1, sym=(0, i, 0))
        assert np.array_equal(mv.n, S.az_search(w, i, SIMS))


# ------------------------------------------------------------------ 2. m > 1
def _check_targets(n, t):
    assert (t <= n).all()
    cs = int(np.argmax(n))
    assert t[cs] == n[cs]
    assert not ((t == 1) & (n != 1)).any()


@pytest.mark.parametrize("m", [2, 3, 4, 8, 16])
def test_batched_counts_sum_to_the_budget_and_targets_keep_the_invariants(roots, m):
    rng = np.random.default_rng(m)
    for w in _sample(roots, 120, seed=m):
        L = len(O.oracle_probe(w)[1])
        eta = np.zeros(81, np.float32)
        eta[O.oracle_probe(w)[1]] = rng.dirichlet(np.full(L, 0.3)).astype(np.float32)
        for sims in (1, m - 1, 7, SIMS):
            if sims < 1:
                continue
            mv = TP.search(w, sims, m, forced_k=2.0, eta=eta, eps=0.25)
            assert len(mv.n) == L and mv.n.sum() == sims
            _check_targets(mv.n, mv.t)
            assert mv.evals == len(mv.leaves) and mv.rounds[0] == 0
            assert (np.diff(mv.rounds) >= 0).all() and np.bincount(mv.rounds)[1:].max(initial=0) <= m
            # the rows of the hash evaluator, fed back in order, reproduce the search
            pol, val = TP.hash_rows(mv.leaves)
            rep = TP.search(w, sims, m, forced_k=2.0, eta=eta, eps=0.25, rows=(pol, val))
            assert np.array_equal(rep.n, mv.n) and np.array_equal(rep.t, mv.t)
            assert np.array_equal(rep.leaves, mv.leaves) and np.array_equal(rep.rounds, mv.rounds)
            with pytest.raises(RuntimeError, match="rows ran out"):
                TP.search(w, sims, m, forced_k=2.0, eta=eta, eps=0.25, rows=(pol[:-1], val[:-1]))


def test_noise_and_symmetry_change_the_search(roots):
    changed_noise = changed_sym = 0
    for i, w in enumerate(_sample(roots, 60, seed=5)):
        legal = O.oracle_probe(w)[1]
        eta = np.zeros(81, np.float32)
        eta[legal[0]] = 1.0
        base = TP.search(w, SIMS, 8)
        changed_noise += int(not np.array_equal(TP.search(w, SIMS, 8, eta=eta, eps=0.25).n, base.n))
        changed_sym += int(not np.array_equal(TP.search(w, SIMS, 8, sym=(3, i, 1)).n, base.n))
    assert changed_noise > 0 and changed_sym > 0


def test_finished_roots_give_an_empty_result():
    for g in range(6):
        w = O.playout_states(11, g)[0][-1]
        mv = TP.search(w, SIMS, 8)
        assert len(mv.n) == 0 and len(mv.leaves) == 0


# ------------------------------------------------------------------ 3. coverage of the GPU tests' position set
def test_every_path_of_the_round_is_exercised_on_the_gpu_position_set():
    total = dict.fromkeys(TP.COVERAGE, 0)
    for m, sims, sts in TP.search_cases():
        for w in sts:
            if len(O.oracle_probe(w)[1]) == 0:
                continue
            mv = TP.search(w, sims, m)
            for k in TP.COVERAGE:
                total[k] += mv.cov[k]
    assert all(v > 0 for v in total.values()), total
