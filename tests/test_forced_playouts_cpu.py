"""CPU: forced playouts and policy target pruning (UTTT_SP_FORCED_PLAYOUTS) without a device -- the C pruning of
tests/forced_oracle.c against a brute-force numpy float32 restatement of the header's rule, the oracle's forced search
against the plain one when nothing can be forced, History.targets() on hand-built histories, and the argument checks."""
import numpy as np
import pytest

import oracle_lib as O

F32 = np.float32


def _lib():
    from test_abi_cpu import _lib_or_skip
    return _lib_or_skip()


def prune_brute(n, w, p, k):
    """the header's pruning rule, literally: for every child the largest r in [0, R] whose steps 1..r ALL score below S*
    (no monotonicity assumed), every operation one float32 rounding"""
    n = np.asarray(n, np.int64)
    w = np.asarray(w, F32)
    p = np.asarray(p, F32)
    k = F32(k)
    t = n.copy()
    if len(n) == 0 or n.max() == 0:
        return t
    N = int(n.sum())
    sq = np.sqrt(F32(N))
    cs = int(np.argmax(n))                                  # first maximum
    best = F32(F32(-w[cs]) / F32(n[cs])) + F32(F32(p[cs] * sq) / F32(1 + n[cs]))
    for i in range(len(n)):
        if i == cs or n[i] == 0:
            continue
        q = F32(-w[i]) / F32(n[i])
        F = np.sqrt(F32(F32(k * p[i]) * F32(N)))
        R = min(int(n[i]), int(F))
        r = 0
        for cand in range(R + 1):
            if all(F32(q + F32(F32(p[i] * sq) / F32(1 + n[i] - j))) < best for j in range(1, cand + 1)):
                r = cand
        t[i] = 0 if (r >= 1 and n[i] - r == 1) else n[i] - r
    return t


def _check(n, w, p, k):
    import forced_lib as FL
    got = FL.prune(n, w, p, k)
    want = prune_brute(n, w, p, k)
    assert np.array_equal(got, want), (n, w, p, k, got, want)
    return got


# ------------------------------------------------------------------ pruning on hand-built roots
def test_most_visited_child_ties_keep_the_first_and_prune_the_other():
    # children 0 and 2 tie at 20 visits: child 0 is c* and keeps them, child 2 is an ordinary child
    n, w, p = [20, 3, 20], [-10.0, 1.0, -12.0], [0.3, 0.4, 0.3]
    t = _check(n, w, p, 2.0)
    assert t[0] == 20 and t[1] <= 3


def test_single_playout_children_and_the_one_playout_rule():
    # a child with one bad playout: F = sqrt(2 * 0.2 * 41) > 1, so r = 1 and it goes to 0 (not left at n - r)
    n, w, p = [40, 1], [-20.0, 1.0], [0.8, 0.2]
    assert list(_check(n, w, p, 2.0)) == [40, 0]
    # two bad playouts with R = 1: r = 1 leaves a single playout, which is pruned outright
    t = _check([40, 2], [-20.0, 2.0], [0.97, 0.03], 2.0)
    assert int(np.sqrt(F32(2 * F32(0.03)) * F32(42))) == 1 and list(t) == [40, 0]


def test_f_below_one_prunes_nothing():
    n, w, p = [30, 5, 2, 1], [-10.0, 3.0, 2.0, 1.0], [0.5, 0.3, 0.15, 0.05]
    assert list(_check(n, w, p, 1e-4)) == n


def test_r_capped_by_floor_f():
    # a terrible child (q = -1): every removal keeps it below S*, so r = floor(F) < n
    n, w, p = [60, 12], [-30.0, 12.0], [0.5, 0.5]
    F = np.sqrt(F32(F32(F32(2.0) * F32(0.5)) * F32(72)))
    t = _check(n, w, p, 2.0)
    assert int(F) < 12 and t[1] == 12 - int(F)


def test_r_capped_by_the_best_score():
    # a child nearly as good as c*: removing playouts raises its exploration term above S* after a few steps
    n, w, p = [30, 20], [-15.0, -5.0], [0.3, 0.7]
    t = _check(n, w, p, 2.0)
    F = int(np.sqrt(F32(F32(F32(2.0) * F32(0.7)) * F32(50))))
    assert 0 < 20 - t[1] < F


def test_single_legal_move_and_unvisited_children():
    assert list(_check([50], [-3.0], [1.0], 2.0)) == [50]
    assert list(_check([0, 0, 0], [0.0, 0.0, 0.0], [0.2, 0.3, 0.5], 2.0)) == [0, 0, 0]
    assert list(_check([10, 0, 3], [-5.0, 0.0, 2.0], [0.4, 0.5, 0.1], 2.0))[1] == 0


@pytest.mark.parametrize("seed", range(6))
def test_random_roots(seed):
    rng = np.random.default_rng(seed)
    pruned = 0
    for _ in range(300):
        L = int(rng.integers(1, 82))
        p = rng.dirichlet(np.full(L, 0.3)).astype(F32)
        n = rng.multinomial(int(rng.integers(1, 400)), rng.dirichlet(np.ones(L))).astype(np.int32)
        w = (rng.uniform(-1, 1, L) * n).astype(F32)
        k = float(rng.choice([0.5, 1.0, 2.0, 4.0, 100.0]))
        t = _check(n, w, p, k)
        assert (t <= n).all() and t[int(np.argmax(n))] == n.max() and not ((t == 1) & (n != 1)).any()
        pruned += int((t != n).any())
    assert pruned > 50


# ------------------------------------------------------------------ the forced search
def _roots():
    st, _ = O.playout_states(4, 2)
    return [st[i] for i in (0, 1, 3, 7, 12, 20) if i < len(st) - 1]


def test_forced_search_with_tiny_k_is_the_plain_search():
    import forced_lib as FL
    import resign_lib as R
    for w in _roots():
        for sims in (8, 50):
            n, ws, t = FL.forced_root(w, sims, 1e-6)
            n0, w0 = R.root_children(w, sims, 1, "az")
            assert np.array_equal(n, n0) and np.array_equal(ws.view(np.uint32), w0.view(np.uint32))
            assert np.array_equal(t, n)


def test_forced_search_forces_and_prunes():
    import forced_lib as FL
    import resign_lib as R
    changed = pruned = 0
    for w in _roots():
        n, ws, t = FL.forced_root(w, 50, 2.0)
        n0, _ = R.root_children(w, 50, 1, "az")
        assert n.sum() == 50 and (t <= n).all() and t[np.argmax(n)] == n.max()
        changed += not np.array_equal(n, n0)
        pruned += int((n - t).sum())
    assert changed > 0 and pruned > 0


# ------------------------------------------------------------------ host side
def test_history_targets_are_the_counts_unless_a_target_was_fetched():
    import engine
    import parallel
    h = engine.History(2, pinned=False)
    h.lens[:] = [3, 2]
    h.counts[:, :3, :5] = 4
    assert h.target is None and h.targets() is h.counts
    nb = h.nbytes
    raw0 = parallel.pack_history_host(h, 2).numpy().reshape(-1, engine.SAMPLE_BYTES)
    h.target = h.counts.copy()
    h.target[:, :, 0] = 0
    assert h.targets() is h.target and h.nbytes == nb + h.target.nbytes
    st, cn, z = h.samples()
    assert np.array_equal(cn, h.target[h.sample_mask()])
    raw = parallel.pack_history_host(h, 2).numpy().reshape(-1, engine.SAMPLE_BYTES)
    assert np.array_equal(raw[:, 32:194].copy().view(np.uint16), cn)
    assert np.array_equal(np.delete(raw, np.s_[32:194], 1), np.delete(raw0, np.s_[32:194], 1))


def test_set_forced_playouts_rejects_bad_values():
    lib = _lib()
    for k in (0.0, -1.0, 100.5, float("nan"), float("inf")):
        assert lib.uttt_set_forced_playouts(None, k) != 0 and b"forced playouts" in lib.uttt_last_error(), k
    assert lib.uttt_set_forced_playouts(None, 2.0) != 0 and b"null engine" in lib.uttt_last_error()
    assert lib.uttt_selfplay_fetch_target(None, 1, None) != 0


def test_self_play_knob_is_validated_before_any_gpu_work(monkeypatch):
    _lib()
    import engine
    import self_play_cpp as sp
    assert sp.SP_FORCED_PLAYOUTS is None and sp._forced_playouts_flags() == 0
    monkeypatch.setattr(sp, "SP_SEARCH_MODE", "throughput")
    for bad in (0, -1.0, 100.5, float("nan"), float("inf"), True, "2"):
        monkeypatch.setattr(sp, "SP_FORCED_PLAYOUTS", bad)
        with pytest.raises(ValueError, match="SP_FORCED_PLAYOUTS"):
            sp._forced_playouts_flags()
        with pytest.raises(ValueError):
            sp.play(None)                                    # refused before the engine or the model is touched
    for ok in (1e-6, 2, 2.0, 100):
        monkeypatch.setattr(sp, "SP_FORCED_PLAYOUTS", ok)
        assert sp._forced_playouts_flags() == engine.SP_FORCED_PLAYOUTS
    monkeypatch.setattr(sp, "SP_SEARCH_MODE", "compat")
    with pytest.raises(ValueError, match="throughput"):
        sp._forced_playouts_flags()
    with pytest.raises(ValueError):
        sp.play(None)
