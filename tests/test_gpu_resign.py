"""GPU: resignation in self-play and matches (UTTT_SP_RESIGN, Engine.set_resign, History.values / .resigned).

1. Every recorded root value is, bit for bit, -w/n of the first most-visited root child of a CPU search of the recorded
   root (tests/resign_oracle.c): reference-exact search with the correct terminal sign at batch 8 and 1, and the
   throughput mode's sequential configuration -- with and without the flag.
2. Prefix property: a run with resignation equals the same run without it cut at would_resign_ply, game by game, for
   the hash and bf16 evaluators (bf16x3 on fewer games), every search mode that allows the flag, with and without random
   symmetries, in one and two lanes; check games are played out in full; resigned / final / match points follow the rule.
3. Boundaries: threshold -1 and check fraction 1 resign nothing.
4. The packed samples and the corrected labels of a resigning run.
5. Errors, and the self_play_cpp drop-in with a threshold and with calibration.
"""
import ctypes as C
import pickle

import numpy as np
import pytest

import oracle_lib as O
import resign_lib as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nets():
    import torch
    from dual_network import DualNetwork
    torch.manual_seed(0)
    a = DualNetwork().eval()
    torch.manual_seed(1)
    return a, DualNetwork().eval()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _root_at(h, g, ply):
    """the position searched at `ply` of game g: the recorded root, or for the ply a game resigned at (not recorded), the
    last recorded root with its move played"""
    if ply < h.lens[g]:
        return h.states[g, ply]
    s = O.state_from_packed(h.states[g, ply - 1])
    nx = O.OrcState()
    O.oracle().orc_next(C.byref(s), int(h.actions[g, ply - 1]), C.byref(nx))
    return O.packed_from_state(nx)


def _recorded_plies(h, g):
    return range(int(h.lens[g]) + int(h.resigned[g]))


# ------------------------------------------------------------------ 1. values against the CPU search
@pytest.mark.parametrize("resign", [False, True])
@pytest.mark.parametrize("mode,batch", [("exact_correct", 8), ("exact_correct", 1), ("az", 1)])
def test_values_equal_the_cpu_search(mode, batch, resign):
    import engine
    n, sims = 40, 50
    flags = engine.SP_THROUGHPUT if mode == "az" else engine.SP_CORRECT_TERMINAL_SIGN
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.set_root_noise(0.3, 0.0)                 # the throughput mode without noise is the CPU az search
        e.set_resign(-0.6, 0.25)
        h = e.selfplay(n, sims=sims, batch=batch, seed=3, evaluator=engine.EVAL_HASH,
                       flags=flags | (engine.SP_RESIGN if resign else 0))
    finally:
        e.close()
    assert bool(h.resigned.any()) == resign
    checked = 0
    for g in range(n):
        for t in _recorded_plies(h, g):
            cn, w = R.root_children(_root_at(h, g, t), sims, batch, mode)
            if t < h.lens[g]:
                assert np.array_equal(h.counts[g, t][O.oracle_probe(h.states[g, t])[1]], cn), (g, t)
            assert _bits(h.values[g, t]) == _bits(R.root_value(cn, w)), (g, t, h.values[g, t], R.root_value(cn, w))
            checked += 1
    assert checked == h.lens.sum() + h.resigned.sum() > 500


# ------------------------------------------------------------------ 2. prefix property
SEARCH = {"exact": ("CORRECT_TERMINAL_SIGN",), "throughput": ("THROUGHPUT",),
          "match": ("MATCH", "CORRECT_TERMINAL_SIGN"), "match_py": ("MATCH", "PYSEARCH", "CORRECT_TERMINAL_SIGN")}


def _flags(search, sym):
    import engine
    f = 0
    for name in SEARCH[search]:
        f |= getattr(engine, "SP_" + name)
    return f | (engine.SP_RANDOM_SYMMETRY if sym else 0)


def _threshold(h, n):
    """a threshold that some games cross: the lower quartile of the values of plies 1.. of the run"""
    rows = (np.arange(81)[None, :] < h.lens[:n, None]) & (np.arange(81)[None, :] >= 1)
    return float(np.quantile(h.values[:n][rows], 0.25).astype(np.float32))


def _check_prefix(engine, off, on, n, thr, frac, seed, game0, match):
    chk = engine.check_games(seed, game0, n, frac)
    p = engine.would_resign_ply(off, thr)[:n]
    res = (p >= 1) & ~chk
    assert res.any() and chk.any()
    assert np.array_equal(on.resigned[:n] != 0, res)
    assert np.array_equal(on.lens[:n], np.where(res, p, off.lens[:n]))
    assert np.array_equal(on.final[:n], np.where(res, 1, off.final[:n]))
    assert on.stats[0] == on.lens[:n].sum() < off.stats[0]
    for g in range(n):
        L = int(on.lens[g])
        assert np.array_equal(on.states[g, :L], off.states[g, :L]), g
        assert np.array_equal(on.counts[g, :L], off.counts[g, :L]), g
        assert np.array_equal(on.actions[g, :L], off.actions[g, :L]), g
        m = L + int(res[g])                              # the resigning ply's value is recorded too
        assert np.array_equal(_bits(on.values[g, :m]), _bits(off.values[g, :m])), g
    if match:
        pts_on, pts_off = engine.match_points(on, game0)[:n], engine.match_points(off, game0)[:n]
        resigner = (game0 + np.arange(n) + on.lens[:n]) & 1            # the slot to move at ply len
        assert np.array_equal(pts_on[res], np.where(resigner[res] == 0, 0.0, 1.0))
        assert np.array_equal(pts_on[~res], pts_off[~res])


def _prefix_case(monkeypatch, nets, evaluator, search, sym, lanes, n):
    import engine
    if lanes == 2:
        monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(n // 2))
    seed, game0, frac, sims = 21, 7, 0.25, 32
    flags = _flags(search, sym)
    ev = engine.evaluator_of(evaluator) if evaluator != "hash" else engine.EVAL_HASH
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        if evaluator != "hash":
            e.upload_model(nets[0])
            e.upload_model(nets[1], slot=1)
        off = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=ev, flags=flags, game0=game0)
        assert not off.resigned.any()
        thr = _threshold(off, n)
        e.set_resign(thr, frac)
        on = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=ev, flags=flags | engine.SP_RESIGN, game0=game0)
    finally:
        e.close()
    _check_prefix(engine, off, on, n, thr, frac, seed, game0, "match" in search)


@pytest.mark.parametrize("lanes", [1, 2])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("search", list(SEARCH))
@pytest.mark.parametrize("evaluator", ["hash", "bf16"])
def test_resigned_games_are_prefixes(monkeypatch, nets, evaluator, search, sym, lanes):
    _prefix_case(monkeypatch, nets, evaluator, search, sym, lanes, 64)


@pytest.mark.parametrize("search", ["exact", "throughput", "match"])
def test_resigned_games_are_prefixes_bf16x3(monkeypatch, nets, search):
    _prefix_case(monkeypatch, nets, "bf16x3", search, False, 1, 24)


# ------------------------------------------------------------------ 3. boundaries
def test_minus_one_and_check_fraction_one_resign_nothing():
    import engine
    n = 48
    f = engine.SP_CORRECT_TERMINAL_SIGN
    e = engine.Engine(n_slots=n, max_sims=32, max_batch=8, max_games=n)
    try:
        off = e.selfplay(n, sims=32, batch=8, seed=4, evaluator=engine.EVAL_HASH, flags=f)
        runs = []
        for thr, frac in ((-1.0, 0.0), (0.99, 1.0)):
            e.set_resign(thr, frac)
            runs.append(e.selfplay(n, sims=32, batch=8, seed=4, evaluator=engine.EVAL_HASH, flags=f | engine.SP_RESIGN))
    finally:
        e.close()
    rows = np.arange(81)[None, :] < off.lens[:, None]
    assert (off.values[rows] >= -1.0).all() and (off.values[rows] <= 1.0).all() and (off.values[rows] < -0.9).any()
    assert (engine.would_resign_ply(off, 0.99) >= 1).any()             # the second run would resign without its checks
    for h in runs:
        assert not h.resigned.any()
        assert np.array_equal(h.lens, off.lens) and np.array_equal(h.final, off.final)
        assert np.array_equal(h.states[rows], off.states[rows]) and np.array_equal(h.counts[rows], off.counts[rows])
        assert np.array_equal(h.actions[rows], off.actions[rows])
        assert np.array_equal(_bits(h.values[rows]), _bits(off.values[rows]))


# ------------------------------------------------------------------ 4. packed samples and labels
def test_pack_and_labels_of_a_resigning_run():
    import engine
    import self_play_cpp as sp
    n = 64
    e = engine.Engine(n_slots=n, max_sims=32, max_batch=8, max_games=n)
    try:
        e.set_resign(-0.3, 0.1)
        e.selfplay_device(n, sims=32, batch=8, seed=9, evaluator=engine.EVAL_HASH,
                          flags=engine.SP_THROUGHPUT | engine.SP_RESIGN)
        h = e.selfplay_fetch(n)
        buf, ns = e.selfplay_pack(n)
        packed = buf.cpu().numpy()
    finally:
        e.close()
    res = h.resigned != 0
    assert res.any() and (~res).any() and (h.final[res] == 1).all()
    st, cn, z = h.samples()
    assert ns == h.lens.sum() == len(z)
    pst, pcn, pz, ply = engine.samples_to_numpy(packed)
    assert np.array_equal(pst, st) and np.array_equal(pcn, cn) and np.array_equal(pz, z)
    assert np.array_equal(ply, np.concatenate([np.arange(L) for L in h.lens]))
    # corrected labels: the resigner (the mover at ply len) and every ply it moved get -1, its opponent +1
    zc = sp._corrected_labels(h)
    off = np.concatenate([[0], np.cumsum(h.lens)])
    for g in np.nonzero(res)[0]:
        L = int(h.lens[g])
        assert zc[off[g]:off[g + 1]].tolist() == [-1 if (L - t) % 2 == 0 else 1 for t in range(L)]


# ------------------------------------------------------------------ 5. errors and the drop-in
def test_resign_errors():
    import engine
    e = engine.Engine(n_slots=8, max_sims=50, max_batch=8, max_games=8)
    try:
        with pytest.raises(RuntimeError, match="CORRECT_TERMINAL_SIGN"):
            e.selfplay(8, evaluator=engine.EVAL_HASH, flags=engine.SP_RESIGN)
        with pytest.raises(RuntimeError, match="CORRECT_TERMINAL_SIGN"):
            e.selfplay(8, evaluator=engine.EVAL_HASH, flags=engine.SP_MATCH | engine.SP_PYSEARCH | engine.SP_RESIGN)
        roots = O.playout_states(1, 0)[0][:2]
        for f in (engine.SP_RESIGN | engine.SP_CORRECT_TERMINAL_SIGN, engine.SP_RESIGN | engine.SP_THROUGHPUT):
            with pytest.raises(RuntimeError, match="self-play mode"):
                e.mcts_search(roots, 10, 2, 1.0, engine.EVAL_HASH, flags=f)
        for thr, frac, word in ((float("nan"), 0.1, "threshold"), (1.01, 0.1, "threshold"), (-2.0, 0.1, "threshold"),
                                (-0.9, -0.01, "fraction"), (-0.9, 2.0, "fraction")):
            with pytest.raises(RuntimeError, match=word):
                e.set_resign(thr, frac)
        h = e.selfplay(8, evaluator=engine.EVAL_HASH, flags=engine.SP_RESIGN | engine.SP_CORRECT_TERMINAL_SIGN)
        h2 = e.selfplay(8, evaluator=engine.EVAL_HASH, flags=engine.SP_RESIGN | engine.SP_THROUGHPUT)
        assert (h.lens >= 1).all() and (h2.lens >= 1).all()
    finally:
        e.close()


def test_self_play_drop_in_resigns_and_calibrates(tmp_path, monkeypatch):
    import torch
    import engine
    import self_play_cpp as sp
    from dual_network import DualNetwork
    monkeypatch.chdir(tmp_path)
    (tmp_path / "model").mkdir()
    torch.manual_seed(0)
    torch.save(DualNetwork().state_dict(), "./model/best.pth")
    n = 48
    for k, v in dict(SP_GAME_COUNT=n, PV_EVALUATE_COUNT=16, SP_SEARCH_MODE="throughput", SP_NUMERICS="bf16", SP_SEED=5,
                     SP_PROGRESS=False, SP_RESIGN_THRESHOLD=None, SP_RESIGN_TARGET_FP=0.5,
                     SP_RESIGN_CHECK_FRACTION=0.25).items():
        monkeypatch.setattr(sp, k, v)
    runs = []
    real_run = sp._run

    def run(*a, **k):
        out = real_run(*a, **k)
        runs.append(out[1])
        return out
    monkeypatch.setattr(sp, "_run", run)
    # cycle 1: resignation off, calibrated on all games
    f1 = sp.self_play()
    h1 = runs[-1]
    with open(f1, "rb") as f:
        assert len(pickle.load(f)) == h1.lens[:n].sum() == sp.last_stats["plies"]
    t1 = engine.resign_threshold(h1, 0.5, np.ones(n, bool))
    assert sp.SP_RESIGN_THRESHOLD == t1 == sp.last_stats["calibrated_threshold"] > -1.0
    assert sp.last_stats["resigned"] == 0 and sp.last_stats["check_games"] == 0
    # cycle 2 (same seed): resigns with t1, calibrates on its check games; its games are cycle 1's cut at the rule
    f2 = sp.self_play()
    h2 = runs[-1]
    with open(f2, "rb") as f:
        assert len(pickle.load(f)) == h2.lens[:n].sum() == sp.last_stats["plies"]
    chk = engine.check_games(5, 0, n, 0.25)
    cal = engine.resign_calibration(h2, t1, chk)
    st = sp.last_stats
    assert st["resigned"] == h2.resigned.sum() > 0 and st["check_games"] == chk.sum()
    assert st["check_would_resign"] == cal["would_resign"] and st["check_false_positives"] == cal["false_positives"]
    assert sp.SP_RESIGN_THRESHOLD == st["calibrated_threshold"] == engine.resign_threshold(h2, 0.5, chk)
    p = engine.would_resign_ply(h1, t1)[:n]
    res = (p >= 1) & ~chk
    assert np.array_equal(h2.lens[:n], np.where(res, p, h1.lens[:n]))
    # a resigning cycle without calibration keeps its threshold; the packed sidecar loads with one sample per ply
    monkeypatch.setattr(sp, "SP_RESIGN_TARGET_FP", None)
    monkeypatch.setattr(sp, "SP_WRITE_PACKED", True)
    thr = sp.SP_RESIGN_THRESHOLD
    f3 = sp.self_play()
    assert sp.SP_RESIGN_THRESHOLD == thr and "calibrated_threshold" not in sp.last_stats
    assert sp.last_stats["resigned"] == runs[-1].resigned.sum()
    xs, _, _ = sp.load_packed_history(f3.replace(".history", ".packed.npz"))
    assert len(xs) == runs[-1].lens[:n].sum()
