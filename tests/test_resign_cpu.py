"""CPU: the host side of resignation (UTTT_SP_RESIGN) -- the check-game rule against the oracle's Philox, the calibration
helpers against a brute-force restatement, the argument checks that need no device, the self_play_cpp knob's error, and
the CPU search that the GPU test checks recorded root values against."""
import numpy as np
import pytest

import oracle_lib as O
import resign_lib as R


def _lib():
    from test_abi_cpu import _lib_or_skip
    return _lib_or_skip()


# ------------------------------------------------------------------ check games
@pytest.mark.parametrize("seed,game0", [(0, 0), (7, 1000), (123456789, (1 << 32) - 40)])
def test_check_games_follow_the_philox_rule(seed, game0):
    import engine
    n = 80
    u = np.zeros(n, np.float64)
    r = np.zeros(4, np.uint32)
    for i in range(n):
        g = game0 + i
        O.oracle().orc_philox4x32(seed, 4, g & 0xFFFFFFFF, g >> 32, 0, 0, r)
        u[i] = (int(r[0]) >> 8) / 16777216.0
    for frac in (0.0, 0.1, 0.5, 1.0):
        assert np.array_equal(engine.check_games(seed, game0, n, frac), u < frac), frac
    assert engine.check_games(seed, game0, n, 1.0).all() and not engine.check_games(seed, game0, n, 0.0).any()


# ------------------------------------------------------------------ calibration helpers vs brute force
class _Hist:
    def __init__(self, lens, final, values, resigned):
        self.lens = np.asarray(lens, np.int32)
        self.final = np.asarray(final, np.int8)
        self.values = np.asarray(values, np.float32)
        self.resigned = np.asarray(resigned, np.int8)


def _synthetic(rng, n):
    """values on a coarse grid (ties with the candidates), draws and wins for both colours, some resigned games"""
    lens = rng.integers(1, 82, n)
    final = rng.integers(0, 2, n)
    resigned = (rng.random(n) < 0.3) & (lens < 81)
    final[resigned] = 1
    values = rng.integers(-8, 9, (n, 81)).astype(np.float32) / 8
    return _Hist(lens, final, values, resigned)


def _bf_would(h, thr, g):
    last = int(h.lens[g]) - 1 + int(h.resigned[g])
    for p in range(1, last + 1):
        if h.values[g, p] < np.float32(thr):
            return p
    return -1


def _bf_calibration(h, thr, games):
    wr = fp = 0
    for g in games:
        p = _bf_would(h, thr, g)
        if p < 1:
            continue
        wr += 1
        mover_lost = h.final[g] == 1 and (int(h.lens[g]) - p) % 2 == 0
        fp += not mover_lost
    return wr, fp


def _bf_threshold(h, target, games):
    cand = sorted({float(h.values[g, p]) for g in games for p in range(int(h.lens[g]) + int(h.resigned[g]))})
    for c in reversed(cand):
        wr, fp = _bf_calibration(h, c, games)
        if wr > 0 and fp / wr <= target:
            return c
    return -1.0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_resign_helpers_match_brute_force(seed):
    import engine
    rng = np.random.default_rng(seed)
    h = _synthetic(rng, 60)
    games = np.nonzero(h.resigned == 0)[0]
    for thr in (-1.0, -0.75, -0.5, -0.125, 0.0, 0.5, 1.0):
        p = engine.would_resign_ply(h, thr)
        assert p.tolist() == [_bf_would(h, thr, g) for g in range(60)]
        cal = engine.resign_calibration(h, thr, games)
        wr, fp = _bf_calibration(h, thr, games)
        assert cal == {"games": len(games), "would_resign": wr, "false_positives": fp}
        mask = h.resigned == 0                               # a bool mask selects the same games
        assert engine.resign_calibration(h, thr, mask) == cal
    for target in (0.0, 0.05, 0.25, 0.5, 1.0):
        assert engine.resign_threshold(h, target, games) == _bf_threshold(h, target, games), target
        assert engine.resign_threshold(h, target, None) == _bf_threshold(h, target, range(60)), target


def test_resign_helpers_edge_cases():
    import engine
    v = np.zeros((4, 81), np.float32)
    v[:, 0] = -1.0                                           # ply 0 never resigns
    v[0, 1:4] = [-0.5, -0.9, -0.5]                           # game 0: 4 plies, final lost: the mover at ply 2 lost
    v[1, 1:3] = [-0.5, 0.25]                                 # game 1: a draw
    v[2, 1:5] = [0.5, -0.5, 0.5, -0.25]                      # game 2: resigned at ply 4 (row len recorded)
    v[3, 1] = 0.75                                           # game 3: 2 plies, the mover at ply 2 lost (row 2 unrecorded)
    v[3, 2] = -1.0
    h = _Hist([4, 3, 4, 2], [1, 0, 1, 1], v, [0, 0, 1, 0])
    assert engine.would_resign_ply(h, -0.5).tolist() == [2, -1, -1, -1]       # strict: -0.5 is not below -0.5
    assert engine.would_resign_ply(h, -0.4).tolist() == [1, 1, 2, -1]
    assert engine.would_resign_ply(h, -0.2).tolist() == [1, 1, 2, -1]
    assert engine.would_resign_ply(h, 0.0).tolist() == [1, 1, 2, -1]
    assert engine.would_resign_ply(h, 1.0).tolist() == [1, 1, 1, 1]
    # game 0 at ply 1: (4 - 1) odd -> the mover won (a false positive); at ply 2: lost.  Game 1: a draw, never lost.
    assert engine.resign_calibration(h, -0.6, [0, 1, 3]) == {"games": 3, "would_resign": 1, "false_positives": 0}
    assert engine.resign_calibration(h, -0.4, [0, 1, 3]) == {"games": 3, "would_resign": 2, "false_positives": 2}
    assert engine.resign_threshold(h, 0.0, [0, 1, 3]) == -0.5                  # "v < -0.5" resigns game 0 at ply 2 only
    assert engine.resign_threshold(h, 0.0, [1]) == -1.0                        # a drawn game alone: nothing qualifies
    assert engine.resign_threshold(h, 1.0, [1]) == 0.25                        # any rate is accepted: the largest value
    # game 3 (len 2, final 1): the mover at ply 2 lost, so the mover at ply 1 won; v < 1 resigns it there
    assert engine.resign_calibration(h, 1.0, [3]) == {"games": 1, "would_resign": 1, "false_positives": 1}


# ------------------------------------------------------------------ argument checks without a device
def test_set_resign_rejects_bad_values():
    lib = _lib()
    for thr, frac, word in ((float("nan"), 0.1, b"threshold"), (-1.01, 0.1, b"threshold"), (1.5, 0.1, b"threshold"),
                            (-0.9, -0.1, b"fraction"), (-0.9, 1.01, b"fraction"), (-0.9, float("nan"), b"fraction")):
        assert lib.uttt_set_resign(None, thr, frac) != 0 and word in lib.uttt_last_error(), (thr, frac)
    assert lib.uttt_set_resign(None, -1.0, 1.0) != 0 and b"null engine" in lib.uttt_last_error()


def test_self_play_knob_needs_the_correct_terminal_sign(monkeypatch):
    _lib()
    import engine
    import self_play_cpp as sp
    assert sp.SP_RESIGN_THRESHOLD is None and sp.SP_RESIGN_CHECK_FRACTION == 0.1 and sp.SP_RESIGN_TARGET_FP is None
    assert sp._resign_flags() == 0
    monkeypatch.setattr(sp, "SP_RESIGN_THRESHOLD", -0.9)
    with pytest.raises(ValueError, match="CORRECTED_TERMINAL_SIGN = True") as ex:
        sp._resign_flags()
    assert 'SP_SEARCH_MODE = "throughput"' in str(ex.value)
    with pytest.raises(ValueError):
        sp.play(None)                                        # refused before the engine or the model is touched
    monkeypatch.setattr(sp, "CORRECTED_TERMINAL_SIGN", True)
    assert sp._resign_flags() == engine.SP_RESIGN
    monkeypatch.setattr(sp, "CORRECTED_TERMINAL_SIGN", False)
    monkeypatch.setattr(sp, "SP_SEARCH_MODE", "throughput")
    assert sp._resign_flags() == engine.SP_RESIGN
    monkeypatch.setattr(sp, "SP_SEARCH_MODE", "compat")
    monkeypatch.setattr(sp, "SP_RESIGN_THRESHOLD", None)
    monkeypatch.setattr(sp, "SP_RESIGN_TARGET_FP", 0.05)     # calibrating only: the later threshold would be refused
    with pytest.raises(ValueError):
        sp._resign_flags()


# ------------------------------------------------------------------ the CPU search with root (n, w)
def test_root_search_matches_the_oracle_searches():
    """the new entry points give the oracle's own visit counts; the correct sign changes values only where a terminal
    position is reached"""
    differ = 0
    for game in range(3):
        for w in O.playout_states(11, game)[0][:-1:4]:
            sc, cn, _ = O.oracle_mcts(w, 1.0, 50, 8)
            n, ws = R.root_children(w, 50, 8, "exact")
            assert np.array_equal(n, cn)
            n1, w1 = R.root_children(w, 50, 8, "exact_correct")
            differ += not (np.array_equal(n1, n) and np.array_equal(w1, ws))
            n2, w2 = R.root_children(w, 50, 1, "az")
            assert np.array_equal(n2, O.oracle_az_search(w, 50))
            v = R.root_value(n, ws)
            i = int(np.argmax(n))
            assert v == np.float32(-ws[i]) / np.float32(n[i]) and -1.0 <= v <= 1.0
    assert differ > 0
