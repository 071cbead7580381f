"""CPU: the host side of playout cap randomization (UTTT_SP_PLAYOUT_CAP) -- the full-search rule against a brute-force
Philox and the oracle's, which plies are samples (History.sample_mask, samples(), parallel.pack_history_host) on
hand-built histories, the argument checks that need no device, and the self_play_cpp knobs' validation."""
import numpy as np
import pytest

import oracle_lib as O


def _lib():
    from test_abi_cpu import _lib_or_skip
    return _lib_or_skip()


# ------------------------------------------------------------------ the full-search rule
def _philox_x(k0, k1, c):
    """word x of Philox4x32-10 on Python ints, one counter at a time"""
    c = list(c)
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k1, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + 0x9E3779B9) & 0xFFFFFFFF, (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c[0]


@pytest.mark.parametrize("seed,game0", [(0, 0), (7, 1000), (123456789, (1 << 32) - 3)])
def test_full_moves_follow_the_philox_rule(seed, game0):
    import engine
    n = 6
    u_bf = np.zeros((n, 81), np.float32)
    u_orc = np.zeros((n, 81), np.float32)
    r = np.zeros(4, np.uint32)
    for i in range(n):
        g = game0 + i
        for p in range(81):
            u_bf[i, p] = np.float32(_philox_x(seed, 5, (g & 0xFFFFFFFF, g >> 32, p, 0)) >> 8) * np.float32(2.0 ** -24)
            O.oracle().orc_philox4x32(seed, 5, g & 0xFFFFFFFF, g >> 32, p, 0, r)
            u_orc[i, p] = np.float32(int(r[0]) >> 8) * np.float32(2.0 ** -24)
    assert np.array_equal(u_bf, u_orc)
    for frac in (0.0, 0.1, 0.25, 0.5, 1.0):
        got = engine.full_moves(seed, game0, n, frac)
        assert got.shape == (n, 81) and got.dtype == bool
        assert np.array_equal(got, u_bf < np.float32(frac)), frac
    assert engine.full_moves(seed, game0, n, 1.0).all() and not engine.full_moves(seed, game0, n, 0.0).any()
    # a different key: the rule does not reuse the move draw (key 1) or the check games (key 4)
    assert not np.array_equal(engine.full_moves(seed, game0, n, 0.5), engine.full_moves(seed + 1, game0, n, 0.5))


# ------------------------------------------------------------------ which plies are samples
def _hand_built(engine, full=None):
    h = engine.History(4, pinned=False)
    h.lens[:] = [3, 5, 0, 81]
    h.final[:] = [1, 0, 1, 1]
    for g in range(4):
        h.states[g, :, 0] = np.arange(81) + 100 * g
        h.counts[g, :, :] = (np.arange(81) + g)[:, None]
    if full is not None:
        h.full[:] = full
    return h


def test_history_full_defaults_to_ones_and_keeps_every_played_ply():
    import engine
    h = _hand_built(engine)
    assert h.full.shape == (4, 81) and h.full.dtype == np.uint8 and (h.full == 1).all()
    assert h.nbytes >= h.full.nbytes + h.states.nbytes
    mask = h.sample_mask()
    assert np.array_equal(mask, np.arange(81)[None, :] < h.lens[:, None])
    st, cn, z = h.samples()
    assert len(z) == 89 and np.array_equal(st[:, 0], np.concatenate([np.arange(L) + 100 * g for g, L in enumerate(h.lens)]))


def test_sample_mask_samples_and_host_pack_drop_fast_plies():
    import engine
    import parallel
    rng = np.random.default_rng(3)
    full = (rng.random((4, 81)) < 0.4).astype(np.uint8)
    h = _hand_built(engine, full)
    mask = h.sample_mask()
    want = (np.arange(81)[None, :] < h.lens[:, None]) & (full != 0)
    assert np.array_equal(mask, want) and 0 < mask.sum() < h.lens.sum()
    assert np.array_equal(h.sample_mask(2), want[:2])
    st, cn, z = h.samples()
    g, p = np.nonzero(want)
    assert np.array_equal(st[:, 0], p + 100 * g) and np.array_equal(cn[:, 0], p + g)
    # z: the reference's label of the ply, by the ply's own parity (a dropped ply does not shift it)
    z0 = np.where(h.final[g] != 0, -1, 0)
    assert np.array_equal(z, (z0 * np.where(p % 2 == 0, 1, -1)).astype(np.int8))
    for n_local in (4, 2):
        raw = parallel.pack_history_host(h, n_local).numpy()
        pst, pcn, pz, ply = engine.samples_to_numpy(raw)
        sel = g < n_local
        assert len(pz) == int(h.sample_mask(n_local).sum()) == sel.sum()
        assert np.array_equal(pst[:, 0], st[sel, 0]) and np.array_equal(pcn, cn[sel]) and np.array_equal(pz, z[sel])
        assert np.array_equal(ply, p[sel])


def test_corrected_labels_follow_the_sample_mask(monkeypatch):
    _lib()
    import engine
    import self_play_cpp as sp
    full = np.zeros((4, 81), np.uint8)
    full[:, ::3] = 1
    h = _hand_built(engine, full)
    zc = sp._corrected_labels(h)
    g, p = np.nonzero(h.sample_mask())
    zf = np.where(h.final[g] != 0, -1, 0)
    assert np.array_equal(zc, np.where((h.lens[g] - p) % 2 == 0, zf, -zf).astype(np.int8))


# ------------------------------------------------------------------ argument checks without a device
def test_set_playout_cap_rejects_bad_values():
    lib = _lib()
    for fast, frac, word in ((0, 0.25, b"fast_sims"), (-3, 0.25, b"fast_sims"), (8, float("nan"), b"fraction"),
                             (8, -0.01, b"fraction"), (8, 1.01, b"fraction")):
        assert lib.uttt_set_playout_cap(None, fast, frac) != 0 and word in lib.uttt_last_error(), (fast, frac)
    assert lib.uttt_set_playout_cap(None, 8, 0.25) != 0 and b"null engine" in lib.uttt_last_error()
    assert lib.uttt_selfplay_fetch_full(None, 1, None) != 0


def test_self_play_knobs_are_validated_before_any_gpu_work(monkeypatch):
    _lib()
    import engine
    import self_play_cpp as sp
    assert sp.SP_FAST_SIMS is None and sp.SP_FULL_FRACTION == 0.25 and sp._playout_cap_flags() == 0
    for bad in (0, -1, sp.PV_EVALUATE_COUNT + 1, 2.5, True):
        monkeypatch.setattr(sp, "SP_FAST_SIMS", bad)
        with pytest.raises(ValueError, match="SP_FAST_SIMS"):
            sp._playout_cap_flags()
        with pytest.raises(ValueError):
            sp.play(None)                                    # refused before the engine or the model is touched
    for ok in (1, 8, sp.PV_EVALUATE_COUNT):
        monkeypatch.setattr(sp, "SP_FAST_SIMS", ok)
        assert sp._playout_cap_flags() == engine.SP_PLAYOUT_CAP
    for bad in (-0.1, 1.5, float("nan")):
        monkeypatch.setattr(sp, "SP_FULL_FRACTION", bad)
        with pytest.raises(ValueError, match="SP_FULL_FRACTION"):
            sp._playout_cap_flags()
