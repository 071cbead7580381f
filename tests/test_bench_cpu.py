"""CPU: bench.py --dump-outputs writes the history it is given as float32 / float64 .npy files within its size limit."""
import os

import numpy as np

import bench
import engine


def _random_history(n_games, seed):
    rng = np.random.RandomState(seed)
    h = engine.History(n_games, pinned=False)
    h.states[:] = rng.randint(0, 2 ** 32, h.states.shape, dtype=np.uint64).astype(np.uint32)
    h.counts[:] = rng.randint(0, 2 ** 16, h.counts.shape).astype(np.uint16)
    h.actions[:] = rng.randint(0, 81, h.actions.shape)
    h.lens[:] = rng.randint(17, 82, n_games)
    h.final[:] = rng.randint(0, 2, n_games)
    return h


def test_dump_writes_every_game_exactly(tmp_path):
    h = _random_history(50, 0)
    stats = np.array([2 ** 40 + 3, 5, 7, 9], np.int64)
    bench.dump_outputs(str(tmp_path), h, stats)
    got = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert set(got) == {"game", "lens", "final", "actions", "counts", "states", "stats"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert (got["game"] == np.arange(50)).all() and (got["stats"] == stats).all() and got["stats"][0] == 2 ** 40 + 3
    assert (got["lens"] == h.lens).all() and (got["final"] == h.final).all()
    for g in range(50):
        n = h.lens[g]
        assert (got["states"][g, :n] == h.states[g, :n]).all() and (got["states"][g, n:] == 0).all()
        assert (got["counts"][g, :n] == h.counts[g, :n]).all() and (got["counts"][g, n:] == 0).all()
        assert (got["actions"][g, :n] == h.actions[g, :n]).all() and (got["actions"][g, n:] == 0).all()


def test_dump_of_many_games_is_a_fixed_sample_under_64_mb(tmp_path):
    h = _random_history(4096, 1)
    a = bench.dump_outputs(str(tmp_path / "a"), h, np.zeros(4, np.int64))
    b = bench.dump_outputs(str(tmp_path / "b"), _random_history(4096, 2), np.zeros(4, np.int64))
    total = sum(os.path.getsize(os.path.join(tmp_path, "a", f)) for f in os.listdir(tmp_path / "a"))
    assert total <= 64 * 10 ** 6
    games = a["game"].astype(np.int64)
    assert 1000 < len(games) < 4096 and (b["game"] == a["game"]).all() and (np.diff(games) > 0).all()
    g = games[len(games) // 2]
    n = h.lens[g]
    assert (a["counts"][len(games) // 2, :n] == h.counts[g, :n]).all()
