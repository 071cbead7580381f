"""GPU: forced playouts and policy target pruning in self-play (UTTT_SP_FORCED_PLAYOUTS, Engine.set_forced_playouts,
History.target).

1. Bit for bit against the CPU: with one leaf per round and no noise every ply's raw counts, root value and targets
   equal the forced search of tests/forced_oracle.c, and every move is the Philox draw over the targets (T = 1) or c*
   (T = 0); with UTTT_SP_PLAYOUT_CAP the fast plies are the plain search and keep their counts as targets.
2. Batched, noisy runs (hash and bf16): the targets obey the rule's invariants, and forcing changes the counts.
3. Identity: k = 1e-6 forces and prunes nothing, so the run is the run without the flag, bit for bit.
4. Reproducibility across slot counts and the lane split.
5. Packed samples carry the targets; a later run without the flag packs the counts again.
6. Errors, and the self_play_cpp drop-in.
"""
import pickle

import numpy as np
import pytest

import forced_lib as FL
import oracle_lib as O
import resign_lib as R
import test_gpu_playout_cap as PC
import test_gpu_resign as RS

pytestmark = pytest.mark.gpu

SIMS, K = 50, 2.0


@pytest.fixture(scope="module")
def net():
    import torch
    from dual_network import DualNetwork
    torch.manual_seed(0)
    return DualNetwork().eval()


def _rows(h, n=None):
    n = len(h.lens) if n is None else n
    return np.arange(81)[None, :] < h.lens[:n, None]


def _draw(seed, game, ply, t):
    """the T = 1 move draw over target counts t in legal order -> legal index"""
    import engine
    x = int(engine._philox4x32_x(seed, 1, game & 0xFFFFFFFF, game >> 32, ply, 0))
    pick = (x * int(t.sum())) >> 32
    return int(np.nonzero(np.cumsum(t) > pick)[0][0])


def _run(n, batch=1, eps=0.0, seed=3, game0=0, flags=0, k=K, temperature=1.0, evaluator=None, model=None, sims=SIMS,
         slots=None, cap=None):
    import engine
    e = engine.Engine(n_slots=slots or n, max_sims=sims, max_batch=8, max_games=n)
    try:
        if model is not None:
            e.upload_model(model)
        e.set_root_noise(0.3, eps)
        e.set_forced_playouts(k)
        e.set_selfplay_temperature(temperature)
        if cap is not None:
            e.set_playout_cap(*cap)
        return e.selfplay(n, sims=sims, batch=batch, seed=seed, game0=game0,
                          evaluator=engine.EVAL_HASH if evaluator is None else evaluator,
                          flags=engine.SP_THROUGHPUT | engine.SP_FORCED_PLAYOUTS | flags)
    finally:
        e.close()


# ------------------------------------------------------------------ 1. bit for bit against the CPU
@pytest.mark.parametrize("temperature", [1.0, 0.0])
def test_every_ply_equals_the_cpu_forced_search(temperature):
    n, seed, game0 = 44, 3, 5
    h = _run(n, seed=seed, game0=game0, temperature=temperature)
    checked = pruned = 0
    for g in range(n):
        for p in range(int(h.lens[g])):
            legal = O.oracle_probe(h.states[g, p])[1]
            cn, w, t = FL.forced_root(h.states[g, p], SIMS, K)
            assert np.array_equal(h.counts[g, p][legal], cn), (g, p)
            assert np.array_equal(h.target[g, p][legal], t), (g, p)
            assert h.counts[g, p].sum() == h.counts[g, p][legal].sum() == SIMS
            assert h.target[g, p].sum() == t.sum()
            assert RS._bits(h.values[g, p]) == RS._bits(R.root_value(cn, w)), (g, p)
            i = _draw(seed, game0 + g, p, t) if temperature == 1.0 else int(np.argmax(cn))
            assert h.actions[g, p] == legal[i], (g, p)
            pruned += int((t != cn).any())
            checked += 1
    assert checked > 800 and pruned > 0


def test_fast_plies_are_the_plain_search_with_the_counts_as_targets():
    import engine
    n, seed, game0, fast = 40, 9, 0, 8
    h = _run(n, seed=seed, game0=game0, flags=engine.SP_PLAYOUT_CAP, cap=(fast, 0.25))
    rows = _rows(h)
    assert np.array_equal(h.full[rows] != 0, engine.full_moves(seed, game0, n, 0.25)[rows])
    n_fast = n_full = 0
    for g in range(n):
        for p in range(int(h.lens[g])):
            legal = O.oracle_probe(h.states[g, p])[1]
            if h.full[g, p]:
                cn, w, t = FL.forced_root(h.states[g, p], SIMS, K)
                n_full += 1
            else:
                cn, w = R.root_children(h.states[g, p], fast, 1, "az")
                t = cn
                n_fast += 1
            assert np.array_equal(h.counts[g, p][legal], cn) and np.array_equal(h.target[g, p][legal], t), (g, p)
            assert RS._bits(h.values[g, p]) == RS._bits(R.root_value(cn, w)), (g, p)
            assert h.actions[g, p] == legal[_draw(seed, game0 + g, p, t)], (g, p)
    assert n_fast > 200 and n_full > 50


# ------------------------------------------------------------------ 2. batched, noisy runs
def _invariants(h, seed, game0, budget):
    # only the played plies: rows past a game's length are never written (unspecified, like hist_counts'), and a fresh
    # target buffer may hold what an earlier engine left in that memory
    rows = _rows(h)
    cn = h.counts.astype(np.int64)
    t = h.target.astype(np.int64)
    assert (cn.sum(2)[rows] == budget).all()
    assert (t <= cn)[rows].all()
    cs = cn.argmax(2)
    assert (np.take_along_axis(t, cs[:, :, None], 2) == np.take_along_axis(cn, cs[:, :, None], 2))[rows].all()
    assert not ((t == 1) & (cn != 1))[rows].any()
    for g in range(len(h.lens)):
        for p in range(int(h.lens[g])):
            legal = O.oracle_probe(h.states[g, p])[1]
            assert h.actions[g, p] == legal[_draw(seed, game0 + g, p, t[g, p][legal])], (g, p)
    assert (t != cn).any(2)[rows].any()


@pytest.mark.parametrize("evaluator", ["hash", "bf16"])
def test_batched_noisy_runs_keep_the_invariants_and_force(net, evaluator):
    import engine
    n, seed, game0 = 48, 4, 17
    ev = engine.EVAL_HASH if evaluator == "hash" else engine.evaluator_of("bf16")
    model = net if evaluator != "hash" else None
    on = _run(n, batch=8, eps=0.25, seed=seed, game0=game0, evaluator=ev, model=model)
    _invariants(on, seed, game0, SIMS)
    e = engine.Engine(n_slots=n, max_sims=SIMS, max_batch=8, max_games=n)
    try:
        if model is not None:
            e.upload_model(model)
        e.set_root_noise(0.3, 0.25)
        off = e.selfplay(n, sims=SIMS, batch=8, seed=seed, game0=game0, evaluator=ev, flags=engine.SP_THROUGHPUT)
    finally:
        e.close()
    assert off.target is None
    assert not np.array_equal(on.counts[:, 0], off.counts[:, 0])      # the first move's root is the same position


# ------------------------------------------------------------------ 3. identity
@pytest.mark.parametrize("lanes", [1, 2])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("evaluator", ["hash", "bf16"])
def test_tiny_k_is_the_run_without_the_flag(monkeypatch, net, evaluator, sym, lanes):
    import engine
    n = 64
    flags = engine.SP_THROUGHPUT | engine.SP_RESIGN | (engine.SP_RANDOM_SYMMETRY if sym else 0)
    if lanes == 2:
        monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(n // 2))
    ev = engine.evaluator_of(evaluator) if evaluator != "hash" else engine.EVAL_HASH
    e = engine.Engine(n_slots=n, max_sims=32, max_batch=8, max_games=n)
    try:
        if evaluator != "hash":
            e.upload_model(net)
        e.set_resign(-0.5 if evaluator == "hash" else -0.05, 0.1)
        off = e.selfplay(n, sims=32, batch=8, seed=21, evaluator=ev, flags=flags, game0=7)
        e.set_forced_playouts(1e-6)
        on = e.selfplay(n, sims=32, batch=8, seed=21, evaluator=ev, flags=flags | engine.SP_FORCED_PLAYOUTS, game0=7)
    finally:
        e.close()
    rows = PC._same_games(off, on)
    assert off.target is None and np.array_equal(on.target[rows], on.counts[rows])
    if evaluator == "hash":
        assert off.resigned.any()


# ------------------------------------------------------------------ 4. reproducibility
def test_same_seed_same_games_across_slots_and_lanes(monkeypatch):
    n, seed, game0 = 64, 5, 3
    runs = []
    for slots, thr in ((n, None), (20, None), (n, n // 2)):
        if thr is None:
            monkeypatch.delenv("UTTT_LANE_THRESHOLD", raising=False)
        else:
            monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(thr))
        runs.append(_run(n, batch=8, eps=0.25, seed=seed, game0=game0, slots=slots))
    a = runs[0]
    for b in runs[1:]:
        rows = PC._same_games(a, b)
        assert np.array_equal(a.target[rows], b.target[rows])


# ------------------------------------------------------------------ 5. packed samples
def test_pack_carries_the_targets_and_an_unflagged_run_the_counts_again():
    import torch
    import engine
    import parallel
    n, slots = 120, 48
    e = engine.Engine(n_slots=slots, max_sims=SIMS, max_batch=8, max_games=n)
    try:
        e.set_forced_playouts(K)
        for forced in (True, False):
            flags = engine.SP_THROUGHPUT | (engine.SP_FORCED_PLAYOUTS if forced else 0)
            e.selfplay_device(n, sims=SIMS, batch=8, seed=8, evaluator=engine.EVAL_HASH, flags=flags)
            h = e.selfplay_fetch(n)
            buf, ns = e.selfplay_pack(n)
            assert (h.target is not None) == forced
            mask = h.sample_mask()
            assert ns == mask.sum() == h.lens.sum()
            assert torch.equal(buf.cpu(), parallel.pack_history_host(h, n))
            st, cn, z, ply = engine.samples_to_numpy(buf.cpu().numpy())
            assert np.array_equal(cn, (h.target if forced else h.counts)[mask])
            if forced:
                assert (cn != h.counts[mask]).any()
            _, p, _ = engine.samples_unpack(buf)
            pw = torch.from_numpy(cn.astype(np.float32) / cn.sum(1, keepdims=True).astype(np.float32)).cuda()
            assert torch.equal(p, pw)
    finally:
        e.close()


# ------------------------------------------------------------------ 6. errors and the drop-in
def test_forced_playouts_errors():
    import engine
    e = engine.Engine(n_slots=8, max_sims=50, max_batch=8, max_games=8)
    try:
        for k in (0.0, -1.0, 100.5, float("nan"), float("inf")):
            with pytest.raises(RuntimeError, match="forced playouts"):
                e.set_forced_playouts(k)
        for f, word in ((0, "UTTT_SP_THROUGHPUT"), (engine.SP_CORRECT_TERMINAL_SIGN, "UTTT_SP_THROUGHPUT"),
                        (engine.SP_THROUGHPUT | engine.SP_MATCH, "UTTT_SP_MATCH")):
            with pytest.raises(RuntimeError, match=word):
                e.selfplay(8, sims=32, evaluator=engine.EVAL_HASH, flags=f | engine.SP_FORCED_PLAYOUTS)
        roots = O.playout_states(1, 0)[0][:2]
        for f in (engine.SP_FORCED_PLAYOUTS, engine.SP_FORCED_PLAYOUTS | engine.SP_THROUGHPUT):
            with pytest.raises(RuntimeError, match="self-play mode"):
                e.mcts_search(roots, 10, 2, 1.0, engine.EVAL_HASH, flags=f)
        h = e.selfplay(8, sims=32, evaluator=engine.EVAL_HASH, flags=engine.SP_THROUGHPUT | engine.SP_FORCED_PLAYOUTS)
        assert (h.lens >= 1).all() and h.target is not None
    finally:
        e.close()


def test_self_play_drop_in_trains_on_the_pruned_targets(tmp_path, monkeypatch):
    import torch
    import self_play_cpp as sp
    from dual_network import DualNetwork
    monkeypatch.chdir(tmp_path)
    (tmp_path / "model").mkdir()
    torch.manual_seed(0)
    torch.save(DualNetwork().state_dict(), "./model/best.pth")
    n = 40
    for k, v in dict(SP_GAME_COUNT=n, PV_EVALUATE_COUNT=32, SP_NUMERICS="bf16", SP_SEED=5, SP_PROGRESS=False,
                     SP_SEARCH_MODE="throughput", SP_FORCED_PLAYOUTS=2.0).items():
        monkeypatch.setattr(sp, k, v)
    runs = []
    real_run = sp._run

    def run(*a, **k):
        out = real_run(*a, **k)
        runs.append(out[1])
        return out
    monkeypatch.setattr(sp, "_run", run)
    f = sp.self_play()
    h = runs[-1]
    with open(f, "rb") as fh:
        rows = pickle.load(fh)
    mask = h.sample_mask(n)
    assert len(rows) == mask.sum()
    pol = np.stack([r[1] for r in rows])
    cn, t = h.counts[:n][mask], h.target[:n][mask]
    assert ((pol > 0) == (t > 0)).all()
    assert ((t == 0) & (cn > 0)).any()
    assert np.allclose(pol, t / t.sum(1, keepdims=True), atol=1e-6)
    assert sp.last_stats["pruned_visits"] == int(cn.astype(np.int64).sum() - t.astype(np.int64).sum()) > 0
