"""GPU: UTTT_SP_RANDOM_SYMMETRY -- every leaf evaluated under a random board symmetry g, its policy read back through
sigma_g.

1. Hash evaluator: search scores / visit counts (C++ semantics, pure-Python semantics, the throughput mode's sequential
   configuration) and self-play histories are bit-exact against the restatement in tests/symmetry_oracle.c.
2. Network evaluator: the trace (untransformed leaf, row in the leaf's own action ids) replays bit-exactly through the
   reference search; every recorded row equals sigma_g^-1 of a stand-alone forward of g(leaf), with g recomputed from
   the documented key; the draws are spread evenly over the 8 symmetries.
3. Self-play with the flag is reproducible (re-runs, slot recycling, two lanes) and differs with the seed and from a run
   without the flag.
"""
import os

import numpy as np
import pytest

import oracle_lib as O
import symmetry_lib as S

pytestmark = pytest.mark.gpu

CHI2_7_LIMIT = 24.32        # chi-square, 7 degrees of freedom, p = 0.001


def _roots(n, seed):
    out, g = [], 0
    while sum(len(x) for x in out) < n:
        out.append(O.playout_states(seed, g)[0][:-1])
        g += 1
    sts = np.concatenate(out)[:n]
    return np.ascontiguousarray(sts[np.random.RandomState(0).permutation(n)])


@pytest.fixture(scope="module")
def eng():
    import engine
    e = engine.Engine(n_slots=256, max_sims=200, max_batch=8, max_games=128)
    yield e
    e.close()


@pytest.fixture(scope="module")
def model():
    import torch
    from dual_network import DualNetwork
    torch.manual_seed(0)
    return DualNetwork().eval()


# ------------------------------------------------------------------ 1. hash evaluator vs the restatement
@pytest.mark.parametrize("sims,batch,T", [(50, 8, 1.0), (50, 1, 1.0), (37, 5, 0.0), (10, 2, 1.0)])
def test_hash_search_cpp_semantics_matches_restatement(eng, sims, batch, T):
    import engine
    sts = _roots(200, seed=606)
    scores, counts, ns = eng.mcts_search(sts, sims, batch, T, engine.EVAL_HASH, flags=engine.SP_RANDOM_SYMMETRY)
    plain = eng.mcts_search(sts, sims, batch, T, engine.EVAL_HASH)[1]
    for i in range(0, len(sts), 3):
        sc, cn = S.cpp_search(sts[i], i, T, sims, batch)
        assert ns[i] == len(sc), i
        assert (counts[i, :ns[i]] == cn).all(), i
        assert scores[i, :ns[i]].tobytes() == sc.tobytes(), i
    if sims > 10:
        assert (counts != plain).any()


@pytest.mark.parametrize("sims,batch", [(50, 8), (50, 1), (37, 5), (10, 2)])
def test_hash_search_python_semantics_matches_restatement(eng, sims, batch):
    import engine
    sts = _roots(200, seed=707)
    _, counts, ns = eng.mcts_search(sts, sims, batch, 1.0, engine.EVAL_HASH,
                                    flags=engine.SP_PYSEARCH | engine.SP_RANDOM_SYMMETRY)
    for i in range(0, len(sts), 3):
        cn = S.py_search(sts[i], i, sims, batch)
        assert ns[i] == len(cn) and (counts[i, :ns[i]] == cn).all(), i


@pytest.mark.parametrize("sims", [50, 200])
def test_hash_search_throughput_sequential_matches_restatement(eng, sims):
    import engine
    sts = _roots(200, seed=808)
    eng.set_root_noise(0.3, 0.0)
    try:
        _, counts, ns = eng.mcts_search(sts, sims, 1, 1.0, engine.EVAL_HASH,
                                        flags=engine.SP_THROUGHPUT | engine.SP_RANDOM_SYMMETRY)
    finally:
        eng.set_root_noise(0.3, 0.25)
    for i in range(0, len(sts), 3):
        cn = S.az_search(sts[i], i, sims)
        assert ns[i] == len(cn) and (counts[i, :ns[i]] == cn).all(), (sims, i)


@pytest.mark.parametrize("slots", [128, 40])           # 40 slots: games are recycled into freed slots
def test_hash_selfplay_histories_match_restatement(slots):
    import engine
    e = engine.Engine(n_slots=slots, max_sims=50, max_batch=8, max_games=96)
    try:
        h = e.selfplay(96, sims=50, batch=8, seed=13, evaluator=engine.EVAL_HASH, flags=engine.SP_RANDOM_SYMMETRY, game0=500)
    finally:
        e.close()
    for gi in range(0, 96, 5):
        n, st, cn, ac = S.selfplay(13, 500 + gi, 50, 8)
        assert h.lens[gi] == n, gi
        assert (h.states[gi, :n] == st[:n]).all() and (h.counts[gi, :n] == cn[:n]).all(), gi
        assert (h.actions[gi, :n] == ac[:n]).all(), gi


# ------------------------------------------------------------------ 2. network evaluator
def _moves(meta, cols):
    """record indices grouped by the columns that identify one move's search, each group in evaluation order"""
    key = meta[:, cols[0]].astype(np.int64)
    if len(cols) > 1:
        key = key * 128 + meta[:, cols[1]]
    order = np.argsort(key, kind="stable")
    keys, first = np.unique(key[order], return_index=True)
    return {int(k): order[a:b] for k, a, b in zip(keys, first, list(first[1:]) + [len(order)])}


def _draws(meta, groups, seed, game_col, ply_col):
    """g of every record, recomputed from the key: (seed, game, ply, j = index of the evaluation in its move's search)"""
    g = np.zeros(len(meta), np.int64)
    for idx in groups.values():
        for j, r in enumerate(idx):
            game = int(meta[r, game_col])
            ply = int(meta[r, ply_col]) if ply_col is not None else 0
            g[r] = S.draw(seed, game, ply, j)
    return g


def _check_rows(e, st, pol, val, g, ev):
    """every recorded row is sigma_g^-1 of a stand-alone forward of g(leaf), bit for bit"""
    import torch
    import engine
    images = np.stack([engine.state_symmetry(st[r], g[r])[0] for r in range(len(st))])
    maps = np.stack([engine.state_symmetry(st[0], k)[1] for k in range(8)])
    p2, v2 = e.net_forward(torch.from_numpy(images.view(np.int32)).cuda(), ev)
    p2, v2 = p2.cpu().numpy(), v2.cpu().numpy()
    want = np.take_along_axis(p2, maps[g], axis=1)
    same = (want == pol).all(1) & (v2 == val)
    assert same.all(), "rows differ from sigma_g^-1(forward(g(leaf))): %d of %d" % ((~same).sum(), len(same))


def _chi2(g):
    c = np.bincount(g, minlength=8).astype(np.float64)
    e = len(g) / 8.0
    return float(((c - e) ** 2 / e).sum())


@pytest.mark.parametrize("evaluator", ["bf16", "bf16x3"])
def test_network_search_replays_and_rows_are_symmetric_forwards(model, evaluator):
    """60 / 148 / 370 / 518 / 700 roots: every band of the tensor-core trunk"""
    import engine
    ev = engine.evaluator_of(evaluator)
    all_g = []
    for n_roots in (60, 148, 370, 518, 700):
        roots = _roots(n_roots, seed=4242 + n_roots)
        e = engine.Engine(n_slots=n_roots, max_sims=50, max_batch=8, max_games=8)
        try:
            e.upload_model(model)
            e.trace(True)
            scores, counts, ns = e.mcts_search(roots, 50, 8, 1.0, ev, flags=engine.SP_RANDOM_SYMMETRY)
            meta, st, pol, val = e.trace_read()
            e.trace(False)
            assert len(val) > 0 and (counts.sum(1)[ns > 0] == 50).all()
            groups = _moves(meta, [0])
            g = _draws(meta, groups, 0, 0, None)
            _check_rows(e, st, pol, val, g, ev)
            all_g.append(g)
            for i in range(n_roots):
                idx = groups.get(i, np.zeros(0, np.int64))
                got, miss, unused = O.table_mcts(roots[i], 1.0, 50, 8, st[idx], pol[idx], val[idx])
                assert miss == 0 and unused == 0, (n_roots, i, miss, unused)
                assert got.tobytes() == scores[i, :ns[i]].tobytes(), (n_roots, i)
        finally:
            e.close()
    assert _chi2(np.concatenate(all_g)) < CHI2_7_LIMIT


@pytest.mark.parametrize("evaluator", ["bf16", "bf16x3"])
def test_network_selfplay_cycle_replays_and_rows_are_symmetric_forwards(model, evaluator):
    """the 500-game / 50-simulation cycle: every move of every game is searched again by the reference MCTS fed the rows
    the engine consumed; the visit counts in the history are identical"""
    import engine
    ev = engine.evaluator_of(evaluator)
    e = engine.Engine(n_slots=500, max_sims=50, max_batch=8, max_games=500)
    try:
        e.upload_model(model)
        e.trace(True)
        h = e.selfplay(500, sims=50, batch=8, seed=11, evaluator=ev, flags=engine.SP_RANDOM_SYMMETRY)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        assert h.stats[2] == len(val)
        groups = _moves(meta, [1, 2])
        g = _draws(meta, groups, 11, 1, 2)
        _check_rows(e, st, pol, val, g, ev)
        assert _chi2(g) < CHI2_7_LIMIT
        n_moves = 0
        for gi in range(500):
            for ply in range(int(h.lens[gi])):
                idx = groups.get(gi * 128 + ply, np.zeros(0, np.int64))
                root = h.states[gi, ply]
                got, miss, unused = O.table_mcts(root, 1.0, 50, 8, st[idx], pol[idx], val[idx])
                assert miss == 0 and unused == 0, (gi, ply, miss, unused)
                legal = O.oracle_probe(root)[1]
                want = h.counts[gi, ply][legal].astype(np.float32) / np.float32(50)
                assert got.tobytes() == want.tobytes(), (gi, ply)
                n_moves += 1
        assert n_moves == h.stats[0]
    finally:
        e.close()


# ------------------------------------------------------------------ 3. reproducibility
def _same(a, b):
    return (a.lens == b.lens).all() and (a.actions == b.actions).all() and (a.counts == b.counts).all()


def test_selfplay_with_symmetry_is_reproducible(model):
    import engine
    flags = engine.SP_RANDOM_SYMMETRY
    e = engine.Engine(n_slots=420, max_sims=50, max_batch=8, max_games=420)
    try:
        e.upload_model(model)
        h1 = e.selfplay(420, sims=50, batch=8, seed=21, evaluator=engine.EVAL_NET_BF16, flags=flags)
        h2 = e.selfplay(420, sims=50, batch=8, seed=21, evaluator=engine.EVAL_NET_BF16, flags=flags)
        assert _same(h1, h2)
        h3 = e.selfplay(420, sims=50, batch=8, seed=22, evaluator=engine.EVAL_NET_BF16, flags=flags)
        assert not _same(h1, h3)
        h4 = e.selfplay(420, sims=50, batch=8, seed=21, evaluator=engine.EVAL_NET_BF16)
        assert not _same(h1, h4)
    finally:
        e.close()
    # more games than slots, the slots split into two lanes on two streams
    os.environ["UTTT_LANE_THRESHOLD"] = "100"
    try:
        e = engine.Engine(n_slots=160, max_sims=50, max_batch=8, max_games=420)
    finally:
        del os.environ["UTTT_LANE_THRESHOLD"]
    try:
        e.upload_model(model)
        h5 = e.selfplay(420, sims=50, batch=8, seed=21, evaluator=engine.EVAL_NET_BF16, flags=flags)
        h6 = e.selfplay(420, sims=50, batch=8, seed=21, evaluator=engine.EVAL_NET_BF16, flags=flags)
        assert _same(h5, h6)
    finally:
        e.close()


# ------------------------------------------------------------------ 4. the drop-in modules' knobs
def test_evaluate_network_knob_runs_both_searches_with_the_flag(eng, monkeypatch):
    """EN_RANDOM_SYMMETRY adds UTTT_SP_RANDOM_SYMMETRY to the gating match's search, with the Python semantics (default)
    and with EN_SEARCH = "cpp"; hash evaluator, checked against the restatement"""
    import engine
    import evaluate_network as en
    roots = _roots(60, seed=909)
    monkeypatch.setattr(en, "EN_RANDOM_SYMMETRY", True)
    sc_py, ns_py = en.pv_mcts_scores_batch(eng, roots, 1.0, engine.EVAL_HASH, search="python")
    sc_cpp, ns_cpp = en.pv_mcts_scores_batch(eng, roots, 1.0, engine.EVAL_HASH, search="cpp")
    for i in range(len(roots)):
        cn = S.py_search(roots[i], i, 50, 8)
        assert ns_py[i] == len(cn) and (sc_py[i, :ns_py[i]] == en.python_scores(cn, 1.0)).all(), i
        sc, _ = S.cpp_search(roots[i], i, 1.0, 50, 8)
        assert ns_cpp[i] == len(sc) and sc_cpp[i, :ns_cpp[i]].tobytes() == sc.tobytes(), i
    monkeypatch.setattr(en, "EN_RANDOM_SYMMETRY", False)
    assert (en.pv_mcts_scores_batch(eng, roots, 1.0, engine.EVAL_HASH, search="python")[0] != sc_py).any()
    assert (en.pv_mcts_scores_batch(eng, roots, 1.0, engine.EVAL_HASH, search="cpp")[0] != sc_cpp).any()


def test_self_play_knob_passes_the_flag(model, monkeypatch):
    """SP_RANDOM_SYMMETRY: the drop-in self-play cycle plays exactly the games of the engine call with the flag"""
    import engine
    import self_play_cpp as sp
    monkeypatch.setattr(sp, "SP_SEED", 77)
    monkeypatch.setattr(sp, "SP_NUMERICS", "bf16")
    monkeypatch.setattr(sp, "SP_RANDOM_SYMMETRY", True)
    eng, h = sp._run(model, 16)
    with_flag = eng.selfplay(16, sims=sp.PV_EVALUATE_COUNT, batch=sp.MCTS_BATCH_SIZE, seed=77, evaluator=engine.EVAL_NET_BF16,
                             flags=engine.SP_RANDOM_SYMMETRY)
    assert _same(h, with_flag)
    monkeypatch.setattr(sp, "SP_RANDOM_SYMMETRY", False)
    _, h_off = sp._run(model, 16)
    assert not _same(h, h_off)
