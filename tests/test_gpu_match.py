"""GPU: matches between two networks on the device (UTTT_SP_MATCH, Engine.match).

1. Queue plumbing under the hash evaluator (which reads no weights): a match's histories equal plain self-play's bit for
   bit in every search mode, with slot recycling and with two lanes -- the leaves of slot 1's moves now travel through the
   second evaluator queue, so an indexing slip there shows up as a different game.
2. The same network in both slots: a match equals plain self-play bit for bit under bf16, bf16x3 and fp32 (a row does not
   depend on the batch it was evaluated in).
3. Two different networks: every recorded row is a stand-alone forward of its leaf by the network of slot (game + ply) & 1,
   and every move's visit counts are the reference search's fed those rows (C++ and pure-Python semantics); the moves
   follow the documented Philox draw and match_points agrees with a replay of the games.
4. Reproducibility, launch counts, argument errors, and the evaluate_network drop-in (EN_DEVICE_MATCH).
"""
import numpy as np
import pytest

import oracle_lib as O
import symmetry_lib as S

pytestmark = pytest.mark.gpu


def _same(a, b, n=None):
    n = len(a.lens) if n is None else n
    return (np.array_equal(a.lens[:n], b.lens[:n]) and np.array_equal(a.final[:n], b.final[:n])
            and np.array_equal(a.actions[:n], b.actions[:n]) and np.array_equal(a.states[:n], b.states[:n])
            and np.array_equal(a.counts[:n], b.counts[:n]))


@pytest.fixture(scope="module")
def nets():
    import torch
    from dual_network import DualNetwork
    from test_gpu_net import _damped
    torch.manual_seed(0)
    model = DualNetwork().eval()
    return model, _damped(DualNetwork().eval())


# ------------------------------------------------------------------ 1. hash evaluator: match == self-play
@pytest.mark.parametrize("flags", ["exact", "symmetry", "throughput"])
@pytest.mark.parametrize("slots,lane_threshold", [(40, None), (40, 32), (1024, None)])
def test_hash_match_equals_selfplay(monkeypatch, flags, slots, lane_threshold):
    """40 slots for 96 games: games recycle into freed slots; lane threshold 32 (and 1024 slots at the default threshold):
    both lanes run, each with its own slice of both queues"""
    import engine
    if lane_threshold is not None:
        monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(lane_threshold))
    f = {"exact": 0, "symmetry": engine.SP_RANDOM_SYMMETRY, "throughput": engine.SP_THROUGHPUT}[flags]
    n_games = 96 if slots < 1024 else 1024
    e = engine.Engine(n_slots=slots, max_sims=50, max_batch=8, max_games=n_games)
    try:
        plain = e.selfplay(n_games, sims=50, batch=8, seed=13, evaluator=engine.EVAL_HASH, flags=f, game0=500)
        plain_launches = e.last_run_profile()["trunk"][1]
        pts, h = e.match(n_games, sims=50, batch=8, seed=13, evaluator=engine.EVAL_HASH, flags=f, game0=500)
        match_launches = e.last_run_profile()["trunk"][1]
    finally:
        e.close()
    assert _same(h, plain)
    assert (h.stats[:3] == plain.stats[:3]).all()
    lanes = 2 if (slots >= (lane_threshold or 1024)) else 1
    assert plain_launches == plain.stats[3] * lanes and match_launches == 2 * h.stats[3] * lanes     # both passes counted
    assert np.array_equal(pts, engine.match_points(h, 500)) and set(np.unique(pts)) <= {0.0, 0.5, 1.0}
    if flags == "symmetry":         # the restatement of self-play with the flag reproduces the match's games
        for gi in range(0, n_games, 5 if n_games < 1024 else 97):
            n, st, cn, ac = S.selfplay(13, 500 + gi, 50, 8)
            assert h.lens[gi] == n, gi
            assert (h.states[gi, :n] == st[:n]).all() and (h.counts[gi, :n] == cn[:n]).all(), gi
            assert (h.actions[gi, :n] == ac[:n]).all(), gi


def test_hash_match_is_reproducible_and_follows_the_seed():
    import engine
    e = engine.Engine(n_slots=64, max_sims=50, max_batch=8, max_games=64)
    try:
        _, a = e.match(64, sims=50, batch=8, seed=3, evaluator=engine.EVAL_HASH, flags=engine.SP_PYSEARCH)
        _, b = e.match(64, sims=50, batch=8, seed=3, evaluator=engine.EVAL_HASH, flags=engine.SP_PYSEARCH)
        _, c = e.match(64, sims=50, batch=8, seed=4, evaluator=engine.EVAL_HASH, flags=engine.SP_PYSEARCH)
    finally:
        e.close()
    assert _same(a, b) and not _same(a, c)


# ------------------------------------------------------------------ 2. one network in both slots: match == self-play
@pytest.mark.parametrize("numerics", ["bf16", "bf16x3", "fp32"])
def test_same_network_in_both_slots_equals_selfplay(nets, numerics):
    import engine
    model, _ = nets
    ev = engine.evaluator_of(numerics)
    n, sims = (96, 50) if numerics != "fp32" else (48, 16)
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.upload_model(model)
        e.upload_model(model, slot=1)
        e.batch_histogram(reset=True)
        plain = e.selfplay(n, sims=sims, batch=8, seed=5, evaluator=ev)
        hist_plain = e.batch_histogram(reset=True)
        _, h = e.match(n, sims=sims, batch=8, seed=5, evaluator=ev)
        hist_match = e.batch_histogram(reset=True)
    finally:
        e.close()
    assert _same(h, plain)
    if numerics != "fp32":          # the trunk launches of both passes are in the batch-size histogram
        assert hist_match.sum() > hist_plain.sum() > 0


# ------------------------------------------------------------------ 3. two networks, replayed
def _philox_pick(seed, game, ply, counts):
    """the documented T = 1 draw (include/uttt_b200.h, hist_actions): index into the legal-order counts"""
    r = np.zeros(4, np.uint32)
    O.oracle().orc_philox4x32(seed, 1, game & 0xFFFFFFFF, game >> 32, ply, 0, r)
    pick = (int(r[0]) * int(counts.sum())) >> 32
    return int(np.argmax(np.cumsum(counts.astype(np.int64)) > pick))


def _replay_points(h, game0):
    """slot 0's point per game from a replay of its actions through uttt_cpp.State (evaluate_network.py:26-30,80-85)"""
    import uttt_cpp
    out = []
    for i in range(len(h.lens)):
        s = uttt_cpp.State()
        for t in range(int(h.lens[i])):
            assert not s.is_done()
            s = s.next(int(h.actions[i, t]))
        assert s.is_done()
        fp = (0 if s.is_first_player() else 1) if s.is_lose() else 0.5
        out.append(fp if (game0 + i) % 2 == 0 else 1 - fp)
    return np.array(out)


@pytest.mark.parametrize("search", ["cpp", "python"])
def test_two_network_match_replays_bit_exactly(nets, search):
    """500 games, 50 simulations, batch 8, bf16, model in slot 0 and its damped copy in slot 1, trace on"""
    import torch
    import engine
    model, damped = nets
    game0, seed, n = 3, 17, 500
    flags = engine.SP_PYSEARCH if search == "python" else 0
    e = engine.Engine(n_slots=n, max_sims=50, max_batch=8, max_games=n)
    try:
        e.upload_model(model)
        e.upload_model(damped, slot=1)
        e.trace(True)
        pts, h = e.match(n, sims=50, batch=8, seed=seed, evaluator=engine.EVAL_NET_BF16, flags=flags, game0=game0)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        # the same match without the trace: identical games (the trace only reads)
        pts2, h2 = e.match(n, sims=50, batch=8, seed=seed, evaluator=engine.EVAL_NET_BF16, flags=flags, game0=game0)
        assert _same(h, h2) and np.array_equal(pts, pts2)
    finally:
        e.close()
    assert h.stats[2] == len(val)                          # every evaluated leaf was recorded
    net = (game0 + meta[:, 1].astype(np.int64) + meta[:, 2]) & 1
    assert 0 < net.sum() < len(net)
    # (1) every row is the forward of its leaf by the network of its slot, and not the other network's
    ref = engine.Engine(n_slots=512, max_sims=50, max_batch=8, max_games=1)
    try:
        fw = []
        for m in (model, damped):
            ref.upload_model(m)                            # that network in slot 0 of a second engine
            p2, v2 = ref.net_forward(torch.from_numpy(st.view(np.int32)).cuda(), engine.EVAL_NET_BF16)
            fw.append((p2.cpu().numpy(), v2.cpu().numpy()))
    finally:
        ref.close()
    for k in (0, 1):
        rows = net == k
        pk, vk = fw[k]
        po, vo = fw[1 - k]
        same = (pk[rows] == pol[rows]).all(1) & (vk[rows] == val[rows])
        assert same.all(), "net %d: %d of %d rows differ from its own forward" % (k, (~same).sum(), rows.sum())
        other = (po[rows] == pol[rows]).all(1) & (vo[rows] == val[rows])
        assert not other.all(), "net %d: the other network's forward gives the same rows" % k
    # (2) every move's visit counts are the reference search's fed that move's rows; (3) the move is the Philox draw
    key = meta[:, 1].astype(np.int64) * 128 + meta[:, 2]
    order = np.argsort(key, kind="stable")
    keys, first = np.unique(key[order], return_index=True)
    bounds = dict(zip(keys.tolist(), zip(first.tolist(), list(first[1:]) + [len(order)])))
    n_moves = 0
    for g in range(n):
        for ply in range(int(h.lens[g])):
            a, b = bounds.get(g * 128 + ply, (0, 0))
            idx = order[a:b]
            root = h.states[g, ply]
            legal = O.oracle_probe(root)[1]
            cn = h.counts[g, ply][legal]
            if search == "python":
                assert len(idx) and (st[idx[0]] == root).all(), (g, ply)      # the first record of a move is its root
                got, miss, unused = O.table_py_mcts(root, 50, 8, st[idx], pol[idx], val[idx])
                assert miss == 0 and unused == 0 and (got == cn).all(), (g, ply)
            else:
                got, miss, unused = O.table_mcts(root, 1.0, 50, 8, st[idx], pol[idx], val[idx])
                assert miss == 0 and unused == 0, (g, ply, miss, unused)
                assert got.tobytes() == (cn.astype(np.float32) / np.float32(50)).tobytes(), (g, ply)
            assert h.actions[g, ply] == legal[_philox_pick(seed, game0 + g, ply, cn)], (g, ply)
            n_moves += 1
    assert n_moves == h.stats[0] and n_moves > 20000
    # (4) the points: the documented rule == a replay of the games; both networks won games
    assert np.array_equal(pts, _replay_points(h, game0))
    assert np.array_equal(pts, engine.match_points(h, game0))


def test_network_match_is_reproducible_and_follows_the_seed(nets):
    import engine
    model, damped = nets
    e = engine.Engine(n_slots=64, max_sims=50, max_batch=8, max_games=64)
    try:
        e.upload_model(model)
        e.upload_model(damped, slot=1)
        p1, a = e.match(64, sims=50, batch=8, seed=8, evaluator=engine.EVAL_NET_BF16X3, flags=engine.SP_PYSEARCH)
        p2, b = e.match(64, sims=50, batch=8, seed=8, evaluator=engine.EVAL_NET_BF16X3, flags=engine.SP_PYSEARCH)
        _, c = e.match(64, sims=50, batch=8, seed=9, evaluator=engine.EVAL_NET_BF16X3, flags=engine.SP_PYSEARCH)
        # swapping the networks' slots swaps who moves first: different games
        e.upload_model(damped)
        e.upload_model(model, slot=1)
        _, d = e.match(64, sims=50, batch=8, seed=8, evaluator=engine.EVAL_NET_BF16X3, flags=engine.SP_PYSEARCH)
    finally:
        e.close()
    assert _same(a, b) and np.array_equal(p1, p2)
    assert not _same(a, c) and not _same(a, d)


# ------------------------------------------------------------------ 4. errors
def test_match_argument_errors(nets):
    import engine
    model, _ = nets
    e = engine.Engine(n_slots=8, max_sims=50, max_batch=8, max_games=8)
    try:
        e.upload_model(model)
        with pytest.raises(RuntimeError, match="slot 1"):
            e.match(8, evaluator=engine.EVAL_NET_BF16)             # no slot-1 upload
        with pytest.raises(RuntimeError):
            e.selfplay(8, evaluator=engine.EVAL_HASH, flags=engine.SP_PYSEARCH)     # plain self-play: still a search option
        with pytest.raises(RuntimeError):
            e.match(8, evaluator=engine.EVAL_HASH, flags=engine.SP_PYSEARCH | engine.SP_THROUGHPUT)
        with pytest.raises(RuntimeError):
            e.mcts_search(O.playout_states(1, 0)[0][:2], 10, 2, 1.0, engine.EVAL_HASH, flags=engine.SP_MATCH)
        with pytest.raises(ValueError):
            e.upload_model(model, slot=2)
        w = engine.UtttWeights()
        assert e.lib.uttt_upload_weights_slot(e.h, 2, w, 0) != 0 and b"slot" in e.lib.uttt_last_error()
        assert e.lib.uttt_upload_weights_slot(e.h, -1, w, 0) != 0
        e.match(8, evaluator=engine.EVAL_HASH)                     # the hash evaluator needs no slot-1 upload
        e.upload_model(model, slot=1)
        e.match(8, evaluator=engine.EVAL_NET_BF16)
    finally:
        e.close()


# ------------------------------------------------------------------ 5. the evaluate_network drop-in
def test_evaluate_network_device_match(tmp_path, monkeypatch, capsys):
    import torch
    import engine
    import evaluate_network as en
    from dual_network import DualNetwork
    monkeypatch.chdir(tmp_path)
    (tmp_path / "model").mkdir()
    torch.manual_seed(3); best = DualNetwork().state_dict(); torch.save(best, "./model/best.pth")
    torch.manual_seed(4); latest = DualNetwork().state_dict(); torch.save(latest, "./model/latest.pth")
    monkeypatch.setattr(en, "EN_DEVICE_MATCH", True)
    monkeypatch.setattr(en, "EN_GAME_COUNT", 24)
    monkeypatch.setattr(en, "EN_SEED", 5)

    def host_path_unused(*a, **k):
        raise AssertionError("the host-driven match ran")
    monkeypatch.setattr(en, "play_matches", host_path_unused)
    promoted = en.evaluate_network()
    out = capsys.readouterr().out
    assert "Evaluate 24/24" in out and "AveragePoint" in out and ("Change BestPlayer" in out) == promoted
    avg = float(out.split("AveragePoint")[1].split()[0])
    assert promoted == (avg > 0.5)
    # the printed average is the mean of match_points of the same match played directly
    e = engine.Engine(n_slots=24, max_sims=en.PV_EVALUATE_COUNT, max_batch=en.MCTS_BATCH_SIZE, max_games=24)
    try:
        e.upload_state_dict(latest)
        e.upload_state_dict(best, slot=1)
        e.set_selfplay_temperature(en.EN_TEMPERATURE)
        flags = engine.SP_PYSEARCH if en.EN_SEARCH == "python" else 0
        pts, _ = e.match(24, sims=en.PV_EVALUATE_COUNT, batch=en.MCTS_BATCH_SIZE, seed=5,
                         evaluator=engine.evaluator_of(en.EN_NUMERICS), flags=flags)
    finally:
        e.close()
    assert avg == sum(pts.tolist()) / 24
    b = torch.load("./model/best.pth", weights_only=True)
    assert all(torch.equal(b[k], (latest if promoted else best)[k]) for k in b)
    # AlphaGo Zero's 400-game gate
    monkeypatch.setattr(en, "EN_GAME_COUNT", 400)
    en.evaluate_network()
    out = capsys.readouterr().out
    assert "Evaluate 400/400" in out and 0.0 <= float(out.split("AveragePoint")[1].split()[0]) <= 1.0
