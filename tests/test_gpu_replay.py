"""GPU: the reference search fed the ENGINE's OWN network rows (north_star: "MCTS visit counts must be bit-exact against
the reference C++ MCTS when both are fed identical network outputs").

With the network evaluator the leaves never leave the GPU (evaluator queue -> trunk_auto_kernel -> fused heads -> tree
kernel), so the engine records, per evaluated leaf, the policy / value row its tree is about to consume
(uttt_debug_trace).  Each root is then searched again by UTTT::pv_mcts_scores (cpp/uttt_mcts.cpp:84-196; the compiled
reference from oracle/_ref when it was built, else the C restatement) with a callback that returns exactly those rows
(cpp/python_bindings.cpp:11-47 contract), and the float scores / visit counts must agree bit for bit.  The recorded rows
are checked against a separate uttt_net_forward of the same leaf states, so a row handed to the wrong tree, or computed
from the wrong planes, cannot hide behind a consistent record.
"""
import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu


def _roots(n, seed=4242):
    out, g = [], 0
    while sum(len(x) for x in out) < n:
        out.append(O.playout_states(seed, g)[0][:-1])
        g += 1
    sts = np.concatenate(out)[:n]
    # vary the phase of the game across the batch (late positions finish their searches early: the batch decays)
    return sts[np.random.RandomState(0).permutation(n)]


@pytest.fixture(scope="module")
def nets():
    import torch
    from dual_network import DualNetwork
    from test_gpu_net import _damped
    torch.manual_seed(0)
    model = DualNetwork().eval()
    return model, _damped(DualNetwork().eval())


def _by_key(meta, col):
    order = np.argsort(meta[:, col], kind="stable")
    keys, first = np.unique(meta[order, col], return_index=True)
    return {int(k): order[a:b] for k, a, b in zip(keys, first, list(first[1:]) + [len(order)])}


def _search_and_replay(e, roots, sims, batch, evaluator, exact_rows, temperature=1.0):
    import torch
    e.trace(True)
    scores, counts, ns = e.mcts_search(roots, sims, batch, temperature, evaluator)
    meta, st, pol, val = e.trace_read()
    e.trace(False)
    assert len(val) > 0 and (counts.sum(1)[ns > 0] == sims).all()
    # (1) the recorded rows are the network's outputs for the recorded leaves
    p2, v2 = e.net_forward(torch.from_numpy(st.view(np.int32)).cuda(), evaluator)
    p2, v2 = p2.cpu().numpy(), v2.cpu().numpy()
    same = (p2 == pol).all(1) & (v2 == val)
    if exact_rows:
        assert same.all(), "rows differ from a separate forward of the same leaves: %d of %d" % ((~same).sum(), len(same))
    # (2) the reference search fed these rows reproduces the engine's scores bit for bit
    groups = _by_key(meta, 0)
    for i in range(len(roots)):
        idx = groups.get(i, np.zeros(0, np.int64))
        want = scores[i, :ns[i]]
        got, miss, unused = O.table_mcts(roots[i], temperature, sims, batch, st[idx], pol[idx], val[idx])
        assert miss == 0 and unused == 0, (i, miss, unused)
        assert got.tobytes() == want.tobytes(), (i, got, want)
    return same, p2, pol, v2, val


@pytest.mark.parametrize("n_roots", [60, 148, 300, 370, 450, 518])
def test_benchmarked_path_search_replays_bit_exactly_in_every_band(nets, n_roots):
    """UTTT_EVAL_NET_BF16 with up to 518 trees = trunk_auto_kernel + fused heads (the benchmarked path):
    <= 148 (one tile per CTA), 149-370 (two tiles), 371-518 (two groups in flight, cta_group::2 MMAs; the one-tile group's
    weight stages issued by one thread in quarter layers).  The recorded rows equal a stand-alone forward of the same leaves bit for
    bit in every band: a row's arithmetic does not depend on the batch it was evaluated in."""
    import engine
    model, damped = nets
    roots = _roots(n_roots)
    e = engine.Engine(n_slots=n_roots, max_sims=50, max_batch=8, max_games=8)
    try:
        e.upload_model(model)
        hist0 = e.batch_histogram()
        _search_and_replay(e, roots, 50, 8, engine.EVAL_NET_BF16, exact_rows=True)
        hist = e.batch_histogram()
        assert hist[(n_roots - 1) >> 4] + hist[min(63, n_roots >> 4)] > 0, hist      # the band did occur
        if n_roots > 370:          # the band with the one-tile group of trunk_pp_body<1>, on a second network
            e.upload_model(damped)
            _search_and_replay(e, roots, 50, 8, engine.EVAL_NET_BF16, exact_rows=True)
        # other search shapes of the same path
        for sims, batch, T in ((50, 1, 1.0), (37, 5, 0.0), (10, 2, 1.0)):
            _search_and_replay(e, roots[: min(n_roots, 96)], sims, batch, engine.EVAL_NET_BF16, exact_rows=False, temperature=T)
    finally:
        e.close()


@pytest.mark.parametrize("n_roots,evaluator", [(700, "bf16"), (1200, "bf16"), (100, "bf16x3"), (450, "bf16x3"), (800, "bf16x3"),
                                               (64, "fp32")])
def test_compacted_queue_search_replays_bit_exactly(nets, n_roots, evaluator):
    """engines above 518 trees (10-positions-per-pair trunk + separate heads kernel), and the bf16x3 / fp32 evaluators"""
    import engine
    model, _ = nets
    ev = {"bf16": engine.EVAL_NET_BF16, "bf16x3": engine.EVAL_NET_BF16X3, "fp32": engine.EVAL_NET_FP32}[evaluator]
    roots = _roots(n_roots, seed=99)
    e = engine.Engine(n_slots=n_roots, max_sims=50, max_batch=8, max_games=8)
    try:
        e.upload_model(model)
        _search_and_replay(e, roots, 50, 8, ev, exact_rows=True)
    finally:
        e.close()


@pytest.mark.parametrize("evaluator", ["bf16x3", "bf16"])
def test_gating_search_with_network_replays_bit_exactly(nets, evaluator):
    """the gating match's search (pv_mcts.py:74-180 semantics, UTTT_SP_PYSEARCH) with the NETWORK evaluator: the root is
    evaluated too, so its row is part of the record; the C restatement of the Python search (pinned against the
    unmodified reference module by tests/golden/pymcts.npz) fed the engine's own rows gives the same visit counts"""
    import torch
    import engine
    model, _ = nets
    ev = engine.evaluator_of(evaluator)
    roots = _roots(200, seed=31)
    e = engine.Engine(n_slots=200, max_sims=50, max_batch=8, max_games=8)
    try:
        e.upload_model(model)
        e.trace(True)
        _, counts, ns = e.mcts_search(roots, 50, 8, 1.0, ev, flags=engine.SP_PYSEARCH)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        p2, v2 = e.net_forward(torch.from_numpy(st.view(np.int32)).cuda(), ev)
        assert (p2.cpu().numpy() == pol).all() and (v2.cpu().numpy() == val).all()
        groups = _by_key(meta, 0)
        for i in range(len(roots)):
            idx = groups[i]
            assert (st[idx[0]] == roots[i]).all()                  # the first evaluated leaf of a tree is its root
            got, miss, unused = O.table_py_mcts(roots[i], 50, 8, st[idx], pol[idx], val[idx])
            assert miss == 0 and unused == 0 and len(got) == ns[i] and (got == counts[i, :ns[i]]).all(), i
        assert (counts.sum(1) == 50 - 8).all()                     # the first flush backs up the root only (pv_mcts.py:150-165)
    finally:
        e.close()


def test_full_selfplay_cycle_replays_bit_exactly(nets):
    """BASELINE config 3 as benchmarked (500 concurrent games, 50 simulations, batch 8, bf16 trunk, fused heads): every move
    of every game is searched again by the reference MCTS fed the rows the engine's network produced for that move's
    leaves; the visit counts in the history must be identical."""
    import engine
    model, _ = nets
    e = engine.Engine(n_slots=500, max_sims=50, max_batch=8, max_games=500)
    try:
        e.upload_model(model)
        e.trace(True)
        h = e.selfplay(500, sims=50, batch=8, seed=11, evaluator=engine.EVAL_NET_BF16)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        assert h.stats[2] == len(val)                      # every evaluated leaf was recorded
        key = meta[:, 1].astype(np.int64) * 128 + meta[:, 2]
        order = np.argsort(key, kind="stable")
        keys, first = np.unique(key[order], return_index=True)
        bounds = dict(zip(keys.tolist(), zip(first.tolist(), list(first[1:]) + [len(order)])))
        n_moves = 0
        for g in range(500):
            for ply in range(int(h.lens[g])):
                a, b = bounds.get(g * 128 + ply, (0, 0))
                idx = order[a:b]
                root = h.states[g, ply]
                got, miss, unused = O.table_mcts(root, 1.0, 50, 8, st[idx], pol[idx], val[idx])
                assert miss == 0 and unused == 0, (g, ply, miss, unused)
                legal = O.oracle_probe(root)[1]
                want = h.counts[g, ply][legal].astype(np.float32) / np.float32(50)
                assert got.tobytes() == want.tobytes(), (g, ply)
                n_moves += 1
        assert n_moves == h.stats[0] and n_moves > 20000
        # the same run without the trace: identical games (the trace only reads)
        h2 = e.selfplay(500, sims=50, batch=8, seed=11, evaluator=engine.EVAL_NET_BF16)
        assert (h.lens == h2.lens).all() and (h.actions == h2.actions).all() and (h.counts == h2.counts).all()
    finally:
        e.close()
