"""GPU: the throughput search (UTTT_SP_THROUGHPUT) in the configuration self-play runs -- several leaves per round with
virtual loss, root noise, forced playouts -- bit for bit against tests/tp_oracle.c.

1. Search calls, hash evaluator, no noise: the visit counts of every root for m = 2..16 leaves per round and budgets
   from 1 to 200 (800 at m = 16), over roots from every phase of the game, one-move roots and finished ones; the trace
   holds the same queued positions in the same rounds.
2. Search calls with noise: eta from uttt_debug_root_noise under the search key (seed 0, root index, ply 0); the result
   does not depend on the seed of a self-play run made earlier on the engine.
3. Self-play, hash evaluator, 8 leaves per round, eps = 0.25: every ply's counts, root value bits, targets and move, alone
   (T = 1 and T = 0) and with forced playouts, the playout cap, the random symmetry, resignation and the lane split.
4. Network replay: the traced rows are stand-alone forwards of the traced leaves, and the oracle fed those rows queues
   the same positions in the same rounds and reproduces counts, values, targets and moves (bf16 with noise, symmetry
   and forced playouts; bf16x3; fp32; a two-network match).
"""

import numpy as np
import pytest

import oracle_lib as O
import tp_lib as TP
import test_gpu_forced_playouts as FP
import test_gpu_resign as RS
import test_gpu_symmetry as SY

pytestmark = pytest.mark.gpu

ALPHA, EPS, K = 0.3, 0.25, 2.0

@pytest.fixture(scope="module")
def net():
    import torch
    from dual_network import DualNetwork
    torch.manual_seed(0)
    return DualNetwork().eval()

def _legal(w):
    return O.oracle_probe(w)[1]

def _eta(seed, states, games, plies):
    import engine
    if len(states) == 0:
        return np.zeros((0, 81), np.float32)
    return engine.root_noise(seed, ALPHA, np.stack(states), np.asarray(games, np.int64), np.asarray(plies, np.int32)).cpu().numpy()

# ------------------------------------------------------------------ 1. search calls, no noise
def test_search_counts_bit_exact_for_every_batch_size_and_budget():
    import engine
    cases = TP.search_cases()
    sts = cases[0][2]
    n_legal = np.array([len(_legal(w)) for w in sts])
    assert (n_legal == 0).any() and (n_legal == 1).any()
    e = engine.Engine(n_slots=len(sts), max_sims=800, max_batch=16, max_games=8)
    try:
        e.set_root_noise(ALPHA, 0.0)
        for m, sims, roots in cases:
            _, counts, ns = e.mcts_search(roots, sims, m, 1.0, engine.EVAL_HASH, flags=engine.SP_THROUGHPUT)
            assert e.counters()["overflow"] == 0
            for i, w in enumerate(roots):
                mv = TP.search(w, sims, m)
                assert ns[i] == len(mv.n) and np.array_equal(counts[i, :ns[i]], mv.n), (m, sims, i)
    finally:
        e.close()

@pytest.mark.parametrize("m", [3, 8, 16])
def test_search_trace_queues_the_oracles_positions_in_its_rounds(m):
    import engine
    sts = TP.search_cases()[0][2][::2]
    e = engine.Engine(n_slots=len(sts), max_sims=50, max_batch=16, max_games=8)
    try:
        e.set_root_noise(ALPHA, 0.0)
        e.trace(True)
        _, counts, ns = e.mcts_search(sts, 50, m, 1.0, engine.EVAL_HASH, flags=engine.SP_THROUGHPUT | engine.SP_RANDOM_SYMMETRY)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
    finally:
        e.close()
    groups = SY._moves(meta, [0])
    for i, w in enumerate(sts):
        mv = TP.search(w, 50, m, sym=(0, i, 0))
        idx = groups.get(i, np.zeros(0, np.int64))
        assert np.array_equal(counts[i, :ns[i]], mv.n), i
        assert np.array_equal(st[idx], mv.leaves) and np.array_equal(meta[idx, 3] - meta[idx[:1], 3], mv.rounds), i
        rep = TP.search(w, 50, m, rows=(pol[idx], val[idx]))
        assert np.array_equal(rep.n, mv.n) and np.array_equal(rep.leaves, mv.leaves), i

# ------------------------------------------------------------------ 2. search calls with noise
def test_noisy_search_bit_exact_with_the_device_noise():
    import engine
    sts = TP.search_cases()[0][2]
    sts = sts[[len(_legal(w)) > 0 for w in sts]]
    eta = _eta(0, list(sts), np.arange(len(sts)), np.zeros(len(sts)))
    for i, w in enumerate(sts):
        legal = _legal(w)
        assert (eta[i][legal] > 0).all() and np.delete(eta[i], legal).sum() == 0
        assert abs(float(eta[i].sum()) - 1.0) < 1e-5
    e = engine.Engine(n_slots=len(sts), max_sims=200, max_batch=16, max_games=8)
    try:
        e.set_root_noise(ALPHA, EPS)
        for m, sims in ((4, 50), (8, 200), (16, 50)):
            _, counts, ns = e.mcts_search(sts, sims, m, 1.0, engine.EVAL_HASH, flags=engine.SP_THROUGHPUT)
            for i, w in enumerate(sts):
                mv = TP.search(w, sims, m, eta=eta[i], eps=EPS)
                assert np.array_equal(counts[i, :ns[i]], mv.n), (m, sims, i)
    finally:
        e.close()

def test_dirichlet_sampler_is_the_root_noise_of_a_first_root():
    import engine
    w = O.playout_states(1, 0)[0][0]
    assert len(_legal(w)) == 81
    eta = _eta(9, [w] * 6, np.arange(100, 106), np.zeros(6))
    d = engine.dirichlet_samples(9, 100, 6, 81, ALPHA).cpu().numpy()
    assert np.array_equal(eta.view(np.uint32), d.view(np.uint32))

def test_noisy_search_does_not_depend_on_an_earlier_selfplay_seed():
    import engine
    sts = np.concatenate([O.playout_states(909, g)[0][:-1:5] for g in range(12)])[:100]
    out = []
    for earlier in (None, 7):
        e = engine.Engine(n_slots=len(sts), max_sims=50, max_batch=8, max_games=8)
        try:
            e.set_root_noise(ALPHA, EPS)
            if earlier is not None:
                e.selfplay(8, sims=16, batch=8, seed=earlier, evaluator=engine.EVAL_HASH, flags=engine.SP_THROUGHPUT)
            out.append(e.mcts_search(sts, 50, 8, 1.0, engine.EVAL_HASH, flags=engine.SP_THROUGHPUT)[1])
        finally:
            e.close()
    assert np.array_equal(out[0], out[1])

# ------------------------------------------------------------------ 3. self-play replay
def _replay(h, n, seed, game0, sims, m, flags, temperature=1.0, eps=EPS, fast=None, frac=None, resign=None, trace=None):
    """every searched ply of the first n games of history h (with the ply a game resigned at) against the oracle:
    counts, value bits, targets, move.  trace = (meta, states, policy, value) feeds the oracle the recorded rows and
    checks the queued positions and their rounds.  -> number of plies checked"""
    import engine
    forced, sym = bool(flags & engine.SP_FORCED_PLAYOUTS), bool(flags & engine.SP_RANDOM_SYMMETRY)
    full = engine.full_moves(seed, game0, n, frac) if flags & engine.SP_PLAYOUT_CAP else np.ones((n, 81), bool)
    plies = [(g, p) for g in range(n) for p in range(int(h.lens[g]) + int(h.resigned[g] != 0))]
    roots = [RS._root_at(h, g, p) for g, p in plies]
    noisy = [i for i, (g, p) in enumerate(plies) if eps > 0 and full[g, p]]
    eta = np.zeros((len(plies), 81), np.float32)
    noisy_s = set(noisy)
    eta[noisy] = _eta(seed, [roots[i] for i in noisy], [game0 + plies[i][0] for i in noisy], [plies[i][1] for i in noisy])
    groups = SY._moves(trace[0], [1, 2]) if trace is not None else None
    if resign is not None:
        checks = engine.check_games(seed, game0, n, resign[1])
    for i, (g, p) in enumerate(plies):
        w, f = roots[i], bool(full[g, p])
        rows = None
        if trace is not None:
            idx = groups[g * 128 + p]
            rows = (trace[2][idx], trace[3][idx])
        mv = TP.search(w, sims if f else fast, m, forced_k=K if forced and f else 0.0, eta=eta[i] if i in noisy_s else None,
                       eps=eps, sym=(seed, game0 + g, p) if sym and trace is None else None, rows=rows)
        if trace is not None:
            assert mv.evals == len(idx), (g, p)
            assert np.array_equal(trace[1][idx], mv.leaves), (g, p)
            assert np.array_equal(trace[0][idx, 3] - trace[0][idx[0], 3], mv.rounds), (g, p)
        assert RS._bits(h.values[g, p]) == RS._bits(mv.value), (g, p)
        if p == h.lens[g]:                            # the ply the game resigned at
            assert mv.value < resign[0] and not checks[g], (g, p)
            continue
        legal = _legal(w)
        assert np.array_equal(h.counts[g, p][legal], mv.n) and h.counts[g, p].sum() == mv.n.sum(), (g, p)
        if forced:
            assert np.array_equal(h.target[g, p][legal], mv.t), (g, p)
        j = FP._draw(seed, game0 + g, p, mv.t) if temperature == 1.0 else int(np.argmax(mv.t))
        assert h.actions[g, p] == legal[j], (g, p)
    return len(plies)

SP_CASES = {
    "alone": dict(),
    "alone_t0": dict(temperature=0.0),
    "forced": dict(flags="SP_FORCED_PLAYOUTS"),
    "playout_cap": dict(flags="SP_PLAYOUT_CAP", cap=(8, 0.25)),
    "forced_playout_cap": dict(flags="SP_FORCED_PLAYOUTS|SP_PLAYOUT_CAP", cap=(8, 0.25)),
    "symmetry": dict(flags="SP_RANDOM_SYMMETRY"),
    "resign": dict(flags="SP_RESIGN|SP_FORCED_PLAYOUTS", resign=(-0.5, 0.1)),
    "lanes": dict(flags="SP_FORCED_PLAYOUTS|SP_RANDOM_SYMMETRY", slots=20, lanes=10),
}

def _flags(names):
    import engine
    f = engine.SP_THROUGHPUT
    for nm in (names.split("|") if names else []):
        f |= getattr(engine, nm)
    return f

@pytest.mark.parametrize("case", list(SP_CASES))
def test_selfplay_every_ply_bit_exact(monkeypatch, case):
    import engine
    c = SP_CASES[case]
    n, seed, game0, sims = 32, 17, 40, 50
    flags = _flags(c.get("flags"))
    if "lanes" in c:
        monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(c["lanes"]))
    temperature = c.get("temperature", 1.0)
    e = engine.Engine(n_slots=c.get("slots", n), max_sims=sims, max_batch=8, max_games=n)
    try:
        e.set_root_noise(ALPHA, EPS)
        e.set_forced_playouts(K)
        e.set_selfplay_temperature(temperature)
        if "cap" in c:
            e.set_playout_cap(*c["cap"])
        if "resign" in c:
            e.set_resign(*c["resign"])
        h = e.selfplay(n, sims=sims, batch=8, seed=seed, game0=game0, evaluator=engine.EVAL_HASH, flags=flags)
    finally:
        e.close()
    if "resign" in c:
        assert h.resigned.any()
    cap = c.get("cap", (None, None))
    assert _replay(h, n, seed, game0, sims, 8, flags, temperature, fast=cap[0], frac=cap[1], resign=c.get("resign")) > 500

# ------------------------------------------------------------------ 4. network replay
def _check_forward_rows(e, meta, st, pol, val, seed, game0, sym, ev, keep=None):
    """the traced rows are sigma_g^-1 of stand-alone forwards of g(leaf), g keyed (seed, game0 + game index, ply, j)"""
    import symmetry_lib as S
    g = np.zeros(len(meta), np.int64)
    if sym:
        for key, idx in SY._moves(meta, [1, 2]).items():
            for j, r in enumerate(idx):
                g[r] = S.draw(seed, game0 + key // 128, key % 128, j)
    sel = np.arange(len(meta)) if keep is None else np.nonzero(keep)[0]
    SY._check_rows(e, st[sel], pol[sel], val[sel], g[sel], ev)

@pytest.mark.parametrize("evaluator,flags", [("bf16", "SP_FORCED_PLAYOUTS|SP_RANDOM_SYMMETRY"), ("bf16x3", ""),
                                             ("fp32", "SP_FORCED_PLAYOUTS")])
def test_network_selfplay_replays_from_the_traced_rows(net, evaluator, flags):
    import engine
    ev = engine.evaluator_of(evaluator)
    n, seed, game0, sims = 16, 23, 3, 32
    f = _flags(flags)
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.upload_model(net)
        e.set_root_noise(ALPHA, EPS)
        e.set_forced_playouts(K)
        e.trace(True)
        h = e.selfplay(n, sims=sims, batch=8, seed=seed, game0=game0, evaluator=ev, flags=f)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        assert h.stats[2] == len(val)
        _check_forward_rows(e, meta, st, pol, val, seed, game0, bool(f & engine.SP_RANDOM_SYMMETRY), ev)
    finally:
        e.close()
    assert _replay(h, n, seed, game0, sims, 8, f, trace=(meta, st, pol, val)) > 200

def test_network_match_replays_from_the_traced_rows(net):
    import torch
    import engine
    from dual_network import DualNetwork
    torch.manual_seed(1)
    other = DualNetwork().eval()
    ev = engine.evaluator_of("bf16")
    n, seed, game0, sims = 16, 31, 2, 32
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.upload_model(net, slot=0)
        e.upload_model(other, slot=1)
        e.set_root_noise(ALPHA, EPS)
        e.trace(True)
        _, h = e.match(n, sims=sims, batch=8, seed=seed, game0=game0, evaluator=ev, flags=engine.SP_THROUGHPUT)
        meta, st, pol, val = e.trace_read()
        e.trace(False)
        net0 = ((game0 + meta[:, 1].astype(np.int64) + meta[:, 2]) & 1) == 0
        assert net0.any() and (~net0).any()
        _check_forward_rows(e, meta, st, pol, val, seed, game0, False, ev, keep=net0)
    finally:
        e.close()
    assert _replay(h, n, seed, game0, sims, 8, engine.SP_THROUGHPUT, trace=(meta, st, pol, val)) > 200
