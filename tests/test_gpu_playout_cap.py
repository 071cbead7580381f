"""GPU: playout cap randomization in self-play (UTTT_SP_PLAYOUT_CAP, Engine.set_playout_cap, History.full).

1. Kinds and budgets: History.full follows engine.full_moves, and a ply's visit counts add up to its budget, in every
   search mode.
2. Every ply is its own search: its counts and root value equal a CPU search of the recorded root at that ply's budget
   (tests/resign_oracle.c); with root noise on, the fast plies still equal the noise-free CPU search.
3. Identity: full_fraction 1 is the run without the flag, bit for bit (hash and bf16, symmetry on and off, with
   resignation, one and two lanes); fast_sims == evaluate_count with fraction 0 plays the same games and packs nothing.
4. Reproducibility across slot counts and the lane threshold.
5. Packed samples: exactly the full plies, byte-equal to the host restatements; unpack; a single-rank SelfPlayCycle.
6. Resignation: a resigning capped run is the capped run cut short.
7. Errors, and the self_play_cpp drop-in.
"""
import pickle
import socket

import numpy as np
import pytest

import oracle_lib as O
import resign_lib as R
import test_gpu_resign as RS

pytestmark = pytest.mark.gpu

SIMS, FAST, FRAC = 50, 8, 0.25
MODES = {"exact": 0, "exact_correct": "CORRECT_TERMINAL_SIGN", "az": "THROUGHPUT"}


@pytest.fixture(scope="module")
def net():
    import torch
    from dual_network import DualNetwork
    torch.manual_seed(0)
    return DualNetwork().eval()


def _mode_flags(mode):
    import engine
    return getattr(engine, "SP_" + MODES[mode]) if MODES[mode] else 0


def _rows(h, n=None):
    n = len(h.lens) if n is None else n
    return np.arange(81)[None, :] < h.lens[:n, None]


def _capped_run(mode, batch, eps, n=40, seed=3, game0=0):
    import engine
    e = engine.Engine(n_slots=n, max_sims=SIMS, max_batch=8, max_games=n)
    try:
        e.set_root_noise(0.3, eps)
        e.set_playout_cap(FAST, FRAC)
        return e.selfplay(n, sims=SIMS, batch=batch, seed=seed, evaluator=engine.EVAL_HASH, game0=game0,
                          flags=_mode_flags(mode) | engine.SP_PLAYOUT_CAP)
    finally:
        e.close()


# ------------------------------------------------------------------ 1. kinds and budgets
@pytest.mark.parametrize("mode,batch,eps", [("exact", 8, 0.0), ("exact", 1, 0.0), ("exact_correct", 8, 0.0),
                                            ("az", 1, 0.0), ("az", 8, 0.0), ("az", 1, 0.25), ("az", 8, 0.25)])
def test_kinds_and_budgets(mode, batch, eps):
    import engine
    n, seed, game0 = 40, 3, 11
    h = _capped_run(mode, batch, eps, n, seed, game0)
    rows = _rows(h)
    want = engine.full_moves(seed, game0, n, FRAC)
    assert np.array_equal(h.full[rows] != 0, want[rows])
    assert 0 < want[rows].sum() < rows.sum()
    tot = h.counts.astype(np.int64).sum(axis=2)
    assert (tot[rows & want] == SIMS).all() and (tot[rows & ~want] == FAST).all()
    assert h.stats[0] == rows.sum()


# ------------------------------------------------------------------ 2. every ply against the CPU search
@pytest.mark.parametrize("mode,batch,eps", [("exact_correct", 8, 0.0), ("exact_correct", 1, 0.0), ("az", 1, 0.0),
                                            ("az", 1, 0.25)])
def test_every_ply_is_its_own_search(mode, batch, eps):
    n = 40
    h = _capped_run(mode, batch, eps, n)
    checked = noisy_differ = 0
    for g in range(n):
        for t in range(int(h.lens[g])):
            full = bool(h.full[g, t])
            cn, w = R.root_children(h.states[g, t], SIMS if full else FAST, batch, mode)
            got = h.counts[g, t][O.oracle_probe(h.states[g, t])[1]]
            if full and eps > 0:                      # the full searches' roots are noisy: the CPU search has none
                noisy_differ += not np.array_equal(got, cn)
                continue
            assert np.array_equal(got, cn), (g, t, full)
            assert RS._bits(h.values[g, t]) == RS._bits(R.root_value(cn, w)), (g, t)
            checked += 1
    assert checked > 500
    if eps > 0:
        assert noisy_differ > 0


# ------------------------------------------------------------------ 3. identity
def _pair(monkeypatch, nets, evaluator, flags, lanes, n, before, seed=21, game0=7, sims=32, frac=1.0, fast=FAST):
    """(run without the flag, run with it) on one engine; before(e) configures both"""
    import engine
    if lanes == 2:
        monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(n // 2))
    ev = engine.evaluator_of(evaluator) if evaluator != "hash" else engine.EVAL_HASH
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        if evaluator != "hash":
            e.upload_model(nets)
        before(e)
        off = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=ev, flags=flags, game0=game0)
        e.set_playout_cap(fast, frac)
        on = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=ev, flags=flags | engine.SP_PLAYOUT_CAP, game0=game0)
    finally:
        e.close()
    return off, on


def _same_games(off, on):
    rows = _rows(off)
    assert np.array_equal(on.lens, off.lens) and np.array_equal(on.final, off.final)
    assert np.array_equal(on.resigned, off.resigned) and np.array_equal(on.stats[0], off.stats[0])
    assert np.array_equal(on.states[rows], off.states[rows]) and np.array_equal(on.counts[rows], off.counts[rows])
    assert np.array_equal(on.actions[rows], off.actions[rows])
    rec = rows | (np.arange(81)[None, :] == (off.lens * (off.resigned != 0) - (off.resigned == 0))[:, None])
    assert np.array_equal(RS._bits(on.values[rec]), RS._bits(off.values[rec]))
    return rows


@pytest.mark.parametrize("lanes", [1, 2])
@pytest.mark.parametrize("sym", [False, True])
@pytest.mark.parametrize("search", ["exact_correct", "az"])
@pytest.mark.parametrize("evaluator", ["hash", "bf16"])
def test_full_fraction_one_is_the_run_without_the_flag(monkeypatch, net, evaluator, search, sym, lanes):
    import engine
    flags = _mode_flags(search) | (engine.SP_RANDOM_SYMMETRY if sym else 0) | engine.SP_RESIGN

    def before(e):
        e.set_resign(-0.5 if evaluator == "hash" else -0.05, 0.1)
    off, on = _pair(monkeypatch, net, evaluator, flags, lanes, 64, before)
    rows = _same_games(off, on)
    assert (on.full[rows] == 1).all() and (off.full[rows] == 1).all()
    if evaluator == "hash":
        assert off.resigned.any()


def test_fast_budget_equal_to_the_full_one_plays_the_same_games_and_packs_nothing(monkeypatch):
    import engine
    n, sims = 48, 32
    off, on = _pair(monkeypatch, None, "hash", 0, 1, n, lambda e: None, sims=sims, frac=0.0, fast=sims)
    rows = _same_games(off, on)
    assert (on.full[rows] == 0).all() and on.sample_mask().sum() == 0 and len(on.samples()[2]) == 0
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.set_playout_cap(sims, 0.0)
        e.selfplay_device(n, sims=sims, batch=8, seed=21, evaluator=engine.EVAL_HASH, game0=7, flags=engine.SP_PLAYOUT_CAP)
        buf, ns = e.selfplay_pack(n)
        assert ns == 0 and buf.numel() == 0
        assert np.array_equal(e.selfplay_fetch(n).lens, off.lens)
    finally:
        e.close()


# ------------------------------------------------------------------ 4. reproducibility
@pytest.mark.parametrize("mode,eps", [("exact", 0.0), ("az", 0.25)])
def test_same_seed_same_games_across_slots_and_lanes(monkeypatch, mode, eps):
    import engine
    n, seed, game0 = 64, 5, 3
    runs = []
    for slots, thr in ((n, None), (20, None), (n, n // 2)):
        if thr is None:
            monkeypatch.delenv("UTTT_LANE_THRESHOLD", raising=False)
        else:
            monkeypatch.setenv("UTTT_LANE_THRESHOLD", str(thr))
        e = engine.Engine(n_slots=slots, max_sims=SIMS, max_batch=8, max_games=n)
        try:
            e.set_root_noise(0.3, eps)
            e.set_playout_cap(FAST, FRAC)
            runs.append(e.selfplay(n, sims=SIMS, batch=8, seed=seed, evaluator=engine.EVAL_HASH, game0=game0,
                                   flags=_mode_flags(mode) | engine.SP_PLAYOUT_CAP))
        finally:
            e.close()
    a = runs[0]
    rows = _rows(a)
    for b in runs[1:]:
        rows_b = _same_games(a, b)
        assert np.array_equal(rows_b, rows) and np.array_equal(b.full[rows], a.full[rows])
    assert np.array_equal(a.full[rows] != 0, engine.full_moves(seed, game0, n, FRAC)[rows])


# ------------------------------------------------------------------ 5. packed samples
@pytest.mark.parametrize("mode", ["exact", "az"])
def test_pack_carries_exactly_the_full_plies(mode):
    import torch
    import engine
    import parallel
    n, slots = 120, 48
    e = engine.Engine(n_slots=slots, max_sims=SIMS, max_batch=8, max_games=n)
    try:
        e.set_playout_cap(FAST, FRAC)
        stats = e.selfplay_device(n, sims=SIMS, batch=8, seed=8, evaluator=engine.EVAL_HASH,
                                  flags=_mode_flags(mode) | engine.SP_PLAYOUT_CAP)
        h = e.selfplay_fetch(n)
        buf, ns = e.selfplay_pack(n)
    finally:
        e.close()
    mask = h.sample_mask()
    assert np.array_equal(mask, _rows(h) & engine.full_moves(8, 0, n, FRAC))
    assert ns == mask.sum() < stats[0] == h.lens.sum() and buf.numel() == ns * engine.SAMPLE_BYTES
    assert torch.equal(buf.cpu(), parallel.pack_history_host(h, n))
    st, cn, z, ply = engine.samples_to_numpy(buf.cpu().numpy())
    st2, cn2, z2 = h.samples()
    assert np.array_equal(st, st2) and np.array_equal(cn, cn2) and np.array_equal(z, z2)
    assert np.array_equal(ply, np.nonzero(mask)[1]) and (cn.astype(np.int64).sum(1) == SIMS).all()
    x, p, v = engine.samples_unpack(buf)
    planes = engine.game_encode(torch.from_numpy(st.view(np.int32)).cuda()).permute(0, 3, 1, 2).contiguous()
    assert torch.equal(x, planes)
    pw = torch.from_numpy(cn.astype(np.float32) / cn.sum(1, keepdims=True).astype(np.float32)).cuda()
    assert torch.equal(p, pw) and torch.equal(v[:, 0].cpu(), torch.from_numpy(z.astype(np.float32)))


def test_selfplay_cycle_with_a_playout_cap_single_rank(net):
    import torch
    import torch.distributed as dist
    import engine
    import parallel
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        n = 48
        cyc = parallel.SelfPlayCycle(n, sims=20, batch=8, numerics="bf16", fast_sims=4, full_fraction=0.25)
        try:
            r = cyc.run(net, seed=1, cycle=1)
            h = cyc.engine.selfplay_fetch(n)
        finally:
            cyc.close()
    finally:
        dist.destroy_process_group()
    mask = h.sample_mask()
    assert np.array_equal(mask, _rows(h) & engine.full_moves(1, n, n, 0.25))          # cycle 1: games n .. 2n - 1
    assert r["n_samples"] == mask.sum() < h.lens.sum() and r["samples_per_rank"] == [r["n_samples"]]
    assert torch.equal(r["samples"].cpu(), parallel.pack_history_host(h, n))
    assert r["x"].shape == (r["n_samples"], 3, 9, 9)
    assert torch.allclose(r["policy"].sum(1), torch.ones(r["n_samples"], device="cuda"))
    assert (h.counts[mask].astype(np.int64).sum(1) == 20).all() and (h.counts[_rows(h) & ~mask].astype(np.int64).sum(1) == 4).all()


# ------------------------------------------------------------------ 6. with resignation
@pytest.mark.parametrize("mode", ["exact_correct", "az"])
def test_resigned_capped_games_are_prefixes(mode):
    import engine
    n, seed, game0, frac, sims = 64, 21, 7, 0.25, 32
    flags = _mode_flags(mode) | engine.SP_PLAYOUT_CAP
    e = engine.Engine(n_slots=n, max_sims=sims, max_batch=8, max_games=n)
    try:
        e.set_playout_cap(FAST, FRAC)
        off = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=engine.EVAL_HASH, flags=flags, game0=game0)
        thr = RS._threshold(off, n)
        e.set_resign(thr, frac)
        on = e.selfplay(n, sims=sims, batch=8, seed=seed, evaluator=engine.EVAL_HASH, flags=flags | engine.SP_RESIGN,
                        game0=game0)
    finally:
        e.close()
    RS._check_prefix(engine, off, on, n, thr, frac, seed, game0, False)
    for g in range(n):
        L = int(on.lens[g])
        assert np.array_equal(on.full[g, :L], off.full[g, :L]), g
    assert (off.full[_rows(off)] == 0).any()


# ------------------------------------------------------------------ 7. errors and the drop-in
def test_playout_cap_errors():
    import engine
    e = engine.Engine(n_slots=8, max_sims=50, max_batch=8, max_games=8)
    try:
        for fast, frac, word in ((0, 0.25, "fast_sims"), (51, 0.25, "max_sims"), (8, float("nan"), "fraction"),
                                 (8, -0.1, "fraction"), (8, 1.1, "fraction")):
            with pytest.raises(RuntimeError, match=word):
                e.set_playout_cap(fast, frac)
        e.set_playout_cap(40, 0.25)
        with pytest.raises(RuntimeError, match="exceeds evaluate_count"):
            e.selfplay(8, sims=32, evaluator=engine.EVAL_HASH, flags=engine.SP_PLAYOUT_CAP)
        e.set_playout_cap(8, 0.25)
        with pytest.raises(RuntimeError, match="UTTT_SP_MATCH"):
            e.selfplay(8, sims=32, evaluator=engine.EVAL_HASH, flags=engine.SP_PLAYOUT_CAP | engine.SP_MATCH)
        roots = O.playout_states(1, 0)[0][:2]
        for f in (engine.SP_PLAYOUT_CAP, engine.SP_PLAYOUT_CAP | engine.SP_THROUGHPUT):
            with pytest.raises(RuntimeError, match="self-play mode"):
                e.mcts_search(roots, 10, 2, 1.0, engine.EVAL_HASH, flags=f)
        h = e.selfplay(8, sims=32, evaluator=engine.EVAL_HASH, flags=engine.SP_PLAYOUT_CAP)
        assert (h.lens >= 1).all()
    finally:
        e.close()


def test_self_play_drop_in_keeps_the_full_plies(tmp_path, monkeypatch):
    import torch
    import engine
    import self_play_cpp as sp
    from dual_network import DualNetwork
    monkeypatch.chdir(tmp_path)
    (tmp_path / "model").mkdir()
    torch.manual_seed(0)
    torch.save(DualNetwork().state_dict(), "./model/best.pth")
    n = 40
    for k, v in dict(SP_GAME_COUNT=n, PV_EVALUATE_COUNT=16, SP_NUMERICS="bf16", SP_SEED=5, SP_PROGRESS=False,
                     SP_FAST_SIMS=4, SP_FULL_FRACTION=0.25, SP_WRITE_PACKED=True).items():
        monkeypatch.setattr(sp, k, v)
    runs = []
    real_run = sp._run

    def run(*a, **k):
        out = real_run(*a, **k)
        runs.append(out[1])
        return out
    monkeypatch.setattr(sp, "_run", run)
    for corrected in (False, True):
        monkeypatch.setattr(sp, "CORRECTED_LABELS", corrected)
        f = sp.self_play()
        h = runs[-1]
        with open(f, "rb") as fh:
            rows = pickle.load(fh)
        mask = h.sample_mask(n)
        assert np.array_equal(mask, _rows(h, n) & engine.full_moves(5, 0, n, 0.25))
        st = sp.last_stats
        assert len(rows) == mask.sum() == st["full_plies"] > 0 and st["fast_plies"] > 0
        assert st["full_plies"] + st["fast_plies"] == st["plies"] == h.lens[:n].sum()
        g, p = np.nonzero(mask)
        xs = engine.game_encode(torch.from_numpy(h.states[:n][mask].view(np.int32)).cuda()).cpu().numpy()
        assert all(np.array_equal(rows[i][0], xs[i]) for i in range(len(rows)))
        cn = h.counts[:n][mask].astype(np.float64)
        assert np.allclose(np.stack([r[1] for r in rows]), cn / cn.sum(1, keepdims=True), atol=1e-6)
        zf = np.where(h.final[g] != 0, -1, 0)
        want = np.where((h.lens[g] - p) % 2 == 0, zf, -zf) if corrected else zf * np.where(p % 2 == 0, 1, -1)
        assert [r[2] for r in rows] == want.tolist()
        xs2, _, _ = sp.load_packed_history(f.replace(".history", ".packed.npz"))
        assert len(xs2) == mask.sum()
    x, pol, val = sp.history_tensors(DualNetwork().to("cuda").eval(), n)
    assert x.shape[0] == runs[-1].sample_mask(n).sum() == sp.last_stats["full_plies"]
