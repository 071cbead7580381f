#!/usr/bin/env python
"""Generate tests/golden/*.npz from the COMPILED REFERENCE (oracle/_ref).  TEST INFRASTRUCTURE.

Run in the build container (where /root/reference exists):
    make -C oracle ref && python oracle/gen_golden.py
Every array below is an output of the reference's own UTTT::State / UTTT::pv_mcts_scores
(cpp/uttt_game.cpp, cpp/uttt_mcts.cpp) driven through oracle/ref_harness.cpp with
deterministic inputs (Philox playouts, integer-hash evaluator).  The vectors pin
oracle/uttt_oracle.c (CPU tests) and the CUDA library (GPU tests).

Two generators read the reference's Python files instead, from the directory given on the command line, and record that
directory's name as `source`:
    python oracle/gen_golden.py --trainer DIR               -> trainer.npz: DIR/train_network.py on the inputs of
                                                               tests/test_train_cpu.py
    python oracle/gen_golden.py --train-cycle-imports DIR   -> train_cycle_imports.json: the import block of DIR/train_cycle.py
"""
import ast
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SEED = 0x5EED


def custom_states():
    """Hand-built positions only reachable through the 5-argument constructor (Q-G3 etc.)."""
    L = O.oracle()
    out = []
    # forced board that is already finished -> falls back to "any open board"
    for game in range(64):
        sts, _ = O.playout_states(99, game)
        for w in sts[10::7]:
            s = O.state_from_packed(w)
            for b in range(9):
                if s.main_pieces[b] or s.main_enemy[b]:
                    s2 = O.OrcState.from_buffer_copy(s)
                    s2.active = b
                    out.append(O.packed_from_state(s2))
                    break
    # every sub-board drawn / empty main flags with stones etc.
    s = O.OrcState()
    L.orc_init(C.byref(s))
    s.active = 4
    out.append(O.packed_from_state(s))
    for b in range(9):
        s.main_pieces[b] = 1
        s.main_enemy[b] = 1
    s.active = -1
    out.append(O.packed_from_state(s))
    return np.stack(out)


def gen_rules():
    R = O.ref()
    n = 4096
    dg = np.zeros(n, np.uint64); pl = np.zeros(n, np.int32); rs = np.zeros(n, np.int32)
    R.ref_playouts(SEED, 0, n, dg, pl, rs)
    # full-size (config 2) checksums: 2^20 playouts
    N = 1 << 20
    xor = np.uint64(0); tot = np.uint64(0); plies = 0; hist = np.zeros(3, np.int64)
    chunk = 1 << 16
    d = np.zeros(chunk, np.uint64); p = np.zeros(chunk, np.int32); r = np.zeros(chunk, np.int32)
    for g0 in range(0, N, chunk):
        R.ref_playouts(SEED, g0, chunk, d, p, r)
        xor ^= np.bitwise_xor.reduce(d)
        tot = np.uint64((int(tot) + int(d.astype(object).sum())) & 0xFFFFFFFFFFFFFFFF)
        plies += int(p.sum())
        hist += np.bincount(r, minlength=3)
    # per-state probes
    states = []
    for game in range(48):
        sts, _ = O.playout_states(SEED + 1, game)
        states.append(sts[::2])
    states = np.concatenate(states + [custom_states()])
    ns = len(states)
    flags = np.zeros(ns, np.int32); nleg = np.zeros(ns, np.int32)
    legal = np.full((ns, 81), -1, np.int32); tens = np.zeros((ns, 243), np.float32)
    nxt = np.zeros((ns, 81, 8), np.uint32)
    strs = []
    for i, w in enumerate(states):
        f, n_ = C.c_int(), C.c_int()
        lg = np.zeros(81, np.int32)
        R.ref_state_probe(w, C.byref(f), C.byref(n_), lg, tens[i])
        flags[i] = f.value; nleg[i] = n_.value; legal[i, :n_.value] = lg[:n_.value]
        for k in range(n_.value):
            R.ref_state_next(w, int(lg[k]), nxt[i, k])
        buf = C.create_string_buffer(2048)
        R.ref_state_to_string(w, buf, 2048)
        strs.append(buf.value.decode())
    # next() does no legality check (Q-G5): a few illegal/occupied actions too
    ill_states = states[5:200:13]
    ill_actions = np.array([(7 * i + 3) % 81 for i in range(len(ill_states))], np.int32)
    ill_next = np.zeros((len(ill_states), 8), np.uint32)
    for i, w in enumerate(ill_states):
        R.ref_state_next(w, int(ill_actions[i]), ill_next[i])
    np.savez_compressed(
        os.path.join(OUT, "rules.npz"), seed=np.uint32(SEED), digests=dg, plies=pl, results=rs,
        full_n=np.int64(N), full_xor=np.uint64(xor), full_sum=np.uint64(tot),
        full_plies=np.int64(plies), full_hist=hist,
        states=states, flags=flags, n_legal=nleg, legal=legal.astype(np.int8),
        tensor=tens.astype(np.uint8), next=nxt, strings=np.array(strs),
        ill_states=ill_states, ill_actions=ill_actions, ill_next=ill_next)
    print("rules.npz:", ns, "states;", N, "playouts: xor=%016x sum=%016x plies=%d hist=%s"
          % (int(xor), int(tot), plies, hist))


def gen_mcts():
    R = O.ref()
    states = []
    for game in range(24):
        sts, _ = O.playout_states(SEED + 2, game)
        states.append(sts[:-1:4])          # non-terminal, spread over the game
        states.append(sts[-3:])            # late positions incl. the terminal one
    states = np.concatenate(states + [custom_states()[:6]])
    configs = [(50, 8), (50, 1), (10, 2), (37, 5), (200, 8), (800, 8)]
    rows = []
    scores = []
    for si, w in enumerate(states):
        for ci, (sims, batch) in enumerate(configs):
            if sims == 800 and si % 8:
                continue
            for T in (1.0, 0.0, 0.5):
                if T == 0.5 and (si % 4 or sims > 50):
                    continue
                sc, st = O.ref_mcts(w, T, sims, batch)
                row = np.zeros(81, np.float32)
                row[:len(sc)] = sc
                rows.append((si, sims, batch, T, len(sc), st[0], st[1]))
                scores.append(row)
    rows = np.array(rows, dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "mcts.npz"), states=states, cases=rows,
                        scores=np.stack(scores).view(np.uint32))
    print("mcts.npz:", len(states), "states,", len(rows), "cases")


def gen_selfplay():
    R = O.ref()
    games = []
    for game, (sims, batch) in enumerate([(50, 8), (50, 8), (50, 8), (50, 8), (20, 4), (50, 1)]):
        st = np.zeros((81, 8), np.uint32); cn = np.zeros((81, 81), np.uint16)
        ac = np.zeros(81, np.uint8); z = np.zeros(81, np.int8)
        n = R.ref_selfplay_hash(SEED, game, sims, batch, st, cn, ac, z)
        games.append((game, sims, batch, n, st[:n].copy(), cn[:n].copy(), ac[:n].copy(), z[:n].copy()))
    np.savez_compressed(
        os.path.join(OUT, "selfplay.npz"), seed=np.uint32(SEED),
        meta=np.array([(g, s, b, n) for g, s, b, n, *_ in games], np.int32),
        states=np.concatenate([g[4] for g in games]), counts=np.concatenate([g[5] for g in games]),
        actions=np.concatenate([g[6] for g in games]), z=np.concatenate([g[7] for g in games]))
    print("selfplay.npz:", [(g[0], g[3]) for g in games])


def gen_boltzman():
    R = O.ref()
    rng = np.random.RandomState(0)
    xs = rng.randint(0, 50, size=(32, 16)).astype(np.float32)
    out = {}
    for T in (1.0, 0.5, 2.0):
        o = np.zeros_like(xs)
        for i in range(len(xs)):
            R.ref_boltzman(xs[i], xs.shape[1], T, o[i])
        out["T%g" % T] = o
    np.savez_compressed(os.path.join(OUT, "boltzman.npz"), xs=xs, **out)


def gen_network():
    """fp32 outputs of the REFERENCE DualNetwork (dual_network.py, imported from /root/reference) with its own
    random init under torch.manual_seed(0), on positions from Philox playouts (planes from the reference State)."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("ref_dual_network", "/root/reference/dual_network.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    torch.manual_seed(0)
    model = ref.DualNetwork().eval()
    R = O.ref()
    states = np.concatenate([O.playout_states(SEED + 3, g)[0][:-1:3] for g in range(10)])[:160]
    planes = np.zeros((len(states), 243), np.float32)
    for i, w in enumerate(states):
        f, n_ = C.c_int(), C.c_int()
        R.ref_state_probe(w, C.byref(f), C.byref(n_), np.zeros(81, np.int32), planes[i])
    x = torch.from_numpy(planes.reshape(-1, 9, 9, 3)).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        p, v = model(x)
    sd = model.state_dict()
    digest = float(sum(t.double().abs().sum() for t in sd.values()))
    np.savez_compressed(os.path.join(OUT, "network.npz"), states=states, policy=p.numpy(), value=v.numpy()[:, 0],
                        n_params=np.int64(sum(t.numel() for t in model.parameters())), n_entries=np.int64(len(sd)),
                        weight_abs_sum=np.float64(digest), torch_version=np.array(torch.__version__))
    print("network.npz:", len(states), "positions; params", sum(t.numel() for t in model.parameters()))


def gen_pymcts():
    """Scores of the REFERENCE's pure-Python search -- /root/reference/pv_mcts.py:74-180, the one its gating match uses
    (evaluate_network.py:73-75) -- imported and run unmodified under the integer-hash evaluator.  `model` is a stand-in
    whose forward returns the hash policy / value of the states the reference code is about to evaluate (recorded by
    wrapping pv_mcts.state_to_input_tensor, which predict_batch calls once per state, pv_mcts.py:24); everything else --
    predict_batch's legal-move renormalisation with np.sum, the tree, PUCT, the queue / flush loop, boltzman -- is the
    reference's own code under this container's NumPy (the version is stored with the vectors)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))      # the reference's own pybind module (self_play_cpp imports it)
    sys.path.insert(0, "/root/reference")
    import pv_mcts as ref_pv                                       # noqa: E402  (prints the device line)
    import game as ref_game
    seen = []
    real_tensor = ref_pv.state_to_input_tensor

    def recording_tensor(state):
        seen.append(state)
        return real_tensor(state)
    ref_pv.state_to_input_tensor = recording_tensor

    class HashModel:
        def eval(self):
            return self

        def __call__(self, x):
            n = x.shape[0]
            states = seen[-n:]
            pol = np.zeros((n, 81), np.float32)
            val = np.zeros((n, 1), np.float32)
            for i, st in enumerate(states):
                o = O.OrcState()
                for b_ in range(9):
                    for c_ in range(9):
                        o.pieces[9 * b_ + c_] = st.pieces[b_][c_]
                        o.enemy[9 * b_ + c_] = st.enemy_pieces[b_][c_]
                    o.main_pieces[b_] = st.main_board_pieces[b_]
                    o.main_enemy[b_] = st.main_board_enemy_pieces[b_]
                o.active = st.active_board
                v = C.c_float()
                O.oracle().orc_hash_eval(C.byref(o), pol[i], C.byref(v))
                val[i, 0] = v.value
            del seen[:]
            return torch.from_numpy(pol), torch.from_numpy(val)

    def py_state(w):
        o = O.state_from_packed(w)
        return ref_game.State([[o.pieces[9 * b_ + c_] for c_ in range(9)] for b_ in range(9)],
                              [[o.enemy[9 * b_ + c_] for c_ in range(9)] for b_ in range(9)],
                              list(o.main_pieces), list(o.main_enemy), o.active)
    states = np.concatenate([O.playout_states(SEED + 4, g)[0][:-1:5] for g in range(20)])
    model = HashModel()
    cases, scores = [], []
    for si, w in enumerate(states):
        for sims, batch in ((50, 8), (50, 1), (10, 2), (37, 5), (200, 8)):
            if sims == 200 and si % 4:
                continue
            ref_pv.PV_EVALUATE_COUNT, ref_pv.MCTS_BATCH_SIZE = sims, batch
            for T in (1.0, 0.0, 0.5):
                if T == 0.5 and si % 3:
                    continue
                sc = np.asarray(ref_pv.pv_mcts_scores(model, py_state(w), T), dtype=np.float64)
                row = np.zeros(81, np.float64)
                row[:len(sc)] = sc
                cases.append((si, sims, batch, T, len(sc)))
                scores.append(row)
    np.savez_compressed(os.path.join(OUT, "pymcts.npz"), states=states, cases=np.array(cases, np.float64),
                        scores=np.stack(scores).view(np.uint64), numpy_version=np.array(np.__version__))
    print("pymcts.npz:", len(states), "states,", len(cases), "cases (numpy %s)" % np.__version__)


def gen_trainer(ref_dir):
    """weights and epoch lines of DIR/train_network.py on tests/test_train_cpu.py's inputs (2 epochs of 200 synthetic
    samples from a seed-0 best.pth, torch seed 123, 4 threads, on the CPU): a SHA-256 per state_dict tensor, plus the
    values at 8 seeded positions of each tensor so that a mismatch shows its size"""
    import tempfile
    import torch
    import test_train_cpu as T
    with tempfile.TemporaryDirectory() as d:
        sd, lines = T.run_recorded_case(d, os.path.abspath(ref_dir))
    rng = np.random.RandomState(0)
    idx = np.stack([rng.randint(0, v.numel(), 8) for v in sd.values()])
    vals = np.stack([v.reshape(-1)[torch.from_numpy(i)].double().numpy() for v, i in zip(sd.values(), idx)])
    np.savez_compressed(os.path.join(OUT, "trainer.npz"), names=np.array(list(sd.keys())), sha256=np.array(T.digests(sd)),
                        sample_idx=idx, sample_val=vals, epoch_lines=np.array(lines), torch_version=np.array(torch.__version__),
                        source=np.array("train_network.py of " + os.path.basename(os.path.abspath(ref_dir))))
    print("trainer.npz:", lines)


def gen_train_cycle_imports(ref_dir):
    """(module, name) of every import in DIR/train_cycle.py (name None for `import module`)"""
    wanted = []
    for node in ast.walk(ast.parse(open(os.path.join(ref_dir, "train_cycle.py"), encoding="utf-8-sig").read())):
        if isinstance(node, ast.ImportFrom):
            wanted += [[node.module, a.name] for a in node.names]
        elif isinstance(node, ast.Import):
            wanted += [[a.name, None] for a in node.names]
    with open(os.path.join(OUT, "train_cycle_imports.json"), "w") as f:
        json.dump({"source": "train_cycle.py of " + os.path.basename(os.path.abspath(ref_dir)), "imports": wanted}, f, indent=1)
    print("train_cycle_imports.json:", wanted)


if __name__ == "__main__":
    if "--trainer" in sys.argv:
        gen_trainer(sys.argv[sys.argv.index("--trainer") + 1])
        sys.exit(0)
    if "--train-cycle-imports" in sys.argv:
        gen_train_cycle_imports(sys.argv[sys.argv.index("--train-cycle-imports") + 1])
        sys.exit(0)
    if not O.ref_available():
        sys.exit("oracle/_ref is not built: run `make -C oracle ref` where /root/reference exists")
    os.makedirs(OUT, exist_ok=True)
    if "--pymcts-only" in sys.argv:
        gen_pymcts()
        sys.exit(0)
    gen_rules()
    gen_mcts()
    gen_selfplay()
    gen_boltzman()
    gen_network()
    gen_pymcts()
