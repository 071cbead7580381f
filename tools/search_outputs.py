"""Compare the search and self-play outputs of two builds bit for bit.

  python tools/search_outputs.py dump OUT.npz [TREE]    search and self-play outputs of the library built in TREE (a
                                                       checkout; default: this one)
  python tools/search_outputs.py compare A.npz B.npz   exit status 1 unless every array is bit-identical

Batched search under the hash evaluator in every mode (reference-exact at batch 1 and 8, the Python semantics, the
throughput mode with 1, 4, 8 and 16 leaves per round with and without root noise), each with and without the random board
symmetry, plus the corrected terminal sign; the step-wise search with a host evaluator, one row per leaf and one per
copy; self-play in both search modes at temperatures 1, 0 and 0.5 with the hash evaluator and a seeded random-init bf16
network, and one run of 1100 games, enough slots for two lanes.  Positions, seeds and the model are fixed.
"""
import ctypes as C
import os
import sys

import numpy as np

from forward_rows import compare

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dump(out, tree):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    sys.path.insert(0, os.path.join(os.path.abspath(tree), "ultimate-tictactoe-alphazero_b200"))
    import torch
    import engine
    import oracle_lib as O
    from dual_network import DualNetwork

    arrays = {}

    def put(kind, name, **outs):
        if "n" in outs:        # a root without legal moves leaves its counts row unwritten
            outs["counts"] = np.where(np.arange(81)[None, :] < outs["n"][:, None], outs["counts"], 0)
        for k, v in outs.items():
            arrays["%s_%d_%s_%s" % (kind, len(arrays), name, k)] = np.asarray(v)

    # positions along seeded playouts; the reference-exact searches also get 30 finished ones (empty results)
    sts = np.concatenate([O.playout_states(4242, g)[0] for g in range(40)])
    live = np.array([len(O.oracle_probe(s)[1]) > 0 for s in sts])
    roots = np.concatenate([sts[live][::2][:270], sts[~live][:30]])

    e = engine.Engine(n_slots=1100, max_sims=200, max_batch=16, max_games=1100)
    SYM, TP = engine.SP_RANDOM_SYMMETRY, engine.SP_THROUGHPUT
    for sym in (0, SYM):
        runs = [("ref-b1", 1, 0), ("ref-b8", 8, 0), ("py-b8", 8, engine.SP_PYSEARCH)]
        runs += [("tp-m%d" % m, m, TP) for m in (1, 4, 8, 16)]
        for name, batch, flags in runs:
            for eps in ((0.0, 0.25) if flags == TP else (0.25,)):
                e.set_root_noise(0.3, eps)
                sc, cn, ns = e.mcts_search(roots[:270] if flags == TP else roots, 100, batch, 1.0, engine.EVAL_HASH,
                                           flags=flags | sym)
                put("search", "%s-eps%g-sym%d" % (name, eps, sym > 0), scores=sc.view(np.uint32), counts=cn, n=ns)
    e.set_root_noise(0.3, 0.25)
    sc, cn, ns = e.mcts_search(roots, 100, 8, 1.0, engine.EVAL_HASH, flags=engine.SP_CORRECT_TERMINAL_SIGN)
    put("search", "ref-b8-correct-sign", scores=sc.view(np.uint32), counts=cn, n=ns)

    L = O.oracle()

    def host_eval(per_copy):
        def fn(states, k):
            pol = np.zeros((len(states), 81), np.float32)
            val = np.zeros(len(states), np.float32)
            v = C.c_float()
            for i, s in enumerate(states):
                L.orc_hash_eval(C.byref(O.state_from_packed(s)), pol[i], C.byref(v))
                val[i] = v.value
            if not per_copy:
                return pol, val
            scale = np.float32(1) + np.arange(e.max_batch, dtype=np.float32) / np.float32(16)
            return pol[:, None, :] * scale[None, :, None], val[:, None] / scale[None, :]
        return fn
    for per_copy in (False, True):
        sc, cn, ns = e.mcts_search_host(roots[::6], 50, 8, 1.0, host_eval(per_copy), per_copy=per_copy)
        put("host", "per-copy%d" % per_copy, scores=sc.view(np.uint32), counts=cn, n=ns)

    torch.manual_seed(0)
    e.upload_model(DualNetwork().eval())
    for evaluator, ename in ((engine.EVAL_HASH, "hash"), (engine.EVAL_NET_BF16, "bf16")):
        for flags, fname in ((0, "ref"), (TP, "tp")):
            for T in (1.0, 0.0, 0.5):
                e.set_selfplay_temperature(T)
                h = e.selfplay(64, sims=50, batch=8, seed=11, evaluator=evaluator, flags=flags, game0=300)
                put("selfplay", "%s-%s-T%g" % (ename, fname, T), lens=h.lens, states=h.states, counts=h.counts,
                    actions=h.actions, final=h.final, stats=h.stats)
    e.set_selfplay_temperature(1.0)
    for flags, fname in ((0, "ref"), (TP, "tp")):
        h = e.selfplay(1100, sims=20, batch=8, seed=12, evaluator=engine.EVAL_NET_BF16, flags=flags)
        put("selfplay", "bf16-%s-1100" % fname, lens=h.lens, states=h.states, counts=h.counts, actions=h.actions,
            final=h.final, stats=h.stats)
    e.close()
    np.savez(out, **arrays)
    print("%s: %d arrays from %s" % (out, len(arrays), engine.LIB_PATH))


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "dump":
        dump(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else ROOT)
    elif len(sys.argv) == 4 and sys.argv[1] == "compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    else:
        sys.exit(__doc__)
