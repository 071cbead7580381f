"""Wall-clock effect of forced playouts and policy target pruning (UTTT_SP_FORCED_PLAYOUTS) on device self-play.

  a  500 games x 50 simulations, throughput mode, batch 8, bf16, k = 2
  b  4096 games x 200 simulations, throughput mode, batch 8, bf16, k = 2

Per configuration one engine with as many slots as games and the default root noise (alpha 0.3, eps 0.25); after one
warm-up run of each arm the runs without ("off") and with the flag ("on") alternate, 3 of each, all with the same seed.
One JSON line per timed run: wall ms (Engine.selfplay_device, ended by a device synchronise), plies/s, the non-empty
tensor-core trunk launches and the mean evaluator batch over them (uttt_debug_batch_histogram), the share of the sample
plies' visits that pruning removed from the policy targets, and the card's name and power limit read in the same
process.  A forced child can end a round's leaf collection early (the descent reaches a leaf already queued), so the
mean batch is the number to watch.  The weights are DualNetwork's random initialisation (seed 0); the numbers would differ
on a trained network, and training strength is not measured here.

python tools/forced_playouts_time.py [--configs a,b] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
import engine  # noqa: E402
from dual_network import DualNetwork  # noqa: E402
from match_time import gpu_info  # noqa: E402

SEED = 0x5EED
REPEATS = 3
K = 2.0
CONFIGS = {
    "a": dict(games=500, sims=50, batch=8, numerics="bf16"),
    "b": dict(games=4096, sims=200, batch=8, numerics="bf16"),
}


def timed_run(e, cfg, forced):
    n = cfg["games"]
    flags = engine.SP_THROUGHPUT | (engine.SP_FORCED_PLAYOUTS if forced else 0)
    e.batch_histogram(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    stats = e.selfplay_device(n, sims=cfg["sims"], batch=cfg["batch"], seed=SEED,
                              evaluator=engine.evaluator_of(cfg["numerics"]), flags=flags)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    h = e.selfplay_fetch(n)
    mask = h.sample_mask(n)
    visits = int(h.counts[:n][mask].astype(np.int64).sum())
    kept = int(h.targets()[:n][mask].astype(np.int64).sum())
    launches = int(e.batch_histogram(reset=True).sum())
    plies, evals = int(stats[0]), int(stats[2])
    return {"arm": "on" if forced else "off", "ms": ms, "plies": plies, "plies_per_s": plies / ms * 1e3,
            "simulations": int(stats[1]), "evals": evals, "rounds": int(stats[3]), "trunk_launches": launches,
            "mean_batch": evals / launches if launches else 0.0, "pruned_fraction": (visits - kept) / visits if visits else 0.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="a,b")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    torch.manual_seed(0)
    model = DualNetwork().eval()
    lines = []
    for name in args.configs.split(","):
        cfg = CONFIGS[name]
        n = cfg["games"]
        e = engine.Engine(n_slots=n, max_sims=cfg["sims"], max_batch=cfg["batch"], max_games=n)
        try:
            e.upload_model(model)
            e.set_forced_playouts(K)
            timed_run(e, cfg, False)                                   # warm-up, both arms
            timed_run(e, cfg, True)
            for rep in range(REPEATS):
                for forced in (False, True):
                    rec = dict(config=name, games=n, sims=cfg["sims"], batch=cfg["batch"], search="throughput",
                               numerics=cfg["numerics"], k=K if forced else None, rep=rep, weights="random-init (seed 0)")
                    rec.update(timed_run(e, cfg, forced))
                    rec.update(info)
                    line = json.dumps(rec)
                    print(line, flush=True)
                    lines.append(line)
        finally:
            e.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
