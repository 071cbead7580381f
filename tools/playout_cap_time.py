"""Wall-clock effect of playout cap randomization (UTTT_SP_PLAYOUT_CAP) on device self-play.

  a  500 games x 50 simulations, reference-exact search with the correct terminal sign, bf16 and bf16x3:
     every move a full search ("flat") against the cap (fast_sims 8, full fraction 0.25)
  b  4096 games x 200 simulations, throughput mode, batch 8, bf16: flat against the cap (32, 0.25)

Per configuration one engine with as many slots as games; after one warm-up run of each arm the flat and capped runs
alternate, 3 of each, all with the same seed.  One JSON line per timed run: wall ms (Engine.selfplay_device, ended by a
device synchronise), games/s, plies/s, full samples/s (the plies that would become training samples), the non-empty
tensor-core trunk launches and the mean evaluator batch over them (uttt_debug_batch_histogram), and the card's name and
power limit read in the same process.  The weights are DualNetwork's random initialisation (seed 0); game lengths, and so
the numbers, would differ on a trained network, and training strength is not measured here.

python tools/playout_cap_time.py [--configs a,b] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
import engine  # noqa: E402
from dual_network import DualNetwork  # noqa: E402
from match_time import gpu_info  # noqa: E402

SEED = 0x5EED
REPEATS = 3
CONFIGS = {
    "a": [dict(games=500, sims=50, batch=8, search="compat+correct_sign", numerics=nm, flags=engine.SP_CORRECT_TERMINAL_SIGN,
               fast_sims=8, full_fraction=0.25) for nm in ("bf16", "bf16x3")],
    "b": [dict(games=4096, sims=200, batch=8, search="throughput", numerics="bf16", flags=engine.SP_THROUGHPUT,
               fast_sims=32, full_fraction=0.25)],
}


def timed_run(e, cfg, capped):
    n = cfg["games"]
    flags = cfg["flags"] | (engine.SP_PLAYOUT_CAP if capped else 0)
    e.batch_histogram(reset=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    stats = e.selfplay_device(n, sims=cfg["sims"], batch=cfg["batch"], seed=SEED,
                              evaluator=engine.evaluator_of(cfg["numerics"]), flags=flags)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    h = e.selfplay_fetch(n)
    full = int(h.sample_mask(n).sum())
    launches = int(e.batch_histogram(reset=True).sum())
    plies, evals = int(stats[0]), int(stats[2])
    return {"arm": "cap" if capped else "flat", "ms": ms, "games_per_s": n / ms * 1e3, "plies": plies,
            "plies_per_s": plies / ms * 1e3, "full_samples": full, "full_samples_per_s": full / ms * 1e3,
            "sims": int(stats[1]), "evals": evals, "rounds": int(stats[3]), "trunk_launches": launches,
            "mean_batch": evals / launches if launches else 0.0}


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
        for cfg in CONFIGS[name]:
            n = cfg["games"]
            e = engine.Engine(n_slots=n, max_sims=cfg["sims"], max_batch=cfg["batch"], max_games=n)
            try:
                e.upload_model(model)
                e.set_playout_cap(cfg["fast_sims"], cfg["full_fraction"])
                timed_run(e, cfg, False)                                   # warm-up, both arms
                timed_run(e, cfg, True)
                for rep in range(REPEATS):
                    for capped in (False, True):
                        rec = dict(config=name, games=n, sims=cfg["sims"], batch=cfg["batch"], search=cfg["search"],
                                   numerics=cfg["numerics"], fast_sims=cfg["fast_sims"] if capped else None,
                                   full_fraction=cfg["full_fraction"] if capped else None, rep=rep,
                                   weights="random-init (seed 0)")
                        rec.update(timed_run(e, cfg, capped))
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
