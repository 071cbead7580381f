"""Wall-clock cost and effect of resignation (UTTT_SP_RESIGN) in self-play -- mechanism numbers on random-init weights.

  a  500 games x 50 simulations, reference-exact search with the correct terminal sign, bf16 and bf16x3
  b  1024 games x 200 simulations, throughput mode, bf16

each with resignation off and at thresholds -0.95, -0.8 and -0.5 (check fraction 0.1), the same seed throughout, so a
resigning run's games are the off-run's cut short.  Every case is timed after one warm-up run of its own; one JSON line
per case: ms (Engine.selfplay, history copy included), plies, resigned games, check games, and the check games'
would-be resignations and false positives under the case's threshold (the off-run: over all its games).  The weights are
DualNetwork's random initialisation (seed 0): the values of an untrained network say nothing about what resignation
saves in training, so these numbers show the mechanism and its cost only.

python tools/resign_time.py [--configs a,b] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import engine  # noqa: E402
from dual_network import DualNetwork  # noqa: E402
from match_time import gpu_info  # noqa: E402

SEED = 0x5EED
THRESHOLDS = (None, -0.95, -0.8, -0.5)
CHECK_FRACTION = 0.1
CONFIGS = {
    "a": [dict(games=500, sims=50, batch=8, search="compat+correct_sign", numerics=nm, flags=engine.SP_CORRECT_TERMINAL_SIGN)
          for nm in ("bf16", "bf16x3")],
    "b": [dict(games=1024, sims=200, batch=8, search="throughput", numerics="bf16", flags=engine.SP_THROUGHPUT)],
}


def case(model, cfg, thr):
    n = cfg["games"]
    e = engine.Engine(n_slots=n, max_sims=cfg["sims"], max_batch=cfg["batch"], max_games=n)
    try:
        e.upload_model(model)
        flags = cfg["flags"]
        if thr is not None:
            flags |= engine.SP_RESIGN
            e.set_resign(thr, CHECK_FRACTION)

        def run(seed):
            return e.selfplay(n, sims=cfg["sims"], batch=cfg["batch"], seed=seed, evaluator=engine.evaluator_of(cfg["numerics"]),
                              flags=flags)
        run(SEED + 1)                                                   # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h = run(SEED)
        ms = (time.perf_counter() - t0) * 1e3
    finally:
        e.close()
    chk = engine.check_games(SEED, 0, n, CHECK_FRACTION) if thr is not None else np.ones(n, bool)
    out = {"ms": ms, "plies": int(h.stats[0]), "resigned": int(h.resigned.sum()),
           "check_games": int(chk.sum()) if thr is not None else 0}
    for t in ([thr] if thr is not None else [x for x in THRESHOLDS if x is not None]):
        cal = engine.resign_calibration(h, t, chk)
        key = "" if thr is not None else "_at_%g" % t
        out["calib_would_resign" + key] = cal["would_resign"]
        out["calib_false_positives" + key] = cal["false_positives"]
    return out


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
            for thr in THRESHOLDS:
                rec = dict(config=name, games=cfg["games"], sims=cfg["sims"], search=cfg["search"], numerics=cfg["numerics"],
                           threshold=thr, check_fraction=CHECK_FRACTION if thr is not None else None,
                           weights="random-init (seed 0): mechanism numbers, not a training saving")
                rec.update(case(model, cfg, thr))
                rec.update(info)
                line = json.dumps(rec)
                print(line, flush=True)
                lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
