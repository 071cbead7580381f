"""Cost of UTTT_SP_RANDOM_SYMMETRY on the 500-game / 50-simulation self-play cycle (BASELINE config 3):
python tools/symmetry_cost.py [runs] [numerics ...]

For each numerics, runs with the flag off and on alternate (`runs` of each, after a warm-up of both).  Every run is timed
twice: end to end with CUDA events at profile level 0 (moves/s), then once more at profile level 2 for the tree-kernel
and trunk ms of uttt_last_run_profile (the per-kernel events of level 2 slow the cycle down, so its moves/s are not used)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
import torch  # noqa: E402
import engine  # noqa: E402
from dual_network import DualNetwork  # noqa: E402

GAMES, SIMS, BATCH = 500, 50, 8


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def cycle(e, ev, flags, game0):
    s = torch.cuda.current_stream()
    e.set_profile_level(0)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(s)
    st = e.selfplay_device(GAMES, sims=SIMS, batch=BATCH, seed=0x5EED, evaluator=ev, flags=flags, game0=game0, stream=s)
    t1.record(s)
    t1.synchronize()
    ms = t0.elapsed_time(t1)
    e.set_profile_level(2)
    e.selfplay_device(GAMES, sims=SIMS, batch=BATCH, seed=0x5EED, evaluator=ev, flags=flags, game0=game0, stream=s)
    torch.cuda.synchronize()
    prof = e.last_run_profile()
    return int(st[0]) / (ms / 1e3), ms, prof["tree"][0], prof["trunk"][0]


def main():
    runs = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    numerics = sys.argv[2:] or ["bf16", "bf16x3"]
    print("card: %s" % card())
    torch.manual_seed(0)
    e = engine.Engine(n_slots=GAMES, max_sims=SIMS, max_batch=BATCH, max_games=GAMES)
    e.upload_model(DualNetwork().eval())
    for name in numerics:
        ev = engine.evaluator_of(name)
        res = {0: [], engine.SP_RANDOM_SYMMETRY: []}
        for flags in res:
            cycle(e, ev, flags, 10 ** 6)                                    # warm-up
        for r in range(runs):
            for flags in res:
                res[flags].append(cycle(e, ev, flags, r * GAMES))
        for flags, rows in res.items():
            for mps, ms, tree, trunk in rows:
                print("%-6s symmetry=%s: %9.0f moves/s  cycle %7.2f ms | level 2: tree kernels %7.2f ms, trunk %7.2f ms" % (
                    name, "on " if flags else "off", mps, ms, tree, trunk))
        off, on = [sum(x[i] for x in res[0]) / runs for i in range(4)], [sum(x[i] for x in res[engine.SP_RANDOM_SYMMETRY]) / runs for i in range(4)]
        spread = max(x[0] for x in res[0]) / min(x[0] for x in res[0]) - 1
        print("%-6s mean moves/s off %.0f, on %.0f (%+.2f %%; run-to-run spread off %.2f %%); tree ms off %.2f on %.2f; trunk ms off %.2f on %.2f" % (
            name, off[0], on[0], 100 * (on[0] / off[0] - 1), 100 * spread, off[2], on[2], off[3], on[3]))
    e.close()


if __name__ == "__main__":
    main()
