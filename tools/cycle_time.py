"""Device time of the 500-game cycle (BASELINE config 3) at a given per-kernel event level: python tools/cycle_time.py [level] [steps] [numerics]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
import torch  # noqa: E402
import engine  # noqa: E402
from dual_network import DualNetwork  # noqa: E402

level = int(sys.argv[1]) if len(sys.argv) > 1 else 0
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
ev = engine.evaluator_of(sys.argv[3] if len(sys.argv) > 3 else "bf16")
games = int(os.environ.get("GAMES", "500"))
torch.manual_seed(0)
e = engine.Engine(n_slots=min(games, 4096), max_sims=50, max_batch=8, max_games=games)
e.upload_model(DualNetwork().eval())
e.set_profile_level(level)
s = torch.cuda.current_stream()
for i in range(3):
    e.selfplay_device(games, seed=0x5EED, evaluator=ev, game0=(1000 + i) * games, stream=s)
ms, plies = [], 0
for i in range(steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    st = e.selfplay_device(games, seed=0x5EED, evaluator=ev, game0=i * games, stream=s)
    e1.record(s)
    e1.synchronize()
    ms.append(e0.elapsed_time(e1))
    plies += int(st[0])
prof = e.last_run_profile()
print("level=%d games=%d: %.2f ms/cycle (min %.2f), %.0f moves/s, rounds %d, trunk %.2f ms" % (
    level, games, sum(ms) / len(ms), min(ms), plies / (sum(ms) / 1e3), int(st[3]), prof["trunk"][0]))
e.close()
