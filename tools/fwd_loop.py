"""time back-to-back network forwards: python tools/fwd_loop.py n [reps] [bf16|bf16x3|fp32]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, engine, oracle_lib as O
from dual_network import DualNetwork
n = int(sys.argv[1]); reps = int(sys.argv[2]) if len(sys.argv) > 2 else 200
numerics = sys.argv[3] if len(sys.argv) > 3 else "bf16"
MODE = engine.evaluator_of(numerics)
torch.manual_seed(0)
e = engine.Engine(n_slots=max(n, int(os.environ.get("FWD_SLOTS", "8"))), max_sims=50, max_batch=8, max_games=8)
e.upload_model(DualNetwork().eval())
sts = np.concatenate([O.playout_states(1, g)[0][:-1] for g in range(n // 40 + 2)])[:n]
d = torch.from_numpy(sts.view(np.int32)).cuda()
for _ in range(5):
    e.net_forward(d, MODE)
torch.cuda.synchronize()
t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
t0.record()
for _ in range(reps):
    e.net_forward(d, MODE)
t1.record(); torch.cuda.synchronize()
us = 1e3 * t0.elapsed_time(t1) / reps
print("n=%d  %s  %.1f us per forward = %.0f TFLOP/s useful (gather + trunk + heads + 2 copies)" % (
    n, numerics, us, n * 764411904 / us / 1e6))
