"""Trainer drop-in (SURVEY 8f-2): ultimate-tictactoe-alphazero_b200/train_network.py on a fixed history file, best.pth
and torch seed must give the weights and epoch lines in tests/golden/trainer.npz, bit for bit, on the CPU (the batch
order is the DataLoader's, reproduced from the global RNG).  `python oracle/gen_golden.py --trainer DIR` records that
file from DIR/train_network.py on the same inputs -- from the reference's trainer wherever its checkout is at hand --
and stores in `source` whose trainer it ran."""
import hashlib
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "trainer.npz")


def _synthetic_history(n, seed=7):
    rng = np.random.RandomState(seed)
    hist = []
    for _ in range(n):
        x = (rng.rand(9, 9, 3) < 0.3).astype(np.float32)
        pi = rng.rand(81) * (rng.rand(81) < 0.2)
        pi[rng.randint(81)] += 0.5
        pi = pi / pi.sum()                                   # float64, sums to 1 over a sparse support
        hist.append([x, pi, int(rng.randint(-1, 2))])
    return hist


def _run(tmp, module_dir, tag):
    code = ("import sys; sys.path.insert(0, %r); import torch; torch.set_num_threads(4); import train_network as t; "
            "t.RN_EPOCHS = 2; torch.manual_seed(123); t.train_network()" % module_dir)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, "-c", code], cwd=tmp, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    sd = torch.load(os.path.join(tmp, "model", "latest.pth"), weights_only=True)
    os.rename(os.path.join(tmp, "model", "latest.pth"), os.path.join(tmp, "model", "latest_%s.pth" % tag))
    return sd, [l for l in out.stdout.splitlines() if l.startswith("Epoch")]


def run_recorded_case(tmp, module_dir=PKG):
    """2 epochs of module_dir's train_network() on 200 synthetic samples (2 batches per epoch: 128 + 72, ragged) from a
    seed-0 best.pth, in the scratch directory tmp"""
    sys.path.insert(0, PKG)
    from dual_network import DualNetwork
    os.makedirs(os.path.join(tmp, "data")); os.makedirs(os.path.join(tmp, "model"))
    with open(os.path.join(tmp, "data", "20260101000000.history"), "wb") as f:
        pickle.dump(_synthetic_history(200), f)
    torch.manual_seed(0)
    torch.save(DualNetwork().state_dict(), os.path.join(tmp, "model", "best.pth"))
    return _run(tmp, module_dir, "ours")


def digests(sd):
    return [hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() for v in sd.values()]


def test_trainer_reproduces_recorded_weights_bit_for_bit(tmp_path):
    tmp = str(tmp_path)
    our_sd, our_log = run_recorded_case(tmp)
    with np.load(GOLDEN) as g:
        g = {k: g[k] for k in g.files}
    names, want_digests, log = g["names"].tolist(), g["sha256"].tolist(), g["epoch_lines"].tolist()
    assert our_log == log and len(log) == 2, (log, our_log)
    assert list(our_sd.keys()) == names
    best = torch.load(os.path.join(tmp, "model", "best.pth"), weights_only=True)
    assert not torch.equal(best["conv_input.weight"], our_sd["conv_input.weight"])        # it did train
    for i, (k, got, want) in enumerate(zip(names, digests(our_sd), want_digests)):
        vals = our_sd[k].reshape(-1)[torch.from_numpy(g["sample_idx"][i])].double().numpy()
        assert got == want, "%s: max |difference| %.3e at the recorded sample positions (recorded from %s)" % (
            k, np.abs(vals - g["sample_val"][i]).max(), g["source"])


def test_epoch_order_is_the_dataloader_order():
    """the shuffle protocol alone, against a live DataLoader (no reference needed)"""
    sys.path.insert(0, PKG)
    import train_network as t
    from torch.utils.data import DataLoader, TensorDataset
    n = 1000
    ds = TensorDataset(torch.arange(n))
    torch.manual_seed(99)
    seen = [torch.cat([b[0] for b in DataLoader(ds, batch_size=128, shuffle=True)]) for _ in range(3)]
    after_ref = torch.rand(1)
    torch.manual_seed(99)
    ours = [t._loader_epoch_order(n) for _ in range(3)]
    after_ours = torch.rand(1)
    assert all(torch.equal(a, b) for a, b in zip(seen, ours)) and torch.equal(after_ref, after_ours)


def test_train_tensors_learns_and_follows_the_schedule():
    sys.path.insert(0, PKG)
    import train_network as t
    assert [t.lr_lambda(e) for e in (0, 49, 50, 79, 80, 99)] == [1.0, 1.0, 0.5, 0.5, 0.25, 0.25]
    xs, ps, vs = t.history_to_tensors(_synthetic_history(64), torch.device("cpu"))
    assert xs.shape == (64, 3, 9, 9) and ps.shape == (64, 81) and vs.shape == (64, 1) and xs.dtype == torch.float32
    torch.manual_seed(1)
    # a tiny stand-in with the DualNetwork output contract keeps this test fast

    class Tiny(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.p = torch.nn.Linear(243, 81); self.v = torch.nn.Linear(243, 1)

        def forward(self, x):
            x = x.flatten(1)
            return torch.softmax(self.p(x), 1), torch.tanh(self.v(x))
    model = Tiny()
    lines = []
    losses = t.train_tensors(model, xs, ps, vs, epochs=6, batch_size=16, bf16=False, log=lines.append)
    assert len(losses) == 6 and losses[-1] < losses[0] and lines[0].startswith("Epoch 1/6, Loss: ")
