"""CPU: the point rule of a device match (engine.match_points), the argument checks that need no device, the
EN_DEVICE_MATCH switch, and the register budgets of the tree-search kernels that route leaves to two networks."""
import importlib
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200", "csrc")


def _lib():
    from test_abi_cpu import _lib_or_skip
    return _lib_or_skip()


class _Hist:
    def __init__(self, lens, final):
        self.lens = np.asarray(lens, np.int32)
        self.final = np.asarray(final, np.int8)


def test_match_points_rule():
    import engine
    # game g, plies n: the last mover is slot (g + n - 1) & 1; final == 0 is a draw
    h = _Hist([10, 10, 11, 11, 30, 81], [1, 1, 1, 1, 0, 0])
    assert engine.match_points(h, 0).tolist() == [0.0, 1.0, 1.0, 0.0, 0.5, 0.5]
    assert engine.match_points(h, 1).tolist() == [1.0, 0.0, 0.0, 1.0, 0.5, 0.5]
    assert engine.match_points(h, 2).tolist() == engine.match_points(h, 0).tolist()


def test_match_points_agree_with_a_replay_of_random_games():
    """random playouts stand in for match games: the rule on (len, is_lose of the end) == first_player_point of the
    reference's evaluate_network.py:26-30 with the colours alternating by game (evaluate_network.py:80-85)"""
    _lib()
    import engine
    import uttt_cpp
    for game0 in (0, 7):
        lens, final, want = [], [], []
        for g in range(40):
            _, acts = O.playout_states(99, g)
            s = uttt_cpp.State()
            for a in acts:
                s = s.next(int(a))
            assert s.is_done()
            lens.append(len(acts))
            final.append(1 if s.is_lose() else 0)
            fp = (0 if s.is_first_player() else 1) if s.is_lose() else 0.5
            want.append(fp if (game0 + g) % 2 == 0 else 1 - fp)
        assert engine.match_points(_Hist(lens, final), game0).tolist() == want
        assert 0.0 in want and 1.0 in want


def test_weight_slot_must_be_0_or_1():
    import engine
    lib = _lib()
    w = engine.UtttWeights()
    for slot in (-1, 2):
        assert lib.uttt_upload_weights_slot(None, slot, w, 0) != 0 and b"slot" in lib.uttt_last_error()
        assert lib.uttt_upload_weights_scattered_slot(None, slot, engine.UtttWeightsScattered(), 0) != 0
        assert b"slot" in lib.uttt_last_error()
    e = object.__new__(engine.Engine)                # (no device here: the slot is checked before the engine is used)
    with pytest.raises(ValueError):
        e.upload_state_dict({}, slot=2)


def test_device_match_switch(monkeypatch):
    _lib()
    import evaluate_network as en
    try:
        monkeypatch.delenv("UTTT_DEVICE_MATCH", raising=False)
        assert importlib.reload(en).EN_DEVICE_MATCH is False
        monkeypatch.setenv("UTTT_DEVICE_MATCH", "1")
        assert importlib.reload(en).EN_DEVICE_MATCH is True
        monkeypatch.setenv("UTTT_DEVICE_MATCH", "0")
        assert importlib.reload(en).EN_DEVICE_MATCH is False
        with pytest.raises(ValueError):
            en.device_match(None, None, 4, 1, search="lua")
    finally:
        monkeypatch.delenv("UTTT_DEVICE_MATCH", raising=False)
        importlib.reload(en)


def _ptxas(src, kernel):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not shutil.which(nvcc):
        pytest.skip("nvcc not available")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--ptxas-options=-v",
                          "-c", os.path.join(CSRC, src), "-o", os.devnull], capture_output=True, text=True, check=True)
    log = out.stdout + out.stderr
    m = re.search(r"Compiling entry function '\w*%s\w*'.*?(\d+) bytes spill stores, (\d+) bytes spill loads.*?Used (\d+) registers"
                  % kernel, log, re.S)
    assert m, log
    return int(m.group(1)), int(m.group(2)), int(m.group(3))


def test_tree_round_kernels_keep_their_register_budgets():
    """the net selection of UTTT_SP_MATCH spills nothing in either tree-round kernel, and tree_round_kernel keeps 7
    blocks of 128 threads per SM (at most 65536 / (7 * 128) = 73 registers)"""
    st, ld, regs = _ptxas("tree_kernels.cu", "tree_round_kernel")
    assert st == 0 and ld == 0 and regs <= 73, (st, ld, regs)
    st, ld, regs = _ptxas("tree_tp_kernels.cu", "tree_tp_round_kernel")
    assert st == 0 and ld == 0 and regs <= 102, (st, ld, regs)
