"""CPU: the C-ABI library loads and exports every symbol include/uttt_b200.h declares (no device
compute), and the host-side `uttt_cpp.State` shim matches the oracle / the reference goldens."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib_or_skip():
    import engine
    if not os.path.exists(engine.LIB_PATH):
        import importlib.util
        spec = importlib.util.spec_from_file_location("uttt_build", os.path.join(os.path.dirname(engine.__file__), "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    return engine.load_library()


def test_header_symbols_exported():
    import engine
    lib = _lib_or_skip()
    hdr = open(os.path.join(ROOT, "include", "uttt_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(uttt_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    for name in sorted(declared):
        assert hasattr(lib, name), "libuttt_b200.so does not export %s" % name
    assert declared == set(engine.ABI.keys()), declared ^ set(engine.ABI.keys())
    assert lib.uttt_abi_version() == 1


def test_no_device_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import engine
    lib = _lib_or_skip()
    assert lib.uttt_device_check(0) != 0
    assert b"no CPU fallback" in lib.uttt_last_error()
    with pytest.raises(RuntimeError):
        engine.Engine(n_slots=4, max_sims=10, max_batch=2, max_games=4, device=0)


def test_state_shim_matches_reference_goldens(golden_dir):
    _lib_or_skip()
    import uttt_cpp
    with np.load(os.path.join(golden_dir, "rules.npz")) as z:
        g = {k: z[k] for k in z.files}
    for i in range(0, len(g["states"]), 3):
        s = uttt_cpp.State._from_packed(g["states"][i])
        f = g["flags"][i]
        assert (s.is_lose(), s.is_draw(), s.is_done(), s.is_first_player()) == (bool(f & 1), bool(f & 2), bool(f & 4), bool(f & 8))
        n = g["n_legal"][i]
        legal = s.legal_actions()
        assert legal == g["legal"][i, :n].tolist()
        assert s.to_input_tensor() == g["tensor"][i].astype(np.float32).tolist()
        assert str(s) == str(g["strings"][i]) == s.to_string()
        for k, a in enumerate(legal):
            assert (s.next(a).packed() == g["next"][i, k]).all()
        # 5-argument constructor + read-only properties round trip (cpp/python_bindings.cpp:54-74)
        s2 = uttt_cpp.State(s.pieces, s.enemy_pieces, s.main_board_pieces, s.main_board_enemy_pieces, s.active_board)
        assert (s2.packed() == s.packed()).all()
    for w, a, ref in zip(g["ill_states"], g["ill_actions"], g["ill_next"]):
        assert (uttt_cpp.State._from_packed(w).next(int(a)).packed() == ref).all()


def test_state_shim_random_playouts_vs_oracle():
    _lib_or_skip()
    import uttt_cpp
    for game in range(20):
        sts, acts = O.playout_states(4242, game)
        s = uttt_cpp.State()
        for t, a in enumerate(acts):
            assert (s.packed() == sts[t]).all()
            flags, legal, tens = O.oracle_probe(sts[t])
            assert s.legal_actions() == legal.tolist()
            s = s.next(int(a))
        assert s.is_done() and (s.packed() == sts[-1]).all()


def test_state_shim_errors():
    _lib_or_skip()
    import uttt_cpp
    s = uttt_cpp.State()
    with pytest.raises(RuntimeError):
        s.next(81)
    with pytest.raises(ValueError):
        uttt_cpp.State([[2] * 9] * 9, [[0] * 9] * 9, [0] * 9, [0] * 9, -1)
    assert s.active_board == -1 and s.main_board_pieces == [0] * 9 and len(s.pieces) == 9


def test_dual_network_state_dict_layout():
    import torch
    from dual_network import DualNetwork
    import engine
    torch.manual_seed(0)
    m = DualNetwork()
    sd = m.state_dict()
    assert len(sd) == 216                                    # SURVEY 8(b)
    assert sum(p.numel() for p in m.parameters()) == 4765338
    assert sd["conv_input.weight"].shape == (128, 3, 3, 3)
    assert sd["residual_blocks.15.conv2.weight"].shape == (128, 128, 3, 3)
    assert sd["policy_fc.weight"].shape == (81, 162) and sd["value_fc1.weight"].shape == (256, 81)
    packed = engine.pack_state_dict(sd)
    assert packed["res_conv_w"].shape == (16, 2, 128, 128, 3, 3)
    assert np.array_equal(packed["res_conv_w"][3, 1], sd["residual_blocks.3.conv2.weight"].numpy())
    assert np.array_equal(packed["res_bn"][5, 0, 3], sd["residual_blocks.5.bn1.running_var"].numpy())
    p, v = m.eval()(torch.zeros(2, 3, 9, 9))
    assert p.shape == (2, 81) and v.shape == (2, 1)
    assert torch.allclose(p.sum(1), torch.ones(2), atol=1e-5)


def test_history_labels_follow_reference_rule():
    import engine
    h = engine.History(3, pinned=False)
    h.lens[:] = [3, 4, 2]
    h.final[:] = [1, 1, 0]
    h.counts[:] = 0
    st, cn, z = h.samples()
    assert len(z) == 9
    # self_play_cpp.py:95-99: z0 = -1 if final.is_lose() else 0, alternating from ply 0
    assert z.tolist() == [-1, 1, -1, -1, 1, -1, 1, 0, 0]


def test_dual_network_reproduces_reference_golden_outputs(golden_dir):
    """same seed -> same weights and same fp32 outputs as the reference's own DualNetwork (tests/golden/network.npz,
    generated by importing /root/reference/dual_network.py in oracle/gen_golden.py)"""
    import torch
    from dual_network import DualNetwork
    with np.load(os.path.join(golden_dir, "network.npz")) as z:
        g = {k: z[k] for k in z.files}
    torch.manual_seed(0)
    m = DualNetwork().eval()
    sd = m.state_dict()
    assert len(sd) == int(g["n_entries"]) and sum(t.numel() for t in m.parameters()) == int(g["n_params"])
    assert abs(float(sum(t.double().abs().sum() for t in sd.values())) - float(g["weight_abs_sum"])) < 1e-6
    planes = np.stack([O.oracle_probe(w)[2] for w in g["states"]]).reshape(-1, 9, 9, 3)
    x = torch.from_numpy(planes).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        p, v = m(x)
    assert np.abs(p.numpy() - g["policy"]).max() < 1e-5 and np.abs(v.numpy()[:, 0] - g["value"]).max() < 1e-5


def test_reference_train_cycle_imports_resolve_against_the_package(golden_dir):
    """the reference's driver (train_cycle.py:6-18) imports by module name; with the package directory first on sys.path
    every module / name it asks for must exist there (checked on the syntax trees: importing uttt_cpp needs the GPU
    library).  The import list is tests/golden/train_cycle_imports.json; the GPU test test_train_cycle_iteration runs the
    package's own driver."""
    import ast
    import json
    with open(os.path.join(golden_dir, "train_cycle_imports.json")) as f:
        wanted = [tuple(x) for x in json.load(f)["imports"]]
    pkg = os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200")
    assert ("self_play_cpp", "self_play") in wanted and ("uttt_cpp", None) in wanted
    for mod, name in wanted:
        if mod == "self_play_hybrid":
            continue                                   # the reference's fallback when uttt_cpp is missing: never taken here
        path = os.path.join(pkg, mod + ".py")
        assert os.path.exists(path), "package has no module %s" % mod
        if name is not None:
            tree = ast.parse(open(path).read())
            defined = {n.name for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef))}
            defined |= {t.id for n in tree.body if isinstance(n, ast.Assign) for t in n.targets if isinstance(t, ast.Name)}
            assert name in defined, "%s.%s missing" % (mod, name)
