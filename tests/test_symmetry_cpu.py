"""CPU: the board symmetries of UTTT_SP_RANDOM_SYMMETRY (uttt_state_symmetry, the host face of sym_state / sym_action in
csrc/uttt_rules.cuh) against the restatement on the oracle's arrays, the numpy picture transforms, the rules and the
group structure -- over the golden positions and random playouts."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
import symmetry_lib as S


@pytest.fixture(scope="module")
def positions(golden_dir):
    with np.load(os.path.join(golden_dir, "rules.npz")) as z:
        golden = z["states"]
    played = np.concatenate([O.playout_states(7171, g)[0] for g in range(12)])
    return np.ascontiguousarray(np.concatenate([golden, played]), dtype=np.uint32)


def _encode(w):
    import engine
    out = np.zeros(243, np.float32)
    assert engine.load_library().uttt_state_encode(np.ascontiguousarray(w, np.uint32), out) == 0
    return out.reshape(9, 9, 3)


def _legal(w):
    import engine
    out = np.zeros(81, np.int32)
    n = C.c_int()
    assert engine.load_library().uttt_state_legal_actions(np.ascontiguousarray(w, np.uint32), out, C.byref(n)) == 0
    return out[:n.value].copy()


def _next(w, a):
    import engine
    out = np.zeros(8, np.uint32)
    assert engine.load_library().uttt_state_next(np.ascontiguousarray(w, np.uint32), int(a), out) == 0
    return out


def _flags(w):
    import engine
    f = C.c_int()
    assert engine.load_library().uttt_state_flags(np.ascontiguousarray(w, np.uint32), C.byref(f)) == 0
    return f.value


def _picture(x, g):
    """symmetry g of an (9, 9, ...) picture: transpose if g >= 4, then numpy.rot90 by g % 4"""
    if g >= 4:
        x = np.swapaxes(x, 0, 1)
    return np.rot90(x, k=g % 4, axes=(0, 1))


def test_engine_agrees_with_the_array_restatement(positions):
    import engine
    assert len(positions) > 1732
    for g in range(8):
        amap = S.action_map(g)
        for w in positions:
            out, am = engine.state_symmetry(w, g)
            assert (out == S.symmetry(w, g)).all(), (g, w)
            assert (am == amap).all(), g


def test_planes_of_the_image_are_the_transformed_picture(positions):
    import engine
    for g in range(8):
        for w in positions[::3]:
            assert (_encode(engine.state_symmetry(w, g)[0]) == _picture(_encode(w), g)).all(), (g, w)


def test_rules_commute_with_every_symmetry(positions):
    import engine
    for g in range(8):
        for w in positions[::2]:
            gw, amap = engine.state_symmetry(w, g)
            legal = _legal(w)
            assert (_legal(gw) == np.sort(amap[legal])).all(), (g, w)
            assert _flags(gw) == _flags(w)
            for a in legal:
                assert (_next(gw, amap[a]) == engine.state_symmetry(_next(w, a), g)[0]).all(), (g, w, a)


def test_the_eight_maps_form_the_dihedral_group(positions):
    import engine
    maps = [engine.state_symmetry(positions[0], g)[1] for g in range(8)]
    assert (maps[0] == np.arange(81)).all()
    assert len({m.tobytes() for m in maps}) == 8 and all(sorted(m) == list(range(81)) for m in maps)
    # the action map of g is the picture transform: the cell of action a moves to the cell of sigma_g(a)
    R, Cc = np.divmod(np.arange(81), 9)
    act_of_cell = ((R // 3) * 3 + Cc // 3) * 9 + (R % 3) * 3 + Cc % 3            # picture cell -> action
    for g in range(8):
        ids = np.zeros((9, 9), np.int64)
        ids.reshape(-1)[:] = act_of_cell
        moved = _picture(ids, g).reshape(-1)            # action now at each picture cell
        want = np.zeros(81, np.int64)
        want[moved] = act_of_cell
        assert (maps[g] == want).all(), g
    # composition table: sigma_g after sigma_h is sigma_k with k the product in the group of picture transforms
    index = {m.tobytes(): g for g, m in enumerate(maps)}
    probe = np.arange(81).reshape(9, 9)
    for g in range(8):
        for h in range(8):
            k = index[maps[g][maps[h]].tobytes()]
            assert (_picture(_picture(probe, h), g) == _picture(probe, k)).all(), (g, h, k)
        inv = [h for h in range(8) if (maps[g][maps[h]] == np.arange(81)).all()]
        assert len(inv) == 1
        for w in positions[::50]:
            assert (engine.state_symmetry(engine.state_symmetry(w, g)[0], inv[0])[0] == w).all()


def test_rejects_out_of_range_symmetry():
    import engine
    with pytest.raises(RuntimeError, match="symmetry"):
        engine.state_symmetry(np.zeros(8, np.uint32), 8)


def test_symmetry_draw_is_the_documented_philox_word():
    out = np.zeros(4, np.uint32)
    for seed, game, ply, j in ((0, 0, 0, 0), (11, 499, 37, 12), (2025, 1 << 33, 80, 400)):
        O.oracle().orc_philox4x32(seed, 2, game & 0xFFFFFFFF, game >> 32, ply, j, out)
        assert S.draw(seed, game, ply, j) == out[0] >> 29
