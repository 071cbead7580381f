"""Drop-in replacement for the reference's self_play_cpp.py: `play(model)`, `self_play()` and the
module constants keep their names, defaults, printed progress line and output format
(./data/YYYYMMDDHHMMSS.history = pickle of [[x (9,9,3) f32, pi (81,) f64, z int], ...]), but the
SP_GAME_COUNT games of a cycle run CONCURRENTLY on the GPU inside one C-ABI call
(uttt_selfplay_run): trees, leaves, network forward, sampling and the history all stay in HBM.

Differences that cannot be avoided: moves are sampled with the engine's counter-based Philox
stream (seeded from numpy's global RNG, so np.random.seed still makes a run reproducible) instead
of np.random.choice (self_play_cpp.py:86).  Labelling follows self_play_cpp.py:95-99 verbatim
unless CORRECTED_LABELS is set (SURVEY.md B3).
"""
import os
import pickle
from datetime import datetime

import numpy as np
import torch

import engine as _eng
import uttt_cpp  # noqa: F401  (fails loudly when the CUDA library is missing)
from dual_network import DualNetwork, device

CPP_AVAILABLE = True
print("Using B200 CUDA backend for MCTS")

SP_GAME_COUNT = 500       # self_play_cpp.py:26
SP_TEMPERATURE = 1.0      # self_play_cpp.py:27
PV_EVALUATE_COUNT = 50    # self_play_cpp.py:30
MCTS_BATCH_SIZE = 8       # self_play_cpp.py:31

# knobs that do not exist in the reference (defaults reproduce it)
SP_NUMERICS = _eng.DEFAULT_NUMERICS   # "bf16x3" (split-bf16 tcgen05 trunk: within 1e-2 of the fp32 reference forward on
                              # any weights), "bf16" (plain bf16 operands: 3x faster, within 1e-2 on trained weights) or
                              # "fp32" (CUDA cores)
SP_PROGRESS = True            # print the reference's per-game progress line (self_play_cpp.py:121) as games finish
SP_MAX_SLOTS = 4096           # concurrent games per GPU
SP_SEED = None                # None: draw from np.random
CORRECTED_LABELS = False      # True: label from the true winner instead of self_play_cpp.py:95-99
CORRECTED_TERMINAL_SIGN = False
SP_SEARCH_MODE = "compat"     # "compat": reference-exact search; "throughput": AlphaZero-standard search
                              #   (evaluated root + Dirichlet noise, virtual loss, MCTS_BATCH_SIZE leaves / round)
SP_DIRICHLET_ALPHA = 0.3      # throughput mode only
SP_DIRICHLET_EPS = 0.25
SP_RANDOM_SYMMETRY = False    # evaluate every leaf under a random board symmetry, policy mapped back (AlphaGo Zero)
SP_WRITE_PACKED = False       # also write ./data/<timestamp>.packed.npz (357 B/sample instead of ~1.7 KB; SURVEY 8f-3)
SP_RESIGN_THRESHOLD = None    # a float: a mover resigns when its root value is below it (AlphaGo Zero; engine.SP_RESIGN).
                              # Needs CORRECTED_TERMINAL_SIGN = True or SP_SEARCH_MODE = "throughput"
SP_RESIGN_CHECK_FRACTION = 0.1    # fraction of games never resigned, to measure the false positives
SP_RESIGN_TARGET_FP = None    # a float: after each cycle SP_RESIGN_THRESHOLD becomes the largest threshold whose false-positive
                              # rate on that cycle's played-out games (the check games; all games while resignation is off)
                              # is at most this (engine.resign_threshold)

_engine = None
last_stats = {}


def _get_engine(n_games):
    global _engine
    slots = min(max(n_games, 1), SP_MAX_SLOTS)
    if (_engine is None or _engine.n_slots < slots or _engine.max_games < n_games
            or _engine.max_sims < PV_EVALUATE_COUNT or _engine.max_batch < MCTS_BATCH_SIZE):
        if _engine is not None:
            _engine.close()
        _engine = _eng.Engine(n_slots=slots, max_sims=PV_EVALUATE_COUNT, max_batch=MCTS_BATCH_SIZE,
                              max_games=n_games)
    return _engine


def _history_arrays(eng, hist):
    """packed History -> (xs (N,9,9,3) f32, pis (N,81) f64, zs (N,) int) in game-major order"""
    st, cn, z = hist.samples()
    n = st.shape[0]
    dev = torch.device("cuda", eng.device)
    st_d = torch.from_numpy(st.view(np.int32)).to(dev)
    xs = _eng.game_encode(st_d).cpu().numpy()                         # cpp/uttt_game.cpp:244-280 on device
    legal = xs.reshape(n, 81, 3)[:, :, 2] > 0                          # by picture cell
    # action id of picture cell (R,C): cpp/uttt_game.cpp:256-257
    R, Ccol = np.divmod(np.arange(81), 9)
    act_of_cell = ((R // 3) * 3 + (Ccol // 3)) * 9 + (R % 3) * 3 + (Ccol % 3)
    legal_by_action = np.zeros((n, 81), bool)
    legal_by_action[:, act_of_cell] = legal
    # scores over the legal actions: float32 n/sum (cpp/uttt_mcts.cpp:199-216, T=1) -> float64 renormalised
    # with numpy's own summation over exactly the legal entries (self_play_cpp.py:74-78), grouped by L
    sc32 = _scores_from_counts(cn)
    pis = np.zeros((n, 81), np.float64)
    L = legal_by_action.sum(axis=1)
    for l in np.unique(L):
        rows = np.nonzero(L == l)[0]
        cols = np.nonzero(legal_by_action[rows])[1].reshape(len(rows), l)
        s64 = np.ascontiguousarray(sc32[rows[:, None], cols].astype(np.float64))
        s64 = s64 / np.sum(s64, axis=1)[:, None]
        pis[rows[:, None], cols] = s64
    if CORRECTED_LABELS:
        z = _corrected_labels(hist)
    return xs, pis, z.astype(np.int64)


def _scores_from_counts(cn):
    """what pv_mcts_scores returns for these root visit counts at SP_TEMPERATURE (cpp/uttt_mcts.cpp:177-216): fp32
    n / sum at T = 1, one-hot at the first maximum at T = 0, n^(1/T) / sum otherwise (zeros stay zeros)"""
    x = cn.astype(np.float32)
    if SP_TEMPERATURE == 0:
        out = np.zeros_like(x)
        out[np.arange(len(x)), x.argmax(axis=1)] = 1.0
        return out
    if SP_TEMPERATURE != 1.0:
        x = np.power(x, np.float32(1.0) / np.float32(SP_TEMPERATURE), dtype=np.float32)
    return x / x.sum(axis=1, dtype=np.float32)[:, None]


def _corrected_labels(hist):
    """value from each mover's own perspective (the labelling of the reference's self_play.py:21-25,96)"""
    lens = hist.lens.astype(np.int64)
    mask = np.arange(81)[None, :] < lens[:, None]
    # the final position's mover lost iff final != 0; ply t has the same mover as the final position
    # iff (len - t) is even
    par = ((lens[:, None] - np.arange(81)[None, :]) % 2) == 0
    zf = np.where(hist.final != 0, -1, 0)[:, None]
    return np.where(par, zf, -zf)[mask].astype(np.int8)


def _to_reference_format(xs, pis, zs):
    return [[xs[i], pis[i], int(zs[i])] for i in range(len(zs))]


def _resign_flags():
    """engine.SP_RESIGN if SP_RESIGN_THRESHOLD is set, else 0; ValueError if resignation is asked for (a threshold or a
    calibration target) under the reference's terminal sign, where a move that wins at once backs up as a loss"""
    if SP_RESIGN_THRESHOLD is None and SP_RESIGN_TARGET_FP is None:
        return 0
    if not (CORRECTED_TERMINAL_SIGN or SP_SEARCH_MODE == "throughput"):
        raise ValueError("resignation needs root values with the correct terminal sign: set CORRECTED_TERMINAL_SIGN = True "
                         "or SP_SEARCH_MODE = \"throughput\"")
    return _eng.SP_RESIGN if SP_RESIGN_THRESHOLD is not None else 0


def _resign_stats(hist, n_games, seed, resign):
    """resigned games and the false positives of the played-out calibration games (the check games while resigning, all
    games otherwise); with SP_RESIGN_TARGET_FP, the threshold calibrated on them becomes SP_RESIGN_THRESHOLD"""
    global SP_RESIGN_THRESHOLD
    calib = (_eng.check_games(seed, 0, n_games, SP_RESIGN_CHECK_FRACTION) if resign
             else np.ones(n_games, bool))
    out = {"resigned": int((hist.resigned[:n_games] != 0).sum()), "check_games": int(calib.sum()) if resign else 0}
    if resign:
        cal = _eng.resign_calibration(hist, SP_RESIGN_THRESHOLD, calib)
        out.update(check_would_resign=cal["would_resign"], check_false_positives=cal["false_positives"])
    if SP_RESIGN_TARGET_FP is not None:
        SP_RESIGN_THRESHOLD = _eng.resign_threshold(hist, SP_RESIGN_TARGET_FP, calib)
        out["calibrated_threshold"] = SP_RESIGN_THRESHOLD
    return out


def _run(model, n_games, progress=False):
    resign = _resign_flags()
    eng = _get_engine(n_games)
    model.eval()
    eng.upload_model(model)
    seed = int(np.random.randint(0, 2 ** 31 - 1)) if SP_SEED is None else int(SP_SEED)
    ev = _eng.evaluator_of(SP_NUMERICS)
    flags = _eng.SP_CORRECT_TERMINAL_SIGN if CORRECTED_TERMINAL_SIGN else 0
    if SP_SEARCH_MODE == "throughput":
        flags |= _eng.SP_THROUGHPUT
        eng.set_root_noise(SP_DIRICHLET_ALPHA, SP_DIRICHLET_EPS)
    if SP_RANDOM_SYMMETRY:
        flags |= _eng.SP_RANDOM_SYMMETRY
    if resign:
        flags |= resign
        eng.set_resign(SP_RESIGN_THRESHOLD, SP_RESIGN_CHECK_FRACTION)
    eng.set_selfplay_temperature(SP_TEMPERATURE)
    if SP_PROGRESS and progress:
        shown = [0]

        def progress(done, total):         # self_play_cpp.py:121, one line per finished game
            for i in range(shown[0], done):
                print(f"\rSelfPlay {i + 1}/{total} (Backend: C++)", end="")
            shown[0] = done
        eng.set_progress_callback(progress)
    try:
        hist = eng.selfplay(n_games, sims=PV_EVALUATE_COUNT, batch=MCTS_BATCH_SIZE, seed=seed, evaluator=ev, flags=flags)
    finally:
        eng.set_progress_callback(None)
        eng.set_selfplay_temperature(1.0)
    last_stats.update(plies=int(hist.stats[0]), sims=int(hist.stats[1]), evals=int(hist.stats[2]),
                      rounds=int(hist.stats[3]), seed=seed)
    for k in ("check_would_resign", "check_false_positives", "calibrated_threshold"):     # only what this cycle reports
        last_stats.pop(k, None)
    last_stats.update(_resign_stats(hist, n_games, seed, bool(resign)))
    return eng, hist


def history_tensors(model, n_games=None):
    """Trainer feed without the pickle round trip (SURVEY 8f-2): runs a self-play cycle and returns CUDA tensors
    in exactly the layout train_network.py:30-60 builds from the .history file:
    xs (N,3,9,9) float32, policies (N,81) float32, values (N,1) float32."""
    n_games = SP_GAME_COUNT if n_games is None else n_games
    eng, hist = _run(model, n_games)
    xs, pis, zs = _history_arrays(eng, hist)
    dev = torch.device("cuda", eng.device)
    x = torch.from_numpy(xs).to(dev).permute(0, 3, 1, 2).contiguous()
    return x, torch.from_numpy(pis.astype(np.float32)).to(dev), torch.from_numpy(zs.astype(np.float32)).to(dev).unsqueeze(1)


def play(model, use_cpp=True):
    """self_play_cpp.py:34-101: one game -> [[x, pi, z], ...]"""
    eng, hist = _run(model, 1)
    return _to_reference_format(*_history_arrays(eng, hist))


def self_play(use_cpp=True):
    """self_play_cpp.py:104-130: SP_GAME_COUNT games -> ./data/<timestamp>.history"""
    model = DualNetwork().to(device)
    model.load_state_dict(torch.load("./model/best.pth", map_location=device, weights_only=True))
    model.eval()
    eng, hist = _run(model, SP_GAME_COUNT, progress=True)
    history = _to_reference_format(*_history_arrays(eng, hist))
    print("")
    now = datetime.now()
    file_name = "./data/{:04}{:02}{:02}{:02}{:02}{:02}.history".format(
        now.year, now.month, now.day, now.hour, now.minute, now.second)
    os.makedirs("./data", exist_ok=True)
    with open(file_name, mode="wb") as f:
        pickle.dump(history, f)
    if SP_WRITE_PACKED:
        save_packed_history(file_name.replace(".history", ".packed.npz"), hist)
    return file_name


def save_packed_history(path, hist):
    """packed sidecar of a cycle: per sample the 32-byte position, the 81 visit counts and the label"""
    st, cn, z = hist.samples()
    np.savez_compressed(path, states=st, counts=cn, z=z, lens=hist.lens.copy(), final=hist.final.copy())


def load_packed_history(path, device_index=0):
    """-> (xs (N,3,9,9) f32, policies (N,81) f32, values (N,) f32) numpy arrays, i.e. what train_network.py:41-60
    derives from the .history pickle (x planes are re-encoded on the GPU from the packed positions)"""
    with np.load(path) as z:
        st, cn, zz = z["states"], z["counts"], z["z"]
    dev = torch.device("cuda", device_index)
    xs = _eng.game_encode(torch.from_numpy(st.view(np.int32)).to(dev)).permute(0, 3, 1, 2).contiguous().cpu().numpy()
    tot = cn.sum(axis=1, keepdims=True).astype(np.float32)
    return xs, cn.astype(np.float32) / tot, zz.astype(np.float32)


if __name__ == "__main__":
    from pv_mcts_cpp import check_cpp_compatibility
    check_cpp_compatibility()
    self_play()
