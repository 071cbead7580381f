"""Drop-in for the reference's evaluate_network.py (gating match, SURVEY 8f-1): same names, constants,
printed lines and promotion rule (evaluate_network.py:22-23,62-104), but the EN_GAME_COUNT games are played
CONCURRENTLY: at every ply all positions in which the same network is to move are searched as one batch on the
GPU (uttt_mcts_search), so a 50-game match costs ~160 batched searches instead of ~2,900 sequential ones.

Search semantics: the reference's gating match calls the pure-Python pv_mcts.pv_mcts_action (evaluate_network.py:73-75),
whose search differs from the C++ one used for self-play (evaluated root, replaced child lists, np.sum renormalisation,
float64 scores; pv_mcts.py:74-180).  EN_SEARCH = "python" (default) runs exactly that search on the engine
(UTTT_SP_PYSEARCH; pinned bit-exactly against the unmodified pv_mcts.py by tests/golden/pymcts.npz); EN_SEARCH = "cpp"
selects the C++ semantics (cpp/uttt_mcts.cpp:84-196) instead.

EN_DEVICE_MATCH (environment UTTT_DEVICE_MATCH=1; off by default) plays the whole match inside one engine instead
(device_match): both networks' games live on the device as in self-play, see evaluate_network().
"""
import os
from shutil import copy

import numpy as np
import torch

import engine as _eng
import uttt_cpp  # noqa: F401
from dual_network import DualNetwork, device

EN_GAME_COUNT = 50        # evaluate_network.py:22
EN_TEMPERATURE = 1.0      # evaluate_network.py:23
PV_EVALUATE_COUNT = 50    # pv_mcts.py:16
MCTS_BATCH_SIZE = 8       # pv_mcts.py:17
EN_SEED = None            # None: derived from numpy's global RNG
EN_SEARCH = "python"      # "python": pv_mcts.py semantics (what the reference's gating match runs); "cpp": uttt_mcts.cpp semantics
EN_NUMERICS = _eng.DEFAULT_NUMERICS    # "bf16x3" | "bf16" | "fp32" (engine.evaluator_of)
EN_RANDOM_SYMMETRY = False             # evaluate every leaf under a random board symmetry, policy mapped back (AlphaGo Zero)
EN_DEVICE_MATCH = os.environ.get("UTTT_DEVICE_MATCH") == "1"    # play the match on the device (device_match)


def first_player_point(ended_state):
    """evaluate_network.py:26-30: 1 first player won, 0 lost, 0.5 draw"""
    if ended_state.is_lose():
        return 0 if ended_state.is_first_player() else 1
    return 0.5


def python_scores(counts, temperature):
    """pv_mcts.py:166-180 on the root visit counts: one-hot at np.argmax for T == 0, else boltzman in Python floats"""
    if temperature == 0:
        scores = np.zeros(len(counts))
        scores[int(np.argmax(counts))] = 1
        return scores
    xs = [int(x) ** (1 / temperature) for x in counts]
    total = sum(xs)
    return np.array([x / total for x in xs])


def pv_mcts_scores_batch(engine, roots, temperature, evaluator, search=None, evaluate_count=None, batch_size=None):
    """the gating match's search for many positions at once -> (scores (n,81) in legal order, n_legal (n,)); float64
    probabilities with the Python semantics, float32 scores with the C++ ones"""
    search = EN_SEARCH if search is None else search
    sims = PV_EVALUATE_COUNT if evaluate_count is None else evaluate_count
    batch = MCTS_BATCH_SIZE if batch_size is None else batch_size
    sym = _eng.SP_RANDOM_SYMMETRY if EN_RANDOM_SYMMETRY else 0
    if search == "cpp":
        sc, _, ns = engine.mcts_search(roots, sims, batch, temperature, evaluator, flags=sym)
        return sc, ns                  # float32, renormalised in float64 by the caller (pv_mcts_cpp.py:129-133)
    if search != "python":
        raise ValueError("EN_SEARCH must be 'python' or 'cpp', not %r" % (search,))
    _, counts, ns = engine.mcts_search(roots, sims, batch, 1.0, evaluator, flags=_eng.SP_PYSEARCH | sym)
    sc = np.zeros((len(ns), 81), np.float64)
    for i, n in enumerate(ns):
        if n:
            sc[i, :n] = python_scores(counts[i, :n], temperature)
    return sc, ns


class NetworkActor:
    """one side of a match: a DualNetwork evaluated by its own engine"""

    def __init__(self, model, temperature, n_slots, numerics=None, search=None):
        self.evaluator = _eng.evaluator_of(EN_NUMERICS if numerics is None else numerics)
        self.search = EN_SEARCH if search is None else search
        self.engine = _eng.Engine(n_slots=n_slots, max_sims=PV_EVALUATE_COUNT, max_batch=MCTS_BATCH_SIZE, max_games=1)
        model.eval()
        self.engine.upload_model(model)
        self.temperature = temperature

    def scores(self, roots):
        return pv_mcts_scores_batch(self.engine, roots, self.temperature, self.evaluator, self.search)

    def close(self):
        self.engine.close()


class RandomActor:
    """game.random_action (game.py:234-236): uniform over the legal actions"""

    def scores(self, roots):
        dev = torch.device("cuda", torch.cuda.current_device())
        masks, _ = _eng.game_legal_mask(torch.from_numpy(np.ascontiguousarray(roots).view(np.int32)).to(dev))
        ns = masks[:, 3].cpu().numpy().astype(np.int32)
        sc = np.zeros((len(roots), 81), np.float32)
        for i, n in enumerate(ns):
            sc[i, :n] = 1.0 / n
        return sc, ns

    def close(self):
        pass


def play_matches(actors, n_games, seed):
    """All games of a match at once.  Game i uses actors as given when i is even and swapped when odd
    (evaluate_network.py:80-85); returns the list of points of actors[0] per game.
    Moves are drawn with a per-game RandomState(seed, i) so the result does not depend on batching."""
    dev = torch.device("cuda", torch.cuda.current_device())
    states = np.zeros((n_games, 8), np.uint32)
    plies = np.zeros(n_games, np.int64)
    alive = np.ones(n_games, bool)
    rngs = [np.random.RandomState([seed & 0x7FFFFFFF, i]) for i in range(n_games)]
    points = [None] * n_games
    while alive.any():
        idx = np.nonzero(alive)[0]
        # who moves: the first player moves at even plies; odd games have the actors swapped
        side = (plies[idx] % 2) ^ (idx % 2)
        for a in (0, 1):
            sel = idx[side == a]
            if len(sel) == 0:
                continue
            sc, ns = actors[a].scores(states[sel])
            st_d = torch.from_numpy(states[sel].view(np.int32)).to(dev)
            masks, _ = _eng.game_legal_mask(st_d)
            masks = masks.cpu().numpy().view(np.uint32)
            acts = np.zeros(len(sel), np.int32)
            for j, g in enumerate(sel):
                legal = [x for x in range(81) if (masks[j, x // 27] >> (x % 27)) & 1]
                p = sc[j, :ns[j]]
                if p.dtype != np.float64:                 # float32 scores of the C++ semantics (pv_mcts_cpp.py:129-133)
                    p = p.astype(np.float64)
                    p = p / p.sum()
                acts[j] = rngs[g].choice(legal, p=p)
            nxt = _eng.game_step(st_d, torch.from_numpy(acts).to(dev))
            _, status = _eng.game_legal_mask(nxt)
            states[sel] = nxt.cpu().numpy().view(np.uint32)
            status = status.cpu().numpy()
            plies[sel] += 1
            for j, g in enumerate(sel):
                if status[j] != 0:                         # 1: mover has lost, 2: draw
                    alive[g] = False
                    mover_is_first = (plies[g] % 2 == 0)
                    fp = 0.5 if status[j] == 2 else (0 if mover_is_first else 1)      # first_player_point
                    points[g] = fp if g % 2 == 0 else 1 - fp
    return points


def device_match(model0, model1, n_games, seed, temperature=None, numerics=None, search=None):
    """The match of play_matches (model0 first in even games, model1 in odd ones) played by ONE engine, all games
    device-resident like self-play (Engine.match, UTTT_SP_MATCH): model0 in weight slot 0, model1 in slot 1, every leaf
    evaluated by the network whose side is to move, no host work between plies.  Same searches (EN_SEARCH, EN_NUMERICS,
    EN_RANDOM_SYMMETRY) and the same temperature rule; the one difference: moves are drawn by the engine's Philox sampler
    from the same distribution (the visit counts, or n^(1/T), the first maximum at T = 0) instead of by
    RandomState(seed, i).choice, so both paths play the same kind of match but not identical games.
    Returns the points of model0 per game (a list, as play_matches)."""
    temperature = EN_TEMPERATURE if temperature is None else temperature
    search = EN_SEARCH if search is None else search
    if search not in ("python", "cpp"):
        raise ValueError("EN_SEARCH must be 'python' or 'cpp', not %r" % (search,))
    flags = (_eng.SP_PYSEARCH if search == "python" else 0) | (_eng.SP_RANDOM_SYMMETRY if EN_RANDOM_SYMMETRY else 0)
    evaluator = _eng.evaluator_of(EN_NUMERICS if numerics is None else numerics)
    e = _eng.Engine(n_slots=n_games, max_sims=PV_EVALUATE_COUNT, max_batch=MCTS_BATCH_SIZE, max_games=n_games)
    try:
        model0.eval()
        model1.eval()
        e.upload_model(model0, slot=0)
        e.upload_model(model1, slot=1)
        e.set_selfplay_temperature(temperature)
        points, _ = e.match(n_games, sims=PV_EVALUATE_COUNT, batch=MCTS_BATCH_SIZE, seed=seed & 0xFFFFFFFF,
                            evaluator=evaluator, flags=flags)
    finally:
        e.close()
    return points.tolist()


def update_best_player():
    """evaluate_network.py:57-59"""
    copy('./model/latest.pth', './model/best.pth')
    print('Change BestPlayer')


def evaluate_network():
    """evaluate_network.py:62-104.  With EN_DEVICE_MATCH the games are played by device_match (one engine, latest.pth in
    weight slot 0, best.pth in slot 1, same seed); the printed lines and the promotion rule do not change."""
    model0 = DualNetwork().to(device)
    model0.load_state_dict(torch.load('./model/latest.pth', map_location=device, weights_only=True))
    model1 = DualNetwork().to(device)
    model1.load_state_dict(torch.load('./model/best.pth', map_location=device, weights_only=True))
    seed = int(np.random.randint(0, 2 ** 31 - 1)) if EN_SEED is None else int(EN_SEED)
    if EN_DEVICE_MATCH:
        points = device_match(model0, model1, EN_GAME_COUNT, seed)
    else:
        actors = (NetworkActor(model0, EN_TEMPERATURE, EN_GAME_COUNT), NetworkActor(model1, EN_TEMPERATURE, EN_GAME_COUNT))
        try:
            points = play_matches(actors, EN_GAME_COUNT, seed)
        finally:
            for a in actors:
                a.close()
    print('\rEvaluate {}/{}'.format(EN_GAME_COUNT, EN_GAME_COUNT), end='')
    print('')
    average_point = sum(points) / EN_GAME_COUNT
    print('AveragePoint', average_point)
    del model0
    del model1
    if average_point > 0.5:
        update_best_player()
        return True
    return False


if __name__ == '__main__':
    evaluate_network()
