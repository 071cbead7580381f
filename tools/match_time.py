"""Wall-clock time of a whole gating match, host-driven against device-resident.

  host    evaluate_network.play_matches: per ply one batched search per network (two engines), legal masks and the next
          positions copied to the host, moves drawn there with RandomState(seed, i).choice
  device  Engine.match (UTTT_SP_MATCH): one engine with the two networks in weight slots 0 and 1, every game on the device
          as in self-play, each leaf evaluated by the network to move
  floor   plain self-play (one network) of the same number of games on the same kind of engine

for 50 and 400 games, bf16 and bf16x3, EN_SEARCH "python" (UTTT_SP_PYSEARCH) and "cpp".  Each case is timed after one
warm-up match of its own; one JSON line per case: ms, plies, rounds (device and floor: tree rounds; host: not counted),
trunk launches (device and floor: all evaluator passes; host and every case: "trunk_nonempty", the tensor-core trunk
launches that evaluated at least one position, from the batch-size histogram), searches (host: batched searches).

python tools/match_time.py [--games 50,400] [--numerics bf16,bf16x3] [--search python,cpp] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200"))
import torch  # noqa: E402
import engine  # noqa: E402
import evaluate_network as en  # noqa: E402
from dual_network import DualNetwork  # noqa: E402

SEED = 0x5EED


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def trunk_nonempty(engines):
    return int(sum(e.batch_histogram(reset=True).sum() for e in engines))


class CountingActor:
    """a NetworkActor that counts its batched searches and the positions they searched (= plies)"""

    def __init__(self, actor):
        self.actor, self.searches, self.plies = actor, 0, 0

    def scores(self, roots):
        self.searches += 1
        self.plies += len(roots)
        return self.actor.scores(roots)


def host_case(models, games, numerics, search):
    actors = [en.NetworkActor(m, en.EN_TEMPERATURE, games, numerics=numerics, search=search) for m in models]
    try:
        engines = [a.engine for a in actors]
        en.play_matches(actors, games, SEED + 1)                      # warm-up
        counted = [CountingActor(a) for a in actors]
        trunk_nonempty(engines)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        points = en.play_matches(counted, games, SEED)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        return {"ms": ms, "plies": sum(c.plies for c in counted), "rounds": None, "trunk_launches": None,
                "trunk_nonempty": trunk_nonempty(engines), "searches": sum(c.searches for c in counted),
                "average_point": sum(points) / games}
    finally:
        for a in actors:
            a.close()


def device_case(models, games, numerics, search, floor=False):
    e = engine.Engine(n_slots=games, max_sims=en.PV_EVALUATE_COUNT, max_batch=en.MCTS_BATCH_SIZE, max_games=games)
    try:
        ev = engine.evaluator_of(numerics)
        flags = engine.SP_PYSEARCH if (search == "python" and not floor) else 0
        e.upload_model(models[0])
        if not floor:
            e.upload_model(models[1], slot=1)
        e.set_selfplay_temperature(en.EN_TEMPERATURE)

        def run(seed):
            if floor:
                return None, e.selfplay(games, sims=en.PV_EVALUATE_COUNT, batch=en.MCTS_BATCH_SIZE, seed=seed, evaluator=ev)
            return e.match(games, sims=en.PV_EVALUATE_COUNT, batch=en.MCTS_BATCH_SIZE, seed=seed, evaluator=ev, flags=flags)
        run(SEED + 1)                                                   # warm-up
        trunk_nonempty([e])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        points, h = run(SEED)
        ms = (time.perf_counter() - t0) * 1e3                           # (selfplay() returns after the history copy)
        out = {"ms": ms, "plies": int(h.stats[0]), "rounds": int(h.stats[3]),
               "trunk_launches": int(e.last_run_profile()["trunk"][1]), "trunk_nonempty": trunk_nonempty([e]),
               "searches": None}
        if points is not None:
            out["average_point"] = float(points.mean())
        return out
    finally:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", default="50,400")
    ap.add_argument("--numerics", default="bf16,bf16x3")
    ap.add_argument("--search", default="python,cpp")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = gpu_info()
    torch.manual_seed(1); m0 = DualNetwork().eval()
    torch.manual_seed(2); m1 = DualNetwork().eval()
    lines = []

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        lines.append(line)
    for games in [int(x) for x in args.games.split(",")]:
        for numerics in args.numerics.split(","):
            emit(dict(path="floor", games=games, numerics=numerics, search=None, **device_case((m0, m1), games, numerics, "cpp",
                                                                                                floor=True)))
            for search in args.search.split(","):
                for path in ("host", "device"):
                    fn = host_case if path == "host" else device_case
                    emit(dict(path=path, games=games, numerics=numerics, search=search, **fn((m0, m1), games, numerics, search)))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
