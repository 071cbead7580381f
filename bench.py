#!/usr/bin/env python
"""bench.py -- self-play throughput of the B200 engine on BASELINE.json's metric.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference ...                    (the reference's CPU path on the host cores)

One "step" = one self-play cycle of --games games per GPU (default 500 = SP_GAME_COUNT of the
reference, BASELINE.json configs[2]) at 50 simulations/move, MCTS_BATCH_SIZE 8, random-init
DualNetwork 128x16, reference-exact ("compat") search semantics.  Games are independent, so
ranks shard them with no collective on the search path (weak scaling: fixed games per GPU).

value : plies of all ranks / device time (CUDA events on the launching stream, max over ranks),
        weights and buffers resident in HBM
e2e   : the same cycle through the public host API -- Engine.upload_state_dict(host weights) +
        Engine.selfplay(...) -> host History -- with the H2D / D2H copies inside the timed region

The headline numerics are plain bf16 operands (BASELINE.json configs[2]: "DualNetwork 128x16 bf16"); the same line carries
the same two measurements for the split-bf16 mode ("bf16x3": the tensor-core numerics that meet north_star's 1e-2 bar on
random-init weights, 3x the MMAs), the other BASELINE configs as extra keys -- "c2_rules" (2^20 playouts), "c4_stress"
(4096 trees x 800 simulations, throughput mode) -- and "cycle": BASELINE config 5's self-play stage (4096 games per GPU,
weight broadcast + packed history gather to rank 0 over NCCL when N > 1).  `--numerics bf16x3` makes bf16x3 the line itself.

`--dump-outputs DIR` writes the history of rank 0's last timed step (see dump_outputs) so that two builds can be compared
output for output: the model, the seeds and the game indices depend on the arguments only.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "ultimate-tictactoe-alphazero_b200")
for p in (PKG, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

TRUNK_FLOP_PER_POSITION = 32 * 2 * 81 * 128 * 1152          # SURVEY 8(d): 764,411,904 (dense 3x3 convs)
NET_FLOP_PER_POSITION = 765102212
DUMP_LIMIT_BYTES = 60 << 20                          # --dump-outputs: below 64 MB with the .npy headers


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, \
        "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, rank):
    """reference arm: the reference's own CPU implementation (compiled C++ MCTS + rules from
    oracle/_ref, DualNetwork fp32 through PyTorch on all host threads); each step is a bounded
    sample of the same workload (args.ref_moves plies of 50-simulation self-play)."""
    if rank != 0:
        return
    import torch
    import cpu_selfplay
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    from dual_network import DualNetwork
    try:
        ref = cpu_selfplay.load_reference_module()
        kind = "reference"
    except FileNotFoundError as e:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built: %s" % e}))
        return
    model = DualNetwork().eval()
    rng = np.random.RandomState(0)
    for _ in range(args.warmup):
        cpu_selfplay.play_moves(ref, model, 2, args.sims, args.batch, rng=rng)
    stats = {"forward_s": 0.0, "forwards": 0, "positions": 0}
    t0 = time.perf_counter()
    plies = 0
    for _ in range(args.steps):
        plies += cpu_selfplay.play_moves(ref, model, args.ref_moves, args.sims, args.batch, rng=rng, stats=stats)
    dt = time.perf_counter() - t0
    v = plies / dt
    sample = "%d plies/step of %d-sim batch-%d self-play (reference C++ MCTS + PyTorch fp32 forward on %d host threads)" % (
        args.ref_moves, args.sims, args.batch, cores)
    print(json.dumps({
        "impl": "reference", "metric": "self-play moves/sec (50 sims/move)", "value": v, "unit": "moves/s",
        "sims_per_s": v * args.sims, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (random-init weights, games from the initial position)",
        "config": workload_config(args), "forward_frac": stats["forward_s"] / dt,
        "cpu_baseline": {"value": v, "unit": "moves/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": v, "unit": "moves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))

def workload_config(args):
    return {"workload": "C3 (BASELINE.json configs[2]): %d-game self-play cycle per GPU, %d sims/move, "
                        "MCTS_BATCH_SIZE=%d, DualNetwork 128fx16 random-init" % (args.games, args.sims, args.batch),
            "games_per_gpu": args.games, "sims_per_move": args.sims, "mcts_batch_size": args.batch,
            "search": "compat (reference-exact queue/flush semantics)", "numerics": args.numerics,
            "l2": "flushed between timed steps (256 MiB device write)"}


class Ctx:
    pass


def dump_outputs(out_dir, hist, stats):
    """Write a History of self-play games and the run's stats [plies, sims, evals, rounds] as out_dir/<name>.npy: integers
    below 2^24 as float32, packed states (uint32 words) and stats as float64.  Plies past a game's length hold whatever
    earlier runs left in the engine's buffers and are written as zeros.  Above DUMP_LIMIT_BYTES a fixed seeded sample of
    the games is written; `game` holds their indices within the step."""
    n = hist.n_games
    per_game = 81 * 8 * 8 + 81 * 81 * 4 + 81 * 4 + 3 * 8
    games = np.arange(n)
    if n * per_game > DUMP_LIMIT_BYTES:
        games = np.sort(np.random.RandomState(0).choice(n, DUMP_LIMIT_BYTES // per_game, replace=False))
    live = np.arange(81)[None, :] < hist.lens[games, None]
    arrays = {"game": games.astype(np.float64), "lens": hist.lens[games].astype(np.float32),
              "final": hist.final[games].astype(np.float32),
              "actions": np.where(live, hist.actions[games], 0).astype(np.float32),
              "counts": np.where(live[:, :, None], hist.counts[games], 0).astype(np.float32),
              "states": np.where(live[:, :, None], hist.states[games], 0).astype(np.float64),
              "stats": np.asarray(stats, dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return arrays


def timed_selfplay(c, eng, ev_kind, steps, warmup, games, seed0):
    """device-resident leg: CUDA events on the launching stream around every cycle -> dict of rank-local sums"""
    import torch
    a = c.args

    def step(i):
        return eng.selfplay_device(games, sims=a.sims, batch=a.batch, seed=0x5EED, evaluator=ev_kind,
                                   game0=(seed0 + i * c.world + c.rank) * games, stream=c.stream)
    for i in range(warmup):
        step(1000 + i)
    # trunk_*: the trunk launches that were bracketed by CUDA events (the engine brackets every 4th window of 8 rounds: an event
    # record on either side of every trunk launch costs 1.6 % of the step)
    out = {"dev_ms": 0.0, "plies": 0, "sims": 0, "evals": 0, "rounds": 0, "trunk_ms": 0.0, "trunk_launches": 0, "trunk_evals": 0,
           "launches": 0}
    c.barrier()
    for i in range(steps):
        c.flush.fill_(i & 0xFF)                    # evict L2 between timed steps (not timed)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(c.stream)
        st = step(i)
        e1.record(c.stream)
        e1.synchronize()
        out["dev_ms"] += e0.elapsed_time(e1)
        out["last_stats"] = st
        out["plies"] += int(st[0]); out["sims"] += int(st[1]); out["evals"] += int(st[2]); out["rounds"] += int(st[3])
        prof = eng.last_run_profile()
        tt = prof["trunk_timed"]
        out["trunk_ms"] += tt[0]; out["trunk_launches"] += tt[1]; out["trunk_evals"] += tt[2]; out["launches"] += prof["all"][1]
    c.barrier()
    return out


def timed_e2e(c, eng, ev_kind, steps, games, hist):
    """the same cycle through the public host API: pinned host weights in, host History out, wall clock"""
    a = c.args
    eng.upload_state_dict(c.sd_host)
    eng.selfplay(games, sims=a.sims, batch=a.batch, seed=1, evaluator=ev_kind, game0=10 ** 6, history=hist)       # warm-up
    c.barrier()
    t0 = time.perf_counter()
    plies = 0
    for i in range(steps):
        eng.upload_state_dict(c.sd_host)
        h = eng.selfplay(games, sims=a.sims, batch=a.batch, seed=0x5EED, evaluator=ev_kind,
                         game0=(i * c.world + c.rank) * games, history=hist)
        plies += int(h.stats[0])
    c.barrier()
    return plies, time.perf_counter() - t0


def reduce_leg(c, leg, e2e_plies, e2e_s):
    """max over ranks of the times, sums over ranks of the counts"""
    import torch
    import torch.distributed as dist
    red = torch.tensor([leg["dev_ms"], e2e_s], dtype=torch.float64, device=c.dev)
    tot = torch.tensor([leg["plies"], leg["sims"], leg["evals"], e2e_plies, leg["launches"]], dtype=torch.float64, device=c.dev)
    if c.world > 1:
        dist.all_reduce(red, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    return [float(x) for x in red.tolist()], [float(x) for x in tot.tolist()]


def c2_rules(c):
    """BASELINE config 2: 2^20 concurrent random playouts (legal mask, forced board, winner); bit-exactness is checked
    against checksums of the compiled reference's own playouts (tests/golden/rules.npz, minted by oracle/gen_golden.py)"""
    import numpy as np
    import torch
    import engine
    n = 1 << 20
    engine.game_playout(1, 0, n)
    torch.cuda.synchronize()
    ms = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); dg, pl, rs = engine.game_playout(0x5EED, 0, n); e1.record(); torch.cuda.synchronize()
        ms = min(ms, e0.elapsed_time(e1))
    plies = int(pl.sum().item())
    out = {"playouts": n, "transitions": plies, "ms": ms, "transitions_per_s": plies / (ms / 1e3), "bit_exact": None}
    gpath = os.path.join(ROOT, "tests", "golden", "rules.npz")
    if os.path.exists(gpath):
        with np.load(gpath) as z:
            d = dg.cpu().numpy().view(np.uint64)
            xor = int(np.bitwise_xor.reduce(d))
            tot = int(d.astype(object).sum()) & 0xFFFFFFFFFFFFFFFF
            hist = np.bincount(rs.cpu().numpy(), minlength=3)
            out["bit_exact"] = bool(int(z["seed"]) == 0x5EED and int(z["full_n"]) == n and xor == int(z["full_xor"]) and
                                    tot == int(z["full_sum"]) and plies == int(z["full_plies"]) and
                                    (hist == z["full_hist"]).all())
            out["checked_against"] = "xor / sum of the 2^20 per-game digests, plies and results of the compiled reference"
    return out


def c4_stress(c, trees=4096, sims=800, leaves=8):
    """BASELINE config 4: 4096 concurrent trees x 800 simulations per move, throughput mode (evaluated root with Dirichlet
    noise eps 0.25 alpha 0.3 from Philox, virtual loss, 8 leaves per tree and round): one move of every tree"""
    import numpy as np
    import engine
    import uttt_cpp
    rng = np.random.RandomState(4)
    roots = []
    while len(roots) < 256:                       # 256 distinct mid-game positions (host rules helpers), tiled to 4096 trees
        s = uttt_cpp.State()
        for _ in range(rng.randint(6, 36)):
            if s.is_done():
                break
            la = s.legal_actions()
            s = s.next(la[rng.randint(len(la))])
        if not s.is_done():
            roots.append(s.packed())
    roots = np.tile(np.stack(roots), (trees // 256, 1))
    e = engine.Engine(n_slots=trees, max_sims=sims, max_batch=leaves, max_games=1, device=c.local_rank)
    try:
        e.upload_state_dict(c.sd_host)
        e.set_root_noise(0.3, 0.25)
        ev = engine.EVAL_NET_BF16
        e.mcts_search(roots, 64, leaves, 1.0, ev, flags=engine.SP_THROUGHPUT)       # warm-up
        import torch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, counts, _ = e.mcts_search(roots, sims, leaves, 1.0, ev, flags=engine.SP_THROUGHPUT)
        dt = time.perf_counter() - t0
        k = e.counters()
        assert (counts.sum(1) == sims).all() and k["overflow"] == 0
        return {"trees": trees, "sims_per_move": sims, "leaves_per_tree_per_round": leaves, "wall_s": dt,
                "sims_per_s": k["sims"] / dt, "nn_evals_per_s": k["evals"] / dt,
                "trunk_tflops_equiv": k["evals"] * TRUNK_FLOP_PER_POSITION / dt / 1e12,
                "note": "rank 0's GPU; whole pipeline (tree + trunk + heads kernels), host wall clock around one synchronous search"}
    finally:
        e.close()


def cycle_leg(c, ev_name):
    """BASELINE config 5, the self-play stage of one train_cycle iteration: weights broadcast from rank 0, 4096 games per
    GPU, every rank's history packed on its GPU and sent to rank 0 in one exact-length transfer, expanded there into the
    trainer's tensors.  One warm-up cycle, then one timed cycle per numerics; time = max over ranks of the wall clock."""
    import torch
    import torch.distributed as dist
    import parallel
    from dual_network import DualNetwork
    a = c.args
    torch.manual_seed(0)
    model = DualNetwork().eval()
    n_games = a.cycle_games * c.world
    cyc = parallel.SelfPlayCycle(n_games, sims=a.sims, batch=a.batch, numerics=ev_name, device=c.local_rank)
    try:
        cyc.run(model, seed=1, cycle=0)
        c.barrier()
        res = cyc.run(model, seed=2, cycle=1)
        t = dict(cyc.timings)
        red = torch.tensor([t["total_ms"], t["broadcast_ms"], t["selfplay_ms"], t["pack_ms"], t["gather_ms"], t["unpack_ms"]],
                           dtype=torch.float64, device=c.dev)
        if c.world > 1:
            dist.all_reduce(red, op=dist.ReduceOp.MAX)
        if c.rank != 0:
            return None
        n = int(res["n_samples"])
        assert res["x"].shape == (n, 3, 9, 9) and float(res["policy"].sum()) > 0.99 * n
        tot, bc, sp, pk, ga, up = [float(x) for x in red.tolist()]
        return {"games": n_games, "games_per_gpu": a.cycle_games, "numerics": ev_name, "samples": n,
                "moves_per_s_e2e": n / (tot / 1e3), "total_ms": tot, "broadcast_ms": bc, "selfplay_ms": sp, "pack_ms": pk,
                "gather_ms": ga, "unpack_ms": up, "gather_bytes": int(t["gather_bytes"]),
                "broadcast_bytes": int(c.w_bytes),
                "collectives": "dist.broadcast of one flat 19.1 MB buffer; one tiny all_gather of sizes + one send/recv per rank "
                               "of its exact-length packed history (196 B/sample) into rank 0's buffer" if c.world > 1 else "none (1 GPU)",
                "note": "times are max over ranks of wall clock between device synchronisations; engine and buffers persist across cycles"}
    finally:
        cyc.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--games", type=int, default=500, help="self-play games per GPU per step (SP_GAME_COUNT)")
    ap.add_argument("--sims", type=int, default=50)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--numerics", default="bf16", choices=["bf16", "bf16x3", "fp32"])
    ap.add_argument("--ref-moves", type=int, default=24, help="plies per step of the reference arm")
    ap.add_argument("--cpu-baseline-moves", type=int, default=96)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--saturated-games", type=int, default=4096,
                    help="also time one cycle of this many concurrent games per GPU (0 = skip)")
    ap.add_argument("--cycle-games", type=int, default=4096, help="games per GPU of the config-5 cycle leg (0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the bf16x3 / c2 / c4 / cycle legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the history of rank 0's last timed step as DIR/<name>.npy (float32 / float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the B200 engine's history; the reference arm has none")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import engine
    from dual_network import DualNetwork

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if "MASTER_PORT" not in os.environ:              # not under torchrun: a single-process group on a free port
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            os.environ["MASTER_PORT"] = str(sk.getsockname()[1])
    dist.init_process_group("nccl", device_id=dev, rank=rank, world_size=world)      # world 1: the cycle leg's plumbing only

    c = Ctx()
    c.args, c.rank, c.world, c.local_rank, c.dev = args, rank, world, local_rank, dev

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    c.barrier = barrier

    ev_kind = engine.evaluator_of(args.numerics)
    eng = engine.Engine(n_slots=min(args.games, 4096), max_sims=args.sims, max_batch=args.batch,
                        max_games=args.games, device=local_rank)
    torch.manual_seed(0)
    model = DualNetwork().eval()
    c.sd_host = {k: v.pin_memory() for k, v in model.state_dict().items()}
    c.w_bytes = sum(v.numel() * v.element_size() for v in c.sd_host.values())
    eng.upload_state_dict(c.sd_host)
    c.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    c.stream = torch.cuda.current_stream()

    # ---------------- device-resident timed region (the headline `value`)
    sampler = ClockSampler(local_rank)
    for i in range(args.warmup):
        eng.selfplay_device(args.games, sims=args.sims, batch=args.batch, seed=0x5EED, evaluator=ev_kind,
                            game0=(1000 + i) * args.games, stream=c.stream)
    barrier()
    if rank == 0:
        sampler.start()
    t_wall0 = time.perf_counter()
    leg = timed_selfplay(c, eng, ev_kind, args.steps, 0, args.games, 0)
    wall_s = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng.selfplay_fetch(args.games), leg["last_stats"])
    dev_ms, plies, evals, rounds = leg["dev_ms"], leg["plies"], leg["evals"], leg["rounds"]
    trunk_ms, trunk_launches, trunk_evals = leg["trunk_ms"], leg["trunk_launches"], leg["trunk_evals"]
    # diagnostic, outside the timed region: one more cycle with every kernel bracketed by events (level 2 costs ~1.5 %
    # of a cycle in GPU idle time at the extra event boundaries, which is why the timed steps only bracket the trunk)
    eng.set_profile_level(2)
    st = eng.selfplay_device(args.games, sims=args.sims, batch=args.batch, seed=0x5EED, evaluator=ev_kind,
                             game0=2000 * args.games, stream=c.stream)
    torch.cuda.synchronize()
    prof = eng.last_run_profile()
    split = {"tree_kernels": prof["tree"][0], "trunk": prof["trunk"][0], "heads": prof["heads"][0],
             "device_total": prof["all"][0], "rounds": int(st[3])}
    eng.set_profile_level(1)

    # ---------------- end-to-end through the public host API (H2D weights, D2H history inside the timed region)
    hist = engine.History(args.games)
    e2e_plies, e2e_s = timed_e2e(c, eng, ev_kind, args.steps, args.games, hist)
    (dev_ms_max, e2e_s_max), (plies_all, sims_all, evals_all, e2e_plies_all, launches_all) = reduce_leg(c, leg, e2e_plies, e2e_s)

    # ---------------- the same two measurements with split-bf16 numerics (the mode that meets the 1e-2 parity bar)
    x3 = None
    if args.numerics == "bf16" and not args.no_extras:
        k3 = args.steps
        leg3 = timed_selfplay(c, eng, engine.EVAL_NET_BF16X3, k3, 3, args.games, 50)
        p3, s3 = timed_e2e(c, eng, engine.EVAL_NET_BF16X3, k3, args.games, hist)
        (d3, es3), (pl3, _, ev3, ep3, _) = reduce_leg(c, leg3, p3, s3)
        x3 = {"leg": leg3, "steps": k3, "dev_ms_max": d3, "e2e_s_max": es3, "plies_all": pl3, "evals_all": ev3, "e2e_plies_all": ep3}

    # ---------------- secondary: the machine-filling workload (C5's per-GPU share: 4096 concurrent games)
    sat = None
    if args.saturated_games > 0:
        eng.close()
        eng = engine.Engine(n_slots=min(args.saturated_games, 4096), max_sims=args.sims, max_batch=args.batch,
                            max_games=args.saturated_games, device=local_rank)
        eng.upload_state_dict(c.sd_host)
        eng.selfplay_device(args.saturated_games, sims=args.sims, batch=args.batch, seed=7, evaluator=ev_kind,
                            game0=5 * 10 ** 6, stream=c.stream)                       # warm-up
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(c.stream)
        st = eng.selfplay_device(args.saturated_games, sims=args.sims, batch=args.batch, seed=8, evaluator=ev_kind,
                                 game0=6 * 10 ** 6 + rank * args.saturated_games, stream=c.stream)
        e1.record(c.stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        sat = {"games_per_gpu": args.saturated_games, "moves_per_s_rank0": int(st[0]) / (ms / 1e3),
               "nn_evals_per_s_rank0": int(st[2]) / (ms / 1e3),
               "trunk_tflops_equiv_rank0": int(st[2]) * TRUNK_FLOP_PER_POSITION / (ms / 1e3) / 1e12,
               "note": "whole-pipeline rate (tree + trunk + heads, two overlapped lanes); trunk_tflops_equiv = evals x "
                       "764.4 MFLOP / wall, i.e. a lower bound on the trunk kernels' own rate"}
    eng.close()
    extras = {}
    if not args.no_extras:
        if args.cycle_games > 0:
            cyc = {}
            for name in ([args.numerics] if args.numerics != "bf16" else ["bf16", "bf16x3"]):
                r = cycle_leg(c, name)
                if rank == 0:
                    cyc[name] = r
            extras["cycle"] = cyc
        if rank == 0:
            extras["c2_rules"] = c2_rules(c)
            extras["c4_stress"] = c4_stress(c)
        barrier()

    if rank == 0:
        peaks, peak_src = measured_peaks()
        value = plies_all / (dev_ms_max / 1e3)
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
        # dominant kernel = the residual trunk (tcgen05 implicit GEMM); rank 0's launches
        achieved_tf = (trunk_evals * TRUNK_FLOP_PER_POSITION / (trunk_ms / 1e3)) / 1e12 if trunk_ms > 0 else 0.0
        trunk_est_ms = trunk_ms / max(trunk_launches, 1) * rounds          # all launches of the timed region at the sampled average
        kernel = {"bf16": "trunk_auto_kernel (one launch per round; on the device: trunk_tc2_body<2> up to 370 positions -- with "
                          "cta_group::2 MMAs up to 148 --, trunk_pp_body<1> with cta_group::2 MMAs above)",
                  "bf16x3": "trunk_x3_kernel (trunk_tc2_body<2, X3, PAIR>: 3 cta_group::2 MMAs per K-block, hi*hi + lo*hi + hi*lo)",
                  "fp32": "conv3x3_fp32_kernel"}[args.numerics]
        out = {
            "metric": "self-play moves/sec (50 sims/move)", "value": value, "unit": "moves/s",
            "sims_per_s": sims_all / (dev_ms_max / 1e3), "nn_evals_per_s": evals_all / (dev_ms_max / 1e3),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "bf16x3": "bf16x3 (split-bf16 operands, fp32 accumulation)", "fp32": "f32"}[args.numerics],
            "data": "synthetic (random-init DualNetwork weights, seed 0; games from the initial position)",
            "config": workload_config(args),
            "clocks": clocks,
            "e2e": {"value": e2e_plies_all / e2e_s_max, "unit": "moves/s", "h2d_bytes_per_step": int(c.w_bytes),
                    "d2h_bytes_per_step": int(hist.nbytes)},
            "gpu_launches": int(launches_all),
            "roofline": {"bound": "tensor", "kernel": kernel,
                         "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": achieved_tf / peak_tf if peak_tf else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture at a batch of ~500 positions
                         # (profiles/r2_trunkpp_full.md, r2_trunkx3_full.md): weights (9.4 MB bf16, 18.9 MB split-bf16), planes, head
                         # features, policy / value rows; activations and the skip connection never reach DRAM
                         "traffic": {"bf16": 15.49e6, "bf16x3": 20.89e6}.get(args.numerics),
                         "traffic_unit": "bytes per launch from a cold-cache ncu capture (bf16: 1.56x the 9.9 MB algorithmic -- the weights "
                                         "come from DRAM once per capture, from L2 in steady state); tensor-bound kernel: informational",
                         "peak_source": peak_src + ", sustained bf16 (kernel timed inside a long step)",
                         "flop_per_launch": trunk_evals * TRUNK_FLOP_PER_POSITION / max(trunk_launches, 1),
                         "flop_convention": "useful (algorithmic) FLOPs: 764.4 MFLOP per evaluated position, SURVEY 8(d)"
                                            + ("; the kernel issues 3x that on the tensor pipe" if args.numerics == "bf16x3" else ""),
                         "avg_launch_ms": trunk_ms / max(trunk_launches, 1), "launches": trunk_launches,
                         "timed_with": "CUDA events on the launching stream around %d of the %d trunk launches of the timed region (every "
                                       "launch of every 4th window of 8 rounds: a uniform sample of the cycle's batch sizes), which "
                                       "evaluated %d of its %d positions; bracketing every launch costs 1.6 %% of the step and gives the same "
                                       "average (UTTT_PROFILE_SAMPLE=1)"
                                       % (trunk_launches, rounds, trunk_evals, evals)},
            "breakdown_ms_rank0": {"trunk_timed_launches": trunk_ms, "trunk_all_launches_at_that_average": trunk_est_ms,
                                   "tree_heads_and_gaps": dev_ms - trunk_est_ms, "device_total": dev_ms,
                                   "rounds": rounds, "evals": evals, "plies": plies,
                                   "one_extra_cycle_with_all_kernels_timed": split},
            "wall_s": wall_s,
            "saturated": sat,
        }
        if x3 is not None:
            l3 = x3["leg"]
            a3 = (l3["trunk_evals"] * TRUNK_FLOP_PER_POSITION / (l3["trunk_ms"] / 1e3)) / 1e12 if l3["trunk_ms"] > 0 else 0.0
            out["bf16x3"] = {
                "what": "the same workload and the same two measurements with UTTT_EVAL_NET_BF16X3 (split-bf16 operands: policy / "
                        "value within 1e-2 of the fp32 reference forward on these random-init weights, tests/test_gpu_net.py)",
                "value": x3["plies_all"] / (x3["dev_ms_max"] / 1e3), "unit": "moves/s", "steps": x3["steps"],
                "ms_per_step": x3["dev_ms_max"] / x3["steps"],
                "e2e": {"value": x3["e2e_plies_all"] / x3["e2e_s_max"], "unit": "moves/s", "h2d_bytes_per_step": int(c.w_bytes),
                        "d2h_bytes_per_step": int(hist.nbytes)},
                "roofline": {"bound": "tensor", "kernel": "trunk_x3_kernel", "achieved": a3, "peak": peak_tf, "unit": "TFLOP/s",
                             "frac": a3 / peak_tf if peak_tf else None, "mma_tflops_issued": 3 * a3,
                             "flop_convention": "useful FLOPs (764.4 MFLOP / position); the tensor pipe executes 3x that",
                             "avg_launch_ms": l3["trunk_ms"] / max(l3["trunk_launches"], 1), "launches": l3["trunk_launches"]}}
        out.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            try:
                import cpu_selfplay
                r = cpu_selfplay.time_cpu_selfplay(args.cpu_baseline_moves, args.sims, args.batch)
                out["cpu_baseline"] = {
                    "value": r["moves_per_s"], "unit": "moves/s", "cores": r["cores"], "kind": "reference",
                    "sample": "%d plies of %d-sim batch-%d self-play: reference C++ MCTS (oracle/_ref) + PyTorch fp32 "
                              "DualNetwork on %d host threads, %.1f s, %.0f%% in forward" % (
                                  r["moves"], args.sims, args.batch, r["cores"], r["seconds"], 100 * r["forward_frac"])}
            except Exception as e:  # noqa: BLE001
                out["cpu_baseline"] = {"value": None, "unit": "moves/s", "cores": os.cpu_count(), "kind": "reference",
                                       "sample": "unavailable: %s" % e}
        print(json.dumps(out))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
