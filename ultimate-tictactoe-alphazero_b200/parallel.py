"""Multi-GPU plumbing around the self-play path (one process per GPU, torch.distributed).

Games are independent, so the search path has NO collective: each rank plays a contiguous block of
game ids on its own GPU.  Collectives are used off the path only, once per cycle:
  * broadcast_state_dict: the new ./model/best.pth weights, one flattened buffer from `src`
  * gather_samples:       every rank's history as ONE exact-length buffer of 196-byte samples
                          (engine.SAMPLE_BYTES: packed position, visit counts, label, ply) to `dst`:
                          the sizes travel in one tiny all_gather, the payload in one send / recv
                          per rank straight into its slice of the destination buffer (device memory
                          over NVLink with "nccl": no padding to the longest rank, no host staging)
Backend "nccl" (GPU tensors) in production, "gloo" (CPU tensors) in the CPU tests.
SelfPlayCycle keeps the engine and the buffers alive across cycles (engine creation allocates GBs).
"""
import time

import numpy as np
import torch
import torch.distributed as dist

import engine as _eng


def shard_games(n_games, world, rank):
    """contiguous block of game ids for `rank`: (game0, count); blocks differ by at most one game"""
    base, rem = divmod(n_games, world)
    count = base + (1 if rank < rem else 0)
    game0 = rank * base + min(rank, rem)
    return game0, count


def _comm_device():
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


def broadcast_state_dict(sd, src=0):
    """In-place broadcast of a DualNetwork state_dict (216 tensors, 19.1 MB fp32) as ONE flat buffer."""
    dev = _comm_device()
    keys = list(sd.keys())
    flat = torch.cat([sd[k].detach().reshape(-1).to(torch.float32) for k in keys]).to(dev)
    dist.broadcast(flat, src=src)
    off = 0
    for k in keys:
        n = sd[k].numel()
        sd[k].copy_(flat[off:off + n].reshape(sd[k].shape).to(sd[k].dtype))
        off += n
    return sd


def gather_samples(samples, dst=0, out=None):
    """samples: this rank's packed history, a 1-D uint8 tensor of n_local * SAMPLE_BYTES bytes on the communication device.
    On `dst` returns (buffer, counts): all ranks' samples concatenated in rank order (= global game-id order for
    shard_games blocks) and the number of samples per rank; (None, counts) elsewhere.  `out`: optional destination
    buffer on `dst` (re-used across cycles) of at least the total size."""
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = samples.device
    assert samples.dtype == torch.uint8 and samples.dim() == 1 and samples.numel() % _eng.SAMPLE_BYTES == 0
    sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(sizes, torch.tensor([samples.numel()], dtype=torch.int64, device=dev))
    sizes = [int(s.item()) for s in sizes]
    counts = [s // _eng.SAMPLE_BYTES for s in sizes]
    if rank != dst:
        if sizes[rank]:
            dist.send(samples, dst=dst)
        return None, counts
    total = sum(sizes)
    if out is None or out.numel() < total:
        out = torch.empty(total, dtype=torch.uint8, device=dev)
    ops, off = [], 0
    for r in range(world):
        if r == dst:
            out[off:off + sizes[r]].copy_(samples)
        elif sizes[r]:
            ops.append(dist.irecv(out[off:off + sizes[r]], src=r))
        off += sizes[r]
    for op in ops:
        op.wait()
    return out[:total], counts


def pack_history_host(hist, n_local):
    """engine.History (host arrays) -> uint8 tensor of packed samples, the layout of uttt_selfplay_pack (csrc/history_kernels.cu):
    one per ply of hist.sample_mask"""
    mask = hist.sample_mask(n_local)
    n = int(mask.sum())
    raw = np.zeros((n, _eng.SAMPLE_BYTES), np.uint8)
    if n:
        raw[:, :32] = hist.states[:n_local][mask].view(np.uint8).reshape(n, 32)
        raw[:, 32:194] = np.ascontiguousarray(hist.targets()[:n_local][mask]).view(np.uint8).reshape(n, 162)
        ply = np.broadcast_to(np.arange(81)[None, :], mask.shape)[mask]
        z0 = np.where(hist.final[:n_local] != 0, -1, 0).astype(np.int8)
        z = np.broadcast_to(z0[:, None], mask.shape)[mask] * np.where(ply % 2 == 0, 1, -1).astype(np.int8)
        raw[:, 194] = z.astype(np.int8).view(np.uint8)
        raw[:, 195] = ply.astype(np.uint8)
    return torch.from_numpy(raw.reshape(-1))


def gather_histories(hist, n_local, dst=0):
    """hist: engine.History of this rank (first n_local games valid).  Returns on `dst` a dict of numpy arrays over all
    samples of all ranks in global game order -- states (N,8) u32, counts (N,81) u16, z (N,) i8, ply (N,) u8, and
    samples_per_rank -- None elsewhere.  (Host-side packing; SelfPlayCycle packs on the device.)"""
    buf = pack_history_host(hist, n_local).to(_comm_device())
    out, counts = gather_samples(buf, dst=dst)
    if out is None:
        return None
    st, cn, z, ply = _eng.samples_to_numpy(out.cpu().numpy())
    return {"states": st, "counts": cn, "z": z, "ply": ply, "samples_per_rank": np.array(counts, np.int64)}


class SelfPlayCycle:
    """BASELINE config 5, the self-play stage of a multi-GPU train_cycle iteration, repeated: rank `src` broadcasts the
    weights (new best.pth), every rank plays its block of games on its own GPU (no collective on the search path), the
    packed histories go to rank `dst` in one transfer per rank and are expanded there into the trainer's tensors.
    The engine, the pack buffer and the gather buffer live as long as the object.  fast_sims (None: every move is a full
    search) turns on playout cap randomization (engine.SP_PLAYOUT_CAP): a move gets a full search of `sims` simulations with
    probability full_fraction and a fast one of fast_sims otherwise, and only the full searches become samples."""

    def __init__(self, n_games, sims=50, batch=8, numerics=None, device=None, max_slots=4096, fast_sims=None, full_fraction=0.25):
        self.world, self.rank = dist.get_world_size(), dist.get_rank()
        self.n_games, self.sims, self.batch = n_games, sims, batch
        self.game0, self.count = shard_games(n_games, self.world, self.rank)
        self.evaluator = _eng.evaluator_of(_eng.DEFAULT_NUMERICS if numerics is None else numerics)
        cnt = max(self.count, 1)
        self.engine = _eng.Engine(n_slots=min(cnt, max_slots), max_sims=sims, max_batch=batch, max_games=cnt, device=device)
        self.flags = 0
        if fast_sims is not None:
            self.engine.set_playout_cap(fast_sims, full_fraction)
            self.flags = _eng.SP_PLAYOUT_CAP
        self.dev = torch.device("cuda", self.engine.device)
        self.pack_buf = torch.empty(81 * cnt * _eng.SAMPLE_BYTES, dtype=torch.uint8, device=self.dev)
        self.gather_buf = None
        self.timings = {}

    def close(self):
        self.engine.close()

    def run(self, model, seed=0, cycle=0, src=0, dst=0, unpack=True):
        """-> on `dst`: dict(samples, n_samples, samples_per_rank[, x, policy, value]); elsewhere dict(n_samples=local).
        self.timings: broadcast_ms, selfplay_ms, pack_ms, gather_ms, unpack_ms (wall clock around synchronised steps),
        gather_bytes (received by `dst`)."""
        def tick():
            torch.cuda.synchronize(self.dev)
            return time.perf_counter()
        t0 = tick()
        broadcast_state_dict(model.state_dict(), src=src)
        self.engine.upload_model(model)
        t1 = tick()
        stats = self.engine.selfplay_device(self.count, sims=self.sims, batch=self.batch, seed=seed, evaluator=self.evaluator,
                                            flags=self.flags, game0=cycle * self.n_games + self.game0)
        t2 = tick()
        samples, n_local = self.engine.selfplay_pack(self.count, out=self.pack_buf)
        t3 = tick()
        if self.rank == dst and self.gather_buf is None:
            self.gather_buf = torch.empty(81 * self.n_games * _eng.SAMPLE_BYTES, dtype=torch.uint8, device=self.dev)
        out, counts = gather_samples(samples, dst=dst, out=self.gather_buf)
        t4 = tick()
        res = {"n_samples": n_local, "stats": stats}
        if self.rank == dst:
            res.update(samples=out, n_samples=sum(counts), samples_per_rank=counts)
            if unpack:
                res["x"], res["policy"], res["value"] = _eng.samples_unpack(out, sum(counts))
        t5 = tick()
        self.timings = {"broadcast_ms": 1e3 * (t1 - t0), "selfplay_ms": 1e3 * (t2 - t1), "pack_ms": 1e3 * (t3 - t2),
                        "gather_ms": 1e3 * (t4 - t3), "unpack_ms": 1e3 * (t5 - t4), "total_ms": 1e3 * (t5 - t0),
                        "gather_bytes": (sum(counts) - counts[dst]) * _eng.SAMPLE_BYTES if self.rank == dst else 0}
        return res


def sharded_self_play(model, n_games, sims=50, batch=8, seed=0, numerics=None, cycle_obj=None):
    """One self-play cycle over all ranks (see SelfPlayCycle).  Returns (result dict, the SelfPlayCycle that ran it:
    pass it back as `cycle_obj` to re-use the engine)."""
    c = cycle_obj or SelfPlayCycle(n_games, sims=sims, batch=batch, numerics=numerics)
    return c.run(model, seed=seed), c
