"""ctypes binding of libuttt_b200.so (include/uttt_b200.h) and the host-side Engine object.

PyTorch is used only for device memory, streams and (optionally) torch.distributed; every
computation on the self-play path is a kernel of the CUDA library.  There is no CPU fallback:
creating an Engine without the built library or without an sm_100 GPU raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libuttt_b200.so")

EVAL_NET_BF16, EVAL_NET_FP32, EVAL_HASH, EVAL_HOST, EVAL_NET_BF16X3 = 0, 1, 2, 3, 4
NUMERICS = {"bf16": EVAL_NET_BF16, "bf16x3": EVAL_NET_BF16X3, "fp32": EVAL_NET_FP32}


def evaluator_of(numerics):
    """"bf16x3" (default of the drop-in modules: split-bf16 tcgen05 trunk, within 1e-2 of the fp32 reference forward on any
    weights), "bf16" (plain bf16 operands: 3x the throughput, within 1e-2 on trained weights only), "fp32" (CUDA cores)"""
    try:
        return NUMERICS[numerics]
    except KeyError:
        raise ValueError("numerics must be one of %s, not %r" % (sorted(NUMERICS), numerics)) from None


DEFAULT_NUMERICS = os.environ.get("UTTT_NUMERICS", "bf16x3")
SP_CORRECT_TERMINAL_SIGN = 1
SP_THROUGHPUT = 2
SP_PYSEARCH = 4
SP_RANDOM_SYMMETRY = 8     # evaluate every leaf under a random board symmetry (include/uttt_b200.h)
SP_MATCH = 16              # self-play as a match: weight slot (game + ply) & 1 moves (include/uttt_b200.h)
SP_RESIGN = 32             # a mover whose root value falls below the threshold resigns (include/uttt_b200.h)

_vp = C.c_void_p
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_F32 = np.float32


class UtttConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("n_slots", C.c_int32), ("max_sims", C.c_int32),
                ("max_batch", C.c_int32), ("max_games", C.c_int64)]


_WEIGHT_FIELDS = ["conv_input_w", "bn_input", "res_conv_w", "res_bn", "policy_conv_w", "policy_bn",
                  "policy_fc_w", "policy_fc_b", "value_conv_w", "value_bn", "value_fc1_w", "value_fc1_b",
                  "value_fc2_w", "value_fc2_b"]


class UtttWeights(C.Structure):
    _fields_ = [(n, _vp) for n in _WEIGHT_FIELDS]


class UtttWeightsScattered(C.Structure):
    _fields_ = [("small", UtttWeights), ("res_conv_w", _vp * 32), ("res_bn", (_vp * 4) * 32)]


# every symbol include/uttt_b200.h declares: name -> (argtypes, restype)
ABI = {
    "uttt_last_error": ([], C.c_char_p),
    "uttt_abi_version": ([], C.c_int),
    "uttt_device_check": ([C.c_int], C.c_int),
    "uttt_state_init": ([_u32p], C.c_int),
    "uttt_state_next": ([_u32p, C.c_int, _u32p], C.c_int),
    "uttt_state_legal_actions": ([_u32p, _i32p, C.POINTER(C.c_int)], C.c_int),
    "uttt_state_flags": ([_u32p, C.POINTER(C.c_int)], C.c_int),
    "uttt_state_encode": ([_u32p, _f32p], C.c_int),
    "uttt_state_to_string": ([_u32p, C.c_char_p, C.c_int, C.POINTER(C.c_int)], C.c_int),
    "uttt_state_symmetry": ([_u32p, C.c_int, _u32p, _vp], C.c_int),
    "uttt_game_step": ([_vp, _vp, _vp, C.c_int64, _vp], C.c_int),
    "uttt_game_legal_mask": ([_vp, _vp, _vp, C.c_int64, _vp], C.c_int),
    "uttt_game_encode": ([_vp, _vp, C.c_int64, _vp], C.c_int),
    "uttt_game_gather_planes": ([_vp, _vp, C.c_int64, _vp], C.c_int),
    "uttt_game_playout": ([C.c_uint32, C.c_uint64, C.c_int64, _vp, _vp, _vp, _vp], C.c_int),
    "uttt_create": ([C.POINTER(UtttConfig), C.POINTER(_vp)], C.c_int),
    "uttt_destroy": ([_vp], C.c_int),
    "uttt_upload_weights": ([_vp, C.POINTER(UtttWeights), C.c_int], C.c_int),
    "uttt_upload_weights_scattered": ([_vp, C.POINTER(UtttWeightsScattered), C.c_int], C.c_int),
    "uttt_upload_weights_slot": ([_vp, C.c_int, C.POINTER(UtttWeights), C.c_int], C.c_int),
    "uttt_upload_weights_scattered_slot": ([_vp, C.c_int, C.POINTER(UtttWeightsScattered), C.c_int], C.c_int),
    "uttt_net_forward": ([_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp], C.c_int),
    "uttt_mcts_search": ([_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_int32, _vp, _vp, _vp],
                         C.c_int),
    "uttt_set_root_noise": ([_vp, C.c_float, C.c_float], C.c_int),
    "uttt_set_selfplay_temperature": ([_vp, C.c_float], C.c_int),
    "uttt_set_progress_callback": ([_vp, _vp, _vp], C.c_int),
    "uttt_debug_dirichlet": ([C.c_uint32, C.c_uint64, C.c_int64, C.c_int32, C.c_float, _vp, _vp], C.c_int),
    "uttt_mcts_begin": ([_vp, _vp, C.c_int32, C.c_int32, C.c_int32], C.c_int),
    "uttt_mcts_advance": ([_vp, C.POINTER(C.c_int32)], C.c_int),
    "uttt_mcts_get_leaves": ([_vp, _vp, _vp, _vp], C.c_int),
    "uttt_mcts_put_results": ([_vp, _vp, _vp, C.c_int], C.c_int),
    "uttt_mcts_finish": ([_vp, C.c_float, _vp, _vp, _vp], C.c_int),
    "uttt_boltzman": ([_f32p, C.c_int32, C.c_float, _f32p], C.c_int),
    "uttt_selfplay_run": ([_vp, C.c_int64, C.c_uint64, C.c_int32, C.c_int32, C.c_uint32, C.c_int32, C.c_int32,
                           _vp, _vp, _vp, _vp, _vp, _vp], C.c_int),
    "uttt_selfplay_run_device": ([_vp, C.c_int64, C.c_uint64, C.c_int32, C.c_int32, C.c_uint32, C.c_int32,
                                  C.c_int32, _vp, _vp], C.c_int),
    "uttt_selfplay_fetch": ([_vp, C.c_int64, _vp, _vp, _vp, _vp, _vp], C.c_int),
    "uttt_set_resign": ([_vp, C.c_float, C.c_float], C.c_int),
    "uttt_selfplay_fetch_values": ([_vp, C.c_int64, _vp, _vp], C.c_int),
    "uttt_selfplay_pack": ([_vp, C.c_int64, _vp, C.c_int64, C.POINTER(C.c_int64), _vp], C.c_int),
    "uttt_samples_unpack": ([_vp, C.c_int64, _vp, _vp, _vp, _vp], C.c_int),
    "uttt_debug_trunk_timeline": ([_vp, _vp], C.c_int),
    "uttt_debug_batch_histogram": ([_vp, _vp, C.c_int32], C.c_int),
    "uttt_last_run_profile": ([_vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)], C.c_int),
    "uttt_set_profile_level": ([_vp, C.c_int], C.c_int),
    "uttt_debug_counters": ([_vp, _vp], C.c_int),
    "uttt_debug_trace": ([_vp, C.c_int], C.c_int),
    "uttt_debug_trace_read": ([_vp, C.c_int64, C.POINTER(C.c_int64), _vp, _vp, _vp, _vp], C.c_int),
}

PROGRESS_FN = C.CFUNCTYPE(None, C.c_int64, C.c_int64, _vp)
_lib = None


def load_library():
    """Load the CUDA library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libuttt_b200.so is not built (run `python __graft_entry__.py` or "
                              "`python ultimate-tictactoe-alphazero_b200/build.py`); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        for name, (argtypes, restype) in ABI.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def _check(rc):
    if rc != 0:
        raise RuntimeError("libuttt_b200: " + load_library().uttt_last_error().decode())


def _ptr(a):
    """device pointer of a torch tensor / host pointer of a numpy array / None"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    assert a.is_contiguous()
    return a.data_ptr()


def _stream(stream=None):
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream


# ------------------------------------------------------------------------------------ single-state helpers
def state_symmetry(state, g):
    """image of one packed state under board symmetry g (0..7: transpose if g >= 4, then numpy.rot90 by g % 4 of the 9x9
    picture) -> (packed state (8,) uint32, action map (81,) int32: [a] = the action at the image of action a's cell)"""
    st = np.ascontiguousarray(state, dtype=np.uint32).reshape(8)
    out = np.zeros(8, np.uint32)
    amap = np.zeros(81, np.int32)
    _check(load_library().uttt_state_symmetry(st, int(g), out, amap.ctypes.data))
    return out, amap


# ------------------------------------------------------------------------------------ rules on device tensors
def game_step(states, actions, out=None, stream=None):
    """states: cuda int32/uint32 (n,8); actions: cuda int32 (n,) -> next states (cpp/uttt_game.cpp:97-145)"""
    import torch
    out = torch.empty_like(states) if out is None else out
    _check(load_library().uttt_game_step(_ptr(states), _ptr(actions), _ptr(out), states.shape[0], _stream(stream)))
    return out


def game_legal_mask(states, stream=None):
    """-> (masks int32 (n,4): 3x27 action bits + count, status uint8 (n,)) (cpp/uttt_game.cpp:77-89,148-191)"""
    import torch
    n = states.shape[0]
    masks = torch.empty((n, 4), dtype=torch.int32, device=states.device)
    status = torch.empty((n,), dtype=torch.uint8, device=states.device)
    _check(load_library().uttt_game_legal_mask(_ptr(states), _ptr(masks), _ptr(status), n, _stream(stream)))
    return masks, status


def game_encode(states, stream=None, out=None):
    """-> float32 (n,9,9,3) HWC planes exactly like State.to_input_tensor (cpp/uttt_game.cpp:244-280);
    `out`: optional contiguous float32 destination of n*243 elements (any 4-byte alignment)"""
    import torch
    n = states.shape[0]
    planes = torch.empty((n, 9, 9, 3), dtype=torch.float32, device=states.device) if out is None else out
    _check(load_library().uttt_game_encode(_ptr(states), _ptr(planes), n, _stream(stream)))
    return planes


def game_gather_planes(states, stream=None, out=None):
    """-> bfloat16 (n,3,9,9) network input batch (pv_mcts_cpp.py:47-60);
    `out`: optional contiguous bfloat16 destination of n*243 elements (any 2-byte alignment)"""
    import torch
    n = states.shape[0]
    planes = torch.empty((n, 3, 9, 9), dtype=torch.bfloat16, device=states.device) if out is None else out
    _check(load_library().uttt_game_gather_planes(_ptr(states), _ptr(planes), n, _stream(stream)))
    return planes


def game_playout(seed, game0, n, device="cuda", stream=None):
    """n Philox random playouts -> (digests int64 (n,), plies int32, results int32)"""
    import torch
    dg = torch.empty((n,), dtype=torch.int64, device=device)
    pl = torch.empty((n,), dtype=torch.int32, device=device)
    rs = torch.empty((n,), dtype=torch.int32, device=device)
    _check(load_library().uttt_game_playout(seed, game0, n, _ptr(dg), _ptr(pl), _ptr(rs), _stream(stream)))
    return dg, pl, rs


def dirichlet_samples(seed, game0, n, n_children, alpha, device="cuda", stream=None):
    """(n, n_children) float32: the root-noise draws of games game0 .. game0 + n - 1 at ply 0 (diagnostics)"""
    import torch
    out = torch.empty((n, n_children), dtype=torch.float32, device=device)
    _check(load_library().uttt_debug_dirichlet(seed, game0, n, n_children, float(alpha), _ptr(out), _stream(stream)))
    return out


# ------------------------------------------------------------------------------------ weights
_SMALL_SHAPES = {"conv_input_w": (128, 3, 3, 3), "bn_input": (4, 128), "policy_conv_w": (2, 128), "policy_bn": (4, 2),
                 "policy_fc_w": (81, 162), "policy_fc_b": (81,), "value_conv_w": (1, 128), "value_bn": (4, 1),
                 "value_fc1_w": (256, 81), "value_fc1_b": (256,), "value_fc2_w": (1, 256), "value_fc2_b": (1,)}
_BN_KEYS = (".weight", ".bias", ".running_mean", ".running_var")


def _check_shapes(out, shapes):
    for k, shp in shapes.items():
        out[k] = np.ascontiguousarray(out[k], dtype=np.float32)
        if out[k].shape != shp:
            raise ValueError("state_dict tensor %s has shape %s, expected %s" % (k, out[k].shape, shp))
    return out


def _np(sd, k):
    return sd[k].detach().to("cpu").float().numpy()


def _bn(sd, prefix):
    return np.stack([_np(sd, prefix + k) for k in _BN_KEYS])


def pack_small(sd):
    """the 12 small arrays of the C ABI (everything but the residual tower) from a DualNetwork state_dict"""
    out = {
        "conv_input_w": _np(sd, "conv_input.weight"), "bn_input": _bn(sd, "bn_input"),
        "policy_conv_w": _np(sd, "policy_conv.weight").reshape(2, 128), "policy_bn": _bn(sd, "policy_bn"),
        "policy_fc_w": _np(sd, "policy_fc.weight"), "policy_fc_b": _np(sd, "policy_fc.bias"),
        "value_conv_w": _np(sd, "value_conv.weight").reshape(1, 128), "value_bn": _bn(sd, "value_bn"),
        "value_fc1_w": _np(sd, "value_fc1.weight"), "value_fc1_b": _np(sd, "value_fc1.bias"),
        "value_fc2_w": _np(sd, "value_fc2.weight"), "value_fc2_b": _np(sd, "value_fc2.bias"),
    }
    return _check_shapes(out, _SMALL_SHAPES)


def pack_state_dict(sd):
    """DualNetwork state_dict (dual_network.py:47-75; 216 entries) -> dict of the 14 contiguous fp32
    arrays the C ABI takes (numpy, host)."""
    n_blocks = 16
    out = pack_small(sd)
    out["res_conv_w"] = np.stack([np.stack([_np(sd, "residual_blocks.%d.conv1.weight" % i),
                                            _np(sd, "residual_blocks.%d.conv2.weight" % i)]) for i in range(n_blocks)])
    out["res_bn"] = np.stack([np.stack([_bn(sd, "residual_blocks.%d.bn1" % i), _bn(sd, "residual_blocks.%d.bn2" % i)])
                              for i in range(n_blocks)])
    return _check_shapes(out, {"res_conv_w": (16, 2, 128, 128, 3, 3), "res_bn": (16, 2, 4, 128)})


def scattered_residual_tensors(sd):
    """-> (32 conv tensors, 32 x 4 BatchNorm tensors) of the residual tower in layer order if every one of them is a
    contiguous fp32 tensor in host or CUDA memory (what torch.load(..., map_location=...) gives), else None"""
    import torch
    convs, bns = [], []
    for i in range(16):
        for j in (1, 2):
            convs.append(sd["residual_blocks.%d.conv%d.weight" % (i, j)])
            bns.append([sd["residual_blocks.%d.bn%d%s" % (i, j, k)] for k in _BN_KEYS])
    for t, shp in [(c, (128, 128, 3, 3)) for c in convs] + [(b, (128,)) for row in bns for b in row]:
        if not (isinstance(t, torch.Tensor) and t.dtype == torch.float32 and t.device.type in ("cpu", "cuda") and t.is_contiguous()):
            return None
        if tuple(t.shape) != shp:
            raise ValueError("state_dict tensor has shape %s, expected %s" % (tuple(t.shape), shp))
    return convs, bns


SAMPLE_BYTES = 196      # UTTT_SAMPLE_BYTES: packed position 32 B, visit counts u16[81], z int8, ply u8


def samples_unpack(samples, n=None, stream=None):
    """device uint8 buffer of packed samples -> (x (n,3,9,9) f32, policy (n,81) f32, value (n,1) f32) CUDA tensors: the
    arrays train_network.py:41-60 builds from the .history pickle"""
    import torch
    n = samples.numel() // SAMPLE_BYTES if n is None else int(n)
    x = torch.empty((n, 3, 9, 9), dtype=torch.float32, device=samples.device)
    p = torch.empty((n, 81), dtype=torch.float32, device=samples.device)
    v = torch.empty((n, 1), dtype=torch.float32, device=samples.device)
    _check(load_library().uttt_samples_unpack(_ptr(samples), n, _ptr(x), _ptr(p), _ptr(v), _stream(stream)))
    return x, p, v


def samples_to_numpy(samples):
    """host view of packed samples: (states (n,8) u32, counts (n,81) u16, z (n,) i8, ply (n,) u8)"""
    raw = np.ascontiguousarray(samples).view(np.uint8).reshape(-1, SAMPLE_BYTES)
    st = raw[:, :32].copy().view(np.uint32)
    cn = raw[:, 32:194].copy().view(np.uint16)
    return st, cn, raw[:, 194].copy().view(np.int8), raw[:, 195].copy()


def match_points(history, game0=0):
    """points of the network in weight slot 0 in the games of an SP_MATCH run (include/uttt_b200.h): 0.5 for a draw
    (final == 0), else 1 if the last mover -- slot (game + len - 1) & 1, game = game0 + i -- is slot 0 and 0 if not.
    `history`: a History or any object with `lens` and `final` arrays -> float64 array of n_games points"""
    lens = np.asarray(history.lens, np.int64)
    final = np.asarray(history.final)
    games = int(game0) + np.arange(len(lens), dtype=np.int64)
    last_mover = (games + lens - 1) & 1
    return np.where(final == 0, 0.5, np.where(last_mover == 0, 1.0, 0.0))


# ------------------------------------------------------------------------------------ resignation (host side)
def _philox4x32_x(k0, k1, c0, c1, c2, c3):
    """word x of Philox4x32-10 (the engine's counter-based generator, csrc/uttt_rules.cuh), vectorised over numpy
    uint64 arrays holding 32-bit values"""
    M = np.uint64(0xFFFFFFFF)
    k0, k1, c0, c1, c2, c3 = (np.asarray(a, np.uint64) & M for a in (k0, k1, c0, c1, c2, c3))
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M
        k0 = (k0 + np.uint64(0x9E3779B9)) & M
        k1 = (k1 + np.uint64(0xBB67AE85)) & M
    return c0


def check_games(seed, game0, n, check_fraction):
    """SP_RESIGN's check games among games game0 .. game0 + n - 1 -> bool array (n,): game g is a check game (never
    resigned) iff (philox4x32(key=(seed, 4), ctr=(g_lo, g_hi, 0, 0)).x >> 8) * 2^-24 < check_fraction (compared in fp32)"""
    g = np.uint64(int(game0)) + np.arange(int(n), dtype=np.uint64)
    x = _philox4x32_x(int(seed), 4, g & np.uint64(0xFFFFFFFF), g >> np.uint64(32), 0, 0)
    u = (x >> np.uint64(8)).astype(_F32) * _F32(1.0 / 16777216.0)
    return u < _F32(check_fraction)


def _recorded_values(history):
    """(values (n,81) f32, mask of the recorded rows): rows 0..len-1, plus row len of a resigned game"""
    lens = np.asarray(history.lens, np.int64)
    resigned = np.asarray(history.resigned) != 0
    last = lens + resigned - 1
    return np.asarray(history.values, _F32), np.arange(81)[None, :] <= last[:, None]


def would_resign_ply(history, threshold):
    """per game, the first ply p >= 1 whose recorded root value is below `threshold` (strictly, in fp32), over the rows
    `history` recorded (0..len-1, and row len of a game that resigned); -1 where there is none -> int64 array (n,).
    For a game played out with resignation off, p is where SP_RESIGN with that threshold would have ended it."""
    values, rec = _recorded_values(history)
    hit = rec & (values < _F32(threshold))
    hit[:, 0] = False
    return np.where(hit.any(axis=1), hit.argmax(axis=1), -1).astype(np.int64)


def _games(history, games):
    n = len(history.lens)
    idx = np.arange(n) if games is None else np.asarray(games)
    return np.nonzero(idx)[0] if idx.dtype == bool else idx.astype(np.int64)


def resign_calibration(history, threshold, games=None):
    """over the played-out games `games` (indices or a bool mask; None: all) of `history`: how many would resign with
    `threshold` (would_resign_ply >= 1) and how many of those are false positives -- the would-be resigner, the mover
    at that ply, did not lose the game (it won or drew) -> dict(games, would_resign, false_positives)"""
    g = _games(history, games)
    p = would_resign_ply(history, threshold)[g]
    w = p >= 1
    # the mover at ply p lost iff the final position is lost for its mover and (len - p) is even
    lost = (np.asarray(history.final)[g] == 1) & ((np.asarray(history.lens, np.int64)[g] - p) % 2 == 0)
    return {"games": int(len(g)), "would_resign": int(w.sum()), "false_positives": int((w & ~lost).sum())}


class _Rows:
    """the lens / final / values / resigned rows `g` of a history"""

    def __init__(self, history, g):
        self.lens = np.asarray(history.lens)[g]
        self.final = np.asarray(history.final)[g]
        self.values = np.asarray(history.values)[g]
        self.resigned = np.asarray(history.resigned)[g]


def resign_threshold(history, target_fp, games=None):
    """AlphaGo Zero's calibration: the largest threshold whose false-positive rate over the played-out games `games`
    (false positives / would-resign games, see resign_calibration) is at most `target_fp`.  Candidates are the distinct
    recorded root values of those games; a candidate that resigns no game does not qualify.  -> float, or -1.0 (never
    resigns: values are >= -1 and the rule is strict) if no candidate qualifies.  Calibrate on the check games of a run
    with resignation on and on all games of a run without it: resigned games have no known outcome."""
    h = _Rows(history, _games(history, games))
    values, rec = _recorded_values(h)
    cand = np.unique(values[rec])
    if len(cand) == 0:
        return -1.0
    # for a game, "resign if v < c" fires at the first ply p >= 1 whose value is below c: as c rises past each new low of
    # the running minimum over plies 1.., that ply moves to the ply of the low.  Candidate i (sorted) fires at the last
    # low l_k < cand[i], i.e. at the low's ply for every candidate above it up to and including the previous low.
    wr = np.zeros(len(cand) + 1, np.int64)
    fp = np.zeros(len(cand) + 1, np.int64)
    lens = np.asarray(h.lens, np.int64)
    for gi in range(len(lens)):
        prev = np.inf
        for p in np.nonzero(rec[gi])[0]:
            v = values[gi, p]
            if p == 0 or not v < prev:
                continue
            lo = np.searchsorted(cand, v, side="right")          # candidates c > v ...
            hi = np.searchsorted(cand, prev, side="right")       # ... and c <= the previous low
            lost = bool(h.final[gi] == 1 and (lens[gi] - p) % 2 == 0)
            wr[lo] += 1; wr[hi] -= 1
            if not lost:
                fp[lo] += 1; fp[hi] -= 1
            prev = v
    wr = np.cumsum(wr)[:-1]
    fp = np.cumsum(fp)[:-1]
    ok = (wr > 0) & (fp <= np.float64(target_fp) * wr)
    return float(cand[np.nonzero(ok)[0][-1]]) if ok.any() else -1.0


class History:
    """Packed self-play history of n_games games (host numpy arrays; rows = game*81 + ply)."""

    def __init__(self, n_games, pinned=True):
        import torch
        self.n_games = n_games
        self._keep = []
        pinned = pinned and torch.cuda.is_available()

        def alloc(shape, tdtype, view=None):
            t = torch.zeros(shape, dtype=tdtype)
            if pinned:
                t = t.pin_memory()
            self._keep.append(t)
            a = t.numpy()
            return a.view(view) if view is not None else a
        self.states = alloc((n_games, 81, 8), torch.int32, np.uint32)
        self.counts = alloc((n_games, 81, 81), torch.int16, np.uint16)
        self.actions = alloc((n_games, 81), torch.uint8)
        self.lens = alloc((n_games,), torch.int32)
        self.final = alloc((n_games,), torch.int8)
        self.values = alloc((n_games, 81), torch.float32)     # the mover's root value of every decided move
        self.resigned = alloc((n_games,), torch.int8)         # 1: the game ended by resignation (SP_RESIGN)
        self.stats = np.zeros(4, np.int64)

    @property
    def nbytes(self):
        return (self.states.nbytes + self.counts.nbytes + self.actions.nbytes + self.lens.nbytes + self.final.nbytes
                + self.values.nbytes + self.resigned.nbytes)

    def samples(self):
        """-> (states (N,8) uint32, counts (N,81) uint16, z (N,) int8) over all plies, game-major order.
        z follows self_play_cpp.py:95-99 verbatim (value of the FINAL position from its mover's view,
        assigned to ply 0 and alternating), i.e. the reference's labelling including its sign quirk."""
        lens = self.lens.astype(np.int64)
        mask = np.arange(81)[None, :] < lens[:, None]
        st = self.states[mask]
        cn = self.counts[mask]
        z0 = np.where(self.final != 0, -1, 0).astype(np.int8)
        sign = np.where((np.arange(81) % 2) == 0, 1, -1).astype(np.int8)
        z = (z0[:, None] * sign[None, :])[mask]
        return st, cn, z


class Engine:
    """Owns one uttt_engine handle on one GPU."""

    def __init__(self, n_slots=512, max_sims=50, max_batch=8, max_games=512, device=None):
        import torch
        self.lib = load_library()
        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        _check(self.lib.uttt_device_check(int(device)))
        cfg = UtttConfig(int(device), int(n_slots), int(max_sims), int(max_batch), int(max_games))
        h = _vp()
        _check(self.lib.uttt_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.cfg = cfg
        self.device = int(device)
        self.n_slots, self.max_sims, self.max_batch, self.max_games = n_slots, max_sims, max_batch, max_games
        self.weights_version = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.uttt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights
    def upload_state_dict(self, sd, slot=0):
        """best.pth state_dict -> device (BN folded, tensor-core layouts) into weight slot `slot`: 0 is what every evaluator
        reads, 1 the second network of match().  Contiguous fp32 tensors (host, pinned or not, or CUDA memory) are copied
        from where they lie; anything else goes through one packed host copy first."""
        if slot not in (0, 1):
            raise ValueError("weight slot must be 0 or 1, not %r" % (slot,))
        res = scattered_residual_tensors(sd)
        if res is None:
            packed = pack_state_dict(sd)
            w = UtttWeights(*[packed[k].ctypes.data for k in _WEIGHT_FIELDS])
            _check(self.lib.uttt_upload_weights_slot(self.h, slot, C.byref(w), 0))
            return
        small = pack_small(sd)
        w = UtttWeightsScattered()
        for k in _WEIGHT_FIELDS:
            if k in small:
                setattr(w.small, k, small[k].ctypes.data)
        convs, bns = res
        for l in range(32):
            w.res_conv_w[l] = convs[l].data_ptr()
            for j in range(4):
                w.res_bn[l][j] = bns[l][j].data_ptr()
        _check(self.lib.uttt_upload_weights_scattered_slot(self.h, slot, C.byref(w), 0))   # synchronous: sd may go away after

    def upload_model(self, model, slot=0):
        self.upload_state_dict(model.state_dict(), slot)

    # ---- network forward on packed states (cuda tensor (n,8) int32)
    def net_forward(self, states, mode=EVAL_NET_BF16, stream=None):
        import torch
        n = states.shape[0]
        pol = torch.empty((n, 81), dtype=torch.float32, device=states.device)
        val = torch.empty((n,), dtype=torch.float32, device=states.device)
        _check(self.lib.uttt_net_forward(self.h, _ptr(states), n, mode, _ptr(pol), _ptr(val), _stream(stream)))
        return pol, val

    # ---- search over many roots (host numpy in / out)
    def set_root_noise(self, alpha=0.3, eps=0.25):
        """Dirichlet root noise of the throughput mode (eps=0 disables)"""
        _check(self.lib.uttt_set_root_noise(self.h, float(alpha), float(eps)))

    def set_progress_callback(self, fn=None):
        """fn(done, total) is called from inside selfplay() whenever the number of finished games has changed"""
        self._progress = PROGRESS_FN(lambda done, total, user: fn(int(done), int(total))) if fn is not None else None
        _check(self.lib.uttt_set_progress_callback(self.h, C.cast(self._progress, _vp) if self._progress else None, None))

    def set_selfplay_temperature(self, temperature=1.0):
        """SP_TEMPERATURE of the self-play loop (1: the reference's setting; 0: always the most visited move)"""
        _check(self.lib.uttt_set_selfplay_temperature(self.h, float(temperature)))

    def set_resign(self, threshold=-0.95, check_fraction=0.1):
        """SP_RESIGN's threshold (a mover at ply >= 1 resigns when its root value is below it; in [-1, 1]) and the fraction
        of check games that are never resigned (in [0, 1]); see include/uttt_b200.h"""
        _check(self.lib.uttt_set_resign(self.h, float(threshold), float(check_fraction)))

    def mcts_search(self, roots, sims, batch, temperature, evaluator, flags=0):
        roots = np.ascontiguousarray(roots, dtype=np.uint32).reshape(-1, 8)
        n = roots.shape[0]
        scores = np.zeros((n, 81), np.float32)
        counts = np.zeros((n, 81), np.int32)
        ns = np.zeros((n,), np.int32)
        _check(self.lib.uttt_mcts_search(self.h, _ptr(roots), n, sims, batch, float(temperature), evaluator, flags,
                                         _ptr(scores), _ptr(counts), _ptr(ns)))
        return scores, counts, ns

    def mcts_search_host(self, roots, sims, batch, temperature, eval_fn, per_copy=False):
        """Step-wise search with a caller-side evaluator.
        eval_fn(states (m,8) uint32, k (m,) int32) -> (policy (m,81) or (m,max_batch,81), value (m,) or (m,max_batch))"""
        roots = np.ascontiguousarray(roots, dtype=np.uint32).reshape(-1, 8)
        n = roots.shape[0]
        _check(self.lib.uttt_mcts_begin(self.h, _ptr(roots), n, sims, batch))
        pend = C.c_int32(0)
        while True:
            _check(self.lib.uttt_mcts_advance(self.h, C.byref(pend)))
            m = pend.value
            if m == 0:
                break
            st = np.zeros((m, 8), np.uint32)
            k = np.zeros((m,), np.int32)
            tr = np.zeros((m,), np.int32)
            _check(self.lib.uttt_mcts_get_leaves(self.h, _ptr(st), _ptr(k), _ptr(tr)))
            pol, val = eval_fn(st, k)
            pol = np.ascontiguousarray(pol, dtype=np.float32)
            val = np.ascontiguousarray(val, dtype=np.float32)
            if per_copy:
                assert pol.shape == (m, self.max_batch, 81) and val.shape == (m, self.max_batch)
            else:
                assert pol.shape == (m, 81) and val.shape == (m,)
            _check(self.lib.uttt_mcts_put_results(self.h, _ptr(pol), _ptr(val), 1 if per_copy else 0))
        scores = np.zeros((n, 81), np.float32)
        counts = np.zeros((n, 81), np.int32)
        ns = np.zeros((n,), np.int32)
        _check(self.lib.uttt_mcts_finish(self.h, float(temperature), _ptr(scores), _ptr(counts), _ptr(ns)))
        return scores, counts, ns

    # ---- self-play
    def selfplay(self, n_games, sims=50, batch=8, seed=0, evaluator=EVAL_NET_BF16, flags=0, game0=0, history=None):
        """Runs n_games concurrent self-play games; returns a History with host copies of everything."""
        hist = history if history is not None else History(n_games)
        _check(self.lib.uttt_selfplay_run(self.h, n_games, game0, sims, batch, seed, evaluator, flags,
                                          _ptr(hist.states), _ptr(hist.counts), _ptr(hist.actions), _ptr(hist.lens),
                                          _ptr(hist.final), _ptr(hist.stats)))
        _check(self.lib.uttt_selfplay_fetch_values(self.h, n_games, _ptr(hist.values), _ptr(hist.resigned)))
        return hist

    def match(self, n_games, sims=50, batch=8, seed=0, evaluator=EVAL_NET_BF16, flags=0, game0=0, history=None):
        """A match between the networks of weight slots 0 and 1, all games on the device: selfplay() with SP_MATCH, so in
        game game0 + i slot (game0 + i + ply) & 1 moves (slot 0 first in even games).  `flags` may add SP_PYSEARCH (the
        reference gating match's search), SP_THROUGHPUT, SP_RANDOM_SYMMETRY, SP_CORRECT_TERMINAL_SIGN; the move draw is
        self-play's (set_selfplay_temperature).  -> (points, history): points[i] = match_points of slot 0 in game game0 + i."""
        hist = self.selfplay(n_games, sims=sims, batch=batch, seed=seed, evaluator=evaluator, flags=int(flags) | SP_MATCH,
                             game0=game0, history=history)
        return match_points(hist, game0)[:n_games], hist

    def selfplay_device(self, n_games, sims=50, batch=8, seed=0, evaluator=EVAL_NET_BF16, flags=0, game0=0,
                        stream=None):
        """Same loop, history stays in HBM (see selfplay_fetch). Returns stats [plies, sims, evals, rounds]."""
        stats = np.zeros(4, np.int64)
        s = _stream(stream) if stream is not None else None
        _check(self.lib.uttt_selfplay_run_device(self.h, n_games, game0, sims, batch, seed, evaluator, flags,
                                                 _ptr(stats), s))
        return stats

    def selfplay_fetch(self, n_games, history=None):
        hist = history if history is not None else History(n_games)
        _check(self.lib.uttt_selfplay_fetch(self.h, n_games, _ptr(hist.states), _ptr(hist.counts), _ptr(hist.actions),
                                            _ptr(hist.lens), _ptr(hist.final)))
        _check(self.lib.uttt_selfplay_fetch_values(self.h, n_games, _ptr(hist.values), _ptr(hist.resigned)))
        return hist

    def selfplay_pack(self, n_games, out=None, stream=None):
        """history of the last selfplay_device() as one device buffer of SAMPLE_BYTES-byte samples -> (uint8 CUDA tensor
        sliced to the exact length, n_samples).  `out`: optional uint8 CUDA tensor to pack into (81 * n_games samples fit)"""
        import torch
        cap = 81 * int(n_games)
        if out is None:
            out = torch.empty(cap * SAMPLE_BYTES, dtype=torch.uint8, device=torch.device("cuda", self.device))
        cap = out.numel() // SAMPLE_BYTES
        n = C.c_int64(0)
        _check(self.lib.uttt_selfplay_pack(self.h, int(n_games), _ptr(out), cap, C.byref(n), _stream(stream)))
        return out[: n.value * SAMPLE_BYTES], n.value

    def trunk_timeline(self):
        """clock64 stamps of CTA 0 of the last tcgen05 trunk launch: (32,4) = MMA start, MMA issued,
        accumulators ready, epilogue done"""
        out = np.zeros(128, np.int64)
        _check(self.lib.uttt_debug_trunk_timeline(self.h, _ptr(out)))
        return out.reshape(32, 4)

    def batch_histogram(self, reset=True):
        """launch counts of the tensor-core trunk by evaluator batch size, 64 buckets of 16 positions"""
        out = np.zeros(64, np.int64)
        _check(self.lib.uttt_debug_batch_histogram(self.h, _ptr(out), 1 if reset else 0))
        return out

    def counters(self):
        """device counters of the last search / self-play run: dict(plies, sims, evals, overflow, finished_trees, finished_games)"""
        out = np.zeros(8, np.uint64)
        _check(self.lib.uttt_debug_counters(self.h, _ptr(out)))
        return {"finished_games": int(out[1]), "plies": int(out[2]), "sims": int(out[3]), "evals": int(out[4]),
                "overflow": int(out[5]), "finished_trees": int(out[6])}

    def trace(self, enable=True):
        """start (and clear) / stop recording every evaluated leaf of the reference-exact search (diagnostics, slow)"""
        _check(self.lib.uttt_debug_trace(self.h, 1 if enable else 0))

    def trace_read(self):
        """-> (meta (n,3) int32 [tree, game index, ply], states (n,8) uint32, policy (n,81) f32, value (n,) f32)"""
        n = C.c_int64(0)
        _check(self.lib.uttt_debug_trace_read(self.h, 0, C.byref(n), None, None, None, None))
        n = n.value
        meta = np.zeros((n, 3), np.int32)
        st = np.zeros((n, 8), np.uint32)
        pol = np.zeros((n, 81), np.float32)
        val = np.zeros((n,), np.float32)
        if n:
            _check(self.lib.uttt_debug_trace_read(self.h, n, C.byref(n_ := C.c_int64(0)), _ptr(meta), _ptr(st), _ptr(pol), _ptr(val)))
        return meta, st, pol, val

    def set_profile_level(self, level):
        """0: no per-kernel events during self-play, 1 (default): the trunk only, 2: tree / trunk / heads"""
        _check(self.lib.uttt_set_profile_level(self.h, int(level)))

    def last_run_profile(self):
        """-> {kind: (ms, launches)} for tree / trunk / heads / all kernels of the last self-play run (ms: of the launches
        bracketed by CUDA events at the engine's profile level, launches: all), plus "trunk_timed": (ms, number, positions) of
        the trunk launches that were bracketed (profile level 1: every 4th window of rounds)"""
        out = {}
        for kind, name in enumerate(("tree", "trunk", "heads", "all")):
            ms, n = C.c_double(), C.c_int64()
            _check(self.lib.uttt_last_run_profile(self.h, kind, C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        ms, n, ev = C.c_double(), C.c_int64(), C.c_int64()
        _check(self.lib.uttt_last_run_profile(self.h, 4, C.byref(ms), C.byref(n)))
        _check(self.lib.uttt_last_run_profile(self.h, 5, None, C.byref(ev)))
        out["trunk_timed"] = (ms.value, n.value, ev.value)
        return out
