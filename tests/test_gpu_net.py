"""GPU: DualNetwork forward kernels vs the fp32 PyTorch module (the reference numerics,
dual_network.py:89-121) on the same weights.

Tolerance (BASELINE.json north_star): |policy - ref| <= 1e-2, |value - ref| <= 1e-2.
  * fp32 CUDA-core trunk ("parity numerics"): must meet it on the reference's RANDOM-INIT weights.
  * bf16x3 tcgen05 trunk (split-bf16 operands, fp32 accumulation and skip connection): must meet it on the RANDOM-INIT
    weights on every position, and on the outputs of the reference's own module (tests/golden/network.npz).
  * bf16 tcgen05 trunk: must meet it on a trained-like (damped) copy; on random-init weights the net is
    ill-conditioned (SURVEY.md H1: logits reach +-400, fp32 softmax is one-hot) and plain bf16 operands
    cannot meet 1e-2 on every position -- there we assert argmax agreement and the exceed fraction and
    print the statistics instead of silently loosening the bound.
    The damped copy's policy is close to uniform, so 1e-2 there is a smoke check, not the accuracy test: every forward
    path is compared row by row, in logit space, with a float64 emulation of its rounding in tests/test_gpu_net_reference.py.
"""
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

TOL = 1e-2


def _positions(n_games=24, seed=31337):
    sts = np.concatenate([O.playout_states(seed, g)[0][:-1] for g in range(n_games)])
    return sts


def _torch_reference(model, sts):
    import torch
    import engine
    planes = engine.game_encode(torch.from_numpy(sts.view(np.int32)).cuda()).cpu()    # (n,9,9,3), checked in test_gpu_rules
    x = planes.permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        p, v = model(x)                      # fp32 PyTorch on the host cores = the reference numerics
    return p.numpy(), v.numpy()[:, 0]


def _damped(model):
    """a 'trained-like' copy: residual branches damped so activations stay O(1) (SURVEY.md H1)"""
    import torch
    with torch.no_grad():
        for blk in model.residual_blocks:
            blk.bn2.weight.mul_(0.3)
        model.policy_fc.weight.mul_(0.05)
        model.value_fc1.weight.mul_(0.1)
        model.value_fc2.weight.mul_(0.2)
        # non-trivial BN statistics so that folding is exercised
        g = torch.Generator().manual_seed(5)
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
    return model


@pytest.fixture(scope="module")
def setup():
    import torch
    import engine
    from dual_network import DualNetwork
    torch.manual_seed(0)
    model = DualNetwork().eval()
    sts = _positions()
    e = engine.Engine(n_slots=256, max_sims=50, max_batch=8, max_games=16)
    yield e, model, sts
    e.close()


def _forward(e, sts, mode):
    import torch
    d = torch.from_numpy(sts.view(np.int32)).cuda()
    p, v = e.net_forward(d, mode)
    torch.cuda.synchronize()
    return p.cpu().numpy(), v.cpu().numpy()


def test_fp32_trunk_random_init_within_tolerance(setup):
    import engine
    e, model, sts = setup
    e.upload_model(model)
    pr, vr = _torch_reference(model, sts)
    p, v = _forward(e, sts, engine.EVAL_NET_FP32)
    perr, verr = np.abs(p - pr).max(), np.abs(v - vr).max()
    print("fp32 trunk, random init: n=%d max|dp|=%.3e max|dv|=%.3e" % (len(sts), perr, verr))
    assert np.allclose(p.sum(1), 1.0, atol=1e-4)
    assert perr <= TOL and verr <= TOL


def test_bf16x3_trunk_random_init_within_tolerance(setup, golden_dir):
    """the tensor-core mode that meets north_star's bar where plain bf16 cannot: all 1,407 random-init positions and the
    reference's own outputs (golden network.npz, minted from /root/reference/dual_network.py:89-121 by gen_golden.py)"""
    import engine
    e, model, sts = setup
    e.upload_model(model)
    pr, vr = _torch_reference(model, sts)
    p, v = _forward(e, sts, engine.EVAL_NET_BF16X3)
    perr, verr = np.abs(p - pr).max(), np.abs(v - vr).max()
    print("bf16x3 tcgen05 trunk, random init: n=%d max|dp|=%.3e max|dv|=%.3e argmax agreement %.4f"
          % (len(sts), perr, verr, (p.argmax(1) == pr.argmax(1)).mean()))
    assert len(sts) >= 1400 and np.allclose(p.sum(1), 1.0, atol=1e-4)
    assert perr <= TOL and verr <= TOL
    with np.load(os.path.join(golden_dir, "network.npz")) as z:
        g = {k: z[k] for k in z.files}
    pg, vg = _forward(e, g["states"], engine.EVAL_NET_BF16X3)
    print("bf16x3 vs reference golden: n=%d max|dp|=%.3e max|dv|=%.3e" % (len(g["states"]), np.abs(pg - g["policy"]).max(),
                                                                            np.abs(vg - g["value"]).max()))
    assert np.abs(pg - g["policy"]).max() <= TOL and np.abs(vg - g["value"]).max() <= TOL


def test_bf16x3_rows_do_not_depend_on_the_batch(setup):
    """one kernel, one arithmetic order per row: any batch size (1 .. several waves of 5-position groups) gives the same bits"""
    import engine
    e, model, sts = setup
    e.upload_model(model)
    big = np.concatenate([sts] * 2)[:1700]
    e3 = engine.Engine(n_slots=1700, max_sims=50, max_batch=8, max_games=8)
    try:
        e3.upload_model(model)
        full_p, full_v = _forward(e3, big, engine.EVAL_NET_BF16X3)
        for n in (1, 2, 4, 5, 6, 73, 74, 75, 148, 149, 222, 223, 296, 297, 370, 371, 500, 740, 741, 1111):
            p, v = _forward(e3, big[:n], engine.EVAL_NET_BF16X3)
            assert (p == full_p[:n]).all() and (v == full_v[:n]).all(), n
        p, v = _forward(e, big[:300], engine.EVAL_NET_BF16X3)          # another engine (256 slots: two calls), same bits
        assert (p == full_p[:300]).all() and (v == full_v[:300]).all()
    finally:
        e3.close()


def test_bf16x3_trained_like_and_selfplay(setup):
    import copy
    import engine
    e, model, sts = setup
    m2 = _damped(copy.deepcopy(model))
    e.upload_model(m2)
    pr, vr = _torch_reference(m2, sts)
    p, v = _forward(e, sts, engine.EVAL_NET_BF16X3)
    print("bf16x3 trained-like: max|dp|=%.2e max|dv|=%.2e" % (np.abs(p - pr).max(), np.abs(v - vr).max()))
    assert np.abs(p - pr).max() <= 1e-4 and np.abs(v - vr).max() <= 1e-4
    e.upload_model(model)
    h = e.selfplay(16, sims=50, batch=8, seed=3, evaluator=engine.EVAL_NET_BF16X3)
    assert (h.lens >= 17).all() and (h.lens <= 81).all() and (h.samples()[1].sum(1) == 50).all()
    h2 = e.selfplay(16, sims=50, batch=8, seed=3, evaluator=engine.EVAL_NET_BF16X3)
    assert (h.lens == h2.lens).all() and (h.actions == h2.actions).all() and (h.counts == h2.counts).all()


def test_bf16_trunk_random_init_statistics(setup):
    import engine
    e, model, sts = setup
    e.upload_model(model)
    pr, vr = _torch_reference(model, sts)
    p, v = _forward(e, sts, engine.EVAL_NET_BF16)
    perr = np.abs(p - pr).max(axis=1)
    verr = np.abs(v - vr)
    agree = (p.argmax(1) == pr.argmax(1)).mean()
    frac = (perr > TOL).mean()
    print("bf16 tcgen05 trunk, random init: n=%d argmax agreement %.3f, frac(|dp|>1e-2)=%.3f, max|dp|=%.3f, "
          "median|dp|=%.2e, max|dv|=%.3e" % (len(sts), agree, frac, perr.max(), np.median(perr), verr.max()))
    assert np.isfinite(p).all() and np.isfinite(v).all()
    assert np.allclose(p.sum(1), 1.0, atol=1e-4)
    assert agree >= 0.97 and frac <= 0.15


def test_bf16_trunk_trained_like_within_tolerance(setup):
    import engine
    e, model, sts = setup
    import copy
    m2 = _damped(copy.deepcopy(model))
    e.upload_model(m2)
    pr, vr = _torch_reference(m2, sts)
    p32, v32 = _forward(e, sts, engine.EVAL_NET_FP32)
    p, v = _forward(e, sts, engine.EVAL_NET_BF16)
    print("trained-like: fp32 max|dp|=%.2e max|dv|=%.2e ; bf16 max|dp|=%.2e max|dv|=%.2e"
          % (np.abs(p32 - pr).max(), np.abs(v32 - vr).max(), np.abs(p - pr).max(), np.abs(v - vr).max()))
    assert np.abs(p32 - pr).max() <= 1e-4 and np.abs(v32 - vr).max() <= 1e-4
    assert np.abs(p - pr).max() <= TOL and np.abs(v - vr).max() <= TOL


def test_forward_ragged_batches_are_row_independent(setup):
    """any batch size (incl. 1, non-multiples of 5 positions per CTA group, > n_slots) gives the same rows"""
    import engine
    e, model, sts = setup
    e.upload_model(model)
    full_p, full_v = _forward(e, sts[:300], engine.EVAL_NET_BF16)
    for n in (1, 4, 5, 6, 127, 256, 257):
        p, v = _forward(e, sts[:n], engine.EVAL_NET_BF16)
        assert (p == full_p[:n]).all() and (v == full_v[:n]).all()
    p32, _ = _forward(e, sts[:7], engine.EVAL_NET_FP32)
    q32, _ = _forward(e, sts[:300], engine.EVAL_NET_FP32)
    assert (p32 == q32[:7]).all()


def test_selfplay_with_network_produces_valid_history(setup):
    import torch
    import engine
    import self_play_cpp
    e, model, sts = setup
    e.upload_model(model)
    h = e.selfplay(16, sims=50, batch=8, seed=3, evaluator=engine.EVAL_NET_BF16)
    assert (h.lens >= 17).all() and (h.lens <= 81).all()
    st, cn, z = h.samples()
    assert (cn.sum(1) == 50).all()                       # sum of root visits == evaluate_count (Q-M4)
    # every recorded action was legal and visited
    masks, _ = engine.game_legal_mask(torch.from_numpy(st.view(np.int32)).cuda())
    masks = masks.cpu().numpy().view(np.uint32)
    acts = np.concatenate([h.actions[g, :h.lens[g]] for g in range(16)]).astype(np.int64)
    assert (((masks[np.arange(len(acts)), acts // 27] >> (acts % 27)) & 1) == 1).all()
    assert (cn[np.arange(len(acts)), acts] > 0).all()
    legal = np.stack([((masks[:, a // 27] >> (a % 27)) & 1) for a in range(81)], 1).astype(bool)
    assert (cn[~legal] == 0).all()
    # reference output format (self_play_cpp.py:34-101)
    xs, pis, zs = self_play_cpp._history_arrays(e, h)
    hist = self_play_cpp._to_reference_format(xs, pis, zs)
    assert len(hist) == h.lens.sum()
    x, pi, zz = hist[0]
    assert x.shape == (9, 9, 3) and x.dtype == np.float32 and pi.shape == (81,) and pi.dtype == np.float64
    assert isinstance(zz, int) and abs(pis.sum(1) - 1).max() < 1e-12
    assert (x[:, :, 2].sum() == 81) and x[:, :, :2].sum() == 0           # initial position


def test_drop_in_play_and_scores_api(setup):
    import uttt_cpp
    import pv_mcts_cpp
    import self_play_cpp
    e, model, sts = setup
    s = uttt_cpp.State()
    sc = pv_mcts_cpp.pv_mcts_scores_cpp(model, s, 1.0, 50, 8)
    assert sc.dtype == np.float64 and len(sc) == 81 and abs(sc.sum() - 1) < 1e-5
    sc0 = pv_mcts_cpp.pv_mcts_scores_cpp(model, s, 0, 50, 8)
    assert sorted(sc0.tolist())[-2:] == [0.0, 1.0]
    a = pv_mcts_cpp.pv_mcts_action_cpp(model, 1.0)(s)
    assert 0 <= int(a) < 81
    np.random.seed(0)
    hist = self_play_cpp.play(model)
    assert 17 <= len(hist) <= 81 and hist[0][1].shape == (81,)
    assert [h[2] for h in hist[:2]] in ([-1, 1], [0, 0])


def test_self_play_writes_reference_history_file(setup, tmp_path, monkeypatch):
    """self_play_cpp.self_play(): ./model/best.pth in, ./data/<timestamp>.history out, loadable the way
    train_network.py:21-60 loads it"""
    import pickle
    import torch
    import self_play_cpp
    from dual_network import dual_network
    monkeypatch.chdir(tmp_path)
    torch.manual_seed(1)
    dual_network()                                        # creates ./model/best.pth (dual_network.py:124-135)
    assert (tmp_path / "model" / "best.pth").exists()
    monkeypatch.setattr(self_play_cpp, "SP_GAME_COUNT", 24)
    monkeypatch.setattr(self_play_cpp, "SP_WRITE_PACKED", True)
    np.random.seed(7)
    path = self_play_cpp.self_play()
    files = sorted((tmp_path / "data").glob("*.history"))
    assert len(files) == 1 and str(files[0]).endswith(os.path.basename(path))
    with open(files[0], "rb") as f:
        history = pickle.load(f)
    xs, ps, vs = zip(*history)                            # train_network.py:44-49
    xs = np.array(xs).transpose(0, 3, 1, 2)
    ps, vs = np.array(ps), np.array(vs)
    assert xs.shape[1:] == (3, 9, 9) and xs.dtype == np.float32 and ps.shape[1] == 81 and ps.dtype == np.float64
    assert len(history) == self_play_cpp.last_stats["plies"] and set(np.unique(vs)) <= {-1, 0, 1}
    assert np.allclose(ps.sum(1), 1.0) and (ps[xs[:, 2].reshape(-1, 81)[:, _cell_to_action()] == 0] == 0).all()
    # the packed sidecar decodes to the same training arrays
    xs2, ps2, vs2 = self_play_cpp.load_packed_history(path.replace(".history", ".packed.npz"))
    assert (xs2 == xs).all() and np.allclose(ps2, ps, atol=1e-7) and (vs2 == vs).all()
    assert os.path.getsize(path.replace(".history", ".packed.npz")) < os.path.getsize(path) / 10
    # ... and the trainer drop-in prefers it over the pickle (same tensors either way)
    import train_network as tn
    a = tn.load_tensors()
    b = tn.history_to_tensors(tn.load_data())
    assert a[0].is_cuda and torch.equal(a[0], b[0]) and torch.allclose(a[1], b[1], atol=1e-7) and torch.equal(a[2], b[2])
    # the tensor feed gives the same layout without the pickle
    np.random.seed(7)
    x, p, v = self_play_cpp.history_tensors(torch.load("./model/best.pth", weights_only=True) and _load_best(), 24)
    assert x.shape[1:] == (3, 9, 9) and p.shape[1] == 81 and v.shape[1] == 1 and x.is_cuda


def _cell_to_action():
    # picture cell (R,C) -> action id, inverse used to index the policy by cell
    R, C = np.divmod(np.arange(81), 9)
    act = ((R // 3) * 3 + (C // 3)) * 9 + (R % 3) * 3 + (C % 3)
    inv = np.zeros(81, np.int64)
    inv[act] = np.arange(81)
    return inv


def _load_best():
    import torch
    from dual_network import DualNetwork
    m = DualNetwork()
    m.load_state_dict(torch.load("./model/best.pth", weights_only=True))
    return m.eval()


def test_fp32_trunk_vs_reference_golden_outputs(setup, golden_dir):
    """engine forward (fp32 numerics) vs outputs of the REFERENCE's own DualNetwork on its seed-0 random init"""
    import engine
    e, model, sts = setup          # `model` is DualNetwork() under torch.manual_seed(0): the golden's weights
    with np.load(os.path.join(golden_dir, "network.npz")) as z:
        g = {k: z[k] for k in z.files}
    e.upload_model(model)
    p, v = _forward(e, g["states"], engine.EVAL_NET_FP32)
    assert np.abs(p - g["policy"]).max() <= TOL and np.abs(v - g["value"]).max() <= TOL
    pb, vb = _forward(e, g["states"], engine.EVAL_NET_BF16)
    print("vs reference golden: fp32 max|dp|=%.2e max|dv|=%.2e ; bf16 argmax agreement %.3f max|dv|=%.2e" % (
        np.abs(p - g["policy"]).max(), np.abs(v - g["value"]).max(), (pb.argmax(1) == g["policy"].argmax(1)).mean(),
        np.abs(vb - g["value"]).max()))
    assert (pb.argmax(1) == g["policy"].argmax(1)).mean() >= 0.9


def test_trunk_variant_boundaries_give_identical_rows(setup):
    """The trunk kernel is chosen on the device from the batch size and the group sizes from ceil(n / pairs): every
    boundary of that dispatch must produce the same rows.  One launch that branches on the device (trunk_auto_kernel,
    net_auto.cu): one group per CTA pair up to 370 positions (net_tc2), two groups in flight above (net_pp), both with
    cta_group::2 MMAs on per-CTA weight halves.  All of them accumulate a row in the
    same order: bit-identical rows -- including the one-tile group of the 6/7-positions-per-pair case (371..518
    positions), whose weight stages are issued by one thread in quarter layers."""
    import copy
    import engine
    e, model, sts = setup
    big = np.concatenate([sts] * 5)[:1600]
    damped = _damped(copy.deepcopy(model))
    e3 = engine.Engine(n_slots=1600, max_sims=50, max_batch=8, max_games=8)
    try:
        for net in (model, damped):
            e3.upload_model(net)
            ref_p, ref_v = _forward(e3, big[:370], engine.EVAL_NET_BF16)     # one group per pair
            big_p, big_v = _forward(e3, big, engine.EVAL_NET_BF16)           # 3 super-groups of 2 x 5 positions on some pairs
            assert (big_p[:370] == ref_p).all() and (big_v[:370] == ref_v).all()
            for n in (1, 2, 3, 73, 74, 75, 147, 148, 149, 221, 222, 223, 295, 296, 297, 369, 370, 371, 372, 443, 444, 445,
                      500, 517, 518, 519, 520, 591, 592, 593, 665, 666, 667, 739, 740, 741, 800, 1111, 1480, 1481):
                p, v = _forward(e3, big[:n], engine.EVAL_NET_BF16)
                assert (p == big_p[:n]).all() and (v == big_v[:n]).all(), n
        e3.upload_model(model)
        ref_p, ref_v = _forward(e3, big[:800], engine.EVAL_NET_BF16)
        f32_p, _ = _forward(e3, big[:64], engine.EVAL_NET_FP32)
        assert (ref_p[:64].argmax(1) == f32_p.argmax(1)).mean() > 0.9
        same_n = (1, 2, 3, 7, 8, 74, 75, 149, 223, 300, 370, 371, 444, 445, 500, 518, 519, 800)
        ref_n = {n: _forward(e3, big[:n], engine.EVAL_NET_BF16) for n in same_n}
    finally:
        e3.close()
    # an engine whose batches cannot exceed one group per CTA pair (<= 518 rows: the 500-game cycle) runs the heads' FC
    # layers in the tail of the trunk kernel; e3 above (1600 rows) ran them as a separate kernel: same bits
    for rows in (518, 500, 8):
        ef = engine.Engine(n_slots=rows, max_sims=50, max_batch=8, max_games=8)
        try:
            ef.upload_model(model)
            for n in same_n:
                if n <= rows:
                    p, v = _forward(ef, big[:n], engine.EVAL_NET_BF16)
                    assert (p == ref_n[n][0]).all() and (v == ref_n[n][1]).all(), (rows, n)
        finally:
            ef.close()


def test_state_dict_upload_paths_give_identical_networks(setup):
    """uttt_upload_weights_scattered (contiguous host tensors read where they lie) == uttt_upload_weights (one packed
    host copy; taken for device-resident / non-contiguous / non-fp32 state_dicts) == device pointers"""
    import torch
    import engine
    e, model, sts = setup
    sd = {k: v.clone() for k, v in _damped(type(model)().eval()).state_dict().items()}
    assert engine.scattered_residual_tensors(sd) is not None
    e.upload_state_dict(sd)
    p0, v0 = _forward(e, sts[:300], engine.EVAL_NET_BF16)
    q0, w0 = _forward(e, sts[:64], engine.EVAL_NET_FP32)
    r0, x0 = _forward(e, sts[:300], engine.EVAL_NET_BF16X3)
    pinned = {k: v.pin_memory() for k, v in sd.items()}
    halves = {k: v.double() for k, v in sd.items()}                  # wrong dtype -> packed path (converted to fp32)
    on_gpu = {k: v.cuda() for k, v in sd.items()}                    # device tensors: read where they lie, too
    strided = {k: (torch.stack([v, v], -1)[..., 0] if v.dim() == 4 else v) for k, v in sd.items()}   # non-contiguous -> packed
    assert engine.scattered_residual_tensors(halves) is None and engine.scattered_residual_tensors(strided) is None
    assert engine.scattered_residual_tensors(on_gpu) is not None
    for other in (pinned, halves, on_gpu, strided):
        e.upload_state_dict({k: torch.zeros_like(v) for k, v in sd.items()})       # really replaced in between
        e.upload_state_dict(other)
        p, v = _forward(e, sts[:300], engine.EVAL_NET_BF16)
        q, w = _forward(e, sts[:64], engine.EVAL_NET_FP32)
        r, x = _forward(e, sts[:300], engine.EVAL_NET_BF16X3)
        assert (p == p0).all() and (v == v0).all() and (q == q0).all() and (w == w0).all()
        assert (r == r0).all() and (x == x0).all()
    bad = dict(sd)
    bad["residual_blocks.3.conv2.weight"] = torch.zeros(128, 64, 3, 3)
    with pytest.raises(ValueError):
        e.upload_state_dict(bad)


def test_profile_levels_and_identical_play(setup):
    """uttt_set_profile_level only changes which kernels are bracketed by CUDA events: same games, same launch counts"""
    import engine
    e, model, sts = setup
    e.upload_model(model)
    hists = []
    try:
        for level, tree_timed, trunk_timed in ((0, False, False), (1, False, True), (2, True, True)):
            e.set_profile_level(level)
            st = e.selfplay_device(12, sims=20, batch=8, seed=3, evaluator=engine.EVAL_NET_BF16)
            prof = e.last_run_profile()
            assert (prof["tree"][0] > 0) == tree_timed and (prof["trunk"][0] > 0) == trunk_timed, (level, prof)
            assert prof["trunk"][1] == st[3] and prof["all"][1] >= 2 * st[3]            # one trunk launch per round
            # the launches that were bracketed: none / every 4th window of 8 rounds / all, with the positions they evaluated
            t_ms, t_n, t_ev = prof["trunk_timed"]
            assert t_ms == prof["trunk"][0] and 0 <= t_ev <= st[2]
            assert t_n == (0 if level == 0 else (st[3] if level == 2 else 8 * ((st[3] // 8 + 3) // 4)))
            if level == 2:
                assert t_ev == st[2]
            h = e.selfplay_fetch(12)
            hists.append((h.lens.copy(), h.actions.copy(), h.counts.copy()))
        for other in hists[1:]:
            assert all((a == b).all() for a, b in zip(hists[0], other))
        with pytest.raises(RuntimeError):
            e.set_profile_level(3)
    finally:
        e.set_profile_level(1)


def test_network_selfplay_is_reproducible_run_to_run(setup):
    """Every bit of a self-play run is a function of the seed: the leaves of a round claim their evaluator rows in the
    order the warps arrive at an atomic counter, which differs from run to run, but a row does not depend on its place
    in the batch and each tree reads back its own row.  420 games on 420 slots keep the batches in the 371..518 band
    (the one-tile group of trunk_pp_body<1>); 200 games on 160 slots recycle slots (later games are claimed in arrival
    order too) and run two lanes, each with its own queue."""
    import engine
    e, model, sts = setup
    for slots, games, n_runs, lane_threshold in ((420, 420, 3, None), (160, 200, 2, "100")):
        if lane_threshold:
            os.environ["UTTT_LANE_THRESHOLD"] = lane_threshold
        try:
            eng = engine.Engine(n_slots=slots, max_sims=16, max_batch=8, max_games=games)
        finally:
            os.environ.pop("UTTT_LANE_THRESHOLD", None)
        try:
            eng.upload_model(model)
            runs = []
            for _ in range(n_runs):
                h = eng.selfplay(games, sims=16, batch=8, seed=5, evaluator=engine.EVAL_NET_BF16)
                assert (h.lens > 0).all()
                runs.append((h.lens.copy(), h.actions.copy(), h.counts.copy()))
            if games == 420:
                hist = eng.batch_histogram()
                assert hist[24:33].sum() > 0, hist             # launches with 384..527 positions did occur
            for other in runs[1:]:
                assert all((a == b).all() for a, b in zip(runs[0], other)), (slots, games)
        finally:
            eng.close()
