"""GPU: every row of every network forward path against the float64 reference of tests/net_reference.py, in logit space.

The reference rounds where the kernels round (bf16, bf16x3) or not at all (fp32), so what is left between a kernel row and
its reference row is the kernel's fp32 accumulation order and the rare bf16 / fp16 rounding that this order flips.  The
comparison is made where faults are visible:
  * policy: log p minus its row mean against the reference logits minus theirs (the kernels return an fp32 softmax);
  * value: atanh(v) against the reference pre-activation where |v| < 0.95, v against tanh(pre-activation) elsewhere.
on the calibrated weight set (net_reference.calibrated: logits of standard deviation ~1.7, nonzero FC biases, negative BN
gammas, running variances from 1e-3 to 10) and, for bf16 and bf16x3, the seed-0 random init.

uttt_net_forward cuts a batch into calls of at most n_slots rows, and each call picks its path from its row count m
(engine.cu run_evaluator, net_auto.cu): bf16 m <= 370 trunk_auto_kernel's tc2 body, 371..518 its pp<1> body (two
groups per CTA pair), both with the heads' FC layers fused into the kernel's tail; m > 518 trunk_pp_large_kernel and the
separate heads_fc_kernel.  bf16x3: trunk_x3_kernel, one wave of 74 groups of <= 5 positions per 370 rows, then
heads_fc_kernel.  fp32: conv3x3_fp32_kernel and the fp32 heads.  (On a B200: 148 SMs, 74 CTA pairs.)

Bounds: each is set from the largest residual measured on a B200 (recorded next to BOUND), and sits at least 3x below
the signals of the faults this file was checked against (the lo term of the BN shift, two swapped weight taps, a skip
chunk, a wrong head shift, an FC bias, a conv tap) -- except the bf16 row bound, see BOUND.
"""
import numpy as np
import pytest

import net_reference as R

pytestmark = pytest.mark.gpu

# Bounds.  "row": the largest residual of any row (policy |dlogit|, value).  "mean": over every row of a check of at least
# MEAN_ROWS rows, the mean signed residual of each logit (the largest of the 81) and of the value.  Measured on an NVIDIA
# B200 (1000 W power limit) over every row of this file, calibrated net:
#   bf16    row 7.27e-2 / 1.38e-1   mean 5.8e-4 / 2.8e-4
#   bf16x3  row 1.44e-4 / 2.95e-4   mean 4.4e-5 / 8.2e-5
#   fp32    row 1.54e-5 / 2.23e-5   (1,784 rows: no mean check)
# bf16 has no better row bound: the net is chaotic under bf16 rounding.  A perturbation of 1e-7 of every pre-activation
# (below one fp32 ulp) moves the emulated logits by up to 7e-2, as far as rounding every activation to bf16 does, so the
# kernel's fp32 accumulation order alone leaves residuals of that size.  A row bound there cannot see a fault smaller than
# that (dropping the lo term of the BN shift: 7.6e-2), but such a fault is systematic and the noise is not: over the ~3,800
# positions of a check the mean residual is 5.8e-4 clean and 7.3e-3 with that fault.
BOUND = {
    "bf16": {"row": (0.1, 0.18), "mean": (2e-3, 2e-3)},
    "bf16x3": {"row": (5e-4, 1e-3), "mean": (2e-4, 3e-4)},
    "fp32": {"row": (1e-4, 1e-4), "mean": (1e-5, 1e-5)},
}
MEAN_ROWS = 3000
# random init, all 3,776 positions: argmax agreement with the emulated reference (measured 0.9730 / 1.0000) and, for
# bf16x3, max |v - tanh(reference pre-activation)| (measured 8.7e-4).  bf16 gets no value bound: on these ill-conditioned
# weights the same sub-ulp differences flip a value outright (measured max 1.7), so it is printed only.
RANDOM_INIT_AGREEMENT = {"bf16": 0.96, "bf16x3": 0.999}
RANDOM_INIT_VALUE = {"bf16x3": 3e-3}

# the trunk dispatch's boundaries (test_gpu_net.py::test_trunk_variant_boundaries_give_identical_rows)
BOUNDARY_N = (1, 2, 3, 73, 74, 75, 147, 148, 149, 221, 222, 223, 295, 296, 297, 369, 370, 371, 372, 443, 444, 445,
              500, 517, 518, 519, 520, 591, 592, 593, 665, 666, 667, 739, 740, 741, 800, 1111, 1480, 1481)
FUSED_SLOTS, LARGE_SLOTS = 518, 1600


@pytest.fixture(scope="module")
def env():
    import torch
    import engine
    sts = np.concatenate([R.playout_states(64, 4242), R.edge_states(16, 9)])        # initial + terminal positions included
    _, first = np.unique(sts, axis=0, return_index=True)
    sts = sts[np.sort(first)]
    d = torch.from_numpy(sts.view(np.int32)).cuda()
    planes = engine.game_encode(d).permute(0, 3, 1, 2).contiguous()                # what the kernels read
    nets = {"calibrated": R.calibrated(), "random_init": R.random_init()}
    engines = {n: engine.Engine(n_slots=n, max_sims=50, max_batch=8, max_games=8) for n in (256, FUSED_SLOTS, LARGE_SLOTS)}
    refs, loaded = {}, {}

    def ref(net, mode):
        if (net, mode) not in refs:
            refs[(net, mode)] = tuple(t.numpy() for t in R.forward(nets[net].state_dict(), planes, mode, device="cuda"))
        return refs[(net, mode)]

    def forward(slots, net, rows, mode):
        e = engines[slots]
        if loaded.get(slots) != net:
            e.upload_model(nets[net])
            loaded[slots] = net
        p, v = e.net_forward(d[torch.from_numpy(np.asarray(rows)).cuda()], mode)
        torch.cuda.synchronize()
        return p.cpu().numpy(), v.cpu().numpy()

    yield sts, ref, forward
    for e in engines.values():
        e.close()


def _rows(n_all, n, k):
    """n distinct positions, the k-th window: consecutive batches see different positions"""
    start = (k * 997) % n_all
    return (start + np.arange(n)) % n_all


def _check(env, mode, slots, sizes, net="calibrated", label=""):
    """every row of batches of `sizes` rows through the engine of `slots` slots against the reference: the largest
    residual of a row, and -- over every row checked -- the mean signed residual of each logit and of the value"""
    sts, ref, forward = env
    import engine
    ev = {"bf16": engine.EVAL_NET_BF16, "bf16x3": engine.EVAL_NET_BF16X3, "fp32": engine.EVAL_NET_FP32}[mode]
    ref_l, ref_v = ref(net, mode)
    worst = []
    sum_l, sum_v, n_rows = np.zeros(81), 0.0, 0
    for k, n in enumerate(sizes):
        rows = _rows(len(sts), n, k)
        p, v = forward(slots, net, rows, ev)
        assert np.isfinite(p).all() and np.isfinite(v).all() and (p > 0).all(), (mode, slots, n)
        dl = R.kernel_logits(p) - R.centered(ref_l[rows])
        dv = R.value_residual(v, ref_v[rows], signed=True)
        worst.append((np.abs(dl).max(), np.abs(dv).max(), n))
        sum_l, sum_v, n_rows = sum_l + dl.sum(0), sum_v + dv.sum(), n_rows + n
    row_l, row_v = max(w[0] for w in worst), max(w[1] for w in worst)
    mean_l, mean_v = np.abs(sum_l / n_rows).max(), abs(sum_v / n_rows)
    print("%-7s engine %4d slots, %2d batches, %6d rows%s: max|dlogit| %.3e  max|dvalue| %.3e  |mean dlogit| %.3e  "
          "|mean dvalue| %.3e" % (mode, slots, len(sizes), n_rows, label, row_l, row_v, mean_l, mean_v))
    b = BOUND[mode]
    assert row_l <= b["row"][0] and row_v <= b["row"][1], [w for w in worst if w[0] > b["row"][0] or w[1] > b["row"][1]]
    if n_rows >= MEAN_ROWS:
        assert mean_l <= b["mean"][0] and mean_v <= b["mean"][1]


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_fused_heads_engine_rows_match_emulation(env, mode):
    """<= 518 rows per call: tc2 (<= 370) and pp<1> (371..518) with fused heads (bf16); x3 one and two waves"""
    _check(env, mode, FUSED_SLOTS, [n for n in BOUNDARY_N if n <= FUSED_SLOTS] + [FUSED_SLOTS])


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_large_engine_rows_match_emulation(env, mode):
    """up to 1600 rows per call: every band of the dispatch, trunk_pp_large_kernel + heads_fc_kernel above 518 (bf16),
    up to five waves of x3 groups"""
    _check(env, mode, LARGE_SLOTS, list(BOUNDARY_N) + [LARGE_SLOTS])


def test_fp32_rows_match_float64(env):
    _check(env, "fp32", LARGE_SLOTS, (1, 7, 8, 255, 256, 257, 1000))


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_batches_larger_than_the_engine_are_chunked_correctly(env, mode):
    """700 rows through 256 slots: calls of 256, 256 and 188 rows; the rows on both sides of each cut are in the check,
    and also compared alone"""
    sts, ref, forward = env
    _check(env, mode, 256, (700,), label=" (chunked)")
    import engine
    ev = engine.EVAL_NET_BF16 if mode == "bf16" else engine.EVAL_NET_BF16X3
    rows = _rows(len(sts), 700, 0)
    p, v = forward(256, "calibrated", rows, ev)
    cut = [254, 255, 256, 257, 510, 511, 512, 513]
    q, w = forward(LARGE_SLOTS, "calibrated", rows[cut], ev)
    assert (q == p[cut]).all() and (w == v[cut]).all()


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_rows_do_not_depend_on_their_neighbours(env, mode):
    """the same positions in reversed and in shuffled order give the same bits per position: nothing leaks across the
    halo rows or the padding rows between positions of a group"""
    sts, ref, forward = env
    import engine
    ev = engine.EVAL_NET_BF16 if mode == "bf16" else engine.EVAL_NET_BF16X3
    rng = np.random.default_rng(11)
    for n in (300, 500, 1200):                         # tc2, pp<1>, pp_large (bf16); one, two and four x3 waves
        rows = _rows(len(sts), n, n)
        p, v = forward(LARGE_SLOTS, "calibrated", rows, ev)
        for order in (np.arange(n)[::-1], rng.permutation(n)):
            q, w = forward(LARGE_SLOTS, "calibrated", rows[order], ev)
            assert (q == p[order]).all() and (w == v[order]).all(), (mode, n)


@pytest.mark.parametrize("mode", ["bf16", "bf16x3"])
def test_random_init_against_emulation(env, mode):
    """the ill-conditioned seed-0 weights (logits up to +-400: log p is not usable): argmax agreement with the emulated
    reference and (bf16x3) a bound on the value, over every position in calls of up to 1600 rows"""
    sts, ref, forward = env
    import engine
    ev = engine.EVAL_NET_BF16 if mode == "bf16" else engine.EVAL_NET_BF16X3
    ref_l, ref_v = ref("random_init", mode)
    rows = np.arange(len(sts))
    p, v = forward(LARGE_SLOTS, "random_init", rows, ev)
    assert np.isfinite(p).all() and np.isfinite(v).all()
    agree = (p.argmax(1) == ref_l.argmax(1)).mean()
    dv = np.abs(v - np.tanh(ref_v))                  # (the pre-activations reach +-100: compared as values)
    print("%-7s random init, engine %4d slots, %6d rows: argmax agreement %.4f  max|dvalue| %.3e  "
          "frac(|dvalue| > 1e-2) %.4f" % (mode, LARGE_SLOTS, len(rows), agree, dv.max(), (dv > 1e-2).mean()))
    assert agree >= RANDOM_INIT_AGREEMENT[mode]
    if mode in RANDOM_INIT_VALUE:
        assert dv.max() <= RANDOM_INIT_VALUE[mode]
