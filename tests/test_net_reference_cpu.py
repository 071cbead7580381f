"""CPU: the float64 reference of tests/net_reference.py -- its plain mode against the PyTorch module, its rounding
helpers against torch's casts, and the calibrated weight set against the properties that make faults visible."""
import numpy as np
import pytest
import torch

import net_reference as R


@pytest.fixture(scope="module")
def positions():
    sts = np.concatenate([R.playout_states(3, 777), R.edge_states(8, 5)])
    return R.planes_of(sts)


@pytest.fixture(scope="module")
def calibrated():
    return R.calibrated()


def _module_outputs(model, x):
    with torch.no_grad():
        p, v = model(x)
    return p, v[:, 0]


@pytest.mark.parametrize("net", ["random_init", "calibrated"])
def test_plain_mode_matches_the_module_in_float64(positions, net):
    import copy
    model = R.random_init() if net == "random_init" else R.calibrated()
    logits, pre = R.forward(model.state_dict(), positions, "fp32")
    p, v = _module_outputs(copy.deepcopy(model).double(), positions.double())
    assert (torch.softmax(logits, 1) - p).abs().max() <= 1e-10
    assert (torch.tanh(pre) - v).abs().max() <= 1e-10


def test_plain_mode_matches_the_module_in_float32(positions, calibrated):
    logits, pre = R.forward(calibrated.state_dict(), positions, "fp32")
    p, v = _module_outputs(calibrated, positions)
    assert p.dtype == torch.float32
    assert (torch.softmax(logits, 1) - p.double()).abs().max() <= 1e-5
    # (the value sums 256 hidden units of a head that is not damped as much: the fp32 module's own rounding reaches 1.03e-5)
    assert (torch.tanh(pre) - v.double()).abs().max() <= 2e-5


def _fp32_samples():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(200000, generator=g, dtype=torch.float64) * 10.0 ** torch.randint(-30, 30, (200000,), generator=g)
    # exact ties of bf16 (low 16 bits 0x8000) with an even and an odd last kept bit, and their neighbours
    bits = torch.randint(0x00800000, 0x7F000000, (20000,), generator=g, dtype=torch.int64) & ~0xFFFF
    ties = torch.cat([bits | 0x8000, bits | 0x18000, bits | 0x7FFF, bits | 0x8001, bits | 0x17FFF])
    ties = ties.to(torch.int32).view(torch.float32).to(torch.float64)
    return torch.cat([x, ties, -ties, torch.tensor([0.0, -0.0, 1.0, 3.0e38, 1e-40])]).to(torch.float32)


def test_bf16_rounding_matches_torch_bit_for_bit():
    x = _fp32_samples()
    mine = R.bf16_round(x).to(torch.float32)
    theirs = x.to(torch.bfloat16).to(torch.float32)
    assert torch.equal(mine.view(torch.int32), theirs.view(torch.int32))
    # round to nearest EVEN: 1 + 2^-8 lies halfway between 1 and 1 + 2^-7
    assert R.bf16_round(torch.tensor([1 + 2.0 ** -8, 1 + 3 * 2.0 ** -8])).tolist() == [1.0, 1 + 2 * 2.0 ** -7]
    # from float64 the value is rounded to fp32 first, as the kernels hold it
    assert torch.equal(R.bf16_round(x.double()), theirs.double())


def test_fp16_rounding_matches_torch_and_saturates():
    x = _fp32_samples()
    x = x[x.abs() < 65504.0]
    ties = torch.tensor([1 + 2.0 ** -11, 1 + 3 * 2.0 ** -11, 2048 + 1.0, 2048 + 3.0], dtype=torch.float32)
    for t in (x, ties):
        mine = R.fp16_satfinite(t).to(torch.float16)
        assert torch.equal(mine.view(torch.int16), t.to(torch.float16).view(torch.int16))
    assert R.fp16_satfinite(ties).tolist() == [1.0, 1 + 2 * 2.0 ** -10, 2048.0, 2052.0]
    # satfinite: what a plain cast turns into inf stays at the largest finite fp16
    big = torch.tensor([65504.0, 65519.0, 65520.0, 1e6, 3e38, -7e4])
    assert torch.isinf(big[2:].to(torch.float16)).all()
    assert R.fp16_satfinite(big).tolist() == [65504.0, 65504.0, 65504.0, 65504.0, 65504.0, -65504.0]


def test_splits_and_bias_terms():
    g = torch.Generator().manual_seed(4)
    x = (torch.randn(10000, generator=g) * 3).double()
    hi, lo = R.bf16_split(x)
    x32 = R.to_fp32(x)
    assert torch.equal(R.bf16_round(hi), hi) and torch.equal(R.bf16_round(lo), lo)
    assert ((hi + lo - x32).abs() <= x32.abs() * 2.0 ** -16).all()          # ~16 mantissa bits
    t2, t3 = R.bf16_terms(x, 2), R.bf16_terms(x, 3)
    assert torch.equal(t2[0], hi) and torch.equal(t2[1], lo) and torch.equal(t3[:2][1], lo)
    assert ((t3[0] + t3[1] + t3[2] - x32).abs() <= x32.abs() * 2.0 ** -24).all()


def test_emulated_modes_stay_near_the_plain_forward(positions, calibrated):
    """the emulations only add rounding: split-bf16 keeps about 16 bits, plain bf16 about 8"""
    sd = calibrated.state_dict()
    l64, v64 = R.forward(sd, positions, "fp32")
    for mode, tol in (("bf16x3", 2e-3), ("bf16", 0.5)):
        l, v = R.forward(sd, positions, mode)
        dl = np.abs(R.centered(l.numpy()) - R.centered(l64.numpy())).max()
        dv = (v - v64).abs().max().item()
        print("%s emulation vs plain float64: max|dlogit| %.2e max|dvalue| %.2e" % (mode, dl, dv))
        assert 0 < dl <= tol and 0 < dv <= tol


def test_calibrated_weight_set_properties(positions, calibrated):
    sd = calibrated.state_dict()
    stats = {}
    logits, pre = R.forward(sd, positions, "bf16", stats=stats)
    p = torch.softmax(logits, 1)
    print("calibrated: n=%d logit std %.2f max p %.3f min p %.2e |value pre| max %.2f, largest activation %.1f"
          % (len(p), logits.std(1).mean(), p.max(), p.min(), pre.abs().max(), stats["max_act"]))
    # logits: spread of about 1-2, softmax neither uniform nor one-hot, log p usable
    assert 1.0 <= logits.std(1).mean() <= 2.0
    assert p.max(1).values.min() > 2.0 / 81 and p.max() < 0.5 and p.min() > 1e-20
    assert (pre.abs() < 2).double().mean() >= 0.95
    # every bf16 activation well inside fp16 range (the skip connection is fp16)
    assert stats["max_act"] < 1000.0
    # nonzero biases in all three Linear layers
    for k in ("policy_fc.bias", "value_fc1.bias", "value_fc2.bias"):
        assert (sd[k] != 0).float().mean() >= 0.99, k
    # BatchNorm statistics far from the identity
    bns = [k[: -len(".weight")] for k in sd if k.endswith(".weight") and k[: -len(".weight")] + ".running_var" in sd]
    trunk = [k for k in bns if k.startswith(("bn_input", "residual_blocks"))]
    assert len(trunk) == 33 and all((sd[k + ".weight"] < 0).any() for k in trunk)
    assert (sd["policy_bn.weight"] < 0).any() and (sd["value_bn.weight"] < 0).any()
    var = torch.cat([sd[k + ".running_var"] for k in bns])
    assert var.min() < 2e-3 and var.max() > 5.0
    for k in bns:
        assert (sd[k + ".running_mean"] != 0).all() and (sd[k + ".bias"] != 0).all(), k
