"""Float64 reference of the network forward in each numerics mode of the engine (TEST INFRASTRUCTURE ONLY).

`forward(sd, planes, mode)` takes a `DualNetwork` state_dict and (N, 3, 9, 9) board planes and returns float64 policy
logits (N, 81) and value pre-activations (N,).  It rounds exactly where the kernels round and computes everything else in
float64, so a kernel row differs from it only by the kernel's fp32 accumulation order (and the rare bf16 / fp16 rounding
that this order flips).  Where each rounding point comes from:

  fold (bf16, bf16x3)  scale = fp32(gamma / fp32(sqrt(fp32(var + 1e-5)))), shift = fp32(beta - fp32(mean * scale)), every
                       weight fp32(w * scale): weights.cu pack_res_kernel (__fdiv_rn / __fsqrt_rn / __fmul_rn / __fsub_rn)
                       for the residual layers, bn_fold and its callers in upload_weights for conv_input and the heads
  bf16                 3x3 weights bf16(w): weights.cu pack_res_kernel (__float2bfloat16), conv_input likewise in
                       upload_weights; BN shift as bf16(s) + bf16(s - bf16(s)) through the bias MMA: weights.cu, the bias
                       blocks (k < 2) in upload_weights, constant A rows (1, 1) in net_tc2_kernel.cuh / net_pp_kernel.cuh;
                       input planes bf16 (exact for 0 / 1); fp32 accumulation in TMEM (float64 here); after a block's
                       second conv the fp16 skip is added (f16x8_add2, tc_common.cuh); the next layer's A operand is
                       bf16(relu(v)) (relu_pack8_bf16); the skip is fp16(relu(v)) with satfinite (relu_pack8_f16), kept for
                       conv_input's and every block's output ("keep" in the epilogues); the last layer's relu(v) feeds the
                       1x1 head convs in fp32 (the `last` epilogue), the heads and FC layers are fp32 (heads_fc.cuh)
  bf16x3               weights hi = bf16(w), lo = bf16(fp32(w - hi)) (pack_res_kernel, upload_weights); activations x =
                       fp32(relu(v)), hi = bf16(x), lo = bf16(x - hi) (net_tc2_kernel.cuh, X3 epilogue: pack8_bf16,
                       bf16x8_residual); products hi*hi + lo*hi + hi*lo, no lo*lo (the three MMAs of the X3 issuer; the
                       input planes have no lo part); the skip connection is x in fp32 (f32x4_add); the shift is three bf16
                       terms (bias blocks k = 0, 1, 2, constant A row (1, 1, 1))
  fp32                 nothing is emulated: the plain float64 forward (BatchNorm folded in float64)

The weight sets: `random_init()` is the reference module's seed-0 initialisation (the weights of tests/golden/network.npz);
`calibrated()` is a damped copy whose faults show in the logits (see its docstring).
"""
import numpy as np
import torch
import torch.nn.functional as F

MODES = ("fp32", "bf16", "bf16x3")
EPS = 1e-5
FP16_MAX = 65504.0
N_BLOCKS = 16


# ---------------------------------------------------------------- rounding
def to_fp32(x):
    """round to fp32 (round to nearest even), as float64"""
    return x.to(torch.float32).to(torch.float64)


def bf16_round(x):
    """bf16(fp32(x)) with round to nearest even, as float64 -- what __float2bfloat16 / cvt.rn.bf16x2.f32 give for the
    finite fp32 values the kernels convert"""
    u = x.to(torch.float32).contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    u = u - ((u >> 31) << 32)                                    # back to the signed range of int32
    return u.to(torch.int32).view(torch.float32).to(torch.float64)


def fp16_satfinite(x):
    """fp16(fp32(x)) with round to nearest even, saturated to +-65504 (cvt.rn.satfinite.f16x2.f32), as float64"""
    return x.to(torch.float32).clamp(-FP16_MAX, FP16_MAX).to(torch.float16).to(torch.float64)


def bf16_split(x):
    """x in fp32 -> (hi, lo) = (bf16(x), bf16(x - hi)); x - hi is exact in fp32"""
    x32 = to_fp32(x)
    hi = bf16_round(x32)
    return hi, bf16_round(x32 - hi)


def bf16_terms(x, n):
    """x in fp32 as n bf16 terms, each the bf16 rounding of what the previous ones leave (weights.cu: the bias blocks)"""
    rest, out = to_fp32(x), []
    for _ in range(n):
        t = bf16_round(rest)
        out.append(t)
        rest = to_fp32(rest - t)
    return out


# ---------------------------------------------------------------- folding
def fold(sd, prefix, fp32):
    """eval-mode BatchNorm `prefix` -> (scale, shift) as float64; fp32: with the kernels' fp32 operations"""
    g, b, m, v = (sd[prefix + k].detach().to(torch.float64) for k in (".weight", ".bias", ".running_mean", ".running_var"))
    if not fp32:
        scale = g / torch.sqrt(v + EPS)
        return scale, b - m * scale
    f = lambda t: t.to(torch.float32)
    scale = f(g) / torch.sqrt(f(v) + np.float32(EPS))             # separate fp32 operations, each rounded once
    shift = f(b) - f(m) * scale
    return scale.to(torch.float64), shift.to(torch.float64)


def folded_conv(sd, conv, bn, fp32):
    """conv weight (co, ci, kh, kw) with its BatchNorm scale folded in, and the shift"""
    w = sd[conv + ".weight"].detach().to(torch.float64)
    scale, shift = fold(sd, bn, fp32)
    w = w * scale.view(-1, 1, 1, 1)
    return (to_fp32(w) if fp32 else w), shift


# ---------------------------------------------------------------- forward
def _conv(x, w):
    return F.conv2d(x, w, padding=w.shape[-1] // 2)


def _trunk_layer(mode, x, layer):
    """one 3x3 conv + BN shift on the activations `x` as the next layer's A operand sees them"""
    w, shift = layer
    if mode == "fp32":
        return _conv(x, w) + shift.view(1, -1, 1, 1)
    if mode == "bf16":
        hi, lo = bf16_terms(shift, 2)
        return _conv(x, bf16_round(w)) + (hi + lo).view(1, -1, 1, 1)
    whi, wlo = bf16_split(w)
    t = bf16_terms(shift, 3)
    xhi, xlo = x
    return (_conv(xhi, whi) + _conv(xlo, whi) + _conv(xhi, wlo)) + (t[0] + t[1] + t[2]).view(1, -1, 1, 1)


def _operand(mode, v):
    """relu(v) as the next layer's A operand"""
    r = torch.relu(v)
    if mode == "fp32":
        return r
    if mode == "bf16":
        return bf16_round(r)
    return bf16_split(r)


def _skip(mode, v):
    """relu(v) as the skip connection keeps it"""
    r = torch.relu(v)
    if mode == "fp32":
        return r
    if mode == "bf16":
        return fp16_satfinite(r)
    return to_fp32(r)


def layers_of(sd, mode):
    """the folded layers the kernels of `mode` read: conv_input, then conv1 / conv2 of every block, and the heads"""
    fp32 = mode != "fp32"
    trunk = [folded_conv(sd, "conv_input", "bn_input", fp32)]
    for i in range(N_BLOCKS):
        for j in (1, 2):
            trunk.append(folded_conv(sd, "residual_blocks.%d.conv%d" % (i, j), "residual_blocks.%d.bn%d" % (i, j), fp32))
    heads = (folded_conv(sd, "policy_conv", "policy_bn", fp32), folded_conv(sd, "value_conv", "value_bn", fp32))
    fc = {k: sd[k].detach().to(torch.float64) for k in ("policy_fc.weight", "policy_fc.bias", "value_fc1.weight",
                                                        "value_fc1.bias", "value_fc2.weight", "value_fc2.bias")}
    return trunk, heads, fc


def forward(sd, planes, mode="fp32", device=None, chunk=1024, stats=None):
    """-> (policy logits (N, 81), value pre-activations (N,)), float64 on the CPU.  `planes`: (N, 3, 9, 9) 0 / 1.
    stats: optional dict that receives the largest |relu(v)| of any trunk layer ("max_act")."""
    assert mode in MODES, mode
    device = torch.device(device or "cpu")
    trunk, heads, fc = layers_of(sd, mode)
    mv = lambda t: t.to(device)
    trunk = [(mv(w), mv(s)) for w, s in trunk]
    heads = [(mv(w), mv(s)) for w, s in heads]
    fc = {k: mv(t) for k, t in fc.items()}
    planes = torch.as_tensor(planes)
    logits, values, max_act = [], [], 0.0
    for c0 in range(0, len(planes), chunk):
        x = planes[c0:c0 + chunk].to(device=device, dtype=torch.float64)
        a = x if mode != "bf16x3" else (x, torch.zeros_like(x))   # the planes are exact in bf16: no lo part
        v = _trunk_layer(mode, a, trunk[0])
        for blk in range(N_BLOCKS):
            skip = _skip(mode, v)
            max_act = max(max_act, float(torch.relu(v).max()))
            h = _trunk_layer(mode, _operand(mode, v), trunk[1 + 2 * blk])
            max_act = max(max_act, float(torch.relu(h).max()))
            v = _trunk_layer(mode, _operand(mode, h), trunk[2 + 2 * blk]) + skip
        feat = torch.relu(v)
        max_act = max(max_act, float(feat.max()))
        (pw, ps), (vw, vs) = heads
        pf = torch.relu(_conv(feat, pw) + ps.view(1, -1, 1, 1)).flatten(1)
        vf = torch.relu(_conv(feat, vw) + vs.view(1, -1, 1, 1)).flatten(1)
        logits.append((pf @ fc["policy_fc.weight"].T + fc["policy_fc.bias"]).cpu())
        hid = torch.relu(vf @ fc["value_fc1.weight"].T + fc["value_fc1.bias"])
        values.append((hid @ fc["value_fc2.weight"].T + fc["value_fc2.bias"])[:, 0].cpu())
    if stats is not None:
        stats["max_act"] = max_act
    return torch.cat(logits), torch.cat(values)


# ---------------------------------------------------------------- logit space
def centered(logits):
    """policy logits up to their per-row constant: minus the row mean"""
    logits = np.asarray(logits, np.float64)
    return logits - logits.mean(1, keepdims=True)


def kernel_logits(p):
    """a softmax row back in logit space: log p minus its row mean"""
    return centered(np.log(np.asarray(p, np.float64)))


def value_residual(v, ref_pre, clip=0.95, signed=False):
    """atanh(v) - pre-activation where |v| < clip (the kernel's tanh is invertible there), v - tanh(pre) elsewhere;
    absolute values unless `signed`"""
    v = np.asarray(v, np.float64)
    ref_pre = np.asarray(ref_pre, np.float64)
    inner = np.abs(v) < clip
    out = v - np.tanh(ref_pre)
    out[inner] = np.arctanh(v[inner]) - ref_pre[inner]
    return out if signed else np.abs(out)


# ---------------------------------------------------------------- weight sets
def random_init(seed=0):
    """the reference module's initialisation under torch.manual_seed(seed) (seed 0: tests/golden/network.npz)"""
    from dual_network import DualNetwork
    torch.manual_seed(seed)
    return DualNetwork().eval()


def calibrated(seed=0):
    """A copy of random_init(seed) on which a fault moves the logits well above the kernels' rounding noise:
      * the residual branches damped as tests/test_gpu_net.py's _damped does (bn2's gamma x 0.3), so activations stay
        O(1) through the 16 blocks;
      * the policy FC scaled so the logits have a standard deviation of about 1.5 (the softmax is neither uniform nor
        one-hot, and log p is finite), the value FCs so that |value pre-activation| is mostly below 2;
      * nonzero biases in all three Linear layers;
      * BatchNorm statistics far from the identity: running_var log-uniform over [1e-3, 10], gamma = +-sqrt(var) times
        U(0.6, 1.4) (so the folded scale stays O(1)) with about a fifth of the trunk's channels and one channel of each
        head BN negative, nonzero running means and betas.  The head convs whose gamma is negative are negated too, so
        their features stay alive."""
    model = random_init(seed)
    g = torch.Generator().manual_seed(1000 + seed)
    with torch.no_grad():
        for name, m in model.named_modules():
            if not isinstance(m, torch.nn.BatchNorm2d):
                continue
            c = m.num_features
            var = 10.0 ** (torch.rand(c, generator=g) * 4.0 - 3.0)
            mag = torch.sqrt(var + EPS) * (0.6 + 0.8 * torch.rand(c, generator=g))
            sign = torch.where(torch.rand(c, generator=g) < 0.2, -1.0, 1.0)
            if name in ("policy_bn", "value_bn"):
                sign = torch.ones(c)
                sign[-1] = -1.0                                  # one channel of each head BN
            m.running_var.copy_(var)
            m.weight.copy_(sign * mag)
            m.running_mean.copy_(torch.randn(c, generator=g) * 0.5 * torch.sqrt(var))
            m.bias.copy_(torch.randn(c, generator=g) * 0.2)
        for blk in model.residual_blocks:
            blk.bn2.weight.mul_(0.3)
        model.policy_conv.weight[-1].neg_()
        model.value_conv.weight[-1].neg_()
        model.policy_fc.weight.mul_(0.18)
        model.policy_fc.bias.copy_(torch.randn(81, generator=g) * 0.5)
        model.value_fc1.weight.mul_(0.2)
        model.value_fc1.bias.copy_(torch.randn(256, generator=g) * 0.1)
        model.value_fc2.weight.mul_(0.8)
        # value_fc2's bias centres the value: pre-activation 0.1 at the initial position (empty board, all cells legal)
        model.value_fc2.bias.zero_()
        start = torch.zeros(1, 3, 9, 9, dtype=torch.float64)
        start[:, 2] = 1.0
        model.value_fc2.bias.fill_(0.1 - float(forward(model.state_dict(), start)[1][0]))
    return model


# ---------------------------------------------------------------- positions (packed states, oracle_lib's format)
def playout_states(n_games, seed):
    """every position of `n_games` seeded playouts, the terminal ones included, without repeats (in first-seen order)"""
    import oracle_lib as O
    sts = np.concatenate([O.playout_states(seed, g)[0] for g in range(n_games)])
    _, first = np.unique(sts, axis=0, return_index=True)
    return sts[np.sort(first)]


def terminal_states(n_games, seed):
    import oracle_lib as O
    return np.stack([O.playout_states(seed, g)[0][-1] for g in range(n_games)])


def edge_states(n, seed):
    """positions with every cell of the picture's border (rows 0, 8, columns 0, 8) occupied, by a random player, and a
    third of the inner cells too: the rows next to the padding between positions in the kernels' GEMM layout"""
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 8), np.uint32)
    for i in range(n):
        for R in range(9):
            for C in range(9):
                if not (R in (0, 8) or C in (0, 8) or rng.random() < 1 / 3):
                    continue
                b, c = (R // 3) * 3 + C // 3, (R % 3) * 3 + C % 3
                out[i, (b // 3) + (3 if rng.random() < 0.5 else 0)] |= np.uint32(1 << ((b % 3) * 9 + c))
    return out


def planes_of(states):
    """(N, 3, 9, 9) float32 input planes of packed states, by the oracle's encoder"""
    import oracle_lib as O
    t = np.stack([O.oracle_probe(w)[2] for w in states]).reshape(-1, 9, 9, 3)
    return torch.from_numpy(t).permute(0, 3, 1, 2).contiguous()
