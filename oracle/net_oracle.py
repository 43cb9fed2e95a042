"""fp64 ORACLE for the floating-point kernels (TEST INFRASTRUCTURE): the trunks (csrc/trunk_rows.cu,
csrc/trunk.cu, csrc/trunk_wide.cu), the fused heads (csrc/heads.cu) and the policy head on the legal moves
(policy_legal_kernel, csrc/mcts.cu), restated from the torch modules of architectures.py.

Everything is computed in float64 on the device of the inputs.  With `rounding=True` (the default) the
oracle rounds where the kernels round, and nowhere else:
  * folded weights: BatchNorm scale times weight in fp32 (as the packers in trunk.py / trunk_wide.py compute
    them), then to bf16 where a kernel feeds them to the tensor core, fp32 where it reads them in an epilogue;
  * activations: fp64 -> fp32 -> bf16 (the cast chain of cvt.rn) at each bf16 store, fp64 -> fp32 where a
    kernel keeps an fp32 value (a TMEM accumulator, an fp32 register sum).
The remaining difference to a kernel is the order of its fp32 accumulation, so most bf16 outputs agree bit
for bit.  With `rounding=False` every function is the module's eval-mode forward in pure fp64.

The oracle reads the torch module, never the packed buffers: a packing bug shows up as kernel != oracle.
"""
import torch
import torch.nn.functional as F

from tetris_reinforcement_learning_b200.architectures import CELLS, SIDE_FEATS

K_IN = CELLS + 16 + 2 * SIDE_FEATS + 1      # 521 inputs of AlphaSame's heads (kernels = 1, o_side_neurons = 16)
K_PAD = 528                                 # x row of csrc/heads.cu: 7 zero columns after the inputs


def _bf16(v, rounding):
    return v.float().bfloat16().double() if rounding else v


def _fp32(v, rounding):
    return v.float().double() if rounding else v


def _dtype(rounding):
    """Arithmetic of the weight folding: the packers' fp32, or fp64."""
    return torch.float32 if rounding else torch.float64


def _param(t, device, rounding):
    return t.detach().to(device=device, dtype=_dtype(rounding))


def fold_bn(bn, device, rounding=True):
    """Eval-mode BatchNorm as y = s * x + b per channel: s = gamma / sqrt(var + eps), b = beta - mean * s.
    (fp32 like trunk._fold_bn with rounding, else fp64.)"""
    g, beta, mean, var = (_param(t, device, rounding) for t in (bn.weight, bn.bias, bn.running_mean, bn.running_var))
    s = g / torch.sqrt(var + bn.eps)
    return s, beta - mean * s


def fold_linear_bn(linear, bn, device, rounding=True):
    """Linear followed by eval-mode BatchNorm1d -> (W * s[:, None], bias * s + b), fp32 or fp64."""
    s, b = fold_bn(bn, device, rounding)
    return _param(linear.weight, device, rounding) * s[:, None], _param(linear.bias, device, rounding) * s + b


def _conv(x, w):
    return F.conv2d(x, w.double(), padding=w.shape[-1] // 2)


def _mma_weight(w, rounding):
    """A folded fp32 weight as the tensor core reads it: bf16."""
    return _bf16(w.double(), rounding)


def _ch(v):
    return v.double()[None, :, None, None]


def _grids(grids):
    return grids.reshape(-1, 1, 40, 10).double()


def alphasame_trunk(net, grids, layout="rows", rounding=True):
    """AlphaSame.grid_features (pre-activation blocks, kernels = 1) -> fp64 [n, 400].

    layout 'rows' (trunk_rows.cu, 16 filters): bf16 stem weights, residual stream X in fp32 (TMEM);
    'taps' (trunk.cu, 16 filters): the same with the stem as an fp32 table (unrounded weights);
    'wide' (trunk_wide.cu, 32 / 64 filters): fp32 stem table, X stored as bf16 after the stem and every block.
    In every layout T = bf16(relu(s1 X + b1)) is taken from the unrounded fp32 sum, U = bf16(relu(conv1'(T) + b2))
    with conv1' = bf16(w1 * s2), X += conv2(U) with bf16(w2), and the head is
    bf16(relu(sb * sum_c k_c relu(sa X + ba) + bb)) with X, the inner terms and the sum in fp32."""
    assert layout in ("rows", "taps", "wide")
    dev = grids.device
    p = lambda t: _param(t, dev, rounding)  # noqa: E731
    w_stem = p(net.conv1.weight)
    w_stem = _mma_weight(w_stem, rounding) if layout == "rows" else w_stem.double()
    d = _fp32(_conv(_grids(grids), w_stem), rounding)           # fp32 accumulator (TMEM / fp32 table sums)
    x = _bf16(d, rounding) if layout == "wide" else d
    for blk in net.res_blocks:
        s1, b1 = fold_bn(blk.conv_block1[0], dev, rounding)
        s2, b2 = fold_bn(blk.conv_block2[0], dev, rounding)
        t = _bf16(torch.relu(_fp32(_ch(s1) * d + _ch(b1), rounding)), rounding)
        w1 = _mma_weight(p(blk.conv_block1[2].weight) * s2[:, None, None, None], rounding)
        u = _bf16(torch.relu(_fp32(_conv(t, w1) + _ch(b2), rounding)), rounding)
        d = _fp32(_conv(u, _mma_weight(p(blk.conv_block2[3].weight), rounding)) + x, rounding)
        x = _bf16(d, rounding) if layout == "wide" else d
    sa, ba = fold_bn(net.batchnorm1, dev, rounding)
    sb, bb = fold_bn(net.batchnorm2, dev, rounding)
    k = p(net.kernel1.weight).reshape(-1).double()
    t = torch.relu(_fp32(_ch(sa) * d + _ch(ba), rounding))
    inner = _fp32(torch.einsum("nchw,c->nhw", t, k), rounding)
    return _bf16(torch.relu(sb.double() * inner + bb.double()), rounding).reshape(-1, CELLS)


def post_act_trunk(net, grids, rounding=True):
    """BaseResNet / AuxBaseResNet trunk as trunk_wide.cu writes it -> fp64 [n, 5 * 400], channel-major:
    channels 0-3 = so * own_collapse_conv(t) (bn scale only, no ReLU: the bias joins the FiLM term in the heads),
    channel 4 = the finished opponent collapse relu(sp * opp_collapse_conv(t) + bp).

    X0 = bf16(relu(stem' + b0)) with stem' = fp32 table of w * s0; per block U = bf16(relu(conv1'(X) + b1)) and
    X' = bf16(relu(conv2'(U) + b2 + X)) with bf16 weights w * s; the head reads the last block's unrounded
    fp32 t = relu(conv2'(U) + b2 + X)."""
    dev = grids.device
    p = lambda t: _param(t, dev, rounding)  # noqa: E731
    s0, b0 = fold_bn(net.stem[1], dev, rounding)
    d = _fp32(_conv(_grids(grids), p(net.stem[0].weight) * s0[:, None, None, None]) + _ch(b0), rounding)
    x = _bf16(torch.relu(d), rounding)
    for blk in net.trunk:
        s1, b1 = fold_bn(blk.bn1, dev, rounding)
        s2, b2 = fold_bn(blk.bn2, dev, rounding)
        u = _bf16(torch.relu(_fp32(_conv(x, _mma_weight(p(blk.conv1.weight) * s1[:, None, None, None], rounding)) + _ch(b1),
                                   rounding)), rounding)
        d = _fp32(_conv(u, _mma_weight(p(blk.conv2.weight) * s2[:, None, None, None], rounding)) + _ch(b2) + x, rounding)
        x = _bf16(torch.relu(d), rounding)
    t = torch.relu(d)
    so, _ = fold_bn(net.own_collapse[1], dev, rounding)
    sp, bp = fold_bn(net.opp_collapse[1], dev, rounding)
    f = t.shape[1]
    own = _fp32(torch.einsum("nchw,oc->nohw", t, p(net.own_collapse[0].weight).reshape(-1, f).double()), rounding)
    opp = _fp32(torch.einsum("nchw,oc->nohw", t, p(net.opp_collapse[0].weight).reshape(-1, f).double()), rounding)
    own = _bf16(_ch(so) * own, rounding)
    opp = _bf16(torch.relu(_ch(sp) * opp + _ch(bp)), rounding)
    return torch.cat([own, opp], dim=1).flatten(1)


def trunk(net, grids, layout=None, rounding=True):
    """The trunk kernel's output rows for any supported net: AlphaSame (layout 'rows', 'taps' or 'wide';
    default 'rows' for 16 filters, 'wide' otherwise) or BaseResNet / AuxBaseResNet."""
    from tetris_reinforcement_learning_b200.architectures import AlphaSame
    if isinstance(net, AlphaSame):
        if layout is None:
            layout = "rows" if net.conv1.out_channels == 16 else "wide"
        return alphasame_trunk(net, grids, layout, rounding)
    return post_act_trunk(net, grids, rounding)


def alphasame_heads(net, own, opp, extras, rounding=True):
    """csrc/heads.cu: own / opp trunk rows [G, 400], extras [G, 105] -> (x [G, 528], o16 [G, 16], value [G]), fp64.

    o16 = bf16(relu(Wo' f_opp + bo')), x = [own | extras[:52] | o16 | extras[52:] | 7 zeros],
    value = bf16(sigmoid|tanh(w2 . relu(Wv' x + bv') + b2)); the folded weights stay fp32 (no bf16 rounding)."""
    dev = own.device
    wo, bo = fold_linear_bn(net.osidedense[0], net.osidedense[1], dev, rounding)
    o16 = _bf16(torch.relu(_fp32(opp.double() @ wo.double().t() + bo.double(), rounding)), rounding)
    ex = extras.double()
    g = own.shape[0]
    x = torch.cat([own.double(), ex[:, :SIDE_FEATS], o16, ex[:, SIDE_FEATS:],
                   torch.zeros((g, K_PAD - K_IN), dtype=torch.float64, device=dev)], dim=1)
    wv, bv = fold_linear_bn(net.value_head[0], net.value_head[1], dev, rounding)
    h = torch.relu(x[:, :K_IN] @ wv.double().t() + bv.double())
    lin2 = net.value_head[3]
    v = h @ _param(lin2.weight, dev, rounding).double().reshape(-1) + _param(lin2.bias, dev, rounding).double()
    v = torch.tanh(v) if isinstance(net.value_head[-1], torch.nn.Tanh) else torch.sigmoid(v)
    return x, o16, _bf16(v, rounding)


def policy_logits(x, w, b, moves=None, rounding=True):
    """logit[g, c] = b[m] + sum_k x[g, k] w[m, k] at m = moves[g, c] (every row of w when moves is None), fp64.
    With rounding x, w and b are taken as the bf16 values policy_legal_kernel reads."""
    def val(t):
        return t.detach().bfloat16().double() if rounding else t.detach().double()
    x, w, b = val(x), val(w), val(b)
    k = min(x.shape[1], w.shape[1])
    x, w = x[:, :k], w[:, :k]
    if moves is None:
        return x @ w.t() + b
    moves = moves.long()
    return torch.bmm(w[moves], x[:, :, None])[:, :, 0] + b[moves]


def alphasame_forward_packed(net, grids, extras, layout=None, rounding=True):
    """AlphaSame.forward_packed as the fused evaluator computes it: trunk kernel on both boards, heads.cu,
    then the policy head -> (value [B], logits [B, 11583])."""
    b = extras.shape[0]
    f = trunk(net, grids, layout, rounding)
    x, _, value = alphasame_heads(net, f[:b], f[b:], extras, rounding)
    return value, policy_logits(x[:, :K_IN], net.policy_head.weight, net.policy_head.bias, rounding=rounding)
