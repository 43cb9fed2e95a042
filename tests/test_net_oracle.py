"""CPU checks of oracle/net_oracle.py, the fp64 reference of the floating-point kernels: without rounding it
must be the module's own fp64 forward, with rounding it must stay within the fp32-module tolerances the GPU
tests of the kernels have always used."""
import copy

import pytest
import torch

from oracle import net_oracle
from tetris_reinforcement_learning_b200 import architectures as arch

CASES = [("alphasame", 16, False), ("alphasame", 16, True), ("alphasame", 32, False), ("alphasame", 64, True),
         ("base", 32, False), ("base", 64, True), ("aux", 32, False)]


def _net(family, filters, use_tanh, blocks=2, seed=0):
    torch.manual_seed(seed)
    if family == "alphasame":
        net = arch.AlphaSame(arch.AlphaSameConfig(blocks=blocks, filters=filters), use_tanh=use_tanh)
    elif family == "base":
        net = arch.BaseResNet(arch.BaseResNetConfig(blocks=blocks, filters=filters), use_tanh=use_tanh)
    else:
        net = arch.AuxBaseResNet(arch.AuxBaseResNetConfig(blocks=blocks, filters=filters), use_tanh=use_tanh)
    for m in net.modules():  # non-trivial BatchNorm statistics
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
            m.running_mean.normal_(0, 0.3); m.running_var.uniform_(0.5, 1.5)
            m.weight.data.uniform_(0.7, 1.3); m.bias.data.normal_(0, 0.2)
    return net.eval()


def _inputs(b, seed=1):
    g = torch.Generator().manual_seed(seed)
    grids = (torch.rand((2 * b, 1, 40, 10), generator=g) < 0.35).float()
    grids[0] = 0
    grids[-1] = 1
    extras = torch.randint(0, 2, (b, 105), generator=g).float()
    return grids, extras


def _module_trunk(net, grids):
    """What one row of the trunk kernel's output holds, from the module itself (fp64 when the net is)."""
    with torch.no_grad():
        if isinstance(net, arch.AlphaSame):
            return net.grid_features(grids)
        feat = net._process_grid(grids)
        bn = net.own_collapse[1]
        so = bn.weight / torch.sqrt(bn.running_var + bn.eps)
        own = net.own_collapse[0](feat) * so[None, :, None, None]
        return torch.cat([own, net.opp_collapse(feat)], dim=1).flatten(1)


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-30)).item()


@pytest.mark.parametrize("family,filters,use_tanh", CASES)
def test_unrounded_oracle_is_the_fp64_module(family, filters, use_tanh):
    net = _net(family, filters, use_tanh)
    net64 = copy.deepcopy(net).double()
    grids, extras = _inputs(6)
    g64, e64 = grids.double(), extras.double()
    ref = _module_trunk(net64, g64)
    layouts = (("rows", "taps") if filters == 16 else ("wide",)) if family == "alphasame" else (None,)
    for layout in layouts:
        got = net_oracle.trunk(net, grids, layout, rounding=False)
        assert got.dtype == torch.float64 and got.shape == ref.shape
        assert _rel(got, ref) <= 1e-9, (layout, _rel(got, ref))
    if family != "alphasame":
        return
    with torch.no_grad():
        v_ref, l_ref = net64.forward_packed(g64, e64)
        o16_ref = net64.osidedense(ref[6:])
    feats = net_oracle.trunk(net, grids, layouts[0], rounding=False)
    x, o16, v = net_oracle.alphasame_heads(net, feats[:6], feats[6:], extras, rounding=False)
    assert _rel(o16, o16_ref) <= 1e-9
    assert _rel(v, v_ref.reshape(-1)) <= 1e-9
    assert x.shape == (6, net_oracle.K_PAD) and (x[:, net_oracle.K_IN:] == 0).all()
    v2, logits = net_oracle.alphasame_forward_packed(net, grids, extras, rounding=False)
    assert _rel(v2, v_ref.reshape(-1)) <= 1e-9
    assert _rel(logits, l_ref) <= 1e-9
    moves = torch.tensor([[0, 11582, 5, 5], [7, 0, 11582, 100]])
    got = net_oracle.policy_logits(x[:2], net.policy_head.weight, net.policy_head.bias, moves, rounding=False)
    assert _rel(got, torch.gather(l_ref[:2], 1, moves)) <= 1e-9


@pytest.mark.parametrize("family,filters,use_tanh", CASES)
def test_rounded_oracle_stays_within_the_fp32_tolerances(family, filters, use_tanh):
    """The bf16 roundings move the oracle away from the fp32 module by no more than the GPU tests of the
    kernels allow the kernels themselves (test_gpu_trunk.py, test_gpu_trunk_wide.py)."""
    net = _net(family, filters, use_tanh, seed=2)
    grids, extras = _inputs(4, seed=3)
    ref = _module_trunk(net, grids).double()
    layouts = (("rows", "taps") if filters == 16 else ("wide",)) if family == "alphasame" else (None,)
    for layout in layouts:
        got = net_oracle.trunk(net, grids, layout)
        assert (got == got.float().bfloat16().double()).all(), "trunk outputs are bf16 values"
        err, scale = (got - ref).abs(), ref.abs().max().item()
        assert err.max().item() <= 0.04 * scale + 0.03, (layout, err.max().item(), scale)
        assert err.mean().item() <= 0.015 * ref.abs().mean().item() + 1e-3
    if family != "alphasame":
        return
    with torch.no_grad():
        v_ref, l_ref = net.forward_packed(grids, extras)
    v, logits = net_oracle.alphasame_forward_packed(net, grids, extras)
    assert (v - v_ref.double().reshape(-1)).abs().max().item() < 0.03
    assert (logits - l_ref.double()).abs().max().item() < 0.05 * l_ref.abs().max().item() + 0.05
