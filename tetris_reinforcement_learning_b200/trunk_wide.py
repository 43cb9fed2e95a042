"""Host side of the wide fused tcgen05 trunk (csrc/trunk_wide.cu): 32 or 64 filters,
AlphaSame (pre-activation blocks) and BaseResNet / AuxBaseResNet (post-activation blocks).

BatchNorm folding, weight packing into the UMMA core-matrix order of the row-Toeplitz MMAs, the
stem as a table over input bit patterns, and the engine evaluators (plain and with exact
trunk-feature reuse).  The nets this covers are the reference's Config default
(AuxBaseResNetConfig, ai.py:83; architectures.py:159-353) and BASELINE config 5
(AlphaSame(blocks=20, filters=64), architectures.py:60-142).
"""
import torch

from . import _native
from .architectures import CELLS, SIDE_FEATS, AlphaSame, BaseResNet
from .trunk import CachedTrunkEvaluator, _fold_bn, _fold_linear_bn

WIDTHS = (32, 64)


def _is_alphasame(net):
    return isinstance(net, AlphaSame)


def filters_of(net):
    return net.conv1.out_channels if _is_alphasame(net) else net.stem[0].out_channels


def supports(net):
    """Nets the wide kernel evaluates: AlphaSame with kernels = 1 and the 16-wide heads of csrc/heads.cu,
    BaseResNet / AuxBaseResNet with own_kernels = 4; 32 or 64 filters."""
    if _is_alphasame(net):
        return (net.conv1.out_channels in WIDTHS and net.kernel1.out_channels == 1 and
                net.osidedense[0].out_features == 16 and net.value_head[0].out_features == 16)
    if isinstance(net, BaseResNet):
        return net.stem[0].out_channels in WIDTHS and net.own_collapse[0].out_channels == 4
    return False


def _pack_conv_rows(w):
    """(F out, F in, 3 dy, 3 dx) -> [dy 3][k chunk F/8][n group 3F/8][n 8][k 8]: per vertical tap the 3F x F
    matrix B[(j, oc), ic] = w[oc, ic, dy, 2 - j] mapping input column x_in to output columns x_in - 1 + j."""
    f = w.shape[0]
    t = w.permute(2, 3, 0, 1).flip(1)                                   # [dy][j][oc][ic]
    t = t.reshape(3, 3 * f, f).reshape(3, 3 * f // 8, 8, f // 8, 8)      # [dy][ng][n][kc][k]
    return t.permute(0, 3, 1, 2, 4).contiguous()                        # [dy][kc][ng][n][k]


def _stem_table(w):
    """(F, taps, taps) -> [dy][pattern][F]: partial sums of one kernel row over the 2^taps input bit patterns
    (bit i of the pattern = cell x - taps//2 + i)."""
    taps = w.shape[-1]
    bits = ((torch.arange(1 << taps)[:, None] >> torch.arange(taps)[None, :]) & 1).to(w)   # [pat][i]
    return torch.einsum("pi,cdi->dpc", bits, w).contiguous()


def pack_wide_trunk(net, device=None):
    """-> dict(w_packed bf16, consts f32, stem_lut f32, filters, n_blocks, post_act, stem_taps, n_out)."""
    assert supports(net)
    device = device or next(net.parameters()).device
    f = filters_of(net)
    zero = torch.zeros(f, device=device)
    convs, slots = [], []

    def slot(bias=None, nscale=None, nbias=None):
        slots.append(torch.stack([x if x is not None else zero for x in (bias, nscale, nbias)]))

    if _is_alphasame(net):
        post, blocks = 0, list(net.res_blocks)
        lut = _stem_table(net.conv1.weight.detach().float()[:, 0])
        folds = [_fold_bn(b.conv_block1[0]) for b in blocks] + [_fold_bn(net.batchnorm1)]   # bn1 of block b; final bn last
        slot(None, *folds[0])
        for i, blk in enumerate(blocks):
            s2, b2 = _fold_bn(blk.conv_block2[0])
            convs.append(_pack_conv_rows(blk.conv_block1[2].weight.detach().float() * s2[:, None, None, None]))
            slot(b2)
            convs.append(_pack_conv_rows(blk.conv_block2[3].weight.detach().float()))
            slot(None, *folds[i + 1])
        sb, bb = _fold_bn(net.batchnorm2)
        head = [net.kernel1.weight.detach().float().reshape(1, f), sb.reshape(1), bb.reshape(1)]
        n_out = 1
    else:
        post, blocks = 1, list(net.trunk)
        s0, b0 = _fold_bn(net.stem[1])
        lut = _stem_table(net.stem[0].weight.detach().float()[:, 0] * s0[:, None, None])
        slot(b0)
        for blk in blocks:
            s1, b1 = _fold_bn(blk.bn1)
            s2, b2 = _fold_bn(blk.bn2)
            convs.append(_pack_conv_rows(blk.conv1.weight.detach().float() * s1[:, None, None, None]))
            slot(b1)
            convs.append(_pack_conv_rows(blk.conv2.weight.detach().float() * s2[:, None, None, None]))
            slot(b2)
        so, _ = _fold_bn(net.own_collapse[1])          # the bias joins the FiLM term in the heads
        sp, bp = _fold_bn(net.opp_collapse[1])
        w_head = torch.cat([net.own_collapse[0].weight.detach().float().reshape(4, f),
                            net.opp_collapse[0].weight.detach().float().reshape(1, f)])
        head = [w_head, torch.cat([so, sp]), torch.cat([torch.zeros(4, device=so.device), bp])]
        n_out = 5
    consts = torch.cat([torch.stack(slots).reshape(-1)] + [h.reshape(-1) for h in head])
    return {"kind": "wide", "filters": f, "n_blocks": len(blocks), "post_act": post, "stem_taps": lut.shape[0], "n_out": n_out,
            "w_packed": torch.stack(convs).reshape(-1).to(device=device, dtype=torch.bfloat16).contiguous(),
            "consts": consts.to(device=device, dtype=torch.float32).contiguous(),
            "stem_lut": lut.to(device=device, dtype=torch.float32).contiguous()}


class WideTrunk:
    """A packed trunk + the per-device scratch the kernel streams activations through."""

    def __init__(self, packed, device):
        self.p = packed
        self.device = torch.device(device)
        lib = _native.lib()
        with torch.cuda.device(self.device):
            n = int(lib.trl_trunk_wide_scratch_bytes(packed["filters"]))
        self.scratch = torch.zeros(n, dtype=torch.uint8, device=self.device)     # pad rows must stay zero
        self.status = torch.zeros(8, dtype=torch.int32, device=self.device)
        self.row_elems = packed["n_out"] * CELLS

    def __call__(self, images, out, n_images=None, n_images_dev=None, out_row=None, pdl=False):
        """images bf16 [>= n][400] -> out bf16 [rows][n_out * 400] (row k, or out_row[k] with a device count)."""
        p = self.p
        n = images.numel() // CELLS if n_images is None else int(n_images)
        with torch.cuda.device(self.device):    # the library launches on the current device
            rc = _native.lib().trl_trunk_wide(
                images.data_ptr(), n, n_images_dev.data_ptr() if n_images_dev is not None else None,
                out_row.data_ptr() if out_row is not None else None, p["filters"], p["n_blocks"], p["post_act"], p["stem_taps"],
                p["w_packed"].data_ptr(), p["consts"].data_ptr(), p["stem_lut"].data_ptr(), out.data_ptr(),
                self.scratch.data_ptr(), self.scratch.numel(), self.status.data_ptr(), int(bool(pdl)),
                torch.cuda.current_stream(self.device).cuda_stream)
        _native.check(rc, "trl_trunk_wide")
        return out

    def check(self):
        """Raise if a wait inside any launch so far timed out (synchronises)."""
        st = self.status.cpu().tolist()
        if st[0]:
            raise RuntimeError(f"trl_trunk_wide: pipeline wait timed out (tag {st[1]}, block {st[2]}, warp {st[3]}, "
                               f"parity {st[4]}, stream index {st[5]})")


def wide_trunk_forward(trunk, grids, out=None):
    """grids: CUDA tensor with n*400 0/1 cells -> bf16 [n, n_out*400] trunk outputs."""
    n = grids.numel() // CELLS
    if grids.dtype != torch.bfloat16 or not grids.is_contiguous():
        grids = grids.to(torch.bfloat16).contiguous()
    if out is None:
        out = torch.empty((n, trunk.row_elems), dtype=torch.bfloat16, device=grids.device)
    return trunk(grids, out, n_images=n)


def _pad_linear(linear, k_pad, dtype, n_pad=None):
    n_pad = n_pad or linear.out_features
    w = torch.zeros((n_pad, k_pad), dtype=dtype, device=linear.weight.device)
    w[:linear.out_features, :linear.in_features] = linear.weight.detach().to(dtype)
    b = torch.zeros(n_pad, dtype=dtype, device=linear.weight.device)
    b[:linear.out_features] = linear.bias.detach().to(dtype)
    return w.contiguous(), b.contiguous()


class BaseResNetHeads:
    """Everything of BaseResNet.forward after the trunk (architectures.py:235-271), eval mode, BatchNorm folded:
    opponent encoding, FiLM-add bias (pushed through the linear 1x1 own collapse), heads.  `own` / `opp` are
    the 5-channel trunk outputs [B, 5*400] of the two boards: channels 0-3 = bn scale * own_collapse conv,
    channel 4 = the finished opponent collapse."""

    def __init__(self, net, dtype=torch.bfloat16):
        f = filters_of(net)
        dev = net.policy_head.weight.device
        w, b = _fold_linear_bn(net.opp_encode[0], net.opp_encode[1])
        self.w_opp, self.b_opp = w.to(dtype).contiguous(), b.to(dtype).contiguous()
        self.w_bias = net.bias_project.weight.detach().to(dtype).contiguous()
        self.b_bias = net.bias_project.bias.detach().to(dtype).contiguous()
        so, bo = _fold_bn(net.own_collapse[1])
        wc = net.own_collapse[0].weight.detach().float().reshape(4, f) * so[:, None]
        self.w_film, self.b_film = wc.to(dtype).contiguous(), bo.to(dtype).contiguous()    # bias_vec [B,F] -> [B,4]
        k_in = net.policy_head.in_features
        self.k_in, self.k_pad = k_in, (k_in + 15) // 16 * 16
        self.w_pol, self.b_pol = _pad_linear(net.policy_head, self.k_pad, dtype, (net.policy_head.out_features + 7) // 8 * 8)
        wv, bv = _fold_linear_bn(net.value_head[0], net.value_head[1])
        self.w_val = torch.zeros((wv.shape[0], self.k_pad), dtype=dtype, device=dev)
        self.w_val[:, :k_in] = wv.to(dtype)
        self.b_val = bv.to(dtype).contiguous()
        self.w_val2 = net.value_head[3].weight.detach().to(dtype).contiguous()
        self.b_val2 = net.value_head[3].bias.detach().to(dtype).contiguous()
        self.tanh = isinstance(net.value_head[-1], torch.nn.Tanh)
        self.dtype = dtype
        self._pad = {}

    def __call__(self, own, opp, extras):
        x = self.features(own, opp, extras)
        return self.value(x), torch.nn.functional.linear(x, self.w_pol, self.b_pol)

    def value(self, x):
        F = torch.nn.functional
        v = F.linear(torch.relu(F.linear(x, self.w_val, self.b_val)), self.w_val2, self.b_val2).reshape(-1)
        return torch.tanh(v) if self.tanh else torch.sigmoid(v)

    def features(self, own, opp, extras):
        """-> head input [B, k_pad] (flattened collapsed own map, own pieces / scalars, colour, zero padding)."""
        F = torch.nn.functional
        b = extras.shape[0]
        own_x, opp_x, color = extras[:, :SIDE_FEATS], extras[:, SIDE_FEATS:2 * SIDE_FEATS], extras[:, 2 * SIDE_FEATS:]
        opp_repr = torch.relu(F.linear(torch.cat([opp[:, 4 * CELLS:], opp_x], dim=1), self.w_opp, self.b_opp))
        bias = F.linear(torch.cat([opp_repr, own_x, color], dim=1), self.w_bias, self.b_bias)
        film = F.linear(bias, self.w_film, self.b_film)                                   # [B,4]
        flat = torch.relu(own[:, :4 * CELLS].reshape(b, 4, CELLS) + film[:, :, None]).reshape(b, 4 * CELLS)
        if b not in self._pad:
            self._pad[b] = torch.zeros((b, self.k_pad - self.k_in), dtype=self.dtype, device=extras.device)
        return torch.cat([flat, own_x, color, self._pad[b]], dim=1)


def make_wide_evaluator(net, dtype=torch.bfloat16):
    """Engine evaluator for the wide nets: grids [2G,1,40,10], extras [G,105] -> (values [G], logits [G, >= 11583])."""
    from . import trunk as trunk16
    assert supports(net) and dtype == torch.bfloat16
    net = net.eval()
    dev = next(net.parameters()).device
    wt = WideTrunk(pack_wide_trunk(net), dev)
    lib = _native.lib()
    if _is_alphasame(net):
        use_tanh = int(isinstance(net.value_head[-1], torch.nn.Tanh))
        w_heads = trunk16.pack_alphasame_heads(net)
        k_in = net.policy_head.in_features
        k_pad = (k_in + 15) // 16 * 16
        w_pol, b_pol = _pad_linear(net.policy_head, k_pad, dtype, (net.policy_head.out_features + 7) // 8 * 8)

        def evaluate(grids, extras):
            b = extras.shape[0]
            feats = wide_trunk_forward(wt, grids)
            x = torch.empty((b, k_pad), dtype=dtype, device=extras.device)
            value = torch.empty(b, dtype=dtype, device=extras.device)
            if extras.dtype != dtype or not extras.is_contiguous():
                extras = extras.to(dtype).contiguous()
            with torch.cuda.device(extras.device):
                _native.check(lib.trl_alphasame_heads(feats.data_ptr(), extras.data_ptr(), b, w_heads.data_ptr(), use_tanh,
                                                      x.data_ptr(), value.data_ptr(), torch.cuda.current_stream(extras.device).cuda_stream),
                              "trl_alphasame_heads")
            return value, torch.nn.functional.linear(x, w_pol, b_pol)

        def heads_indexed(b, extras, G, st):
            with torch.cuda.device(extras.device):
                _native.check(lib.trl_alphasame_heads_indexed(
                    b["cache"].data_ptr(), b["own"].data_ptr(), b["opp"].data_ptr(), extras.data_ptr(), G,
                    w_heads.data_ptr(), use_tanh, b["x"].data_ptr(), b["value"].data_ptr(), st), "trl_alphasame_heads_indexed")
            return b["value"]
    else:
        heads = BaseResNetHeads(net, dtype)
        k_pad = heads.k_pad

        def evaluate(grids, extras):
            b = extras.shape[0]
            feats = wide_trunk_forward(wt, grids)
            return heads(feats[:b], feats[b:], extras.to(dtype))

        def heads_indexed(b, extras, G, st):
            # a skipped leaf (own row < 0) reads row 0: its outputs are ignored by the search kernel
            own = b["cache"].index_select(0, b["own"].clamp(min=0))
            opp = b["cache"].index_select(0, b["opp"].clamp(min=0))
            b["x"].copy_(heads.features(own, opp, extras))
            return heads.value(b["x"])
        w_pol, b_pol = heads.w_pol, heads.b_pol

    evaluate.packed = wt.p
    evaluate.trunk = wt
    evaluate.cached = CachedWideEvaluator(wt, heads_indexed, k_pad, w_pol, b_pol)
    return evaluate


class CachedWideEvaluator:
    """trunk.CachedTrunkEvaluator for the wide nets (same engine contract: make_buffers / encode / __call__):
    per simulation only the board the last move changed goes through the trunk (exact, include/trl.h).  Every library
    call runs on the device of the buffers it is handed."""

    overlap_mode = "heads"     # the leaf enumeration is forked after the trunk (its CTAs own the SMs)
    gather_policy = True       # policy head on the legal moves only (trl_search_policy_legal)

    def __init__(self, wide_trunk, heads_indexed, k_pad, w_pol, b_pol):
        self.trunk, self.heads_indexed, self.k_pad = wide_trunk, heads_indexed, k_pad
        self.w_pol, self.b_pol = w_pol, b_pol
        self.stamp = None

    policy = CachedTrunkEvaluator.policy

    def make_buffers(self, n_states, n_leaves, device, moves_cap=512):
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=device)  # noqa: E731
        return {"cache": z((n_states * 2, self.trunk.row_elems), torch.bfloat16), "images": z((2 * n_leaves, CELLS), torch.bfloat16),
                "dest": z(2 * n_leaves, torch.int32), "count": z(1, torch.int32),
                "own": z(n_leaves, torch.int32), "opp": z(n_leaves, torch.int32), "rowof": z(n_states * 2, torch.int32),
                "x": z((n_leaves, self.k_pad), torch.bfloat16), "value": z(n_leaves, torch.bfloat16),
                "logits_legal": z((n_leaves, moves_cap), torch.float32)}

    def trunk_step(self, b, G):
        self.trunk(b["images"], b["cache"], n_images=2 * G, n_images_dev=b["count"], out_row=b["dest"], pdl=True)

    def heads_step(self, b, extras, G):
        return self.heads_indexed(b, extras, G, torch.cuda.current_stream(extras.device).cuda_stream)

    def encode(self, b, states, leaf_state, leaf_parent, extras):
        st = torch.cuda.current_stream(extras.device).cuda_stream
        with torch.cuda.device(extras.device):
            _native.check(_native.lib().trl_encode_features_cached(
                states.data_ptr(), leaf_state.data_ptr(), leaf_parent.data_ptr(), leaf_state.numel(), b["cache"].data_ptr(),
                b["images"].data_ptr(), b["dest"].data_ptr(), b["count"].data_ptr(), extras.data_ptr(),
                b["own"].data_ptr(), b["opp"].data_ptr(), b["rowof"].data_ptr(), st), "trl_encode_features_cached")

    def __call__(self, b, states, leaf_state, leaf_parent, extras, after_trunk=None, before_trunk=None, encoded=False,
                 search_buffers=None, join_movegen=None):
        G = leaf_state.numel()
        st = torch.cuda.current_stream(extras.device).cuda_stream
        if not encoded:
            self.encode(b, states, leaf_state, leaf_parent, extras)
        stamp = self.stamp or (lambda k, s: None)
        stamp(2, st)
        if before_trunk is not None:
            before_trunk()
        self.trunk_step(b, G)
        stamp(3, st)
        if after_trunk is not None:
            after_trunk()
        value = self.heads_step(b, extras, G)
        stamp(4, st)
        return value, self.policy(b, search_buffers, join_movegen)
