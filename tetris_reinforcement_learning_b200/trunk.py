"""Host side of the fused tcgen05 trunk (csrc/trunk.cu): BatchNorm folding, weight packing into
the UMMA core-matrix order, and the evaluator that runs trunk kernel + PyTorch heads.

Applies to AlphaSame with filters = 16 and kernels = 1 (BASELINE's blocks=10 filters=16 net and
any other depth); other nets use the plain PyTorch evaluator (selfplay.make_net_evaluator)."""
import torch

from . import _native
from .architectures import SIDE_FEATS, AlphaSame


def supports(net):
    """csrc/trunk_rows.cu / trunk.cu hard-code 16 filters and one 1x1 kernel; csrc/heads.cu the 16-wide
    opponent summary and value hidden layer."""
    return (isinstance(net, AlphaSame) and net.conv1.out_channels == 16 and net.kernel1.out_channels == 1
            and len(net.res_blocks) <= 20 and net.osidedense[0].out_features == 16
            and net.value_head[0].out_features == 16)


def _fold_bn(bn):
    s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return s, bn.bias.detach().float() - bn.running_mean.detach().float() * s


def _pack_conv_taps(w):
    """(16 out, 16 in, 3, 3) -> [9 taps][k chunk 2][n group 2][n 8][k 8] (K-major core matrices)."""
    t = w.permute(2, 3, 0, 1).reshape(9, 16, 16)          # [tap][o][i]
    t = t.reshape(9, 2, 8, 2, 8)                           # [tap][ng][n][kc][k]
    return t.permute(0, 3, 1, 2, 4).contiguous()           # [tap][kc][ng][n][k]


def _pack_conv_rows(w):
    """(16 out, 16 in, 3 dy, 3 dx) -> [dy 3][k chunk 2][n group 6][n 8][k 8]: per vertical tap the
    48 x 16 matrix B[(j, oc), ic] = w[oc, ic, dy, 2 - j] that maps input column x_in to the output
    columns x_in - 1 + j (row-Toeplitz form of csrc/trunk_rows.cu), in K-major core-matrix order."""
    t = w.permute(2, 3, 0, 1).flip(1)                      # [dy][j = 2 - dx][oc][ic]
    t = t.reshape(3, 48, 16).reshape(3, 6, 8, 2, 8)        # [dy][ng][n][kc][k]
    return t.permute(0, 3, 1, 2, 4).contiguous()           # [dy][kc][ng][n][k]


def rows_kernel_supports(net):
    """The row-Toeplitz kernel keeps every layer's weights resident in shared memory."""
    return supports(net) and len(net.res_blocks) <= _native.lib().trl_alphasame_trunk_rows_max_blocks()


def pack_alphasame_trunk(net, device=None, layout=None):
    """-> dict(w_packed bf16 [2*blocks, 9*256], consts f32, stem_lut f32 [5,32,16], n_blocks, layout).

    layout 'rows' (csrc/trunk_rows.cu, default when the depth allows it) or 'taps' (csrc/trunk.cu)."""
    assert supports(net)
    if layout is None:
        layout = "rows" if rows_kernel_supports(net) else "taps"
    assert layout in ("rows", "taps")
    _pack_conv = _pack_conv_rows if layout == "rows" else _pack_conv_taps
    device = device or next(net.parameters()).device
    convs, consts = [], []
    for blk in net.res_blocks:
        s1, b1 = _fold_bn(blk.conv_block1[0])
        s2, b2 = _fold_bn(blk.conv_block2[0])
        w1 = blk.conv_block1[2].weight.detach().float() * s2[:, None, None, None]  # bn2 scale folded
        w2 = blk.conv_block2[3].weight.detach().float()
        convs += [_pack_conv(w1), _pack_conv(w2)]
        consts += [s1, b1, b2]
    sa, ba = _fold_bn(net.batchnorm1)
    sb, bb = _fold_bn(net.batchnorm2)
    consts += [sa, ba, net.kernel1.weight.detach().float().reshape(16), sb.reshape(1), bb.reshape(1)]
    w_stem = net.conv1.weight.detach().float()[:, 0]                               # [16][5][5]
    bits = ((torch.arange(32)[:, None] >> torch.arange(5)[None, :]) & 1).float().to(w_stem.device)  # [pat][k]
    lut = torch.einsum("pk,crk->rpc", bits, w_stem).contiguous()                  # [r][pat][c]
    # row-Toeplitz stem (csrc/trunk_rows.cu): per kernel row dy the 160 x 16 matrix
    # B[(x_out, oc), k] = w[oc][dy][k - x_out] (k = input column + 2), K-major core-matrix order
    kk, xo = torch.arange(16)[None, :], torch.arange(10)[:, None]
    dx = (kk - xo)                                                                 # [x_out][k]
    ok = ((dx >= 0) & (dx < 5)).to(w_stem.device)
    tz = w_stem.permute(1, 0, 2)[:, :, dx.clamp(0, 4).to(w_stem.device)] * ok     # [dy][oc][x_out][k]
    tz = tz.permute(0, 2, 1, 3).reshape(5, 160, 16).reshape(5, 20, 8, 2, 8)       # [dy][ng][n][kc][k]
    stem_w = tz.permute(0, 3, 1, 2, 4).contiguous()                               # [dy][kc][ng][n][k]
    return {"stem_w": stem_w.reshape(-1).to(device=device, dtype=torch.bfloat16).contiguous(),
            "w_packed": torch.stack(convs).reshape(len(convs), -1).to(device=device, dtype=torch.bfloat16).contiguous(),
            "consts": torch.cat([c.reshape(-1) for c in consts]).to(device).contiguous(),
            "consts_host": torch.cat([c.reshape(-1) for c in consts]).float().cpu().contiguous(),
            "stem_lut": lut.to(device).contiguous(), "n_blocks": len(net.res_blocks), "layout": layout}


def trunk_forward(packed, grids, out=None):
    """grids: bf16 CUDA tensor with n*400 elements ([n,1,40,10] or [n,400]) -> bf16 [n,400]."""
    n = grids.numel() // 400
    if grids.dtype != torch.bfloat16 or not grids.is_contiguous():
        grids = grids.to(torch.bfloat16).contiguous()
    if out is None:
        out = torch.empty((n, 400), dtype=torch.bfloat16, device=grids.device)
    rows = packed.get("layout") == "rows"
    fn = _native.lib().trl_alphasame_trunk_rows if rows else _native.lib().trl_alphasame_trunk
    stem = packed["stem_w"] if rows else packed["stem_lut"]
    consts = packed["consts_host"] if rows else packed["consts"]   # rows kernel: by-value kernel parameter
    with torch.cuda.device(grids.device):   # the library launches on the current device
        rc = fn(grids.data_ptr(), n, packed["n_blocks"], packed["w_packed"].data_ptr(), consts.data_ptr(),
                stem.data_ptr(), out.data_ptr(), torch.cuda.current_stream(grids.device).cuda_stream)
    _native.check(rc, "trl_alphasame_trunk")
    return out


def _fold_linear_bn(linear, bn):
    """Linear followed by eval-mode BatchNorm1d -> (weight [out, in], bias [out]) in fp32."""
    s, t = _fold_bn(bn)
    return linear.weight.detach().float() * s[:, None], linear.bias.detach().float() * s + t


def pack_alphasame_heads(net, device=None):
    """fp32 weights of csrc/heads.cu: Wo_t[400][16], bo[16], Wv_t[528][16], bv[16], w2[16], b2, pad."""
    device = device or next(net.parameters()).device
    wo, bo = _fold_linear_bn(net.osidedense[0], net.osidedense[1])
    wv, bv = _fold_linear_bn(net.value_head[0], net.value_head[1])
    wv_t = torch.zeros((528, 16), dtype=torch.float32, device=wv.device)
    wv_t[:wv.shape[1]] = wv.t()
    lin2 = net.value_head[3]
    parts = [wo.t().contiguous().reshape(-1), bo, wv_t.reshape(-1), bv, lin2.weight.detach().float().reshape(16),
             lin2.bias.detach().float().reshape(1), torch.zeros(3, device=wv.device)]
    out = torch.cat(parts).to(device).contiguous()
    assert out.numel() == _native.lib().trl_alphasame_heads_weight_floats()
    return out


def make_fused_evaluator(net, dtype=torch.bfloat16, layout=None, fused_heads=True):
    """Engine evaluator: fused tcgen05 trunk on both grids, one fused kernel for the opponent
    summary + concatenation + value head (csrc/heads.cu), and the policy head as a library GEMM."""
    assert supports(net) and dtype == torch.bfloat16
    net = net.eval()
    packed = pack_alphasame_trunk(net, layout=layout)
    use_tanh = int(isinstance(net.value_head[-1], torch.nn.Tanh))
    # The head input has 521 features; cuBLAS needs K % 8 == 0 for its tensor-core kernels, so the
    # policy / first value layer weights get zero columns up to 528 and x gets matching zeros.
    k_in = net.policy_head.in_features
    k_pad = (k_in + 15) // 16 * 16
    dev = net.policy_head.weight.device

    def padded(linear):
        n_pad = (linear.out_features + 7) // 8 * 8     # row pitch of the output must be 16-byte aligned too
        w = torch.zeros((n_pad, k_pad), dtype=dtype, device=dev)
        w[:linear.out_features, :k_in] = linear.weight.detach().to(dtype)
        b = torch.zeros(n_pad, dtype=dtype, device=dev)
        b[:linear.out_features] = linear.bias.detach().to(dtype)
        return w.contiguous(), b.contiguous()

    w_pol, b_pol = padded(net.policy_head)
    if fused_heads:
        w_heads = pack_alphasame_heads(net)
        lib = _native.lib()

        def evaluate(grids, extras):
            b = extras.shape[0]
            feats = trunk_forward(packed, grids)
            x = torch.empty((b, k_pad), dtype=dtype, device=extras.device)
            value = torch.empty(b, dtype=dtype, device=extras.device)
            if extras.dtype != dtype or not extras.is_contiguous():
                extras = extras.to(dtype).contiguous()
            with torch.cuda.device(extras.device):
                rc = lib.trl_alphasame_heads(feats.data_ptr(), extras.data_ptr(), b, w_heads.data_ptr(), use_tanh,
                                             x.data_ptr(), value.data_ptr(), torch.cuda.current_stream(extras.device).cuda_stream)
            _native.check(rc, "trl_alphasame_heads")
            return value, torch.nn.functional.linear(x, w_pol, b_pol)   # logits [G, 11584], last column unused
    else:
        osidedense, value_head = net.osidedense.to(dtype), net.value_head.to(dtype)
        w_val, b_val = padded(value_head[0])
        value_tail = value_head[1:]
        zeros = {}

        def evaluate(grids, extras):
            b = extras.shape[0]
            feats = trunk_forward(packed, grids)
            if b not in zeros:
                zeros[b] = torch.zeros((b, k_pad - k_in), dtype=dtype, device=extras.device)
            x = torch.cat([feats[:b], extras[:, :SIDE_FEATS], osidedense(feats[b:]), extras[:, SIDE_FEATS:], zeros[b]], dim=1)
            value = value_tail(torch.nn.functional.linear(x, w_val, b_val))
            return value, torch.nn.functional.linear(x, w_pol, b_pol)

    evaluate.packed = packed
    if fused_heads and packed["layout"] == "rows":
        evaluate.cached = CachedTrunkEvaluator(packed, w_heads, use_tanh, w_pol, b_pol, k_pad)
    return evaluate


class CachedTrunkEvaluator:
    """Network evaluation for SelfPlayEngine with exact trunk-feature reuse (include/trl.h,
    trl_encode_features_cached): per simulation only the board that the last move changed goes
    through the trunk; the features of the other board are the parent state's.  Outputs are
    bit-identical to the plain fused evaluator (same kernels, same per-image arithmetic).
    Every library call runs on the device of the buffers it is handed."""

    gather_policy = True   # policy head on the legal moves only (trl_search_policy_legal) instead of the dense GEMM

    def __init__(self, packed, w_heads, use_tanh, w_pol, b_pol, k_pad):
        self.packed, self.w_heads, self.use_tanh = packed, w_heads, use_tanh
        self.w_pol, self.b_pol, self.k_pad = w_pol, b_pol, k_pad
        self.stamp = None   # profiling hook (SelfPlayEngine.enable_timeline)

    def make_buffers(self, n_states, n_leaves, device, moves_cap=512):
        """Per-ENGINE buffers (the engine owns them, so they are freed with it): the feature cache
        [n_states * 2, 400] and the per-step staging of images, indices, head inputs and values."""
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=device)  # noqa: E731
        return {"cache": z((n_states * 2, 400), torch.bfloat16), "images": z((2 * n_leaves, 400), torch.bfloat16),
                "dest": z(2 * n_leaves, torch.int32), "count": z(1, torch.int32),
                "own": z(n_leaves, torch.int32), "opp": z(n_leaves, torch.int32), "rowof": z(n_states * 2, torch.int32),
                "x": z((n_leaves, self.k_pad), torch.bfloat16), "value": z(n_leaves, torch.bfloat16),
                "logits_legal": z((n_leaves, moves_cap), torch.float32)}

    def policy(self, b, search_buffers=None, join_movegen=None):
        """Policy logits of the leaves: gathered over the legal moves (fp32 [G, moves_cap]) when the engine hands in
        its buffers, else the dense head [G, 11584]."""
        if self.gather_policy and search_buffers is not None:
            if join_movegen is not None:
                join_movegen()      # the legal lists of this step come from the forked enumeration
            with torch.cuda.device(b["x"].device):
                _native.check(_native.lib().trl_search_policy_legal(
                    search_buffers, b["x"].data_ptr(), self.k_pad, self.w_pol.data_ptr(), self.b_pol.data_ptr(),
                    b["logits_legal"].data_ptr(), torch.cuda.current_stream(b["x"].device).cuda_stream), "trl_search_policy_legal")
            return b["logits_legal"]
        return torch.nn.functional.linear(b["x"], self.w_pol, self.b_pol)

    def trunk_step(self, b, G):
        """Trunk over the queued images b["images"][: b["count"]] -> cache rows b["dest"] (resets the count)."""
        p = self.packed
        with torch.cuda.device(b["cache"].device):
            _native.check(_native.lib().trl_alphasame_trunk_rows_indexed(
                b["images"].data_ptr(), b["count"].data_ptr(), 2 * G, b["dest"].data_ptr(), p["n_blocks"],
                p["w_packed"].data_ptr(), p["consts_host"].data_ptr(), p["stem_w"].data_ptr(), b["cache"].data_ptr(),
                torch.cuda.current_stream(b["cache"].device).cuda_stream), "trl_alphasame_trunk_rows_indexed")

    def heads_step(self, b, extras, G):
        """Opponent summary, head input b["x"] and value b["value"] of the leaves whose b["own"] row is >= 0."""
        with torch.cuda.device(extras.device):
            _native.check(_native.lib().trl_alphasame_heads_indexed(
                b["cache"].data_ptr(), b["own"].data_ptr(), b["opp"].data_ptr(), extras.data_ptr(), G,
                self.w_heads.data_ptr(), self.use_tanh, b["x"].data_ptr(), b["value"].data_ptr(),
                torch.cuda.current_stream(extras.device).cuda_stream), "trl_alphasame_heads_indexed")
        return b["value"]

    def encode(self, b, states, leaf_state, leaf_parent, extras):
        """Feature encoding of the selected leaves (a separate kernel; the engine normally has it done by
        the fused expand + select + encode kernel of the previous step)."""
        st = torch.cuda.current_stream(extras.device).cuda_stream   # b["count"] is zero here: the trunk kernel resets it
        with torch.cuda.device(extras.device):
            _native.check(_native.lib().trl_encode_features_cached(
                states.data_ptr(), leaf_state.data_ptr(), leaf_parent.data_ptr(), leaf_state.numel(), b["cache"].data_ptr(),
                b["images"].data_ptr(), b["dest"].data_ptr(), b["count"].data_ptr(), extras.data_ptr(),
                b["own"].data_ptr(), b["opp"].data_ptr(), b["rowof"].data_ptr(), st), "trl_encode_features_cached")

    def __call__(self, b, states, leaf_state, leaf_parent, extras, after_trunk=None, before_trunk=None, encoded=False,
                 search_buffers=None, join_movegen=None):
        """b: make_buffers(); states uint8 [n_states*400], leaf_state / leaf_parent int32 [G], extras bf16
        [G,105] (written here unless `encoded`) -> (values bf16 [G], logits: bf16 [G, 11584], or fp32
        [G, moves_cap] over the legal moves when the engine passes its search buffers)."""
        lib = _native.lib()
        dev = extras.device
        G = leaf_state.numel()
        st = torch.cuda.current_stream(dev).cuda_stream
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
        self.heads_step(b, extras, G)
        stamp(4, st)
        return b["value"], self.policy(b, search_buffers, join_movegen)
