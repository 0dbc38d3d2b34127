"""Execution engine shared by the drop-in modules: parameter containers that reproduce the reference's
state_dict layout (SURVEY.md Appendix E) and the channels-last kernel schedule that replaces their ATen forward.

The nn.Conv2d / nn.GroupNorm / nn.MultiheadAttention / nn.Linear objects created here are PARAMETER HOLDERS only:
they are never called.  Every forward goes through ops.* -> libcnb200.so; a CPU tensor raises (no fallback).
Kernel-side weight copies (tap-major K-major packing, tf32 rounding) are derived caches attached to the
parameter object and invalidated by (version counter, data_ptr); they never appear in state_dict().
"""
import torch
import torch.nn as nn

from .. import ops
from .. import runtime as rt


# ----------------------------------------------------------------------------------------------------------
# parameter-holder factories (registration order == reference, so seeded default init is identical)
# ----------------------------------------------------------------------------------------------------------
def gn_act_conv3(groups, cin, cout):
    return nn.Sequential(nn.GroupNorm(groups, cin), nn.SiLU(), nn.Conv2d(cin, cout, 3, 1, 1))


def act_linear(din, dout):
    return nn.Sequential(nn.SiLU(), nn.Linear(din, dout))


def zero_(module):
    for prm in module.parameters():
        prm.detach().zero_()
    return module


# ----------------------------------------------------------------------------------------------------------
# derived weight cache
# ----------------------------------------------------------------------------------------------------------
def _cached(params, key, builder):
    """builder()'s result, kept on params[0] under `key` and rebuilt when any of `params` is changed in place (version
    counter) or replaced (data_ptr)."""
    store = params[0].__dict__.setdefault("_cnb_pack", {})
    stamp = tuple((p._version, p.data_ptr()) for p in params)
    ent = store.get(key)
    if ent is None or ent[0] != stamp:
        with torch.no_grad():
            ent = (stamp, builder())
        store[key] = ent
    return ent[1]


def _tc_shape(o, i):
    """mirror of conv2d_tma_supported (csrc/conv_tma.cu): only layers that reach the tensor core get tf32-rounded weights."""
    return i % 4 == 0 and i > 4 and o % 16 == 0      # Cin <= 4 / Cout <= 4 layers run the exact direct kernels


def packed_conv(param, mode):
    r = mode != rt.MODE_F32 and _tc_shape(param.shape[0], param.shape[1])
    return _cached((param,), ("conv", r), lambda: ops.pack_conv_weight(param, r))


def packed_conv_f16(param):
    """fp16 copy of the packed (unrounded) weights: B operand of the kind::f16 convolution."""
    return _cached((param,), ("conv_f16",), lambda: ops.cast_f16(ops.pack_conv_weight(param, False)))


def use_f16(mode, cin, cout):
    """GroupNorm -> conv pairs run with fp16 operands in the tensor-core mode (same 10-bit mantissa as tf32, half the
    bytes, twice the MMA rate) when the layer is tensor-core eligible."""
    return mode != rt.MODE_F32 and cin % 8 == 0 and cout % 16 == 0


_F16_ENABLED = True      # the tensor-core mode computes with fp16 operands; bench.py reads this to label its dtype


def act16(mode):
    """Tensor-core modes keep the whole activation stream (block inputs / outputs, skips, concat buffers) in fp16:
    half the bytes of every HBM-bound kernel, every convolution runs kind::f16.  Statistics, accumulators, biases,
    time-embedding rows and the softmax stay fp32."""
    return mode != rt.MODE_F32


def conv16(x, param, kind, cout, mode, *, packed=None, packed_lp=None, out_f16=None, **kw):
    """ops.conv with the operand / output dtypes the mode implies: fp16 weights when x is fp16, fp16 output when the
    activation stream is fp16 (unless the caller overrides out_f16)."""
    w = packed_conv(param, mode) if packed is None else packed
    lp = None
    if x.dtype == torch.float16:
        lp = packed_conv_f16(param) if packed_lp is None else packed_lp
    if out_f16 is None:
        out_f16 = act16(mode) and cout % 16 == 0
    return ops.conv(x, w, kind, cout, mode=mode, weight_lp=lp, out_f16=out_f16, **kw)
ATTN_F16_DIMS = (4, 8, 16, 24, 32, 48, 64, 96, 128, 192)     # head dims attention_f16.cu instantiates


def fuse_residual(mode, x, h, cout):
    """K-concatenation needs both operands fp16 and TMA-friendly channel counts."""
    if not (act16(mode) and x.dtype == torch.float16 and h.dtype == torch.float16):
        return False
    return h.shape[3] % 16 == 0 and x.shape[3] % 8 == 0 and cout % 16 == 0


def packed_cat_f16(param3x3, param1x1):
    """fp16 [Cout][9*C + Cin] rows: the second 3x3's packed taps followed by the 1x1 residual conv's columns."""
    def build():
        a = ops.pack_conv_weight(param3x3, False)
        b = ops.pack_conv_weight(param1x1, False)
        o = a.shape[0]
        return ops.cast_f16(torch.cat([a.reshape(o, -1), b.reshape(o, -1)], dim=1).contiguous())
    return _cached((param3x3, param1x1), ("cat_f16",), build)


def packed_convT_f16(param):
    return _cached((param,), ("convT_f16",), lambda: ops.cast_f16(ops.pack_convT_weight(param, False)))


def cast_like(x, ref):
    """dtype bridge for the rare mixed case (a block called on its own with fp32 inputs while the stream is fp16)."""
    if x.dtype == ref.dtype:
        return x
    if ref.dtype == torch.float16:
        return ops.cast_f16(x)
    raise rt.CnbError("cannot widen an fp16 activation into an fp32 buffer")


def packed_convT(param, mode):
    r = mode != rt.MODE_F32 and _tc_shape(param.shape[1], param.shape[0])
    return _cached((param,), ("convT", r), lambda: ops.pack_convT_weight(param, r))


def raw(param):
    """fp32 contiguous parameter used in place (bias, GroupNorm affine, small linears)."""
    rt.require_cuda(param)
    if param.dtype != torch.float32 or not param.is_contiguous():
        raise rt.CnbError("parameters must be contiguous fp32 (the reference's state_dict dtype)")
    return param.detach()


_FACTOR = {}


def temb_factor(dim, device):
    key = (dim, str(device))
    if key not in _FACTOR:
        half = dim // 2
        # same expression as get_time_embedding (models/unet_base.py:20-22), evaluated once on the host
        f = 10000 ** (torch.arange(start=0, end=half, dtype=torch.float32) / half)
        _FACTOR[key] = f.to(device)
    return _FACTOR[key]


def as_t(t, device):
    """torch.as_tensor(t).long(), on the device, at least 1-d (get_time_embedding :16-17)."""
    t = torch.as_tensor(t)
    if t.dtype != torch.int64:
        t = t.long()
    if t.device != device:
        t = t.to(device)
    if t.dim() == 0:
        t = t.unsqueeze(0)
    return t.contiguous()


def check_t(t, batch, device):
    """t as the kernels want it, with the shape rule the reference enforces by broadcasting: one row for the whole batch
    ((1,) / 0-d, the sampling tools) or one per sample ((B,), training / compare / student tools).  Anything else is the
    reference's broadcast RuntimeError (`out + t_emb_layers(t_emb)[:, :, None, None]`, unet_base.py:98)."""
    t = as_t(t, device)
    if t.dim() != 1 or t.numel() not in (1, batch):
        raise RuntimeError("The size of tensor t (%d) must match the batch size (%d) or be 1" % (t.numel(), batch))
    return t


def sinusoid(t, dim, device):
    assert dim % 2 == 0, "time embedding dimension must be divisible by 2"
    return ops.time_embedding(as_t(t, device), temb_factor(dim, device), dim)


def t_proj_mlp(seq, emb):
    """Linear -> SiLU -> Linear (Unet.t_proj, unet_base.py:313-317)."""
    h = ops.linear_small(emb, raw(seq[0].weight), raw(seq[0].bias), silu_out=True)
    return ops.linear_small(h, raw(seq[2].weight), raw(seq[2].bias))


class Temb:
    """Per-layer time-embedding rows for one block: either precomputed (one batched launch per U-Net) or
    computed lazily from a raw t_emb tensor when a block is called on its own."""

    def __init__(self, table=None, offsets=None, raw_temb=None):
        self.table, self.offsets, self.raw_temb = table, offsets, raw_temb

    def row(self, block, j):
        if self.table is not None:
            off = self.offsets[j]
            return self.table[:, off:], self.table.shape[1], self.table.shape[0] > 1
        lin = block.t_emb_layers[j][1]
        r = ops.linear_small(self.raw_temb, raw(lin.weight), raw(lin.bias), silu_in=True)
        return r, r.shape[1], r.shape[0] > 1


def _check_x(x):
    rt.require_cuda(x)
    if x.dtype != torch.float32:
        raise rt.CnbError("activations must be fp32 (the reference path is fp32 end to end)")
    return x.contiguous()


# ----------------------------------------------------------------------------------------------------------
# the residual + self-attention stack common to Down / Mid / Up blocks
# ----------------------------------------------------------------------------------------------------------
class ResAttnStack(nn.Module):
    """Holds resnet_conv_first / t_emb_layers / resnet_conv_second / attention_norms / attentions /
    residual_input_conv exactly as the reference blocks do (unet_base.py:39-89, blocks.py:40-112)."""

    def _build(self, cin, cout, t_emb_dim, n_res, n_attn, groups, heads, cross_attn=False):
        if cross_attn:
            raise NotImplementedError("cross-attention branches are dead for every shipped config (SURVEY.md section 2)")
        self._groups, self._heads, self.t_emb_dim = groups, heads, t_emb_dim
        self.resnet_conv_first = nn.ModuleList(
            [gn_act_conv3(groups, cin if i == 0 else cout, cout) for i in range(n_res)])
        if t_emb_dim is not None:
            self.t_emb_layers = nn.ModuleList([act_linear(t_emb_dim, cout) for _ in range(n_res)])
        self.resnet_conv_second = nn.ModuleList([gn_act_conv3(groups, cout, cout) for _ in range(n_res)])
        if n_attn:
            self.attention_norms = nn.ModuleList([nn.GroupNorm(groups, cout) for _ in range(n_attn)])
            self.attentions = nn.ModuleList(
                [nn.MultiheadAttention(cout, heads, batch_first=True) for _ in range(n_attn)])
        self.residual_input_conv = nn.ModuleList(
            [nn.Conv2d(cin if i == 0 else cout, cout, kernel_size=1) for i in range(n_res)])

    # ---- kernels -------------------------------------------------------------------------------------
    def _resnet(self, j, x, temb, mode):
        first, second = self.resnet_conv_first[j], self.resnet_conv_second[j]
        cout = first[2].out_channels
        h16 = use_f16(mode, first[2].in_channels, cout)
        h = ops.groupnorm(x, raw(first[0].weight), raw(first[0].bias), self._groups, silu=True, out_f16=h16)
        if temb is not None and self.t_emb_dim is not None:
            trow, tld, tps = temb.row(self, j)
        else:
            trow, tld, tps = None, 0, False
        h = conv16(h, first[2].weight, "3x3", cout, mode, bias=raw(first[2].bias),
                   temb=trow, temb_ld=tld, temb_per_sample=tps)
        h16 = use_f16(mode, cout, cout)
        h = ops.groupnorm(h, raw(second[0].weight), raw(second[0].bias), self._groups, silu=True, out_f16=h16)
        rc = self.residual_input_conv[j]
        if fuse_residual(mode, x, h, cout):
            # "+ residual_input_conv(resnet_input)" (unet_base.py:100) as extra K of the second 3x3: one launch, no
            # round trip of the 1x1 result through HBM; its bias rides in the epilogue's broadcast-row slot
            w = packed_conv(second[2].weight, mode)
            return ops.conv(h, w, "3x3", cout, bias=raw(second[2].bias), temb=raw(rc.bias), temb_ld=cout,
                            mode=mode, weight_lp=packed_cat_f16(second[2].weight, rc.weight), out_f16=True, x2=x)
        r = conv16(x, rc.weight, "1x1", cout, mode, bias=raw(rc.bias))
        return conv16(h, second[2].weight, "3x3", cout, mode, bias=raw(second[2].bias), residual=r)

    def _attention(self, j, x, mode):
        norm, att = self.attention_norms[j], self.attentions[j]
        E = att.embed_dim
        h16 = use_f16(mode, E, 3 * E)
        a = ops.groupnorm(x, raw(norm.weight), raw(norm.bias), self._groups, silu=False, out_f16=h16)
        # tensor-core modes: q|k|v and the attention output stay fp16 between the three kernels
        f16_core = h16 and (E // att.num_heads) in ATTN_F16_DIMS
        qkv = conv16(a, att.in_proj_weight, "1x1", 3 * E, mode, bias=raw(att.in_proj_bias), out_f16=f16_core)
        o = ops.attention(qkv, att.num_heads, mode=mode)
        return conv16(o, att.out_proj.weight, "1x1", E, mode, bias=raw(att.out_proj.bias), residual=x)

    def temb_channels(self):
        return [seq[1].out_features for seq in self.t_emb_layers] if self.t_emb_dim is not None else []


def run_down(block, x, temb, mode):
    for j in range(block.num_layers):
        x = block._resnet(j, x, temb, mode)
        if block.attn:
            x = block._attention(j, x, mode)
    if block.down_sample:
        dc = block.down_sample_conv
        x = conv16(x, dc.weight, "4x4s2", dc.out_channels, mode, bias=raw(dc.bias))
    return x


def run_mid(block, x, temb, mode):
    x = block._resnet(0, x, temb, mode)
    for j in range(block.num_layers):
        x = block._attention(j, x, mode)
        x = block._resnet(j + 1, x, temb, mode)
    return x


def run_up(block, x, skip, temb, mode, cat=None):
    """ConvTranspose (4 parity phases) or identity into the first half of the concat buffer, skip in the second
    half (unet_base.py:267-269).  `cat` may arrive with its second half already written by the producer of the
    skip (ControlNet zero-conv epilogue), which makes torch.cat free."""
    B, H, W, C = x.shape
    if block.up_sample:
        up = block.up_sample_conv
        cu = up.out_channels
        OH, OW = 2 * H, 2 * W
    else:
        cu, OH, OW = C, H, W
    if cat is None:
        dt = torch.float16 if (act16(mode) and (skip is None or skip.dtype == torch.float16)) else torch.float32
        if skip is None:
            cat = ops.empty(B, OH, OW, cu, device=x.device, dtype=dt)
        else:
            cat = ops.empty(B, OH, OW, cu + skip.shape[3], device=x.device, dtype=dt)
            ops.copy_channels(cast_like(skip, cat), cat, d_coff=cu)
    if block.up_sample:
        wp = packed_convT(up.weight, mode)
        wl = packed_convT_f16(up.weight) if x.dtype == torch.float16 else None
        for ph in range(4):
            ops.conv(x, wp[ph], None, cu, bias=raw(up.bias), out=cat, out_coff=0, mode=mode, phase=(ph >> 1, ph & 1),
                     weight_lp=None if wl is None else wl[ph])
    else:
        ops.copy_channels(cast_like(x, cat), cat, d_coff=0)
    x = cat
    for j in range(block.num_layers):
        x = block._resnet(j, x, temb, mode)
        if block.attn:                                     # always on in the U-Nets, per-level in the VAE decoder
            x = block._attention(j, x, mode)
    return x


# ----------------------------------------------------------------------------------------------------------
# U-Net level helpers (used by Unet / ControlNet / students)
# ----------------------------------------------------------------------------------------------------------
def unet_blocks(unet, with_ups=True):
    blocks = list(unet.downs) + list(unet.mids)
    if with_ups and hasattr(unet, "ups"):
        blocks += list(unet.ups)
    return blocks


def temb_plan(unet, temb_vec, with_ups=True):
    """One launch for all t_emb_layers of a U-Net: rows = SiLU(temb) @ Wcat^T + bcat, Wcat = concat over blocks.
    Returns {block: Temb}."""
    blocks = unet_blocks(unet, with_ups)
    lins = [seq[1] for b in blocks for seq in b.t_emb_layers]

    def build():
        w = torch.cat([raw(lin.weight) for lin in lins], dim=0).contiguous()
        bias = torch.cat([raw(lin.bias) for lin in lins], dim=0).contiguous()
        return w, bias

    wcat, bcat = _cached([lin.weight for lin in lins] + [lin.bias for lin in lins], ("tcat", with_ups), build)
    table = ops.linear_small(temb_vec, wcat, bcat, silu_in=True)
    plan, off = {}, 0
    for b in blocks:
        offs = []
        for c in b.temb_channels():
            offs.append(off)
            off += c
        plan[b] = Temb(table=table, offsets=offs)
    return plan


def unet_time(unet, t, device):
    return t_proj_mlp(unet.t_proj, sinusoid(t, unet.t_emb_dim, device))


def pad16_f16(x_nhwc):
    """fp32 (B, H, W, C <= 8) -> fp16 (B, H, W, 16) zero-padded copy, memoised on the tensor object (the frozen and the
    control conv_in read the same x)."""
    memo = x_nhwc.__dict__.get("_cnb_pad16")
    if memo is not None and memo[0] == x_nhwc._version:
        return memo[1]
    B, H, W, C = x_nhwc.shape
    buf = torch.zeros((B, H, W, 16), device=x_nhwc.device, dtype=torch.float16)
    ops.copy_channels(ops.cast_f16(x_nhwc), buf, d_coff=0)
    x_nhwc.__dict__["_cnb_pad16"] = (x_nhwc._version, buf)
    return buf


def narrow_in_tc(conv, x_nhwc, mode, residual=None):
    """True when conv3x3_narrow_in runs `conv` on the tensor core from the zero-padded fp16 copy of x."""
    cin, cout = conv.in_channels, conv.out_channels
    return (mode != rt.MODE_F32 and cin <= 8 and cout >= 64 and cout % 16 == 0 and x_nhwc.dtype == torch.float32 and
            (residual is None or residual.dtype == torch.float16))


def conv3x3_narrow_in(conv, x_nhwc, mode, residual=None):
    """3x3 conv from a handful of input channels (conv_in of the U-Nets, VAE decoder_conv_in / encoder_conv_in).
    Wide outputs (>= 64 channels: CelebHQ 4 -> 256, VAE 4 -> 384, CIFAR 3 -> 64) run on the tensor core with the input
    channels zero-padded to 16 in fp16: 9 k FMAs per pixel on the FFMA pipe were 0.3 ms per launch at B = 256 (4 -> 256
    @32x32).  Narrow outputs (MNIST 1 -> 32) keep the exact direct kernel."""
    cin, cout = conv.in_channels, conv.out_channels
    if narrow_in_tc(conv, x_nhwc, mode, residual):
        def build():
            w = torch.zeros((cout, 16) + tuple(conv.weight.shape[2:]), device=conv.weight.device, dtype=torch.float32)
            w[:, :cin] = conv.weight.detach()
            packed = ops.pack_conv_weight(w, False)
            return packed, ops.cast_f16(packed)
        packed, packed16 = _cached((conv.weight,), ("cin_pad16",), build)
        return ops.conv(pad16_f16(x_nhwc), packed, "3x3", cout, bias=raw(conv.bias), mode=mode, weight_lp=packed16,
                        out_f16=True, residual=residual)
    return conv16(x_nhwc, conv.weight, "3x3", cout, mode, bias=raw(conv.bias), residual=residual)


def conv_in(unet, x_nhwc, mode, residual=None):
    return conv3x3_narrow_in(unet.conv_in, x_nhwc, mode, residual=residual)


def prewarm_conv_in(unet, x_nhwc, mode):
    """Under CUDA-graph capture, build the memoised padded fp16 copy of x (pad16_f16) on the CURRENT stream when conv_in
    will take the tensor-core route.  The ControlNet forward calls this before it forks its branches: both conv_in
    layers read that one buffer, and whichever branch created it first would otherwise hand it to the other stream
    without an ordering edge.  Outside capture both run on one stream and the first of them builds it."""
    if torch.cuda.is_current_stream_capturing() and narrow_in_tc(unet.conv_in, x_nhwc, mode):
        pad16_f16(x_nhwc)


def gn_silu_conv_tail(norm, conv, h, mode):
    """GroupNorm -> SiLU -> 3x3 conv to a handful of channels (U-Net conv_out, VAE decoder / encoder conv_out).
    Returns the NHWC result, possibly as a channel-narrowed VIEW of a wider buffer (ops.nhwc_to_nchw reads strides).
    Narrow inputs (MNIST / CIFAR: 16 channels) run the exact direct FFMA kernel on fp16 activations.  Wide inputs
    (CelebHQ U-Net 128 -> 4, VAE decoder 128 -> 3 at 128x128: 3.5 k MACs per pixel) run on the tensor core with Cout
    zero-padded to 16: 4-5x wasted MMA work is still ~10x faster than FFMA."""
    cout, cin = conv.out_channels, conv.in_channels
    lowp = mode != rt.MODE_F32 and cout <= 4
    tc = lowp and cin % 16 == 0 and cin >= 64
    h16 = lowp and cin % 4 == 0
    h = ops.groupnorm(h, raw(norm.weight), raw(norm.bias), norm.num_groups, silu=True, out_f16=h16)
    if not tc:
        return ops.conv(h, packed_conv(conv.weight, mode), "3x3", cout, bias=raw(conv.bias), mode=mode)

    def build():
        w = torch.zeros((16,) + tuple(conv.weight.shape[1:]), device=conv.weight.device, dtype=torch.float32)
        w[:cout] = conv.weight.detach()
        b = torch.zeros(16, device=conv.weight.device, dtype=torch.float32)
        b[:cout] = conv.bias.detach()
        packed = ops.pack_conv_weight(w, False)
        return packed, ops.cast_f16(packed), b
    packed, packed16, bias = _cached((conv.weight, conv.bias), ("pad16",), build)
    return ops.conv(h, packed, "3x3", 16, bias=bias, mode=mode, weight_lp=packed16, out_f16=True)[..., :cout]


def conv_out(unet, x, mode):
    """norm_out -> SiLU -> conv_out (unet_base.py:371-373)."""
    return gn_silu_conv_tail(unet.norm_out, unet.conv_out, x, mode)


def run_unet_body(unet, h, plan, mode):
    """downs (saving their inputs as skips) -> mids -> ups -> norm_out/SiLU/conv_out (unet_base.py:355-374)."""
    skips = []
    for d in unet.downs:
        skips.append(h)
        h = run_down(d, h, plan[d], mode)
    for m in unet.mids:
        h = run_mid(m, h, plan[m], mode)
    for u in unet.ups:
        h = run_up(u, h, skips.pop(), plan[u], mode)
    return conv_out(unet, h, mode)


def hint_stack_ddpm(seq, hint_nhwc, mode):
    """3x3 -> SiLU -> 3x3 -> SiLU -> 3x3 -> SiLU -> 1x1 (controlnet.py:69-89); SiLU is fused in the epilogue."""
    h = hint_nhwc
    for idx in (0, 2, 4):
        c = seq[idx]
        h = conv16(h, c.weight, "3x3", c.out_channels, mode, bias=raw(c.bias), act=1)
    c = seq[6]
    return conv16(h, c.weight, "1x1", c.out_channels, mode, bias=raw(c.bias))


class HintCache:
    """hint_block(hint) depends on neither t nor x (controlnet.py:179): compute once per (hint storage, weights).
    A few entries are kept; every entry holds a reference to its hint tensor, so the storage cannot be recycled under
    the cached key.

    An entry is keyed by the hint's STORAGE (data_ptr, shape, strides), the mode and the hint-block weights; the hint's
    version counter is a stamp inside the entry.  When the same storage is overwritten in place (the way a captured
    CUDA graph is re-used with a new hint) the feature is recomputed INTO THE SAME feature tensor, so a graph that baked
    that tensor's address keeps reading valid, current data (sampler.DDPMSampler calls `refresh` before every replay).
    Recomputing under stream capture would silently bake a one-off update into the graph, so it raises instead."""
    MAX_ENTRIES = 8

    def __init__(self):
        self.entries = {}

    def get(self, hint, params, mode, fn):
        key = (hint.data_ptr(), tuple(hint.shape), tuple(hint.stride()), mode,
               tuple((p._version, p.data_ptr()) for p in params))
        ent = self.entries.get(key)
        if ent is None:
            if len(self.entries) >= self.MAX_ENTRIES:
                self.entries.pop(next(iter(self.entries)))
            ent = [hint, hint._version, fn()]
            self.entries[key] = ent
        elif ent[1] != hint._version:
            if torch.cuda.is_current_stream_capturing():
                raise rt.CnbError("hint tensor was modified in place between warm-up and CUDA-graph capture")
            with torch.no_grad():
                ent[2].copy_(fn())
            ent[1] = hint._version
        return ent[2]

    def pinned(self):
        """The (hint, feature) tensors of every live entry: a sampler that captured them into a graph keeps these
        references so that eviction cannot free memory the graph still reads."""
        return [(e[0], e[2]) for e in self.entries.values()]

    def clear(self):
        self.entries = {}
