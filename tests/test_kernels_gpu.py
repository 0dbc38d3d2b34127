"""Per-kernel parity tests (GPU): every C-ABI entry point against a plain PyTorch fp32 reference of the same op
(computed on the CPU so no TF32 / cuDNN heuristics are involved)."""
import importlib
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import golden, rel_l2, syn, ROOT

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(ROOT, "oracle"))


@pytest.fixture(scope="module")
def pk():
    pkg = importlib.import_module("controlnet-pytorch_b200")
    ops = importlib.import_module("controlnet-pytorch_b200.ops")
    rt = importlib.import_module("controlnet-pytorch_b200.runtime")
    assert torch.cuda.is_available()
    rt.lib()
    return ops, rt


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def nchw(x):
    return x.permute(0, 3, 1, 2).contiguous()


def rnd(*shape, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g)


CONV_CASES = [
    # kind, B, Cin, Cout, H, W
    ("3x3", 2, 32, 64, 28, 28), ("3x3", 3, 16, 16, 7, 7), ("3x3", 2, 1, 32, 28, 28), ("3x3", 2, 3, 64, 9, 11),
    ("3x3", 2, 16, 1, 28, 28), ("3x3", 1, 128, 32, 14, 14), ("3x3", 1, 256, 256, 7, 7), ("1x1", 2, 64, 64, 14, 14),
    ("1x1", 5, 32, 96, 7, 7), ("4x4s2", 2, 64, 64, 28, 28), ("4x4s2", 2, 128, 128, 14, 14), ("3x3s2", 2, 16, 32, 16, 16),
    ("3x3", 1, 36, 48, 5, 5), ("1x1", 1, 16, 48, 28, 28),
    # TMA-im2col persistent kernel: several tiles per CTA, M tails, several N tiles, odd BN, strides
    ("3x3", 32, 64, 64, 28, 28), ("3x3", 5, 64, 384, 9, 7), ("1x1", 40, 64, 192, 28, 28), ("3x3", 3, 128, 512, 7, 7),
    ("3x3s2", 3, 64, 96, 16, 16), ("4x4s2", 33, 64, 48, 14, 14), ("3x3", 1, 32, 16, 3, 3), ("1x1", 1, 64, 16, 1, 1),
    # direct small-channel kernels: conv_in / hint conv0 / conv_out shapes of the three configs
    ("3x3", 3, 4, 256, 8, 8), ("3x3", 2, 128, 4, 8, 8), ("3x3", 2, 16, 3, 9, 11), ("1x1", 2, 4, 4, 5, 5),
    ("3x3", 2, 3, 16, 12, 12), ("4x4s2", 2, 3, 32, 8, 8),
    # >= 3 tiles per CTA on 148 SMs: the resident-weights variant of the TMA kernel
    ("3x3", 80, 64, 64, 28, 28), ("1x1", 75, 64, 192, 28, 28), ("3x3", 77, 16, 16, 28, 28), ("3x3", 300, 128, 32, 14, 14),
]


def _conv_ref(kind, x, w, b):
    if kind == "3x3":
        return F.conv2d(x, w, b, padding=1)
    if kind == "1x1":
        return F.conv2d(x, w, b)
    if kind == "4x4s2":
        return F.conv2d(x, w, b, stride=2, padding=1)
    if kind == "3x3s2":
        return F.conv2d(x, w, b, stride=2, padding=1)
    raise ValueError(kind)


@pytest.mark.parametrize("mode,tol", [("fp32", 2e-6), ("f16", 2e-3)])
@pytest.mark.parametrize("kind,B,Cin,Cout,H,W", CONV_CASES)
def test_conv(pk, kind, B, Cin, Cout, H, W, mode, tol):
    ops, rt = pk
    m = {"fp32": rt.MODE_F32, "f16": rt.MODE_F16}[mode]
    k = {"3x3": 3, "1x1": 1, "4x4s2": 4, "3x3s2": 3}[kind]
    x, w, b = rnd(B, Cin, H, W, seed=1), rnd(Cout, Cin, k, k, seed=2) / math.sqrt(Cin * k * k), rnd(Cout, seed=3)
    want = _conv_ref(kind, x, w, b)
    temb = rnd(B, Cout, seed=4)
    res = rnd(*want.shape, seed=5)
    want_full = F.silu(want + temb[:, :, None, None] + res)
    wp = ops.pack_conv_weight(w.cuda(), round_tf32=(m != rt.MODE_F32 and Cin % 4 == 0 and Cout % 16 == 0))
    got = ops.conv(nhwc(x).cuda(), wp, kind, Cout, bias=b.cuda(), mode=m)
    assert rel_l2(nchw(got.cpu()), want) < tol
    got = ops.conv(nhwc(x).cuda(), wp, kind, Cout, bias=b.cuda(), temb=temb.cuda(), temb_ld=Cout,
                   temb_per_sample=True, residual=nhwc(res).cuda(), act=1, mode=m)
    assert rel_l2(nchw(got.cpu()), want_full) < tol
    if m == rt.MODE_F16:
        assert rt.lib().cnb_tc_error_flag() == 0


@pytest.mark.parametrize("kind,B,Cin,Cout,H,W", [c for c in CONV_CASES if c[2] % 8 == 0 and c[3] % 16 == 0] +
                         [("3x3", 2, 64, 256, 7, 7), ("3x3", 1, 512, 512, 8, 8), ("1x1", 3, 8, 16, 6, 6)])
def test_conv_f16_operands(pk, kind, B, Cin, Cout, H, W):
    """kind::f16 tensor-core path: fp16 activations (as GroupNorm emits them) x fp16 weights, fp32 accumulate."""
    ops, rt = pk
    k = {"3x3": 3, "1x1": 1, "4x4s2": 4, "3x3s2": 3}[kind]
    x, w, b = rnd(B, Cin, H, W, seed=1), rnd(Cout, Cin, k, k, seed=2) / math.sqrt(Cin * k * k), rnd(Cout, seed=3)
    res = rnd(*_conv_ref(kind, x, w, b).shape, seed=5)
    want = _conv_ref(kind, x, w, b) + res
    want_q = _conv_ref(kind, x.half().float(), w.half().float(), b) + res     # same operand rounding, exact math
    wp = ops.pack_conv_weight(w.cuda(), round_tf32=False)
    got = ops.conv(nhwc(x).cuda().half(), wp, kind, Cout, bias=b.cuda(), residual=nhwc(res).cuda(), mode=rt.MODE_F16,
                   weight_lp=ops.cast_f16(wp))
    assert got.dtype == torch.float32
    assert rel_l2(nchw(got.cpu()), want_q) < 5e-6
    assert rel_l2(nchw(got.cpu()), want) < 1e-3
    got16 = ops.conv(nhwc(x).cuda().half(), wp, kind, Cout, bias=b.cuda(), residual=nhwc(res).cuda(), mode=rt.MODE_F16,
                     weight_lp=ops.cast_f16(wp), out_f16=True)
    assert got16.dtype == torch.float16
    assert rel_l2(nchw(got16.float().cpu()), want_q) < 6e-4
    assert rt.lib().cnb_tc_error_flag() == 0


@pytest.mark.parametrize("mode,tol", [("fp32", 2e-6), ("f16", 2e-3)])
@pytest.mark.parametrize("B,C,H,W", [(2, 32, 7, 7), (1, 64, 14, 14), (3, 16, 5, 3)])
def test_conv_transpose_into_concat(pk, B, C, H, W, mode, tol):
    """4 parity phases written into the first half of a 2C-channel concat buffer (UpBlock, unet_base.py:268-269)."""
    ops, rt = pk
    m = {"fp32": rt.MODE_F32, "f16": rt.MODE_F16}[mode]
    x, w, b = rnd(B, C, H, W, seed=1), rnd(C, C, 4, 4, seed=2) / math.sqrt(4 * C), rnd(C, seed=3)
    skip = rnd(B, C, 2 * H, 2 * W, seed=4)
    want = torch.cat([F.conv_transpose2d(x, w, b, stride=2, padding=1), skip], dim=1)
    wp = ops.pack_convT_weight(w.cuda(), round_tf32=(m != rt.MODE_F32 and C % 16 == 0))
    cat = torch.full((B, 2 * H, 2 * W, 2 * C), float("nan"), device="cuda")
    ops.copy_channels(nhwc(skip).cuda(), cat, d_coff=C)
    for ph in range(4):
        ops.conv(nhwc(x).cuda(), wp[ph], None, C, bias=b.cuda(), out=cat, out_coff=0, mode=m, phase=(ph >> 1, ph & 1))
    assert rel_l2(nchw(cat.cpu()), want) < tol


@pytest.mark.parametrize("B,C,G,H,W", [(2, 16, 8, 28, 28), (3, 64, 8, 14, 14), (2, 256, 8, 7, 7), (2, 384, 32, 8, 8),
                                       (1, 768, 32, 4, 4), (2, 32, 8, 1, 1), (1, 128, 8, 28, 28), (2, 96, 8, 5, 7),
                                       (3, 64, 8, 28, 28), (2, 128, 32, 32, 32), (300, 32, 8, 28, 28)])
@pytest.mark.parametrize("silu", [False, True])
def test_groupnorm(pk, B, C, G, H, W, silu):
    ops, rt = pk
    x = rnd(B, C, H, W, seed=1) * 2.0 + 0.7
    g, b = 1 + 0.1 * rnd(C, seed=2), 0.1 * rnd(C, seed=3)
    want = F.group_norm(x, G, g, b, eps=1e-5)
    if silu:
        want = F.silu(want)
    got = ops.groupnorm(nhwc(x).cuda(), g.cuda(), b.cuda(), G, silu)
    assert rel_l2(nchw(got.cpu()), want) < 3e-6
    got16 = ops.groupnorm(nhwc(x).cuda(), g.cuda(), b.cuda(), G, silu, out_f16=True)
    assert got16.dtype == torch.float16
    assert rel_l2(nchw(got16.float().cpu()), want) < 6e-4
    # fp16 activation stream: fp16 in (statistics in fp32 over the rounded input), fp16 / fp32 out
    xh = x.half()
    want_h = F.group_norm(xh.float(), G, g, b, eps=1e-5)
    if silu:
        want_h = F.silu(want_h)
    for o16, tol in ((True, 6e-4), (False, 3e-6)):
        got = ops.groupnorm(nhwc(xh).cuda(), g.cuda(), b.cuda(), G, silu, out_f16=o16)
        assert rel_l2(nchw(got.float().cpu()), want_h) < tol


@pytest.mark.parametrize("B,C,G,H,W", [(1, 128, 32, 128, 128), (3, 256, 32, 64, 64), (2, 384, 32, 64, 64), (5, 256, 8, 32, 32),
                                       (2, 64, 8, 61, 67), (1, 384, 32, 33, 31), (70, 128, 32, 32, 32)])
@pytest.mark.parametrize("silu", [False, True])
def test_groupnorm_large_samples(pk, B, C, G, H, W, silu):
    """Split-statistics GroupNorm (cnb_groupnorm_ws: samples beyond one CTA's shared memory, VAE decoder / CelebHQ
    levels): fp16 in, fp16 and fp32 out, odd spatial sizes, 384 channels (5 rows per sweep), a mean far from zero
    (the shifted sums must not cancel) and batch invariance of the statistics."""
    ops, rt = pk
    x = (rnd(B, C, H, W, seed=4) * 1.5 + 6.0).half()
    g, b = 1 + 0.1 * rnd(C, seed=5), 0.1 * rnd(C, seed=6)
    assert rt.lib().cnb_groupnorm_workspace_bytes(B, H * W, C, G, 1) > 0          # this shape takes the split kernels
    want = F.group_norm(x.float(), G, g, b, eps=1e-5)
    if silu:
        want = F.silu(want)
    xc = nhwc(x).cuda()
    for o16, tol in ((True, 6e-4), (False, 4e-6)):
        got = ops.groupnorm(xc, g.cuda(), b.cuda(), G, silu, out_f16=o16)
        assert rel_l2(nchw(got.float().cpu()), want) < tol, (o16, rel_l2(nchw(got.float().cpu()), want))
    if B > 1:   # the number of row ranges follows the batch size; the result must not
        one = ops.groupnorm(xc[:1].contiguous(), g.cuda(), b.cuda(), G, silu, out_f16=True)
        assert torch.equal(one, ops.groupnorm(xc, g.cuda(), b.cuda(), G, silu, out_f16=True)[:1])


ATTN_SHAPES = [(2, 784, 64, 4), (2, 784, 16, 4), (3, 196, 128, 4), (2, 49, 256, 4),
               (2, 196, 32, 4), (1, 1024, 384, 16), (2, 64, 768, 16), (2, 16, 512, 16),
               (1, 64, 512, 4), (1, 100, 384, 4), (1, 50, 768, 4), (2, 1, 64, 4), (1, 13, 32, 4),
               (2, 1024, 128, 16), (3, 130, 64, 4)]


def _attn_want(qkv, B, L, E, heads):
    d = E // heads
    q, k, v = [t.float().reshape(B, L, heads, d).transpose(1, 2) for t in qkv.split(E, dim=-1)]
    return (torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), -1) @ v).transpose(1, 2).reshape(B, L, E)


@pytest.mark.parametrize("B,L,E,heads", ATTN_SHAPES)
@pytest.mark.parametrize("kernel", [None, "mma"])
def test_attention_f16(pk, B, L, E, heads, kernel):
    """fp16-operand flash attention against exact softmax attention on the same fp16-rounded q|k|v; tolerance = fp16
    rounding of P and of the output.  kernel=None is the library's routing (tcgen05 / TMEM kernel where it is
    instantiated, the mma.sync kernel for head dims above 64); "mma" forces the mma.sync kernel."""
    ops, rt = pk
    qkv = rnd(B, L, 3 * E, seed=1).half()
    want = _attn_want(qkv, B, L, E, heads)
    got = ops.attention(qkv.reshape(B, L, 1, 3 * E).cuda(), heads, kernel=kernel)
    assert got.dtype == torch.float16
    assert rel_l2(got.float().cpu().reshape(B, L, E), want) < 1.5e-3
    assert rt.lib().cnb_tc_error_flag() == 0


@pytest.mark.parametrize("B,L,E,heads", [
    (2, 784, 64, 4), (2, 784, 16, 4), (2, 196, 32, 4), (3, 196, 128, 4), (2, 49, 256, 4), (2, 49, 128, 4), (2, 49, 64, 4),   # MNIST
    (1, 1024, 128, 4), (1, 256, 256, 4), (1, 1024, 16, 4), (1, 256, 64, 4), (2, 64, 256, 4),                                # CIFAR
    (1, 1024, 384, 16), (1, 256, 512, 16), (2, 64, 768, 16), (2, 16, 512, 16), (1, 1024, 128, 16), (1, 256, 256, 16),      # CelebHQ
    (3, 130, 64, 4), (1, 96, 64, 4), (2, 128, 32, 2), (1, 129, 64, 2), (5, 257, 256, 16), (2, 1, 64, 4), (1, 13, 32, 4),
    (1, 113, 16, 4), (2, 225, 64, 4), (1, 897, 32, 4), (130, 49, 64, 4)])
def test_attention_tmem(pk, B, L, E, heads):
    """tcgen05 / TMEM flash attention (csrc/attention_tmem.cu: S = Q K^T from smem operands, P written over S in tensor
    memory and consumed from there by the second MMA, thread-per-row online softmax with lazy rescale, V transposed in
    smem, denominators on the tensor core) against exact softmax attention on the same fp16 q|k|v: every (L, head dim)
    of the shipped configs, ragged tails on both the query and the key side, head dims that are loaded as part of a wider
    channel group (4, 8, 24, 48)."""
    ops, rt = pk
    qkv = rnd(B, L, 3 * E, seed=5).half()
    want = _attn_want(qkv, B, L, E, heads)
    got = ops.attention(qkv.reshape(B, L, 1, 3 * E).cuda(), heads, kernel="tmem")
    assert got.dtype == torch.float16
    assert torch.isfinite(got).all()
    assert rel_l2(got.float().cpu().reshape(B, L, E), want) < 1.5e-3
    assert rt.lib().cnb_tc_error_flag() == 0


def test_attention_tmem_is_batch_invariant(pk):
    """rows of a large batch equal the same samples run alone (the data-parallel shards must reproduce the full job)."""
    ops, rt = pk
    B, L, E, heads = 64, 784, 64, 4
    qkv = rnd(B, L, 3 * E, seed=9).half().reshape(B, L, 1, 3 * E).cuda()
    full = ops.attention(qkv, heads, kernel="tmem")
    part = ops.attention(qkv[5:7].contiguous(), heads, kernel="tmem")
    assert torch.equal(full[5:7], part)


@pytest.mark.parametrize("B,L,E,heads", [(2, 784, 64, 4), (2, 300, 128, 4), (1, 1024, 256, 16), (2, 97, 64, 4)])
@pytest.mark.parametrize("gain", [4.0, 12.0])
@pytest.mark.parametrize("kernel", ["mma", "tmem"])
def test_attention_f16_growing_scores(pk, B, L, E, heads, gain, kernel):
    """Scores whose row maximum keeps growing along the key axis (keys scaled by a ramp): the running maximum of an
    online softmax has to move many times, which exercises the lazy O-rescale path of the tcgen05 kernel (reference
    maximum only moves past a 2^8 headroom) and the peaked-softmax regime (P underflow of the early keys)."""
    ops, rt = pk
    d = E // heads
    qkv = rnd(B, L, 3 * E, seed=3)
    ramp = torch.linspace(0.05, 1.0, L).reshape(1, L, 1)
    q, k, v = qkv.split(E, dim=-1)
    q = torch.sign(q) * (0.5 + q.abs()) * math.sqrt(gain)          # no tiny queries: every row sees the ramp
    k = torch.sign(k) * (0.5 + k.abs()) * ramp * math.sqrt(gain)
    qkv = torch.cat([q, k, v], dim=-1).half()
    q, k, v = [t.float().reshape(B, L, heads, d).transpose(1, 2) for t in qkv.split(E, dim=-1)]
    want = (torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), -1) @ v).transpose(1, 2).reshape(B, L, E)
    got = ops.attention(qkv.reshape(B, L, 1, 3 * E).cuda(), heads, kernel=kernel)
    assert torch.isfinite(got).all()
    assert rel_l2(got.float().cpu().reshape(B, L, E), want) < 2e-3
    assert rt.lib().cnb_tc_error_flag() == 0


@pytest.mark.parametrize("B,C,Cx,Cout,H,W", [(3, 64, 64, 64, 14, 14), (2, 64, 32, 64, 28, 28), (5, 128, 256, 128, 7, 7),
                                             (2, 16, 64, 16, 9, 11), (33, 32, 32, 32, 14, 14), (76, 64, 32, 64, 28, 28)])
def test_conv_k_concat_second_input(pk, B, C, Cx, Cout, H, W):
    """3x3 conv over h plus a 1x1 conv over a second input x folded in as extra K (resnet residual_input_conv)."""
    ops, rt = pk
    h, x = rnd(B, C, H, W, seed=1), rnd(B, Cx, H, W, seed=2)
    w3, w1 = rnd(Cout, C, 3, 3, seed=3) / math.sqrt(9 * C), rnd(Cout, Cx, 1, 1, seed=4) / math.sqrt(Cx)
    b3, b1 = rnd(Cout, seed=5), rnd(Cout, seed=6)
    want = (F.conv2d(h.half().float(), w3.half().float(), b3, padding=1) +
            F.conv2d(x.half().float(), w1.half().float(), b1))
    p3, p1 = ops.pack_conv_weight(w3.cuda(), False), ops.pack_conv_weight(w1.cuda(), False)
    wcat = ops.cast_f16(torch.cat([p3.reshape(Cout, -1), p1.reshape(Cout, -1)], dim=1).contiguous())
    got = ops.conv(nhwc(h).cuda().half(), p3, "3x3", Cout, bias=b3.cuda(), temb=b1.cuda(), temb_ld=Cout,
                   mode=rt.MODE_F16, weight_lp=wcat, out_f16=True, x2=nhwc(x).cuda().half())
    assert got.dtype == torch.float16
    assert rel_l2(nchw(got.float().cpu()), want) < 6e-4
    assert rt.lib().cnb_tc_error_flag() == 0


@pytest.mark.parametrize("kind,B,Cin,Cout,H,W", [("1x1", 3, 64, 16, 7, 7), ("1x1", 5, 64, 48, 7, 7), ("1x1", 2, 32, 64, 14, 14),
                                                 ("1x1", 3, 64, 96, 7, 7), ("1x1", 2, 64, 192, 9, 5), ("1x1", 7, 256, 256, 7, 7),
                                                 ("1x1", 3, 256, 768, 7, 7), ("3x3", 2, 128, 128, 7, 7), ("4x4s2", 2, 64, 64, 14, 14),
                                                 ("1x1", 1, 24, 32, 5, 5), ("1x1", 150, 64, 64, 7, 7)])
@pytest.mark.parametrize("with_res", [False, True])
def test_conv_dense_f16_epilogue_offsets(pk, kind, B, Cin, Cout, H, W, with_res):
    """Dense fp16-stream epilogue (per-warp staging + TMA store, fp16 residual fetched by TMA): every N-tile width, several
    N tiles, ragged M (rows past the end clipped by the tensor map), output and residual at channel offsets of wider
    buffers (the decoder's concat layout) - the neighbouring channels must stay untouched."""
    ops, rt = pk
    k = {"3x3": 3, "1x1": 1, "4x4s2": 4}[kind]
    x, w, b = rnd(B, Cin, H, W, seed=1), rnd(Cout, Cin, k, k, seed=2) / math.sqrt(Cin * k * k), rnd(Cout, seed=3)
    ref = _conv_ref(kind, x.half().float(), w.half().float(), b)
    OH, OW = ref.shape[2], ref.shape[3]
    res = rnd(B, Cout, OH, OW, seed=5).half()
    want = ref + (res.float() if with_res else 0.0)
    wp = ops.pack_conv_weight(w.cuda(), round_tf32=False)
    lo, hi = 16, 8                                        # channels before / after the written window
    big = torch.full((B + 1, OH, OW, lo + Cout + hi), 7.0, device="cuda", dtype=torch.float16)
    out = big[:B]                                         # one guard sample behind the last row the kernel may touch
    resbuf = torch.zeros((B, OH, OW, 8 + Cout), device="cuda", dtype=torch.float16)
    resbuf[..., 8:] = nhwc(res.float()).cuda().half()
    ops.conv(nhwc(x).cuda().half(), wp, kind, Cout, bias=b.cuda(), mode=rt.MODE_F16, weight_lp=ops.cast_f16(wp),
             out=out, out_coff=lo, residual=resbuf if with_res else None, res_coff=8)
    got = out[..., lo:lo + Cout].float().cpu()
    assert rel_l2(nchw(got), want) < 6e-4
    assert (out[..., :lo] == 7.0).all() and (out[..., lo + Cout:] == 7.0).all()
    assert (big[B] == 7.0).all()                          # rows past M are clipped, not written
    assert rt.lib().cnb_tc_error_flag() == 0


def test_conv_out_reads_fp16(pk):
    """conv_out (Cout <= 4) on fp16 activations, as GroupNorm(norm_out) emits them in the tensor-core modes."""
    ops, rt = pk
    x, w, b = rnd(3, 16, 9, 7, seed=1), rnd(1, 16, 3, 3, seed=2) / 12.0, rnd(1, seed=3)
    want = F.conv2d(x.half().float(), w, b, padding=1)
    got = ops.conv(nhwc(x).cuda().half(), ops.pack_conv_weight(w.cuda(), False), "3x3", 1, bias=b.cuda(), mode=rt.MODE_F16)
    assert rel_l2(nchw(got.cpu()), want) < 2e-6


def test_time_embedding_and_linear(pk):
    ops, rt = pk
    import cn_oracle as O
    eng = importlib.import_module("controlnet-pytorch_b200.models._engine")
    for D in (32, 128, 512):
        t = torch.tensor([0, 1, 37, 500, 999])
        want = O.time_embedding(t, D)
        got = eng.sinusoid(t, D, torch.device("cuda"))
        assert (got.cpu() - want).abs().max() < 2e-6
    x, w, b = rnd(3, 128, seed=1), rnd(50, 128, seed=2) / 11.0, rnd(50, seed=3)
    want = F.silu(F.linear(F.silu(x), w, b))
    got = ops.linear_small(x.cuda(), w.cuda(), b.cuda(), silu_in=True, silu_out=True)
    assert rel_l2(got.cpu(), want) < 2e-6


@pytest.mark.parametrize("name,kw", [("ddpm", dict(syn.MNIST_DIFFUSION)),
                                     ("ldm", dict(syn.CELEBHQ_DIFFUSION, ldm_scheduler=True))])
def test_scheduler_bit_exact(pk, name, kw):
    """fp32 bit parity with the reference's sample_prev_timestep outputs (tests/golden, made by the reference)."""
    sched_mod = importlib.import_module("controlnet-pytorch_b200.scheduler.linear_noise_scheduler")
    s = sched_mod.LinearNoiseScheduler(**kw)
    g = golden(f"scheduler_{name}")
    for k in ("betas", "alphas", "alpha_cum_prod", "sqrt_alpha_cum_prod", "sqrt_one_minus_alpha_cum_prod"):
        assert np.array_equal(getattr(s, k).numpy(), g[k])
    xt = syn.det_noise("sched:xt", (3, 4, 9, 7)).cuda()
    eps = syn.det_noise("sched:eps", (3, 4, 9, 7)).cuda()
    z = syn.det_noise("sched:z", (3, 4, 9, 7)).cuda()
    for t in (999, 500, 1, 0):
        a, b = s.sample_prev_timestep(xt, eps, torch.as_tensor(t), z=z)
        assert np.array_equal(a.cpu().numpy(), g[f"prev_{t}"]), t
        assert np.array_equal(b.cpu().numpy(), g[f"x0_{t}"]), t


def test_scheduler_reference_rng_default(pk):
    """Without z the drop-in draws torch.randn on the CPU generator like linear_noise_scheduler.py:71."""
    sched_mod = importlib.import_module("controlnet-pytorch_b200.scheduler.linear_noise_scheduler")
    import cn_oracle as O
    s = sched_mod.LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    so = O.SchedulerOracle(**syn.MNIST_DIFFUSION)
    xt, eps = rnd(2, 1, 28, 28, seed=1), rnd(2, 1, 28, 28, seed=2)
    torch.manual_seed(123)
    a, b = s.sample_prev_timestep(xt.cuda(), eps.cuda(), torch.as_tensor(400))
    torch.manual_seed(123)
    z = torch.randn(xt.shape)
    wa, wb = so.sample_prev_timestep(xt, eps, 400, z)
    assert torch.equal(a.cpu(), wa) and torch.equal(b.cpu(), wb)


def test_philox_properties(pk):
    ops, rt = pk
    n = 1 << 20
    a = ops.philox_normal((n,), "cuda", seed=7, step=3)
    assert abs(float(a.mean())) < 5e-3 and abs(float(a.std()) - 1.0) < 5e-3
    # sharding invariance: two half-shards with global offsets == one full draw
    lo = ops.philox_normal((n // 2,), "cuda", seed=7, step=3, elem_offset=0)
    hi = ops.philox_normal((n // 2,), "cuda", seed=7, step=3, elem_offset=n // 2)
    assert torch.equal(torch.cat([lo, hi]), a)
    odd = ops.philox_normal((1001,), "cuda", seed=7, step=3, elem_offset=3)
    assert torch.equal(odd, a[3:1004])
    b = ops.philox_normal((n,), "cuda", seed=7, step=4)
    assert abs(float((a * b).mean())) < 5e-3
    # the fused scheduler noise is the same stream
    coef = torch.tensor([0.5, 0.8, 0.01, 0.99, 0.3, 1.0], device="cuda")
    xt, eps = torch.zeros(4096, device="cuda"), torch.zeros(4096, device="cuda")
    prev, _ = ops.sched_step(xt, eps, coef, z=None, seed=7, step=3)
    assert torch.allclose(prev, 0.3 * a[:4096], rtol=0, atol=1e-7)


@pytest.mark.parametrize("name", ["sched_step", "ddim_step", "dpm_solver_step"])
def test_update_ops_reject_what_the_kernel_would_overrun(pk, name):
    """The fused updates index every per-element buffer by xt's element count: a shorter, non-contiguous or non-fp32
    buffer, a short coef row or a non-int32 step counter is refused before anything is launched."""
    ops, rt = pk
    op = getattr(ops, name)
    n = 4 * 1024 + 3
    good = dict(xt=torch.zeros(n, device="cuda"), eps=torch.zeros(n, device="cuda"),
                coef=torch.tensor([0.5, 0.8, 0.01, 0.99, 0.3, 1.0], device="cuda"))
    if name == "dpm_solver_step":
        good["hist"] = torch.zeros(n, device="cuda")
    short = torch.zeros(n - 1, device="cuda")
    bad = [dict(eps=short), dict(z=short), dict(out=short), dict(x0_out=short),
           dict(xt=torch.zeros(2 * n, device="cuda")[::2]), dict(xt=good["xt"].half()), dict(coef=good["coef"][:5]),
           dict(step_dev=torch.zeros(1, device="cuda", dtype=torch.int64))]
    if name == "dpm_solver_step":
        bad.append(dict(hist=short))
    c0 = rt.launch_count()
    op(**good)
    assert rt.launch_count() == c0 + 1
    for b in bad:
        with pytest.raises(rt.CnbError):
            op(**{**good, **b})
        assert rt.launch_count() == c0 + 1, b


def test_layout_and_scale(pk):
    ops, rt = pk
    x = rnd(3, 5, 6, 7, seed=1)
    assert torch.equal(ops.nchw_to_nhwc(x.cuda()).cpu(), nhwc(x))
    assert torch.equal(ops.nhwc_to_nchw(nhwc(x).cuda()).cpu(), x)
    a, c = rnd(3, seed=2), rnd(3, seed=3)
    y = rnd(3, 5, 6, 7, seed=4)
    got = ops.scale_rows(a.cuda(), x.cuda(), c.cuda(), y.cuda())
    want = a[:, None, None, None] * x + c[:, None, None, None] * y
    assert torch.equal(got.cpu(), want)
    # EDM pre-conditioning fused with the layout change (consistency_controlnet_distilled.py:92, :132): bit-identical to
    # the reference's fp32 expressions, for fp32 and fp16 body outputs and for a channel-narrowed view of a wider buffer
    assert torch.equal(ops.scale_nchw_to_nhwc(a.cuda(), x.cuda()).cpu(), nhwc(a[:, None, None, None] * x))
    f = nhwc(y).cuda()
    assert torch.equal(ops.edm_combine_to_nchw(a.cuda(), x.cuda(), c.cuda(), f).cpu(), want)
    f16 = f.half()
    want16 = a[:, None, None, None] * x + c[:, None, None, None] * f16.float().cpu().permute(0, 3, 1, 2)
    assert torch.equal(ops.edm_combine_to_nchw(a.cuda(), x.cuda(), c.cuda(), f16).cpu(), want16)
    wide = torch.zeros(3, 6, 7, 16, device="cuda", dtype=torch.float16)
    wide[..., :5] = f16
    assert torch.equal(ops.edm_combine_to_nchw(a.cuda(), x.cuda(), c.cuda(), wide[..., :5]).cpu(), want16)
    with pytest.raises(rt.CnbError):                      # x must be the fp32 NCHW tensor matching f
        ops.edm_combine_to_nchw(a.cuda(), x.cuda()[:, :4].contiguous(), c.cuda(), f)
    # nhwc_to_nchw into a caller-provided batch slice
    big = torch.full((5, 5, 6, 7), -1.0, device="cuda")
    ops.nhwc_to_nchw(nhwc(x).cuda(), out=big[1:4])
    assert torch.equal(big[1:4].cpu(), x) and bool((big[0] == -1).all()) and bool((big[4] == -1).all())
    with pytest.raises(rt.CnbError):
        ops.nhwc_to_nchw(nhwc(x).cuda(), out=big[:, :, :, :6])


def test_no_cpu_fallback(pk):
    """Every op rejects host tensors; the public model forward STAGES them to the device instead (models/_entry.py,
    tests/test_models_gpu.py::test_host_tensors_are_staged_not_computed_on_the_host) - nothing computes on the host."""
    ops, rt = pk
    with pytest.raises(rt.CnbError):
        ops.groupnorm(torch.zeros(1, 2, 2, 16), torch.ones(16), torch.zeros(16), 8, True)
    with pytest.raises(rt.CnbError):
        ops.conv(torch.zeros(1, 4, 4, 16), torch.zeros(16, 1, 16), "1x1", 16)
    mod = importlib.import_module("controlnet-pytorch_b200.scheduler.linear_noise_scheduler")
    s = mod.LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    with pytest.raises(rt.CnbError):
        s.sample_prev_timestep(torch.zeros(1, 1, 4, 4), torch.zeros(1, 1, 4, 4), torch.as_tensor(5))
