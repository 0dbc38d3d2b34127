"""Thin tensor-level wrappers over the C ABI.  Activations are channels-last fp32 CUDA tensors of shape
(B, H, W, C); nothing here does arithmetic in PyTorch - torch only owns the memory."""
import ctypes

import torch

from . import runtime as rt

_TAPS_CACHE = {}


def taps_for(kind):
    """(stride, [(dy, dx), ...]) for the convolution kinds on the path (SURVEY.md Appendix F)."""
    if kind in _TAPS_CACHE:
        return _TAPS_CACHE[kind]
    if kind == "1x1":
        r = (1, [(0, 0)])
    elif kind == "3x3":
        r = (1, [(ky - 1, kx - 1) for ky in range(3) for kx in range(3)])
    elif kind == "3x3s2":
        r = (2, [(ky - 1, kx - 1) for ky in range(3) for kx in range(3)])
    elif kind == "4x4s2":
        r = (2, [(ky - 1, kx - 1) for ky in range(4) for kx in range(4)])
    elif kind.startswith("convT"):
        # one output-parity phase (py, px) of ConvTranspose2d(4, 2, 1): T(0) = dy {0, -1}, T(1) = dy {+1, 0}
        py, px = int(kind[5]), int(kind[6])
        t = {0: (0, -1), 1: (1, 0)}
        r = (1, [(t[py][a], t[px][b]) for a in range(2) for b in range(2)])
    else:
        raise ValueError(kind)
    _TAPS_CACHE[kind] = r
    return r


def out_size(kind, n):
    if kind in ("1x1", "3x3"):
        return n
    if kind == "3x3s2":
        return (n + 2 - 3) // 2 + 1
    if kind == "4x4s2":
        return (n + 2 - 4) // 2 + 1
    raise ValueError(kind)


def empty(*shape, device, dtype=torch.float32):
    return torch.empty(shape, device=device, dtype=dtype)


def _conv_params(x, weight, kind, cout, *, bias=None, temb=None, temb_ld=0, temb_per_sample=False, residual=None,
                 res_coff=0, act=0, out=None, out_coff=0, in_coff=0, cin=None, mode=None, phase=None, weight_lp=None,
                 out_f16=False, x2=None, x2_coff=0, cin2=None):
    """(ConvParams, out) for conv / conv_route; allocates `out` when it is None."""
    rt.require_cuda(x, weight, bias, temb, residual, out, weight_lp, x2)
    half = x.dtype == torch.float16
    if half and weight_lp is None and cout > 4:
        raise rt.CnbError("fp16 activations need the fp16 copy of the packed weights (weight_lp)")
    B, H, W, ldi = x.shape
    cin = ldi - in_coff if cin is None else cin
    if phase is not None:
        py, px = phase
        stride, taps = taps_for(f"convT{py}{px}")
        OH, OW = H, W
        OHf, OWf = 2 * H, 2 * W
        oy_mul, oy_add, ox_mul, ox_add = 2, py, 2, px
    else:
        stride, taps = taps_for(kind)
        OH, OW = out_size(kind, H), out_size(kind, W)
        OHf, OWf = OH, OW
        oy_mul, oy_add, ox_mul, ox_add = 1, 0, 1, 0
    if out is None:
        out = torch.empty((B, OHf, OWf, cout), device=x.device, dtype=torch.float16 if out_f16 else torch.float32)
    assert out.shape[0] == B and out.shape[1] == OHf and out.shape[2] == OWf, (out.shape, (B, OHf, OWf))
    p = rt.ConvParams()
    p.inp, p.weight, p.weight_lp = x.data_ptr(), weight.data_ptr(), rt.ptr(weight_lp)
    p.in_dtype = 1 if half else 0
    p.out_dtype = 1 if out.dtype == torch.float16 else 0
    p.bias, p.temb, p.residual, p.out = rt.ptr(bias), rt.ptr(temb), rt.ptr(residual), out.data_ptr()
    p.B, p.H, p.W, p.Cin, p.ldi, p.in_coff = B, H, W, cin, ldi, in_coff
    p.OH, p.OW, p.OHf, p.OWf = OH, OW, OHf, OWf
    p.oy_mul, p.oy_add, p.ox_mul, p.ox_add = oy_mul, oy_add, ox_mul, ox_add
    p.Cout, p.ldo, p.out_coff = cout, out.shape[3], out_coff
    p.ldr, p.res_coff = (residual.shape[3] if residual is not None else 0), res_coff
    p.res_dtype = 1 if (residual is not None and residual.dtype == torch.float16) else 0
    if x2 is not None:      # second input on the output grid, one extra (0,0) tap appended to K (see cnb200.h)
        if x2.dtype != x.dtype or tuple(x2.shape[:3]) != (B, OH, OW):
            raise rt.CnbError("conv: second input must share the first input's dtype and the output grid")
        p.in2, p.ldi2, p.in2_coff = x2.data_ptr(), x2.shape[3], x2_coff
        p.Cin2 = (x2.shape[3] - x2_coff) if cin2 is None else cin2
    p.stride, p.ntaps = stride, len(taps)
    for i, (dy, dx) in enumerate(taps):
        p.dy[i], p.dx[i] = dy, dx
    p.temb_ld, p.temb_per_sample = temb_ld, 1 if temb_per_sample else 0
    p.act = act
    p.mode = rt.get_mode() if mode is None else mode
    return p, out


def conv(x, weight, kind, cout, **kw):
    """Launch cnb_conv2d.  `x` is (B, H, W, ldi); `weight` is the packed [cout][ntaps][cin] tensor.
    kind in {"1x1","3x3","3x3s2","4x4s2"} or phase=(py,px) for a ConvTranspose2d phase (then `out` is required
    and has spatial size (2H, 2W))."""
    p, out = _conv_params(x, weight, kind, cout, **kw)
    rt.check(rt.lib().cnb_conv2d(ctypes.byref(p), rt.stream()))
    return out


ROUTE_FIELDS = ("path", "rb", "bn", "epi", "halo", "bres", "ctas_per_sm", "epi_alt", "epi_nbuf", "grid", "ntiles",
                "tiles_n", "halo_r", "tiles_y")      # CNB_ROUTE_* order (include/cnb200.h)
PATH_NAMES = ("f32", "small", "tma")                  # CNB_PATH_*


def conv_route(x, weight, kind, cout, **kw):
    """The kernel route conv(...) with the same arguments would take (cnb_conv2d_route), as {ROUTE_FIELDS: int};
    nothing is launched.  Raises what conv would raise before its launch."""
    p, _ = _conv_params(x, weight, kind, cout, **kw)
    r = (ctypes.c_int32 * rt.ROUTE_LEN)()
    rt.check(rt.lib().cnb_conv2d_route(ctypes.byref(p), r))
    return dict(zip(ROUTE_FIELDS, r))


def groupnorm(x, gamma, beta, groups, silu, eps=1e-5, out_f16=False):
    """out_f16: emit the normalised activations as fp16, the operand type of the kind::f16 convolution after it.
    Samples too large for one CTA (VAE decoder levels) take the split-statistics kernel pair, whose scratch buffer is
    allocated here (torch's caching allocator, so it is legal under CUDA-graph capture)."""
    rt.require_cuda(x, gamma, beta)
    B, H, W, C = x.shape
    y = torch.empty((B, H, W, C), device=x.device, dtype=torch.float16 if out_f16 else torch.float32)
    in16 = 1 if x.dtype == torch.float16 else 0
    ws_bytes = rt.lib().cnb_groupnorm_workspace_bytes(B, H * W, C, groups, in16)
    if ws_bytes:
        ws = torch.empty(ws_bytes, device=x.device, dtype=torch.uint8)
        rt.check(rt.lib().cnb_groupnorm_ws(x.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, H * W, C,
                                           groups, eps, 1 if silu else 0, in16, 1 if out_f16 else 0, ws.data_ptr(),
                                           ws_bytes, rt.stream()))
        return y
    rt.check(rt.lib().cnb_groupnorm(x.data_ptr(), y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, H * W, C,
                                    groups, eps, 1 if silu else 0, in16, 1 if out_f16 else 0, rt.stream()))
    return y


def cast_f16(x):
    rt.require_cuda(x)
    y = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    rt.check(rt.lib().cnb_cast_f16(x.data_ptr(), y.data_ptr(), x.numel(), rt.stream()))
    return y


def attention(qkv, heads, mode=None, kernel=None):
    """qkv: (B, H, W, 3E) -> (B, H, W, E).  kernel: None = library default, "tmem" forces the tcgen05 / TMEM kernel,
    "mma" the mma.sync kernel (fp16 tensors only)."""
    rt.require_cuda(qkv)
    B, H, W, E3 = qkv.shape
    E = E3 // 3
    if qkv.dtype == torch.float16:
        out = torch.empty((B, H, W, E), device=qkv.device, dtype=torch.float16)
        fn = {None: rt.lib().cnb_attention_f16, "tmem": rt.lib().cnb_attention_tmem, "mma": rt.lib().cnb_attention_mma}[kernel]
        rt.check(fn(qkv.data_ptr(), out.data_ptr(), B, H * W, E, heads, rt.stream()))
        return out
    out = torch.empty((B, H, W, E), device=qkv.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_attention(qkv.data_ptr(), out.data_ptr(), B, H * W, E, heads,
                                    rt.get_mode() if mode is None else mode, rt.stream()))
    return out


def linear_small(x, w, b, silu_in=False, silu_out=False, out=None, ldy=None):
    rt.require_cuda(x, w, b)
    R, K = x.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((R, N), device=x.device, dtype=torch.float32)
        ldy = N
    rt.check(rt.lib().cnb_linear_small(x.data_ptr(), w.data_ptr(), rt.ptr(b), out.data_ptr(), R, K, N, ldy,
                                       1 if silu_in else 0, 1 if silu_out else 0, rt.stream()))
    return out


def time_embedding(t, factor, dim):
    """t: int64 CUDA tensor (n,) ; factor: fp32 CUDA table (dim/2,)."""
    rt.require_cuda(t, factor)
    n = t.numel()
    out = torch.empty((n, dim), device=t.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_time_embedding(t.data_ptr(), factor.data_ptr(), out.data_ptr(), n, dim, rt.stream()))
    return out


def nchw_to_nhwc(x, out=None, out_coff=0):
    rt.require_cuda(x)
    B, C, H, W = x.shape
    if out is None:
        if C == 1:
            return x.reshape(B, H, W, 1)
        out = torch.empty((B, H, W, C), device=x.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_nchw_to_nhwc(x.data_ptr(), out.data_ptr(), B, C, H * W, out.shape[3], out_coff, rt.stream()))
    return out


def nhwc_to_nchw(x, in_coff=0, c=None, out=None):
    """x: (B, H, W, C) channels-last, contiguous or a channel-narrowed view of a wider contiguous buffer.
    `out`: a contiguous fp32 (B, c, H, W) tensor (e.g. a batch slice of a larger one) to write into."""
    rt.require_cuda(x)
    B, H, W, cv = x.shape
    ld = x.stride(2)
    if x.stride(3) != 1 or x.stride(1) != W * ld or x.stride(0) != H * W * ld or ld < cv:
        raise rt.CnbError("nhwc_to_nchw: expected a channels-last tensor or a channel slice of one")
    c = cv - in_coff if c is None else c
    if out is None:
        if c == 1 and ld == 1 and x.dtype == torch.float32:
            return x.reshape(B, 1, H, W)
        out = torch.empty((B, c, H, W), device=x.device, dtype=torch.float32)
    elif tuple(out.shape) != (B, c, H, W) or out.dtype != torch.float32 or not out.is_contiguous():
        raise rt.CnbError("nhwc_to_nchw: out must be a contiguous fp32 (B, c, H, W) tensor")
    rt.check(rt.lib().cnb_nhwc_to_nchw(x.data_ptr(), ld, in_coff, out.data_ptr(), B, c, H * W,
                                       1 if x.dtype == torch.float16 else 0, rt.stream()))
    return out


def copy_channels(src, dst, d_coff, s_coff=0, c=None):
    rt.require_cuda(src, dst)
    B, H, W, lds = src.shape
    c = lds - s_coff if c is None else c
    if src.dtype != dst.dtype:
        raise rt.CnbError("copy_channels: source and destination must have the same dtype")
    rt.check(rt.lib().cnb_copy_channels(src.data_ptr(), lds, s_coff, dst.data_ptr(), dst.shape[3], d_coff, B * H * W,
                                        c, src.element_size(), rt.stream()))
    return dst


def pack_conv_weight(w, round_tf32):
    """OIHW parameter -> packed [O][KH*KW][I] fp32 (derived cache, never part of a state_dict)."""
    rt.require_cuda(w)
    w = w.detach().contiguous()
    if w.dim() == 2:
        O, I = w.shape
        KH = KW = 1
    else:
        O, I, KH, KW = w.shape
    dst = torch.empty((O, KH * KW, I), device=w.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_pack_conv_weight(w.data_ptr(), dst.data_ptr(), O, I, KH, KW, 1 if round_tf32 else 0,
                                           rt.stream()))
    return dst


def pack_convT_weight(w, round_tf32):
    """ConvTranspose2d (I, O, 4, 4) -> [4][O][4][I]."""
    rt.require_cuda(w)
    w = w.detach().contiguous()
    I, O, KH, KW = w.shape
    assert KH == 4 and KW == 4
    dst = torch.empty((4, O, 4, I), device=w.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_pack_convT_weight(w.data_ptr(), dst.data_ptr(), I, O, 1 if round_tf32 else 0, rt.stream()))
    return dst


def sched_step(xt, eps, coef, z=None, want_x0=True, seed=0, step=0, step_dev=None, elem_offset=0, out=None,
               x0_out=None):
    """out may alias xt (every element is read before it is written by the same thread)."""
    rt.require_cuda(xt, eps, coef, z, step_dev, out, x0_out)
    prev = torch.empty_like(xt) if out is None else out
    x0 = x0_out if x0_out is not None else (torch.empty_like(xt) if want_x0 else None)
    rt.check(rt.lib().cnb_sched_step(xt.data_ptr(), eps.data_ptr(), rt.ptr(z), prev.data_ptr(), rt.ptr(x0),
                                     xt.numel(), coef.data_ptr(), seed, step, rt.ptr(step_dev), elem_offset,
                                     rt.stream()))
    return prev, x0


def ddim_step(xt, eps, coef, z=None, want_x0=True, clip_sample=False, seed=0, step=0, step_dev=None, elem_offset=0,
              out=None, x0_out=None):
    """One DDIM update (cnb_ddim_step); coef is a row of DDIMScheduler.coef_table.  Same conventions as sched_step."""
    rt.require_cuda(xt, eps, coef, z, step_dev, out, x0_out)
    prev = torch.empty_like(xt) if out is None else out
    x0 = x0_out if x0_out is not None else (torch.empty_like(xt) if want_x0 else None)
    rt.check(rt.lib().cnb_ddim_step(xt.data_ptr(), eps.data_ptr(), rt.ptr(z), prev.data_ptr(), rt.ptr(x0), xt.numel(),
                                    coef.data_ptr(), 1 if clip_sample else 0, seed, step, rt.ptr(step_dev),
                                    elem_offset, rt.stream()))
    return prev, x0


def dpm_solver_step(xt, eps, coef, z=None, want_x0=True, clip_sample=False, seed=0, step=0, step_dev=None,
                    elem_offset=0, out=None, x0_out=None, *, hist):
    """One DPM-Solver++ update (cnb_dpm_solver_step); coef is a row of DPMSolverMultistepScheduler.coef_table.  hist
    (fp32, xt's size) holds the previous step's data prediction and receives this step's.  Same conventions as
    sched_step."""
    rt.require_cuda(xt, eps, coef, z, step_dev, out, x0_out, hist)
    if hist.dtype != torch.float32 or hist.numel() != xt.numel() or not hist.is_contiguous():
        raise rt.CnbError("dpm_solver_step: hist must be a contiguous fp32 tensor with xt's number of elements")
    prev = torch.empty_like(xt) if out is None else out
    x0 = x0_out if x0_out is not None else (torch.empty_like(xt) if want_x0 else None)
    rt.check(rt.lib().cnb_dpm_solver_step(xt.data_ptr(), eps.data_ptr(), rt.ptr(z), hist.data_ptr(), prev.data_ptr(),
                                          rt.ptr(x0), xt.numel(), coef.data_ptr(), 1 if clip_sample else 0, seed,
                                          step, rt.ptr(step_dev), elem_offset, rt.stream()))
    return prev, x0


def _f32(name, *tensors):
    for t in tensors:
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise rt.CnbError(f"{name}: expected contiguous fp32 tensors")


def add_noise(x_ref, sqrt_acp, sqrt_one_minus, z=None, seed=0, step=0, elem_offset=0, out=None):
    """sqrt_acp * x_ref + sqrt_one_minus * z (cnb_add_noise): LinearNoiseScheduler.add_noise bit for bit with its fp32
    table values at t.  z=None draws the Philox stream (seed, step, elem_offset + i); out may be x_ref."""
    rt.require_cuda(x_ref, z, out)
    out = torch.empty_like(x_ref) if out is None else out
    _f32("add_noise", x_ref, z, out)
    if (z is not None and z.numel() != x_ref.numel()) or out.numel() != x_ref.numel():
        raise rt.CnbError("add_noise: z and out must have x_ref's number of elements")
    rt.check(rt.lib().cnb_add_noise(x_ref.data_ptr(), rt.ptr(z), out.data_ptr(), x_ref.numel(), float(sqrt_acp),
                                    float(sqrt_one_minus), seed, step, elem_offset, rt.stream()))
    return out


def inpaint_blend(x, x_ref, mask, levels, step=0, step_dev=None, z=None, seed=0, noise_step=0, elem_offset=0):
    """In place on x (NCHW fp32): x = m * x + (1 - m) * (a * x_ref + s * z) with (a, s) = levels[k], k = step_dev[0]
    or step (cnb_inpaint_blend; m == 1 keeps x, m == 0 writes the noised reference exactly).  mask is [B, 1, H, W] or
    [B, C, H, W], 1 = generate, 0 = keep the reference.  z=None draws the Philox stream (seed, noise_step,
    elem_offset + i).  Returns x."""
    rt.require_cuda(x, x_ref, mask, levels, step_dev, z)
    _f32("inpaint_blend", x, x_ref, mask, levels, z)
    B, C, H, W = x.shape
    if tuple(x_ref.shape) != tuple(x.shape) or (z is not None and tuple(z.shape) != tuple(x.shape)):
        raise rt.CnbError("inpaint_blend: x_ref and z must have x's shape")
    if mask.dim() != 4 or tuple(mask.shape) not in ((B, 1, H, W), (B, C, H, W)):
        raise rt.CnbError(f"inpaint_blend: mask must be [{B}, 1 or {C}, {H}, {W}] (got {tuple(mask.shape)})")
    if levels.dim() != 2 or levels.shape[1] != 2 or (step_dev is None and not 0 <= int(step) < levels.shape[0]):
        raise rt.CnbError("inpaint_blend: levels must be [n_steps, 2] and step one of its rows")
    rt.check(rt.lib().cnb_inpaint_blend(x.data_ptr(), x_ref.data_ptr(), mask.data_ptr(), rt.ptr(z), x.numel(), C,
                                        H * W, mask.shape[1], levels.data_ptr(), int(step), rt.ptr(step_dev), seed,
                                        noise_step, elem_offset, rt.stream()))
    return x


def mask_max_pool(mask, f):
    """[B, C, H, W] -> [B, C, H / f, W / f], the maximum over each f x f window (cnb_mask_max_pool): an image-space
    inpainting mask on the latent grid, where a latent cell touching any repainted pixel is repainted."""
    rt.require_cuda(mask)
    _f32("mask_max_pool", mask)
    B, C, H, W = mask.shape
    if f < 1 or H % f or W % f:
        raise rt.CnbError(f"mask_max_pool: H={H} and W={W} must be divisible by f={f}")
    out = torch.empty((B, C, H // f, W // f), device=mask.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_mask_max_pool(mask.data_ptr(), out.data_ptr(), B * C, H, W, f, rt.stream()))
    return out


def philox_normal(shape, device, seed, step, elem_offset=0):
    out = torch.empty(shape, device=device, dtype=torch.float32)
    rt.require_cuda(out)
    rt.check(rt.lib().cnb_philox_normal(out.data_ptr(), out.numel(), seed, step, elem_offset, rt.stream()))
    return out


def x0_from_eps(xt, eps, sqrt_one_minus, sqrt_alpha, t):
    """clamp((xt - sqrt_one_minus[t] * eps) / sqrt_alpha[t], -1, 1); t: int64 (1,) or (B,) on the device."""
    rt.require_cuda(xt, eps, sqrt_one_minus, sqrt_alpha, t)
    if t.dtype != torch.int64 or t.numel() not in (1, xt.shape[0]):
        raise rt.CnbError("x0_from_eps: t must be int64 with 1 or B entries")
    out = torch.empty_like(xt)
    B = xt.shape[0]
    rt.check(rt.lib().cnb_x0_from_eps(xt.data_ptr(), eps.data_ptr(), sqrt_one_minus.data_ptr(), sqrt_alpha.data_ptr(),
                                      t.data_ptr(), t.numel(), sqrt_alpha.numel(), out.data_ptr(), B,
                                      xt.numel() // B, rt.stream()))
    return out


def scale_nchw_to_nhwc(a, x):
    """a[b] * x, NCHW fp32 -> channels-last fp32 in one launch (EDM c_in scaling on the way into conv_in)."""
    rt.require_cuda(a, x)
    B, C, H, W = x.shape
    out = torch.empty((B, H, W, C), device=x.device, dtype=torch.float32)
    rt.check(rt.lib().cnb_scale_nchw_to_nhwc(a.data_ptr(), x.data_ptr(), out.data_ptr(), B, C, H * W, rt.stream()))
    return out


def edm_combine_to_nchw(c_skip, x, c_out, f, in_coff=0, c=None):
    """c_skip[b] * x + c_out[b] * f with f leaving the channels-last workspace (fp32 / fp16, possibly a channel-narrowed
    view): the student's output in NCHW fp32, one launch."""
    rt.require_cuda(c_skip, x, c_out, f)
    B, H, W, cv = f.shape
    ld = f.stride(2)
    if f.stride(3) != 1 or f.stride(1) != W * ld or f.stride(0) != H * W * ld or ld < cv:
        raise rt.CnbError("edm_combine_to_nchw: expected a channels-last tensor or a channel slice of one")
    c = cv - in_coff if c is None else c
    if tuple(x.shape) != (B, c, H, W) or x.dtype != torch.float32 or not x.is_contiguous():
        raise rt.CnbError("edm_combine_to_nchw: x must be the contiguous fp32 NCHW tensor matching f")
    out = torch.empty_like(x)
    rt.check(rt.lib().cnb_edm_combine_to_nchw(c_skip.data_ptr(), x.data_ptr(), c_out.data_ptr(), f.data_ptr(), ld,
                                              in_coff, out.data_ptr(), B, c, H * W,
                                              1 if f.dtype == torch.float16 else 0, rt.stream()))
    return out


def scale_rows(a, x, c=None, y=None):
    rt.require_cuda(a, x, c, y)
    out = torch.empty_like(x)
    B = x.shape[0]
    rt.check(rt.lib().cnb_scale_rows(a.data_ptr(), x.data_ptr(), rt.ptr(c), rt.ptr(y), out.data_ptr(), B,
                                     x.numel() // B, rt.stream()))
    return out
