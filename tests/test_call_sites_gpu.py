"""Every kernel launch of the shipped workloads, at their production batch sizes, against a float64 reference element by
element.

The library picks a kernel route at run time from the batch size, the layout and the dtypes, so hand-picked kernel
shapes miss most of what production runs.  Here one eager forward of each production workload is run with synthetic
weights while ops.conv / ops.groupnorm / ops.attention / ops.linear_small record every call's signature (everything
that reaches the C ABI, plus the convolution route from ops.conv_route).  Each distinct signature is then replayed on
seeded random inputs in exactly that layout and checked for
  - route fidelity: the replay takes the harvested route (otherwise it would check something else);
  - windows: every output byte outside the written window (channels before / after it, one guard sample after the
    batch, the other parities of a ConvTranspose phase) and every input byte is unchanged;
  - values, per element: |got - ref| <= tau * mag * s + rho * |ref| on a subset of samples (the first and the last,
    the samples holding the first tile of a CTA's second round and the last tile, two seeded ones), where ref and mag
    are float64 over the operand values the kernel reads, s = 1.1 when SiLU is applied to the output and rho = 2^-11
    for fp16 outputs (one rounding at the store).
Inputs of the tensor-core convolutions are fp16-representable, so every product is exact and the bound measures the
accumulation and the layout only.  A failure names the signature, the route, the sample and the (y, x, channel) of
the worst element.  The CPU tests at the end show the bounds catch single-term, single-column and single-row errors.
"""
import hashlib
import importlib
import math

import pytest
import torch
import torch.nn.functional as F

from helpers import syn

PK = "controlnet-pytorch_b200."

# Per-element tolerance tau (in units of mag) per kernel family: the power of two between 1x and 4x the largest tau the
# production signatures needed on an NVIDIA B200 (1000 W power limit), shown in the last column of the report.
TAU = {
    "conv_tc": 2.0 ** -19,        # tcgen05 kind::f16 / kind::tf32, fp32 accumulation in TMEM (needed 2^-20.7)
    "conv_cuda": 2.0 ** -20,      # CUDA-core fp32 and small-channel kernels (2^-21.0)
    "linear": 2.0 ** -22,         # cnb_linear_small (2^-23.5)
    "attn_f32": 2.0 ** -19,       # exact-fp32 attention core (2^-19.8)
    "attn_f16": 2.0 ** -11,       # fp16 flash attention, P rounded to fp16 (2^-11.9)
    "groupnorm": 2.0 ** -18,      # every GroupNorm kernel (2^-19.1)
}
RHO_F16 = 2.0 ** -11
SENTINEL = 0x7B                    # fp16 60800, fp32 1.3e36: finite, and far from any value the kernels write


# ---------------------------------------------------------------------------------------------------------------------
# comparator (shared by the GPU replays and the CPU self-checks)
# ---------------------------------------------------------------------------------------------------------------------
def compare(got, ref, mag, tau, silu, out_f16):
    """Per-element check of got against ref (float64 tensors of one sample, any layout; the last three dims are read as
    (y, x, channel)).  Returns (worst ratio, index of the worst element, tau the data needed): ratio <= 1 passes."""
    got, ref, mag = got.double(), ref.double(), mag.double()
    s = 1.1 if silu else 1.0
    rho = RHO_F16 if out_f16 else 0.0
    err = (got - ref).abs()
    lim = tau * mag * s + rho * ref.abs()
    ratio = torch.where(err == 0, torch.zeros_like(err), err / lim)
    ratio = torch.where(torch.isfinite(got), ratio, torch.full_like(err, math.inf))
    ratio = torch.nan_to_num(ratio, nan=math.inf)
    need = ((err - rho * ref.abs()).clamp_min(0) / (mag * s).clamp_min(1e-300)).max().item()
    i = int(ratio.flatten().argmax())
    idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), ratio.shape))
    return float(ratio.flatten()[i]), idx, need


def fill_sentinel(t):
    t.view(torch.uint8).fill_(SENTINEL)


def window_violations(buf, mask):
    """Bytes of `buf` outside `mask` (bool, buf's shape) that no longer hold the sentinel: list of element indices."""
    b = buf.view(torch.uint8).reshape(*buf.shape, buf.element_size())
    bad = (b != SENTINEL).any(-1) & ~mask
    return [tuple(int(v) for v in r) for r in bad.nonzero()[:3].tolist()]


def out_window(shape, B, phase, out_coff, cout, device):
    """Elements of a (B + 1, OHf, OWf, ldo) output buffer a convolution writes."""
    m = torch.zeros(shape, dtype=torch.bool, device=device)
    py, px = phase if phase is not None else (0, 0)
    step = 2 if phase is not None else 1
    m[:B, py::step, px::step, out_coff:out_coff + cout] = True
    return m


# ---------------------------------------------------------------------------------------------------------------------
# float64 references
# ---------------------------------------------------------------------------------------------------------------------
def conv_core(x, w, kind, phase):
    """x NCHW, w OIHW (IOHW for a ConvTranspose phase) -> NCHW on the phase's / kind's output grid."""
    if phase is not None:
        return F.conv_transpose2d(x, w, stride=2, padding=1)[:, :, phase[0]::2, phase[1]::2]
    stride, pad = {"3x3": (1, 1), "1x1": (1, 0), "3x3s2": (2, 1), "4x4s2": (2, 1)}[kind]
    return F.conv2d(x, w, stride=stride, padding=pad)


def conv_reference(kind, phase, x, w, x2=None, w2=None, bias=None, temb=None, res=None, act=0):
    """(ref, mag) NHWC float64.  x / x2 NHWC already narrowed to the channels read; temb (n, Cout) rows; res NHWC on the
    output grid."""
    xn = x.double().permute(0, 3, 1, 2)
    pre = conv_core(xn, w.double(), kind, phase)
    mag = conv_core(xn.abs(), w.double().abs(), kind, phase)
    if x2 is not None:
        x2n = x2.double().permute(0, 3, 1, 2)
        pre = pre + F.conv2d(x2n, w2.double())
        mag = mag + F.conv2d(x2n.abs(), w2.double().abs())
    pre, mag = pre.permute(0, 2, 3, 1), mag.permute(0, 2, 3, 1)
    for add in (bias, temb):
        if add is not None:
            a = add.double().reshape(add.shape[0] if add.dim() == 2 else 1, 1, 1, -1)
            pre, mag = pre + a, mag + a.abs()
    if res is not None:
        pre, mag = pre + res.double(), mag + res.double().abs()
    return (F.silu(pre) if act else pre), mag


def groupnorm_reference(x, gamma, beta, G, eps, silu):
    """x (n, H, W, C) -> (ref, mag), statistics in float64 over the values the kernel reads."""
    n, H, W, C = x.shape
    xs = x.double().reshape(n, H * W, G, C // G)
    mean = xs.mean(dim=(1, 3), keepdim=True)
    var = ((xs - mean) ** 2).mean(dim=(1, 3), keepdim=True)
    xh = ((xs - mean) / torch.sqrt(var + eps)).reshape(n, H, W, C)
    g, b = gamma.double(), beta.double()
    pre = g * xh + b
    return (F.silu(pre) if silu else pre), g.abs() * (xh.abs() + 1) + b.abs()


def attention_reference(qkv, heads, drop_keys=None):
    """qkv (n, H, W, 3E) -> (ref, mag) (n, H, W, E).  drop_keys: a key range left out (CPU mutation check only)."""
    n, H, W, E3 = qkv.shape
    E = E3 // 3
    d = E // heads
    q, k, v = [t.double().reshape(n, H * W, heads, d).transpose(1, 2) for t in qkv.split(E, dim=-1)]
    s = q @ k.transpose(-1, -2) / math.sqrt(d)
    if drop_keys is not None:
        s[..., drop_keys[0]:drop_keys[1]] = -math.inf
    p = torch.softmax(s, -1)
    ref = (p @ v).transpose(1, 2).reshape(n, H, W, E)
    mag = (p @ v.abs()).transpose(1, 2).reshape(n, H, W, E)
    return ref, mag


def linear_reference(x, w, b, silu_in, silu_out):
    xi = F.silu(x.double()) if silu_in else x.double()
    pre = xi @ w.double().t() + (b.double() if b is not None else 0.0)
    mag = xi.abs() @ w.double().abs().t() + (b.double().abs() if b is not None else 0.0)
    return (F.silu(pre) if silu_out else pre), mag


# ---------------------------------------------------------------------------------------------------------------------
# harvest
# ---------------------------------------------------------------------------------------------------------------------
def _mod(name):
    return importlib.import_module(PK + name)


def _dt(t):
    return "f16" if t.dtype == torch.float16 else "f32"


def _contig(t, what):
    assert t.is_contiguous(), f"{what} is not contiguous: the replay rebuilds contiguous buffers"


class Recorder:
    """Pass-through replacements of the four ops entry points; `sigs` maps each distinct signature (a tuple) to its
    record, `seen` counts the distinct signatures per workload tag."""

    def __init__(self, ops, rt):
        self.ops, self.rt = ops, rt
        self.real = {k: getattr(ops, k) for k in ("conv", "groupnorm", "attention", "linear_small")}
        self.sigs, self.seen, self.tag = {}, {}, None

    def _add(self, key, rec):
        self.sigs.setdefault(key, rec)
        self.seen.setdefault(self.tag, set()).add(key)

    def conv(self, x, weight, kind, cout, **kw):
        out = self.real["conv"](x, weight, kind, cout, **kw)
        _contig(x, "conv input")
        res, temb, x2 = kw.get("residual"), kw.get("temb"), kw.get("x2")
        mode = self.rt.get_mode() if kw.get("mode") is None else kw["mode"]
        B, H, W, ldi = x.shape
        in_coff = kw.get("in_coff", 0)
        rec = dict(op="conv", mode=mode, kind=kind, phase=kw.get("phase"), B=B, H=H, W=W, ldi=ldi, in_coff=in_coff,
                   cin=ldi - in_coff if kw.get("cin") is None else kw["cin"], cout=cout, OHf=out.shape[1],
                   OWf=out.shape[2], ldo=out.shape[3], out_coff=kw.get("out_coff", 0), in_dt=_dt(x), out_dt=_dt(out),
                   bias=kw.get("bias") is not None, act=kw.get("act", 0), lp=kw.get("weight_lp") is not None,
                   res=None, temb=None, x2=None)
        if res is not None:
            _contig(res, "residual")
            rec["res"] = (_dt(res), res.shape[3], kw.get("res_coff", 0))
        if temb is not None:
            rows = temb.shape[0] if temb.dim() == 2 else 1
            rec["temb"] = (rows, kw.get("temb_ld", 0), temb.storage_offset(), bool(kw.get("temb_per_sample")))
        if x2 is not None:
            _contig(x2, "second input")
            x2_coff = kw.get("x2_coff", 0)
            rec["x2"] = (x2.shape[3], x2_coff, x2.shape[3] - x2_coff if kw.get("cin2") is None else kw["cin2"])
        key = tuple(sorted((k, v) for k, v in rec.items()))
        if key not in self.sigs:
            rec["route"] = self.ops.conv_route(x, weight, kind, cout, **dict(kw, out=out))
        self._add(key, rec)
        return out

    def groupnorm(self, x, gamma, beta, groups, silu, eps=1e-5, out_f16=False):
        _contig(x, "groupnorm input")
        B, H, W, C = x.shape
        rec = dict(op="groupnorm", B=B, H=H, W=W, C=C, G=groups, silu=bool(silu), eps=eps, in_dt=_dt(x),
                   out_f16=bool(out_f16))
        self._add(tuple(sorted(rec.items())), rec)
        return self.real["groupnorm"](x, gamma, beta, groups, silu, eps=eps, out_f16=out_f16)

    def attention(self, qkv, heads, mode=None, kernel=None):
        _contig(qkv, "qkv")
        B, H, W, E3 = qkv.shape
        rec = dict(op="attention", B=B, H=H, W=W, E=E3 // 3, heads=heads, dt=_dt(qkv), kernel=kernel,
                   mode=self.rt.get_mode() if mode is None else mode)
        self._add(tuple(sorted(rec.items())), rec)
        return self.real["attention"](qkv, heads, mode=mode, kernel=kernel)

    def linear_small(self, x, w, b, silu_in=False, silu_out=False, out=None, ldy=None):
        assert out is None, "linear_small into a caller's buffer: extend the replay to that layout"
        _contig(x, "linear_small input")
        R, K = x.shape
        rec = dict(op="linear", R=R, K=K, N=w.shape[0], bias=b is not None, silu_in=bool(silu_in),
                   silu_out=bool(silu_out))
        self._add(tuple(sorted(rec.items())), rec)
        return self.real["linear_small"](x, w, b, silu_in=silu_in, silu_out=silu_out)


def _fill(m, seed=0):
    m.load_state_dict(syn.det_state_dict(m.state_dict(), seed))
    return m.cuda().eval()


def _hint(B, s, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(B, 1, s, s, generator=g, device="cuda") < 0.1).float().expand(B, 3, s, s).contiguous()


def _run_workloads(rec, rt):
    """One eager no_grad forward of each production workload (bench.py configs 2-5)."""
    cn, cnl, vae = _mod("models.controlnet"), _mod("models.controlnet_ldm"), _mod("models.vae")
    cs, dm = _mod("models.consistency_controlnet_distilled"), _mod("models.distribution_matching_controlnet")
    lat = dict(syn.CELEBHQ_LDM_PARAMS, im_channels=4, im_size=32)
    runs = [
        # (tag, batch sizes in f16 mode, batch size in fp32 mode, builder, call)
        ("config2_mnist_controlnet", (1024, 128), 128, lambda: cn.ControlNet(syn.MNIST_PARAMS),
         lambda m, B: m(torch.randn(B, 1, 28, 28, device="cuda"), torch.tensor([500], device="cuda"), _hint(B, 28, 1))),
        ("config3_celebhq_ldm_controlnet", (256, 32), 32,
         lambda: cnl.ControlNet(4, syn.CELEBHQ_LDM_PARAMS, down_sample_factor=32),
         lambda m, B: m(torch.randn(B, 4, 32, 32, device="cuda"), torch.tensor([500], device="cuda"),
                        _hint(B, 1024, 2))),
        ("config3_celebhq_vae_decode", (256, 32), 32, lambda: vae.VAE(3, syn.CELEBHQ_VAE_PARAMS),
         lambda m, B: m.decode(torch.randn(B, 4, 32, 32, device="cuda"))),
        ("config4_consistency_mnist", (4096,), 64, lambda: cs.ConsistencyControlNet(syn.MNIST_PARAMS),
         lambda m, B: m(torch.randn(B, 1, 28, 28, device="cuda"), torch.full((B,), 80.0, device="cuda"),
                        _hint(B, 28, 3))),
        ("config4_consistency_celebhq_latent", (4096,), 64, lambda: cs.ConsistencyControlNet(lat),
         lambda m, B: m(torch.randn(B, 4, 32, 32, device="cuda"), torch.full((B,), 80.0, device="cuda"),
                        _hint(B, 32, 4))),
        ("config5_dm_cifar", (1, 7, 128, 1000, 8192), 7, lambda: dm.DistributionMatchingControlNet(syn.CIFAR_PARAMS),
         lambda m, B: m(torch.randn(B, 3, 32, 32, device="cuda"), torch.full((B,), 999, device="cuda"),
                        _hint(B, 32, 5))),
    ]
    for tag, f16_batches, f32_batch, build, call in runs:
        m = _fill(build())
        for mode, batches in (("f16", f16_batches), ("fp32", (f32_batch,))):
            rt.set_mode(mode)
            for B in batches:
                rec.tag = f"{tag} {mode} B={B}"
                with torch.no_grad():
                    call(m, B)
                torch.cuda.synchronize()
        del m
        torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def harvest():
    ops, rt = _mod("ops"), _mod("runtime")
    assert torch.cuda.is_available()
    rt.lib()
    rec = Recorder(ops, rt)
    prev = rt._MODE
    mp = pytest.MonkeyPatch()
    for k in rec.real:
        mp.setattr(ops, k, getattr(rec, k))
    try:
        _run_workloads(rec, rt)
    finally:
        mp.undo()
        rt._MODE = prev
    print("\nsignatures per workload and mode:")
    for tag, keys in rec.seen.items():
        print(f"  {tag:55s} {len(keys):4d}")
    print(f"  {'distinct over all':55s} {len(rec.sigs):4d}")
    return ops, rt, list(rec.sigs.values())


# ---------------------------------------------------------------------------------------------------------------------
# replay
# ---------------------------------------------------------------------------------------------------------------------
class Report:
    """Worst ratio / needed tau per route row; failures collected so one run reports every broken signature."""

    def __init__(self):
        self.rows, self.failures = {}, []

    def add(self, label, tau_key, ratio, need):
        r = self.rows.setdefault(label, dict(n=0, ratio=0.0, need=0.0, tau=tau_key))
        r["n"] += 1
        r["ratio"], r["need"] = max(r["ratio"], ratio), max(r["need"], need)

    def fail(self, msg):
        self.failures.append(msg)

    def print(self, title):
        print(f"\n{title}: route | signatures | worst ratio | tau | tau the data needed")
        for label, r in sorted(self.rows.items()):
            print(f"  {label:78s} {r['n']:4d}  {r['ratio']:8.4f}  {r['tau']:>18s}=2^{math.log2(TAU[r['tau']]):.0f}  "
                  f"2^{math.log2(r['need']) if r['need'] > 0 else -math.inf:.1f}")

    def check(self):
        assert not self.failures, f"{len(self.failures)} failure(s):\n" + "\n".join(self.failures[:30])


def _gen(sig):
    seed = int(hashlib.sha256(repr(sorted(sig.items(), key=lambda kv: kv[0])).encode()).hexdigest()[:8], 16)
    return seed, torch.Generator(device="cuda").manual_seed(seed)


def _randn(shape, g, dt, scale=1.0):
    """fp16-representable values (every product of two of them is exact in fp32)."""
    x = (torch.randn(shape, generator=g, device="cuda") * scale).half()
    return x if dt == "f16" else x.float()


def _samples(B, seed, extra=(), ends_only=False):
    picks = {0, B - 1} | set(extra)
    if not ends_only:
        g = torch.Generator().manual_seed(seed)
        picks |= set(torch.randint(0, B, (2,), generator=g).tolist())
    return sorted(p for p in picks if 0 <= p < B)


def _tile_samples(sig, route, OH, OW):
    """Samples holding tile `grid` (the first tile of a CTA's second round) and the last tile."""
    if route["path"] != 2:
        return []
    out = []
    for t in (route["grid"], route["ntiles"] - 1):
        if t >= route["ntiles"]:
            continue
        if route["halo"]:
            out.append(t // route["tiles_y"])
        else:
            m0 = (t // route["tiles_n"]) * 128
            out += [m0 // (OH * OW), min(m0 + 127, sig["B"] * OH * OW - 1) // (OH * OW)]
    return out


def conv_label(sig, route):
    if route["path"] != 2:
        return f"conv {('f32', 'small', 'tma')[route['path']]} in={sig['in_dt']} out={sig['out_dt']}"
    halo = f"halo R={route['halo_r']}{' x2' if sig['x2'] else ''}" if route["halo"] else "im2col"
    return (f"conv tma BN={route['bn']} RB={route['rb']} EPI={route['epi']} {halo} bres={route['bres']} "
            f"cta/SM={route['ctas_per_sm']} alt={route['epi_alt']} nbuf={route['epi_nbuf']}")


def replay_conv(ops, rt, sig, rep):
    seed, g = _gen(sig)
    B, H, W, cin, cout, phase, kind = sig["B"], sig["H"], sig["W"], sig["cin"], sig["cout"], sig["phase"], sig["kind"]
    mode = sig["mode"]
    if phase is not None:
        K = 4 * cin
        w = _randn((cin, cout, 4, 4), g, "f32", 1 / math.sqrt(K))
        wp = ops.pack_convT_weight(w, mode != rt.MODE_F32)
        lp = ops.cast_f16(wp)[phase[0] * 2 + phase[1]] if sig["lp"] else None
        wp = wp[phase[0] * 2 + phase[1]]
        OH, OW = H, W
    else:
        k = {"3x3": 3, "1x1": 1, "3x3s2": 3, "4x4s2": 4}[kind]
        K = k * k * cin + (sig["x2"][2] if sig["x2"] else 0)
        w = _randn((cout, cin, k, k), g, "f32", 1 / math.sqrt(K))
        wp = ops.pack_conv_weight(w, mode != rt.MODE_F32 and cin % 4 == 0 and cin > 4 and cout % 16 == 0)
        lp = ops.cast_f16(wp) if sig["lp"] else None
        OH, OW = ops.out_size(kind, H), ops.out_size(kind, W)
    x = _randn((B, H, W, sig["ldi"]), g, sig["in_dt"])
    kw = dict(mode=mode, in_coff=sig["in_coff"], cin=cin, out_coff=sig["out_coff"], act=sig["act"], phase=phase)
    bias = _randn((cout,), g, "f32") if sig["bias"] else None
    kw["bias"] = bias
    x2 = w2 = None
    if sig["x2"]:
        ldi2, x2_coff, cin2 = sig["x2"]
        x2 = _randn((B, OH, OW, ldi2), g, sig["in_dt"])
        w2 = _randn((cout, cin2, 1, 1), g, "f32", 1 / math.sqrt(K))
        p2 = ops.pack_conv_weight(w2, False)
        lp = ops.cast_f16(torch.cat([wp.reshape(cout, -1), p2.reshape(cout, -1)], dim=1).contiguous())
        kw.update(x2=x2, x2_coff=x2_coff, cin2=cin2)
    kw["weight_lp"] = lp
    temb_t = None
    if sig["temb"]:
        rows, ld, off, per = sig["temb"]
        temb_t = _randn((rows, ld), g, "f32")[:, off:]          # the engine's view of its per-U-Net table
        kw.update(temb=temb_t, temb_ld=ld, temb_per_sample=per)
    res = None
    if sig["res"]:
        rdt, ldr, res_coff = sig["res"]
        res = _randn((B, sig["OHf"], sig["OWf"], ldr), g, rdt)
        kw.update(residual=res, res_coff=res_coff)
    odt = torch.float16 if sig["out_dt"] == "f16" else torch.float32
    buf = torch.empty((B + 1, sig["OHf"], sig["OWf"], sig["ldo"]), device="cuda", dtype=odt)
    fill_sentinel(buf)
    kw["out"] = buf[:B]
    label = conv_label(sig, sig["route"])
    route = ops.conv_route(x, wp, kind, cout, **kw)
    name = (f"conv {kind or 'convT'}{phase or ''} mode={mode} B={B} {H}x{W} cin={cin}@{sig['in_coff']}/{sig['ldi']} "
            f"cout={cout}@{sig['out_coff']}/{sig['ldo']} in={sig['in_dt']} out={sig['out_dt']} res={sig['res']} "
            f"temb={sig['temb']} act={sig['act']} x2={sig['x2']} [{label}]")
    if route != sig["route"]:
        rep.fail(f"{name}: replay route {route} != harvested {sig['route']}")
    inputs = [t for t in (x, x2, res, wp, lp, bias, temb_t) if t is not None]
    before = [t.clone() for t in inputs]
    ops.conv(x, wp, kind, cout, **kw)
    torch.cuda.synchronize()
    bad = window_violations(buf, out_window(buf.shape, B, phase, sig["out_coff"], cout, "cuda"))
    if bad:
        rep.fail(f"{name}: bytes outside the output window changed at (sample, y, x, channel) {bad}")
    if not all(torch.equal(a, b) for a, b in zip(inputs, before)):
        rep.fail(f"{name}: an input buffer changed")
    del before
    idx = _samples(B, seed, _tile_samples(sig, sig["route"], OH, OW), ends_only=sig["OHf"] >= 128)
    it = torch.tensor(idx, device="cuda")
    step, (py, px) = (2, phase) if phase is not None else (1, (0, 0))
    got = buf[it][:, py::step, px::step, sig["out_coff"]:sig["out_coff"] + cout].cpu()
    xs = x[it][..., sig["in_coff"]:sig["in_coff"] + cin].cpu()
    x2s = x2[it][..., kw["x2_coff"]:kw["x2_coff"] + kw["cin2"]].cpu() if x2 is not None else None
    tembs = None
    if temb_t is not None:
        tembs = (temb_t[it] if sig["temb"][3] else temb_t[:1])[:, :cout].cpu()
    ress = None
    if res is not None:
        ress = res[it][:, py::step, px::step, sig["res"][2]:sig["res"][2] + cout].cpu()
    ref, mag = conv_reference(kind, phase, xs, w.cpu(), x2s, None if w2 is None else w2.cpu(),
                              None if bias is None else bias.cpu(), tembs, ress, sig["act"])
    tau_key = "conv_tc" if route["path"] == 2 else "conv_cuda"
    worst = (0.0, None, None)
    need = 0.0
    for j, b in enumerate(idx):
        r, e, n = compare(got[j], ref[j], mag[j], TAU[tau_key], sig["act"], sig["out_dt"] == "f16")
        need = max(need, n)
        if r > worst[0]:
            worst = (r, b, e)
    rep.add(label, tau_key, worst[0], need)
    if worst[0] > 1:
        rep.fail(f"{name}: sample {worst[1]} (y, x, channel) {worst[2]} ratio {worst[0]:.3g}")


def replay_groupnorm(ops, rt, sig, rep):
    seed, g = _gen(sig)
    B, H, W, C, G = sig["B"], sig["H"], sig["W"], sig["C"], sig["G"]
    means = (torch.rand((C,), generator=g, device="cuda") * 12 - 6)           # per-channel means of up to +-6
    x = (torch.randn((B, H, W, C), generator=g, device="cuda") * 1.5 + means)
    x = x.half() if sig["in_dt"] == "f16" else x
    gamma = 1 + 0.5 * torch.randn((C,), generator=g, device="cuda")
    beta = 0.5 * torch.randn((C,), generator=g, device="cuda")
    x0 = x.clone()
    y = ops.groupnorm(x, gamma, beta, G, sig["silu"], eps=sig["eps"], out_f16=sig["out_f16"])
    torch.cuda.synchronize()
    split = rt.lib().cnb_groupnorm_workspace_bytes(B, H * W, C, G, 1 if sig["in_dt"] == "f16" else 0) > 0
    label = f"groupnorm {'split-stats' if split else 'one-CTA'} HW={H * W} C={C} G={G}"
    name = f"groupnorm B={B} {H}x{W} C={C} G={G} silu={sig['silu']} in={sig['in_dt']} out_f16={sig['out_f16']} [{label}]"
    if not torch.equal(x, x0):
        rep.fail(f"{name}: the input changed")
    idx = _samples(B, seed, ends_only=H >= 128)
    it = torch.tensor(idx, device="cuda")
    ref, mag = groupnorm_reference(x[it].cpu(), gamma.cpu(), beta.cpu(), G, sig["eps"], sig["silu"])
    got = y[it].cpu()
    tau_key = "groupnorm"
    worst, need = (0.0, None, None), 0.0
    for j, b in enumerate(idx):
        r, e, n = compare(got[j], ref[j], mag[j], TAU[tau_key], sig["silu"], sig["out_f16"])
        need = max(need, n)
        if r > worst[0]:
            worst = (r, b, e)
    rep.add(label, tau_key, worst[0], need)
    if worst[0] > 1:
        rep.fail(f"{name}: sample {worst[1]} (y, x, channel) {worst[2]} ratio {worst[0]:.3g}")


def _attention_kernels(sig):
    if sig["dt"] != "f16":
        return [None]
    d = sig["E"] // sig["heads"]
    eng = _mod("models._engine")
    return [None] + (["tmem"] if d in (4, 8, 16, 24, 32, 48, 64) else []) + (["mma"] if d in eng.ATTN_F16_DIMS else [])


def replay_attention(ops, rt, sig, rep):
    seed, g = _gen(sig)
    B, H, W, E, heads = sig["B"], sig["H"], sig["W"], sig["E"], sig["heads"]
    qkv = _randn((B, H, W, 3 * E), g, sig["dt"])
    q0 = qkv.clone()
    idx = _samples(B, seed)
    it = torch.tensor(idx, device="cuda")
    ref, mag = attention_reference(qkv[it].cpu(), heads)
    f16 = sig["dt"] == "f16"
    tau_key = "attn_f16" if f16 else "attn_f32"
    for kernel in _attention_kernels(sig):
        out = ops.attention(qkv, heads, mode=sig["mode"], kernel=kernel)
        torch.cuda.synchronize()
        label = f"attention {sig['dt']} {kernel or 'default'} d={E // heads}"
        name = f"attention B={B} L={H * W} E={E} heads={heads} [{label}]"
        if not torch.equal(qkv, q0):
            rep.fail(f"{name}: qkv changed")
        got = out[it].cpu()
        worst, need = (0.0, None, None), 0.0
        for j, b in enumerate(idx):
            r, e, n = compare(got[j], ref[j], mag[j], TAU[tau_key], False, f16)
            need = max(need, n)
            if r > worst[0]:
                worst = (r, b, e)
        rep.add(label, tau_key, worst[0], need)
        if worst[0] > 1:
            rep.fail(f"{name}: sample {worst[1]} (y, x, channel) {worst[2]} ratio {worst[0]:.3g}")


def replay_linear(ops, rt, sig, rep):
    seed, g = _gen(sig)
    R, K, N = sig["R"], sig["K"], sig["N"]
    x = torch.randn((R, K), generator=g, device="cuda")
    w = torch.randn((N, K), generator=g, device="cuda") / math.sqrt(K)
    b = torch.randn((N,), generator=g, device="cuda") if sig["bias"] else None
    y = ops.linear_small(x, w, b, silu_in=sig["silu_in"], silu_out=sig["silu_out"])
    torch.cuda.synchronize()
    idx = _samples(R, seed)
    it = torch.tensor(idx, device="cuda")
    ref, mag = linear_reference(x[it].cpu(), w.cpu(), None if b is None else b.cpu(), sig["silu_in"], sig["silu_out"])
    r, e, need = compare(y[it].cpu().reshape(len(idx), 1, 1, N), ref.reshape(len(idx), 1, 1, N),
                         mag.reshape(len(idx), 1, 1, N), TAU["linear"], sig["silu_out"], False)
    label = f"linear_small silu_in={int(sig['silu_in'])} silu_out={int(sig['silu_out'])}"
    rep.add(label, "linear", r, need)
    if r > 1:
        rep.fail(f"linear_small R={R} K={K} N={N} [{label}]: row {idx[e[0]]} column {e[3]} ratio {r:.3g}")


@pytest.mark.gpu
def test_convolutions_at_every_call_site(harvest):
    ops, rt, sigs = harvest
    rep = Report()
    for sig in (s for s in sigs if s["op"] == "conv"):
        replay_conv(ops, rt, sig, rep)
    rep.print("convolutions")
    assert rt.lib().cnb_tc_error_flag() == 0
    rep.check()


@pytest.mark.gpu
def test_groupnorm_attention_linear_at_every_call_site(harvest):
    ops, rt, sigs = harvest
    rep = Report()
    for sig in sigs:
        {"groupnorm": replay_groupnorm, "attention": replay_attention, "linear": replay_linear,
         "conv": lambda *a: None}[sig["op"]](ops, rt, sig, rep)
    rep.print("GroupNorm / attention / linear_small")
    assert rt.lib().cnb_tc_error_flag() == 0
    rep.check()


@pytest.mark.gpu
def test_routes_reached(harvest):
    """The harvest reaches the routes the small-shape kernel tests never did."""
    ops, rt, sigs = harvest
    conv = [(s, s["route"]) for s in sigs if s["op"] == "conv"]
    f16 = [(s, r) for s, r in conv if r["path"] == 2]
    halo32 = [(s, r) for s, r in f16 if r["halo"] and s["H"] == 32 and r["halo_r"] == 3]
    assert any(s["x2"] for s, _ in halo32) and any(not s["x2"] for s, _ in halo32), "halo mode at 32x32"
    assert any(r["ctas_per_sm"] == 2 and r["bres"] and not r["halo"] for _, r in f16), "2 CTAs/SM + resident weights"
    assert any(r["epi"] == 6 and r["epi_nbuf"] == 3 for _, r in f16), "EPI 6 with 3 buffers"
    assert any(r["epi"] == 3 and s["phase"] is not None and s["out_dt"] == "f16" and s["in_dt"] == "f16"
               for s, r in f16), "EPI 3, fp16 ConvTranspose phase into an fp16 buffer"
    widest = {s["cout"]: next(bn for bn in (256, 192, 128, 96, 64, 48, 32, 16) if s["cout"] % bn == 0) for s, _ in f16}
    assert any(r["bn"] < widest[s["cout"]] and not r["halo"] for s, r in f16), "N-split narrowed BN"
    # csrc/groupnorm.cu: 16 channels per group over 49 pixels is 7 vectors per lane, the warp<7> kernel
    assert any(s["op"] == "groupnorm" and s["H"] * s["W"] == 49 and s["C"] // s["G"] == 16 for s in sigs), "warp<7>"
    att = [s for s in sigs if s["op"] == "attention"]
    dims = {s["E"] // s["heads"] for s in att}
    f32_dims = {s["E"] // s["heads"] for s in att if s["dt"] == "f32"}
    assert {96, 128, 192} <= dims
    assert dims == f32_dims, f"head dims never run on the fp32 core: {sorted(dims - f32_dims)}"


# ---------------------------------------------------------------------------------------------------------------------
# CPU self-checks of the comparator: exact results pass, subtle kernel errors fail
# ---------------------------------------------------------------------------------------------------------------------
def _cpu_randn(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).half().float()


def _conv_case(kind, B, H, W, cin, cout, cin2=None):
    K = 9 * cin + (cin2 or 0)
    x = _cpu_randn((B, H, W, cin), 1)
    w = _cpu_randn((cout, cin, 3, 3), 2, 1 / math.sqrt(K))
    x2 = _cpu_randn((B, H, W, cin2), 3) if cin2 else None
    w2 = _cpu_randn((cout, cin2, 1, 1), 4, 1 / math.sqrt(K)) if cin2 else None
    bias = _cpu_randn((cout,), 5)
    ref, mag = conv_reference(kind, None, x, w, x2, w2, bias)
    return x, w, bias, ref, mag


def _passes(got, ref, mag, key, silu=False, f16=False):
    return all(compare(got[j], ref[j], mag[j], TAU[key], silu, f16)[0] <= 1 for j in range(ref.shape[0]))


# the largest K of the harvest (3x3 over 768 channels: CelebHQ mid block at 4x4) and a K-concatenated resnet conv
CONV_SELF_CASES = [("3x3", 2, 4, 4, 768, 768, None), ("3x3", 2, 8, 8, 256, 256, 512)]


@pytest.mark.parametrize("case", CONV_SELF_CASES)
def test_comparator_conv(case):
    x, w, bias, ref, mag = _conv_case(*case)
    for f16 in (False, True):
        exact = ref.to(torch.float16 if f16 else torch.float32)
        assert _passes(exact, ref, mag, "conv_tc", f16=f16)
        assert _passes(exact, ref, mag, "conv_cuda", f16=f16)
    cout = case[5]
    # one dropped product term (of median magnitude) in one output element
    b, y, xx, n = 1, 2, 1, cout // 3
    xn = F.pad(x[b].permute(2, 0, 1), (1, 1, 1, 1))[:, y:y + 3, xx:xx + 3]
    terms = (xn * w[n]).flatten().double()
    term = terms[terms.abs().argsort()[terms.numel() // 2]]
    got = ref.clone()
    got[b, y, xx, n] -= term
    assert not _passes(got.float(), ref, mag, "conv_tc")
    # one output column shifted by one channel
    got = ref.clone()
    got[..., n] = ref[..., n + 1]
    assert not _passes(got.float(), ref, mag, "conv_tc", f16=True)
    # the bias of the last N tile applied to the wrong column
    got = ref.clone()
    got[..., cout - 1] += bias[cout - 2].double() - bias[cout - 1].double()
    assert not _passes(got.float(), ref, mag, "conv_tc", f16=True)


@pytest.mark.parametrize("dt,key", [("f16", "attn_f16"), ("f32", "attn_f32")])
def test_comparator_attention(dt, key):
    B, H, W, E, heads = 2, 16, 16, 128, 2
    qkv = _cpu_randn((B, H, W, 3 * E), 7)
    ref, mag = attention_reference(qkv, heads)
    f16 = dt == "f16"
    assert _passes(ref.to(torch.float16 if f16 else torch.float32), ref, mag, key, f16=f16)
    # a dropped 16-key tile in one query row
    dropped, _ = attention_reference(qkv, heads, drop_keys=(112, 128))
    got = ref.clone()
    got[1, 5, 9] = dropped[1, 5, 9]
    assert not _passes(got, ref, mag, key, f16=f16)
    # a row taken from the neighbouring query
    got = ref.clone()
    got[0, 3, 4] = ref[0, 3, 5]
    assert not _passes(got, ref, mag, key, f16=f16)


@pytest.mark.parametrize("silu,out_f16", [(False, False), (True, False), (False, True), (True, True)])
def test_comparator_groupnorm(silu, out_f16):
    B, H, W, C, G = 2, 32, 32, 128, 32
    g = torch.Generator().manual_seed(11)
    x = (torch.randn(B, H, W, C, generator=g) * 1.5 + torch.rand(C, generator=g) * 12 - 6).half().float()
    gamma, beta = 1 + 0.5 * torch.randn(C, generator=g), 0.5 * torch.randn(C, generator=g)
    key = "groupnorm"
    ref, mag = groupnorm_reference(x, gamma, beta, G, 1e-5, silu)
    dt = torch.float16 if out_f16 else torch.float32
    assert _passes(ref.to(dt), ref, mag, key, silu, out_f16)
    cg = C // G
    # group 5's statistics taken over group 6's channels
    wrong = x.clone()
    wrong[..., 5 * cg:6 * cg] = x[..., 6 * cg:7 * cg]
    xs = wrong.double().reshape(B, H * W, G, cg)
    mean, var = xs.mean(dim=(1, 3)), xs.var(dim=(1, 3), unbiased=False)
    got = ref.clone()
    sl = slice(5 * cg, 6 * cg)
    pre = (gamma[sl].double() * (x[..., sl].double() - mean[:, None, None, 5:6]) /
           torch.sqrt(var[:, None, None, 5:6] + 1e-5) + beta[sl].double())
    got[..., sl] = F.silu(pre) if silu else pre
    assert not _passes(got.to(dt), ref, mag, key, silu, out_f16)
    # one row range (an eighth of the rows) of the split-statistics sums counted twice, the count unchanged
    rows = H * W // 8
    xs = x.double().reshape(B, H * W, G, cg)
    n = H * W * cg
    s1 = (xs.sum(dim=(1, 3)) + xs[:, :rows].sum(dim=(1, 3))) / n
    s2 = ((xs ** 2).sum(dim=(1, 3)) + (xs[:, :rows] ** 2).sum(dim=(1, 3))) / n
    mean, var = s1, (s2 - s1 ** 2).clamp_min(0)
    pre = (gamma.double() * (xs - mean[:, None, :, None]).reshape(B, H, W, C) /
           torch.sqrt(var + 1e-5).repeat_interleave(cg, dim=1)[:, None, None, :] + beta.double())
    got = F.silu(pre) if silu else pre
    assert not _passes(got.to(dt), ref, mag, key, silu, out_f16)


def test_comparator_linear():
    x, w, b = _cpu_randn((4, 512), 1), _cpu_randn((640, 512), 2, 1 / math.sqrt(512)), _cpu_randn((640,), 3)
    ref, mag = linear_reference(x, w, b, True, True)
    shp = (4, 1, 1, 640)
    assert _passes(ref.float().reshape(shp), ref.reshape(shp), mag.reshape(shp), "linear", silu=True)
    got = ref.clone()
    got[2, 7] = ref[2, 8]
    assert not _passes(got.float().reshape(shp), ref.reshape(shp), mag.reshape(shp), "linear", silu=True)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float32])
def test_window_check_reports_one_byte(dtype):
    B, OHf, OWf, ldo, coff, cout = 3, 6, 6, 40, 8, 16
    for phase in (None, (1, 0)):
        buf = torch.empty((B + 1, OHf, OWf, ldo), dtype=dtype)
        fill_sentinel(buf)
        mask = out_window(buf.shape, B, phase, coff, cout, "cpu")
        buf[mask] = 1.0                                   # what the kernel writes
        assert window_violations(buf, mask) == []
        for where in ((0, 0, 0, coff - 1), (1, 2, 3, coff + cout), (B, 0, 0, coff), (2, 5, 5, ldo - 1)):
            bad = buf.clone()
            bad.view(torch.uint8).reshape(*buf.shape, buf.element_size())[where + (0,)] = 0
            assert window_violations(bad, mask) == [where]
        if phase is not None:                              # another parity of the ConvTranspose output
            bad = buf.clone()
            bad.view(torch.uint8).reshape(*buf.shape, buf.element_size())[0, 0, 0, coff, 1] = 0
            assert window_violations(bad, mask) == [(0, 0, 0, coff)]
