"""Image-to-image and inpainting sampling (sampler.DDPMSampler.img2img, LDMSampler.img2img_images, cnb_add_noise,
cnb_inpaint_blend, cnb_mask_max_pool, the tail schedules of scheduler/*.py).

CPU: strength_to_skip, the tail schedules and tables of the three schedulers, the noise-level table.  GPU: the three
kernels against torch-CPU restatements bit for bit; img2img without a mask against the plain sampler over the tail
(bit for bit); the mask identities; graph replay against the eager loop, sharding and sample_data_parallel;
re-capture; oracle parity for the DDPM and the LDM ControlNet; an MNIST-size run and the launch count.
"""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from helpers import (inputs, rel_l2, syn, ROOT, TRAJ_TOL, _base, _ddim, _dpm, _fill, _hang_guard, _mod, _modes,
                     rt)  # noqa: F401 (fixtures)

sys.path.insert(0, os.path.join(ROOT, "oracle"))


def _sched():
    return _mod("scheduler.schedule")


# ---- CPU ---------------------------------------------------------------------------------------------------
def test_strength_to_skip():
    sk, CnbError = _sched().strength_to_skip, _mod("runtime").CnbError
    assert sk(10, 1.0) == 0 and sk(10, 1) == 0 and sk(10, 0.1) == 9 and sk(1, 1.0) == 0 and sk(1000, 0.001) == 999
    assert sk(10, 0.55) == 5 and sk(10, 0.999) == 1                       # int() truncates
    # the float product is truncated, not rounded: 100 * 0.29 = 28.999999999999996 keeps 28 steps, not 29
    assert 100 * 0.29 < 29 and sk(100, 0.29) == 100 - 28
    assert sk(50, 0.6) == 50 - 30 and sk(20, 0.5) == 10
    for bad in (0, 0.0, -0.5, 1.0000001, 2, float("nan"), float("inf"), True, "0.5", None):
        with pytest.raises(CnbError):
            sk(10, bad)
    with pytest.raises(CnbError, match=r"S=10.*|strength=0\.05"):
        sk(10, 0.05)                                                        # n = int(0.5) = 0
    with pytest.raises(CnbError) as e:
        sk(3, 0.3)
    assert "S=3" in str(e.value) and "strength=0.3" in str(e.value)


@pytest.mark.parametrize("kind", ["ddpm", "ddim", "dpm"])
def test_tail_schedules_and_tables(kind):
    CnbError = _mod("runtime").CnbError
    base = _base()
    s = {"ddpm": lambda: base, "ddim": lambda: _ddim(base, num_inference_steps=10, eta=0.5),
         "dpm": lambda: _dpm(base, num_inference_steps=10, variant="sde")}[kind]()
    steps = 10 if kind == "ddpm" else None
    full = s.timesteps(steps)
    assert s.timesteps(steps, 0) == full and s.graph_key(steps, 0) == s.graph_key(steps)
    keys = set()
    for skip in range(len(full)):
        assert s.timesteps(steps, skip) == full[skip:]
        keys.add(s.graph_key(steps, skip))
    assert len(keys) == len(full)
    for bad in (len(full), len(full) + 3, -1, 1.0, True):
        for fn in (lambda: s.timesteps(steps, bad), lambda: s.coef_table("cpu", steps, bad),
                   lambda: s.graph_key(steps, bad)):
            with pytest.raises(CnbError):
                fn()
    if kind != "dpm":
        # a row depends on its own timestep and the next one only: the tail reads the same table
        for skip in (1, 4, len(full) - 1):
            assert s.coef_table("cpu", steps, skip) is s.coef_table("cpu", steps)
        return
    for skip in (1, 4, len(full) - 1):
        tail = full[skip:]
        tab = s.coef_table_host(skip=skip)
        want = _dpm(base, timesteps=tail, variant="sde").coef_table_host()
        assert torch.equal(torch.nan_to_num(tab, nan=7.0), torch.nan_to_num(want, nan=7.0)), skip
        assert tab[tail[0], 4] == 0.0                                       # first kept row: first order
        dev = s.coef_table("cpu", skip=skip)
        assert dev is not s.coef_table("cpu") and torch.equal(torch.nan_to_num(dev, nan=7.0),
                                                              torch.nan_to_num(tab, nan=7.0))
    assert s.coef_table_host()[full[4], 4] != 0.0                           # ... which is second order in the full run


@pytest.mark.parametrize("ldm", [False, True])
def test_noise_levels(ldm):
    base = _base(ldm)
    ts = _ddim(base, num_inference_steps=7).timesteps(None, 2)
    lv = _sched().noise_levels(base, ts)
    assert lv.dtype == torch.float32 and tuple(lv.shape) == (len(ts), 2)
    for k in range(len(ts) - 1):
        assert lv[k, 0] == base.sqrt_alpha_cum_prod[ts[k + 1]] and lv[k, 1] == base.sqrt_one_minus_alpha_cum_prod[
            ts[k + 1]], k
    assert lv[-1].tolist() == [1.0, 0.0]
    assert _sched().noise_levels(base, (5,)).tolist() == [[1.0, 0.0]]


# ---- GPU ---------------------------------------------------------------------------------------------------
def _xt_noise(shape, seed, elem_offset=0):
    """The x_T stream the start and the blend draw from, on the host."""
    S = _mod("sampler")
    return _mod("ops").philox_normal(shape, "cuda", seed, S._XT_STEP, elem_offset).cpu()


@pytest.mark.gpu
def test_add_noise_kernel_is_add_noise_bit_for_bit(rt):
    ops, S = _mod("ops"), _mod("sampler")
    g = torch.Generator().manual_seed(1)
    for ldm in (False, True):
        base = _base(ldm)
        for n in (4 * 1024, 4 * 257 + 3, 7):
            x, z = (3 * torch.randn(1, n, generator=g) for _ in range(2))
            for t in (999, 421, 0):
                a, s = base.sqrt_alpha_cum_prod[t], base.sqrt_one_minus_alpha_cum_prod[t]
                want = base.add_noise(x, z, torch.tensor([t]))
                got = ops.add_noise(x.cuda(), float(a), float(s), z=z.cuda())
                assert torch.equal(got.cpu(), want), (ldm, n, t)
                buf = x.cuda()                                              # out aliasing x_ref
                assert ops.add_noise(buf, float(a), float(s), z=z.cuda(), out=buf) is buf
                assert torch.equal(buf.cpu(), want)
                for off in (0, 6, 4 * 1001 + 1):
                    zp = _xt_noise((1, n), 5, off)
                    got = ops.add_noise(x.cuda(), float(a), float(s), seed=5, step=S._XT_STEP, elem_offset=off)
                    assert torch.equal(got.cpu(), base.add_noise(x, zp, torch.tensor([t]))), (n, t, off)
    with pytest.raises(rt.CnbError):
        buf = torch.zeros(4 * 64 + 4, device="cuda")
        ops.add_noise(buf[4:], 0.5, 0.5, out=buf[:-4])                       # out overlaps x_ref without aliasing it
    with pytest.raises(rt.CnbError):
        buf = torch.zeros(4 * 64 + 1, device="cuda")
        ops.add_noise(buf[1:], 0.5, 0.5)                                    # misaligned


def _host_blend(x, xr, m, z, a, s):
    """cnb_inpaint_blend restated in torch-CPU fp32, one rounding per operation."""
    a, s = torch.tensor(a, dtype=torch.float32), torch.tensor(s, dtype=torch.float32)
    m = m.expand_as(x)
    known = a * xr + s * z
    return torch.where(m == 1, x, torch.where(m == 0, known, m * x + (1 - m) * known))


def _mask(shape, kind, g):
    u = torch.rand(shape, generator=g)
    m = (u > 0.5).float()
    if kind == "soft":
        m = torch.where(u < 0.25, u * 4, m)                                 # a quarter of the values strictly inside
    return m


@pytest.mark.gpu
def test_inpaint_blend_kernel_matches_the_host_restatement(rt):
    ops = _mod("ops")
    base = _base()
    ts = _ddim(base, num_inference_steps=9).timesteps(None, 3)
    lv = _sched().noise_levels(base, ts)
    lvd = lv.cuda()
    g = torch.Generator().manual_seed(2)
    for shape in ((2, 4, 8, 8), (3, 3, 5, 7), (1, 1, 16, 16)):
        B, C, H, W = shape
        x, xr, z = (3 * torch.randn(shape, generator=g) for _ in range(3))
        for mc in sorted({1, C}):
            for kind in ("binary", "soft"):
                m = _mask((B, mc, H, W), kind, g)
                for k in (0, len(ts) // 2, len(ts) - 1):
                    a, s = float(lv[k, 0]), float(lv[k, 1])
                    want = _host_blend(x, xr, m, z, a, s)
                    got = ops.inpaint_blend(x.cuda(), xr.cuda(), m.cuda(), lvd, step=k, z=z.cuda()).cpu()
                    assert torch.equal(got, want), (shape, mc, kind, k)
                    keep = m.expand_as(x) == 1
                    assert torch.equal(got[keep], x[keep])                   # generated elements untouched
                    if k == len(ts) - 1:
                        assert torch.equal(got[m.expand_as(x) == 0], xr[m.expand_as(x) == 0])
                    step_dev = torch.tensor([k], dtype=torch.int32, device="cuda")
                    got2 = ops.inpaint_blend(x.cuda(), xr.cuda(), m.cuda(), lvd, step=0, step_dev=step_dev,
                                             z=z.cuda()).cpu()
                    assert torch.equal(got2, want)
                # the Philox stream at unaligned global offsets
                for off in (0, 6, 4 * 1001 + 1):
                    zp = _xt_noise(shape, 9, off)
                    got = ops.inpaint_blend(x.cuda(), xr.cuda(), m.cuda(), lvd, step=1, seed=9, noise_step=(1 << 40),
                                            elem_offset=off).cpu()
                    assert torch.equal(got, _host_blend(x, xr, m, zp, float(lv[1, 0]), float(lv[1, 1]))), (shape, off)
    # rejected arguments
    n = 2 * 4 * 8 * 8
    buf = torch.zeros(3 * n + 8, device="cuda")
    xs, m = (2, 4, 8, 8), torch.ones((2, 1, 8, 8), device="cuda")
    bad = [lambda: ops.inpaint_blend(buf[:n].view(xs), buf[4:n + 4].view(xs), m, lvd),           # x overlaps x_ref
           lambda: ops.inpaint_blend(buf[:n].view(xs), buf[n:2 * n].view(xs), buf[4:132].view(2, 1, 8, 8), lvd),
           lambda: ops.inpaint_blend(buf[1:n + 1].view(xs), buf[n + 4:2 * n + 4].view(xs), m, lvd),  # misaligned
           lambda: ops.inpaint_blend(buf[:n].view(xs), buf[n + 1:2 * n + 1].view(xs), m, lvd),
           lambda: ops.inpaint_blend(buf[:n].view(xs), buf[n:2 * n].view(xs), torch.ones((2, 2, 8, 8), device="cuda"),
                                     lvd),
           lambda: ops.inpaint_blend(buf[:n].view(xs), buf[n:2 * n].view(xs), m, lvd, step=len(ts))]
    for i, fn in enumerate(bad):
        with pytest.raises(rt.CnbError):
            fn()
            torch.cuda.synchronize()
            pytest.fail(f"case {i} was accepted")


@pytest.mark.gpu
def test_mask_max_pool_is_max_pool2d(rt):
    ops = _mod("ops")
    g = torch.Generator().manual_seed(3)
    for shape, f in (((2, 1, 32, 32), 4), ((3, 1, 64, 48), 8), ((1, 2, 6, 9), 3), ((2, 1, 5, 5), 1)):
        m = _mask(shape, "soft", g)
        assert torch.equal(ops.mask_max_pool(m.cuda(), f).cpu(), F.max_pool2d(m, f))
    with pytest.raises(_mod("runtime").CnbError):
        ops.mask_max_pool(torch.ones((1, 1, 10, 8), device="cuda"), 4)


def _tiny(rt, B=4):
    rt.set_mode("fp32")
    m = _fill(_mod("models.controlnet").ControlNet(syn.TINY_PARAMS))
    x_ref = torch.tanh(syn.det_noise("img2img:ref", (B, 1, 16, 16))).cuda()
    return m, syn.det_hint(B, 16).cuda(), x_ref


def _plain(kind, base, tail, eta_or_variant):
    if kind == "ddim":
        return _ddim(base, timesteps=tail, eta=eta_or_variant)
    return _dpm(base, timesteps=tail, variant=eta_or_variant)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,arg", [("ddpm", None), ("ddim", 0.0), ("ddim", 1.0), ("dpm", "ode"), ("dpm", "sde")])
def test_img2img_is_the_plain_sampler_over_the_tail_and_the_mask_identities(rt, kind, arg):
    S = _mod("sampler")
    m, hint, x_ref = _tiny(rt)
    base = _base()
    if kind == "ddpm":
        s, steps, strength = base, 12, 0.5
    else:
        s, steps, strength = (_ddim(base, num_inference_steps=10, eta=arg) if kind == "ddim" else
                              _dpm(base, num_inference_steps=10, variant=arg)), None, 0.6
    skip = _sched().strength_to_skip(len(s.timesteps(steps)), strength)
    tail = s.timesteps(steps, skip)
    seed = 13
    smp = S.DDPMSampler(m, s, seed=seed)
    got, got0 = smp.img2img(x_ref, hint, strength=strength, steps=steps)
    n_plain = smp.launches_per_step
    # the plain sampler over the tail, started from add_noise(x_ref, z, tau_skip) on the host
    z = _xt_noise(tuple(x_ref.shape), seed)
    start = base.add_noise(x_ref.cpu(), z, torch.full((x_ref.shape[0],), tail[0])).cuda()
    if kind == "ddpm":
        plain, p_steps = S.DDPMSampler(m, base, seed=seed), len(tail)
        assert tail == base.timesteps(p_steps)
    else:
        plain, p_steps = S.DDPMSampler(m, _plain(kind, base, tail, arg), seed=seed), None
    want, want0 = plain.sample(start, hint, steps=p_steps)
    assert torch.equal(got, want) and torch.equal(got0, want0)
    assert plain.launches_per_step == n_plain
    # a mask of all ones is no mask, with one more launch per step
    ones = torch.ones((x_ref.shape[0], 1, 16, 16), device="cuda")
    a, a0 = smp.img2img(x_ref, hint, strength=strength, mask=ones, steps=steps)
    assert torch.equal(a, got) and torch.equal(a0, got0)
    assert smp.launches_per_step == n_plain + 1
    # all zeros keeps the reference exactly
    a, _ = smp.img2img(x_ref, hint, strength=strength, mask=torch.zeros_like(ones, dtype=torch.bool), steps=steps)
    assert torch.equal(a, x_ref)
    # mixed: the kept region is the reference bit for bit, the repainted region is not
    mix = torch.zeros_like(ones)
    mix[:, :, 4:12, 2:9] = 1.0
    a, _ = smp.img2img(x_ref, hint, strength=strength, mask=mix, steps=steps)
    keep = (mix == 0).expand_as(x_ref)
    assert torch.equal(a[keep], x_ref[keep])
    assert not torch.equal(a[~keep], x_ref[~keep])
    assert torch.isfinite(a).all()


@pytest.mark.gpu
def test_graph_equals_eager_shards_and_data_parallel(rt):
    S = _mod("sampler")
    m, hint, x_ref = _tiny(rt)
    s = _ddim(num_inference_steps=8, eta=1.0)
    B, per = 4, 16 * 16
    mask = torch.zeros((B, 1, 16, 16), device="cuda")
    mask[:, :, 3:13, 5:11] = 1.0
    mask[:, :, 3:13, 11] = 0.5                                               # a soft edge
    g = S.DDPMSampler(m, s, seed=11, use_graph=True)
    e = S.DDPMSampler(m, s, seed=11, use_graph=False)
    for off in (0, 3):                                                       # an unaligned global offset
        a, a0 = g.img2img(x_ref, hint, strength=0.7, mask=mask, elem_offset=off)
        b, b0 = e.img2img(x_ref, hint, strength=0.7, mask=mask, elem_offset=off)
        assert torch.equal(a, b) and torch.equal(a0, b0), off
        lo, _ = e.img2img(x_ref[:1], hint[:1], strength=0.7, mask=mask[:1], elem_offset=off)
        hi, _ = e.img2img(x_ref[1:], hint[1:], strength=0.7, mask=mask[1:], elem_offset=off + per)
        c = torch.cat([lo, hi])
        assert rel_l2(c.cpu(), b.cpu()) < 1e-5, off
        keep = (mask == 0).expand_as(x_ref)
        assert torch.equal(c[keep], b[keep]) and torch.equal(b[keep], x_ref[keep])
    a, _ = g.img2img(x_ref, hint, strength=0.7, mask=mask)
    d = S.sample_data_parallel(m, s, (B, 1, 16, 16), lambda lo, hi: hint[lo:hi], seed=11,
                               x_ref_fn=lambda lo, hi: x_ref[lo:hi], mask_fn=lambda lo, hi: mask[lo:hi], strength=0.7)
    assert torch.equal(d, a)
    with pytest.raises(rt.CnbError):
        S.sample_data_parallel(m, s, (B, 1, 16, 16), lambda lo, hi: hint[lo:hi], x_T_fn=lambda lo, hi: x_ref[lo:hi],
                               x_ref_fn=lambda lo, hi: x_ref[lo:hi])
    for bad in (mask * 2, mask - 0.5, torch.full_like(mask, float("nan")), mask[:, :, :8]):
        with pytest.raises(rt.CnbError):
            g.img2img(x_ref, hint, strength=0.7, mask=bad)
    with pytest.raises(rt.CnbError):
        g.img2img(x_ref, hint, strength=0.01)                                # keeps no step of 8


@pytest.mark.gpu
def test_every_path_rejects_a_hint_of_another_batch_size_before_launching(rt):
    """The ControlNet forward reads the hint by sample, so a hint with fewer samples than x would be read past its end:
    the eager paths check it as the graph paths do, before the first launch."""
    S = _mod("sampler")
    m, hint, x_ref = _tiny(rt)
    s = _ddim(num_inference_steps=4)
    e, g = S.DDPMSampler(m, s, seed=1, use_graph=False), S.DDPMSampler(m, s, seed=1)
    x_T = e.draw_xT(tuple(x_ref.shape), "cuda")
    zs = [torch.zeros(tuple(x_ref.shape)) for _ in range(4)]
    mask = torch.ones((4, 1, 16, 16), device="cuda")
    for h in (hint[:3], torch.cat([hint, hint[:1]])):
        calls = [lambda: e.sample(x_T, h), lambda: e.sample_eager(x_T, h, zs=zs),
                 lambda: e.img2img(x_ref, h, strength=0.5), lambda: e.img2img(x_ref, h, strength=0.5, mask=mask),
                 lambda: e.sample_eager(x_T, h, x_ref=x_ref, mask=mask, strength=0.5),
                 lambda: g.sample(x_T, h), lambda: g.img2img(x_ref, h, strength=0.5, mask=mask)]
        for i, fn in enumerate(calls):
            c0 = rt.launch_count()
            with pytest.raises(rt.CnbError, match="batch size"):
                fn()
            assert rt.launch_count() == c0, (h.shape[0], i)


@pytest.mark.gpu
def test_one_sampler_recaptures_on_every_change(rt):
    S = _mod("sampler")
    rt.set_mode("fp32")
    cfg = syn.TINY_LDM_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
    x_ref, hint = inputs("img2img_recap", 2, 4, 8, hint_size=64, p=0.05)
    x_ref, hint = torch.tanh(x_ref).cuda(), hint.cuda()
    base = _base(ldm=True)
    state = {"s": _ddim(base, num_inference_steps=6, eta=1.0)}
    smp = S.DDPMSampler(m, state["s"], seed=4)
    m1 = torch.zeros((2, 1, 8, 8), device="cuda")
    m1[:, :, 2:6, 1:5] = 1.0
    m2 = torch.roll(m1, 2, dims=3)
    m4 = torch.zeros((2, 4, 8, 8), device="cuda")
    m4[:, 1:3, 2:7, 2:7] = 1.0

    def check(strength, mask):
        got, got0 = smp.img2img(x_ref, hint, strength=strength, mask=mask)
        want, want0 = S.DDPMSampler(m, state["s"], seed=4).img2img(x_ref, hint, strength=strength, mask=mask)
        assert torch.equal(got, want) and torch.equal(got0, want0)
        return got

    outs = [check(0.5, None), check(0.8, None), check(0.8, m1)]
    key = smp._key
    outs.append(check(0.8, m2))
    assert smp._key == key                                                   # new mask values: copied, no re-capture
    outs.append(check(0.8, m4))
    outs.append(check(0.8, None))
    state["s"] = smp.scheduler = _dpm(base, num_inference_steps=6)
    outs.append(check(0.8, m1))
    m.load_state_dict(syn.det_state_dict(m.state_dict(), seed=6))
    outs.append(check(0.8, m1))
    for i in range(len(outs) - 1):
        assert not torch.equal(outs[i], outs[i + 1]), i


def _oracle_img2img(forward, base, ts, x_ref, z, mask):
    """DDIM eta = 0 over the tail `ts` in float64 from the fp32 tables: start add_noise(x_ref, z, ts[0]), after step k
    the blend with the noise level of ts[k + 1] (x_ref after the last step)."""
    sa = base.sqrt_alpha_cum_prod.double()
    s1m = base.sqrt_one_minus_alpha_cum_prod.double()
    xr, z, m = x_ref.double(), z.double(), mask.double()
    xt = sa[ts[0]] * xr + s1m[ts[0]] * z
    for k, t in enumerate(ts):
        last = k + 1 == len(ts)
        eps = forward(xt.float(), torch.as_tensor(t).unsqueeze(0)).double()
        x0 = (xt - s1m[t] * eps) / sa[t]
        a_p, s_p = (1.0, 0.0) if last else (float(sa[ts[k + 1]]), float(s1m[ts[k + 1]]))
        xt = a_p * x0 + s_p * eps
        xt = m * xt + (1 - m) * (a_p * xr + s_p * z)
    return xt.float()


@pytest.mark.gpu
def test_ddpm_controlnet_parity_with_the_oracle(rt):
    import cn_oracle as O
    S = _mod("sampler")
    cfg = syn.TINY_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    x_ref, hint = inputs("img2img_tiny", 2, 1, 16)
    x_ref = torch.tanh(x_ref)
    mask = torch.zeros((2, 1, 16, 16))
    mask[:, :, 2:10, 4:14] = 1.0
    mask[:, :, 10, 4:14] = 0.25
    base = _base()
    s = _ddim(base, num_inference_steps=4, eta=0.0)
    ts = s.timesteps(None, _sched().strength_to_skip(4, 0.6))
    assert len(ts) == 2
    z = _xt_noise((2, 1, 16, 16), 3)
    with torch.no_grad():
        want = _oracle_img2img(lambda a, t: O.controlnet_ddpm_forward(sd, cfg, a, t, hint), base, ts, x_ref, z, mask)
    for mode in _modes(rt):
        rt.set_mode(mode)
        got, _ = S.DDPMSampler(m, s, seed=3).img2img(x_ref.cuda(), hint.cuda(), strength=0.6, mask=mask.cuda())
        assert rel_l2(got.cpu(), want) < TRAJ_TOL[mode], mode
        assert torch.equal(got.cpu()[mask.expand_as(x_ref) == 0], x_ref[mask.expand_as(x_ref) == 0])


@pytest.mark.gpu
def test_ldm_controlnet_with_vae_parity_with_the_oracle(rt):
    import cn_oracle as O
    S = _mod("sampler")
    cfg, vcfg = syn.TINY_LDM_PARAMS, syn.TINY_VAE_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
    vae = _fill(_mod("models.vae").VAE(3, vcfg), seed=1)
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    vsd = {k: v.cpu() for k, v in vae.state_dict().items()}
    images = torch.tanh(syn.det_noise("img2img_ldm:images", (2, 3, 32, 32)))
    hint = syn.det_hint(2, 64, p=0.05)
    mask = torch.zeros((2, 1, 32, 32))
    mask[:, :, 5:19, 9:30] = 1.0                                             # not aligned to the 4x4 latent cells
    lmask = F.max_pool2d(mask, 4)
    base = _base(ldm=True)
    s = _ddim(base, num_inference_steps=4, eta=0.0)
    ts = s.timesteps(None, _sched().strength_to_skip(4, 0.6))
    z = _xt_noise((2, 4, 8, 8), 5)
    with torch.no_grad():
        lat0 = O.vae_encode(vsd, vcfg, images)[1][:, :vcfg["z_channels"]]
        lat_ref = _oracle_img2img(lambda a, t: O.controlnet_ldm_forward(sd, cfg, a, t, hint), base, ts, lat0, z,
                                  lmask)
        want = (torch.clamp(O.vae_decode(vsd, vcfg, lat_ref), -1., 1.) + 1) / 2
    for mode in _modes(rt):
        rt.set_mode(mode)
        smp = S.LDMSampler(m, s, vae, seed=5)
        assert torch.equal(smp.latent_mask(mask.cuda(), torch.empty((2, 4, 8, 8), device="cuda")).cpu(), lmask)
        assert rel_l2(smp.encode_mean(images.cuda()).cpu(), lat0) < TRAJ_TOL[mode], mode
        ims, lat = smp.img2img_images(images.cuda(), hint.cuda(), strength=0.6, mask=mask.cuda())
        assert tuple(ims.shape) == (2, 3, 32, 32)
        assert rel_l2(lat.cpu(), lat_ref) < TRAJ_TOL[mode], mode
        assert rel_l2(ims.cpu(), want) < TRAJ_TOL[mode], mode
        keep = (lmask == 0).expand_as(lat_ref)
        assert torch.equal(lat.cpu()[keep], smp.encode_mean(images.cuda()).cpu()[keep])   # the known latents, exactly
        d = S.sample_data_parallel(m, s, (2, 4, 8, 8), lambda lo, hi: hint[lo:hi].cuda(), seed=5, vae=vae,
                                   x_ref_fn=lambda lo, hi: images[lo:hi].cuda(),
                                   mask_fn=lambda lo, hi: mask[lo:hi].cuda(), strength=0.6)
        assert torch.equal(d, ims)


@pytest.mark.gpu
def test_mnist_size_run_and_launch_count(rt):
    S = _mod("sampler")
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    m = _fill(_mod("models.controlnet").ControlNet(syn.MNIST_PARAMS))
    hint = syn.det_hint(64, 28).cuda()
    x_ref = torch.tanh(syn.det_noise("img2img_mnist:ref", (64, 1, 28, 28))).cuda()
    mask = torch.zeros((64, 1, 28, 28), device="cuda")
    mask[:, :, 6:22, 3:17] = 1.0
    s = _ddim(num_inference_steps=50, eta=1.0)
    g = S.DDPMSampler(m, s, seed=3)
    a, a0 = g.img2img(x_ref, hint, strength=0.5, mask=mask)
    b, b0 = S.DDPMSampler(m, s, seed=3, use_graph=False).img2img(x_ref, hint, strength=0.5, mask=mask)
    assert torch.isfinite(a).all() and torch.isfinite(a0).all()
    assert torch.equal(a, b) and torch.equal(a0, b0)
    d = S.DDPMSampler(m, s, seed=3)
    d.sample(S.DDPMSampler(m, s, seed=3).draw_xT((64, 1, 28, 28), "cuda"), hint, steps=2)
    assert g.launches_per_step == d.launches_per_step + 1
