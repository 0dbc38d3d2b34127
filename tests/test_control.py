"""Control strength (sampler.ControlOptions, ControlNet._forward_controlled, cnb_guidance_combine): a conditioning scale
on the zero convolutions, a start/end control window served by a plain U-Net step graph, and hint guidance.

CPU: ControlOptions validation and the window rule `keep`.  GPU: the combine kernel against a torch-CPU restatement bit
for bit; the scaled forward against a deep copy with scaled zero convolutions; scale 0 and guidance 0 against the
frozen U-Net; the guided forward against its restatement; graph replay against the eager loop for every scheduler and
option set; a hand-written loop; the default path; launch counts; shards, sample_data_parallel and the LDM sampler;
re-capture and two samplers on one model; oracle parity for the DDPM and the LDM ControlNet.
"""
import copy
import ctypes
import os
import sys

import pytest
import torch

from helpers import (inputs, rel_l2, syn, ROOT, TRAJ_TOL, _base, _ddim, _dpm, _fill, _hang_guard, _mod, _modes,
                     rt)  # noqa: F401 (fixtures)

sys.path.insert(0, os.path.join(ROOT, "oracle"))


def _opts(**kw):
    return _mod("sampler").ControlOptions(**kw)


# ---- CPU ---------------------------------------------------------------------------------------------------
def test_control_options_validation():
    CnbError = _mod("runtime").CnbError
    o = _opts()
    assert (o.scale, o.start, o.end, o.guidance) == (1.0, 0.0, 1.0, 1.0)
    _opts(scale=0, guidance=0, start=0.999, end=1)                          # boundaries are legal
    bad = [dict(scale=float("nan")), dict(scale=float("inf")), dict(scale=-0.1), dict(scale=True),
           dict(guidance=float("nan")), dict(guidance=-float("inf")), dict(guidance=-1), dict(guidance=False),
           dict(start=0.5, end=0.5), dict(start=0.6, end=0.4), dict(start=-0.1), dict(end=1.1),
           dict(start=float("nan")), dict(end=True), dict(scale="1")]
    for kw in bad:
        with pytest.raises(CnbError) as e:
            _opts(**kw)
        assert any(repr(v) in str(e.value) for v in kw.values()), (kw, str(e.value))
    with pytest.raises(Exception):
        o.scale = 2.0                                                       # frozen


def _bits(keep):
    return "".join("T" if k else "F" for k in keep)


def test_keep_is_the_diffusers_window_rule():
    assert _bits(_opts(start=0.0, end=0.5).keep(10)) == "T" * 5 + "F" * 5
    assert _bits(_opts(start=0.2, end=1.0).keep(10)) == "FFTTTTTTTT"
    assert _bits(_opts(start=0.0, end=0.5).keep(3)) == "TFF"
    assert [i for i, k in enumerate(_opts(start=0.1, end=0.9).keep(50)) if k] == list(range(5, 45))
    assert _opts(start=0.5).keep(1) == [False]
    assert _opts().keep(7) == [True] * 7
    for kw in (dict(scale=0.0), dict(guidance=0.0), dict(scale=0, start=0.2, guidance=3)):
        assert _opts(**kw).keep(10) == [False] * 10


# ---- GPU ---------------------------------------------------------------------------------------------------
def _combine(ec, eu, w):
    """cnb_guidance_combine restated in torch-CPU fp32, one rounding per operation."""
    return eu + torch.tensor(w, dtype=torch.float32) * (ec - eu)


@pytest.mark.gpu
def test_guidance_combine_kernel_matches_the_host_restatement(rt):
    ops = _mod("ops")
    g = torch.Generator().manual_seed(4)
    for dt in (torch.float32, torch.float16):
        for C in (1, 4):
            for B, H, W in ((3, 5, 7), (2, 28, 28)):
                for narrow in (False, True):
                    if narrow:                                              # ld = 16, channel offset 3 and 9
                        wide = [(3 * torch.randn(B, H, W, 16, generator=g)).to(dt).cuda() for _ in range(2)]
                        hc, hu = wide[0][..., 3:3 + C], wide[1][..., 9:9 + C]
                    else:
                        hc, hu = ((3 * torch.randn(B, H, W, C, generator=g)).to(dt).cuda() for _ in range(2))
                    ec, eu = ops.nhwc_to_nchw(hc).cpu(), ops.nhwc_to_nchw(hu).cpu()
                    for w in (0.0, 0.5, 2.5, 7.5):
                        got = ops.guidance_combine(hc, hu, w).cpu()
                        assert got.dtype == torch.float32 and got.is_contiguous()
                        assert torch.equal(got, _combine(ec, eu, w)), (dt, C, B, narrow, w)
                        if w == 0.0:
                            assert torch.equal(got, eu)
                    out = torch.full((B, C, H, W), float("nan"), device="cuda")
                    assert ops.guidance_combine(hc, hu, 2.5, out=out) is out
                    assert torch.equal(out.cpu(), _combine(ec, eu, 2.5))
    # rejected arguments
    a = torch.randn(2, 4, 4, 4, device="cuda")
    buf = torch.zeros(4 * 2 * 4 * 4 * 4, device="cuda")
    bad = [lambda: ops.guidance_combine(a, a.half(), 1.0),                  # mixed dtypes
           lambda: ops.guidance_combine(a, a[:1], 1.0),                     # shapes differ
           lambda: ops.guidance_combine(a[0], a[0], 1.0),                   # not 4-d
           lambda: ops.guidance_combine(a.permute(0, 3, 1, 2), a.permute(0, 3, 1, 2), 1.0),   # not channels-last
           lambda: ops.guidance_combine(a, a, 1.0, out=torch.empty(2, 4, 4, 3, device="cuda")),
           lambda: ops.guidance_combine(a.int(), a.int(), 1.0)]
    hc = buf[:128].view(2, 4, 4, 4)
    bad.append(lambda: ops.guidance_combine(hc, a, 1.0, out=buf[64:192].view(2, 4, 4, 4)))   # out overlaps h_c
    bad.append(lambda: ops.guidance_combine(a, hc, 1.0, out=buf[:128].view(2, 4, 4, 4)))     # out is h_u
    L = rt.lib()
    out = torch.empty(2, 4, 4, 4, device="cuda")
    raw = [lambda: L.cnb_guidance_combine(a.data_ptr() + 1, 4, a.data_ptr(), 4, out.data_ptr(), 2, 4, 16,
                                          ctypes.c_float(1.0), 0, rt.stream()),          # misaligned fp32 input
           lambda: L.cnb_guidance_combine(a.data_ptr(), 4, a.data_ptr(), 4, out.data_ptr() + 2, 2, 4, 16,
                                          ctypes.c_float(1.0), 0, rt.stream()),          # misaligned out
           lambda: L.cnb_guidance_combine(a.data_ptr(), 3, a.data_ptr(), 4, out.data_ptr(), 2, 4, 16,
                                          ctypes.c_float(1.0), 0, rt.stream())]          # ld < C
    bad += [lambda fn=fn: rt.check(fn()) for fn in raw]
    for i, fn in enumerate(bad):
        with pytest.raises(rt.CnbError):
            fn()
            torch.cuda.synchronize()
            pytest.fail(f"case {i} was accepted")


def _scaled_copy(m, s):
    """The defined semantics of a conditioning scale: a deep copy whose down / mid zero-conv weights and biases were
    multiplied by s (fp32, one rounding each); the hint block's zero conv is left alone."""
    c = copy.deepcopy(m)
    with torch.no_grad():
        for name, p in c.named_parameters():
            if "_down_zero_convs." in name or "_mid_zero_convs." in name:
                p.mul_(s)
    return c


def _model(kind):
    if kind == "mnist":
        m = _fill(_mod("models.controlnet").ControlNet(syn.MNIST_PARAMS))
        x, hint = inputs("control_mnist", 3, 1, 28)
    else:
        m = _fill(_mod("models.controlnet_ldm").ControlNet(4, syn.TINY_LDM_PARAMS, down_sample_factor=8))
        x, hint = inputs("control_ldm", 2, 4, 8, hint_size=64, p=0.05)
    return m, x.cuda(), hint.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mnist", "ldm"])
def test_scaled_and_guided_forwards(rt, kind):
    m, x, hint = _model(kind)
    t = torch.tensor([437], device="cuda")
    with torch.no_grad():
        for mode in _modes(rt):
            rt.set_mode(mode)
            ec = m(x, t, hint)
            eu = m.trained_unet(x, t)
            assert torch.equal(m._forward_controlled(x, t, hint), ec)
            assert not torch.equal(ec, eu)
            for s in (0.5, 1.7):
                want = _scaled_copy(m, s)(x, t, hint)
                got = m._forward_controlled(x, t, hint, scale=s)
                assert torch.equal(got, want), (mode, s)
                assert not torch.equal(got, ec)
                for w in (0.0, 3.0):
                    got = m._forward_controlled(x, t, hint, scale=s, guidance=w).cpu()
                    assert torch.equal(got, _combine(want.cpu(), eu.cpu(), w)), (mode, s, w)
            # scale 0 is the frozen U-Net exactly: the steps outside the window may run it alone
            assert torch.equal(m._forward_controlled(x, t, hint, scale=0.0), eu), mode
            # the unconditional branch of the guided forward is trained_unet bit for bit (w = 0 returns it)
            assert torch.equal(m._forward_controlled(x, t, hint, guidance=0.0), eu), mode
            for w in (0.5, 7.5):
                got = m._forward_controlled(x, t, hint, guidance=w).cpu()
                assert torch.equal(got, _combine(ec.cpu(), eu.cpu(), w)), (mode, w)
            # the scaled copy is replaced, not accumulated, when the scale changes
            E = _mod("models._engine")
            n = len(E.pinned_scaled(m))
            m._forward_controlled(x, t, hint, scale=0.25)
            assert len(E.pinned_scaled(m)) == n == len(m.trained_unet.downs) + len(m.trained_unet.mids)


def _tiny(rt, mode, B=4):
    rt.set_mode(mode)
    m = _fill(_mod("models.controlnet").ControlNet(syn.TINY_PARAMS))
    x_ref = torch.tanh(syn.det_noise("control:ref", (B, 1, 16, 16))).cuda()
    return m, syn.det_hint(B, 16).cuda(), x_ref


def _scheduler(kind):
    if kind == "ddpm":
        return _base(), 10
    if kind.startswith("ddim"):
        return _ddim(num_inference_steps=10, eta=float(kind[4:])), None
    return _dpm(num_inference_steps=10, variant=kind.split("_")[1]), None


OPTION_SETS = {"window": dict(start=0.0, end=0.5), "scale": dict(scale=0.6), "guidance": dict(guidance=3.0),
               "all": dict(scale=1.3, start=0.2, end=0.9, guidance=2.5)}


@pytest.mark.gpu
@pytest.mark.parametrize("opt", list(OPTION_SETS))
@pytest.mark.parametrize("kind", ["ddpm", "ddim0", "ddim1", "dpm_ode", "dpm_sde"])
def test_graph_equals_eager(rt, kind, opt):
    S = _mod("sampler")
    s, steps = _scheduler(kind)
    ctl = _opts(**OPTION_SETS[opt])
    mask = torch.zeros((4, 1, 16, 16), device="cuda")
    mask[:, :, 3:13, 5:11] = 1.0
    for mode in _modes(rt):
        m, hint, x_ref = _tiny(rt, mode)
        g = S.DDPMSampler(m, s, seed=7)
        e = S.DDPMSampler(m, s, seed=7, use_graph=False)
        x_T = g.draw_xT((4, 1, 16, 16), "cuda")
        a, a0 = g.sample(x_T, hint, steps=steps, control=ctl)
        b, b0 = e.sample(x_T, hint, steps=steps, control=ctl)
        assert torch.equal(a, b) and torch.equal(a0, b0), mode
        assert torch.isfinite(a).all()
        plain, _ = S.DDPMSampler(m, s, seed=7).sample(x_T, hint, steps=steps)
        assert not torch.equal(a, plain)
        for mk in (None, mask):
            a, a0 = g.img2img(x_ref, hint, strength=0.7, mask=mk, steps=steps, control=ctl)
            b, b0 = e.img2img(x_ref, hint, strength=0.7, mask=mk, steps=steps, control=ctl)
            assert torch.equal(a, b) and torch.equal(a0, b0), (mode, mk is None)
        assert g._keep == ctl.keep(g._nsteps) and len(g._graphs) == len(set(g._keep))


@pytest.mark.gpu
def test_sample_is_the_hand_written_loop(rt):
    """The loop from public pieces: the scaled deep copy, trained_unet, the torch restatement of the combine and the
    scheduler's update."""
    S = _mod("sampler")
    m, hint, _ = _tiny(rt, "fp32")
    s = _ddim(num_inference_steps=8, eta=1.0)
    ctl = _opts(scale=0.7, start=0.25, end=0.75, guidance=2.0)
    cp = _scaled_copy(m, 0.7)
    smp = S.DDPMSampler(m, s, seed=9)
    x_T = smp.draw_xT((4, 1, 16, 16), "cuda")
    got, got0 = smp.sample(x_T, hint, control=ctl)
    ts = s.timesteps()
    keep = ctl.keep(len(ts))
    assert _bits(keep) == "FFTTTTFF"
    table = s.coef_table(x_T.device)
    xt, t_dev = x_T.clone(), torch.empty((1,), device="cuda", dtype=torch.int64)
    with torch.no_grad():
        for k, t in enumerate(ts):
            t_dev.fill_(t)
            eu = m.trained_unet(xt, t_dev)
            eps = _combine(cp(xt, t_dev, hint).cpu(), eu.cpu(), 2.0).cuda() if keep[k] else eu
            xt, x0 = s.update(xt, eps, table[t], want_x0=True, seed=9, step=k)
    assert torch.equal(got, xt) and torch.equal(got0, x0)


@pytest.mark.gpu
def test_default_path_and_launch_counts(rt):
    S = _mod("sampler")
    for mode in _modes(rt):
        m, hint, x_ref = _tiny(rt, mode)
        s = _ddim(num_inference_steps=6, eta=1.0)
        runs = []
        for kw in ({}, dict(control=None), dict(control=_opts())):
            smp = S.DDPMSampler(m, s, seed=3)
            x_T = smp.draw_xT((4, 1, 16, 16), "cuda")
            runs.append((smp.sample(x_T, hint, **kw), smp.launches_per_step, smp.plain_launches_per_step))
        for r in runs[1:]:
            assert torch.equal(r[0][0], runs[0][0][0]) and torch.equal(r[0][1], runs[0][0][1])
            assert r[1:] == runs[0][1:] and r[2] is None
        n_default = runs[0][1]
        # the eager frozen U-Net's launches, counted after a warm call (which builds the weight caches)
        xt, t = x_T.clone(), torch.tensor([500], device="cuda")
        with torch.no_grad():
            m.trained_unet(xt, t)
            c0 = rt.launch_count()
            m.trained_unet(xt, t)
            n_unet = rt.launch_count() - c0
        smp = S.DDPMSampler(m, s, seed=3)
        smp.sample(x_T, hint, control=_opts(start=0.5))
        assert smp.plain_launches_per_step == n_unet + 3 and smp.launches_per_step == n_default, mode
        mask = torch.ones((4, 1, 16, 16), device="cuda")
        smp.img2img(x_ref, hint, strength=0.7, mask=mask, control=_opts(start=0.5))
        assert smp.plain_launches_per_step == n_unet + 4 and smp.launches_per_step == n_default + 1
        # scale 0: every step is the plain step, and only the plain graph is captured
        smp.sample(x_T, hint, control=_opts(scale=0.0))
        assert smp.launches_per_step is None and list(smp._graphs) == [False]
        assert smp.plain_launches_per_step == n_unet + 3
        # guidance: the guided step adds the frozen U-Net's decoder to the ControlNet step
        smp.sample(x_T, hint, control=_opts(guidance=2.0))
        assert smp.plain_launches_per_step is None and smp.launches_per_step > n_default


@pytest.mark.gpu
def test_shards_data_parallel_and_ldm_sampler(rt):
    S = _mod("sampler")
    m, hint, _ = _tiny(rt, "fp32")
    s = _ddim(num_inference_steps=8, eta=1.0)
    ctl = _opts(scale=1.2, start=0.1, end=0.8, guidance=2.0)
    B, per = 4, 16 * 16
    g = S.DDPMSampler(m, s, seed=11)
    e = S.DDPMSampler(m, s, seed=11, use_graph=False)
    for off in (0, 3):
        x_T = g.draw_xT((B, 1, 16, 16), "cuda", elem_offset=off)
        a, _ = g.sample(x_T, hint, elem_offset=off, control=ctl)
        lo, _ = e.sample(x_T[:1], hint[:1], elem_offset=off, control=ctl)
        hi, _ = e.sample(x_T[1:], hint[1:], elem_offset=off + per, control=ctl)
        assert rel_l2(torch.cat([lo, hi]).cpu(), a.cpu()) < 1e-5, off
    a, _ = g.sample(g.draw_xT((B, 1, 16, 16), "cuda"), hint, control=ctl)
    d = S.sample_data_parallel(m, s, (B, 1, 16, 16), lambda lo, hi: hint[lo:hi], seed=11, control=ctl)
    assert torch.equal(d, a)
    # a model without a control branch
    dm = _fill(_mod("models.distribution_matching_controlnet").DistributionMatchingControlNet(syn.TINY_PARAMS))
    for use_graph in (True, False):
        with pytest.raises(rt.CnbError):
            S.DDPMSampler(dm, s, use_graph=use_graph).sample(a, hint, control=_opts(scale=0.5))
    with pytest.raises(rt.CnbError):
        g.sample(a, hint, control=dict(scale=0.5))
    # the LDM sampler
    lm = _fill(_mod("models.controlnet_ldm").ControlNet(4, syn.TINY_LDM_PARAMS, down_sample_factor=8))
    vae = _fill(_mod("models.vae").VAE(3, syn.TINY_VAE_PARAMS), seed=1)
    lhint = syn.det_hint(2, 64, p=0.05).cuda()
    ls = _ddim(_base(ldm=True), num_inference_steps=6)
    smp = S.LDMSampler(lm, ls, vae, seed=5)
    x_T = smp.draw_xT((2, 4, 8, 8), "cuda")
    ims, lat = smp.sample_images(x_T, lhint, control=ctl)
    want, _ = S.DDPMSampler(lm, ls, seed=5, use_graph=False).sample(x_T, lhint, control=ctl)
    assert tuple(ims.shape) == (2, 3, 32, 32) and torch.equal(lat, want)
    assert not torch.equal(lat, smp.sample_images(x_T, lhint)[1])


@pytest.mark.gpu
def test_recapture_reuse_and_two_samplers_on_one_model(rt):
    S, E = _mod("sampler"), _mod("models._engine")
    m, hint, _ = _tiny(rt, "f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    hint2 = torch.flip(hint, dims=[3]).contiguous()
    s = _dpm(num_inference_steps=6)
    smp = S.DDPMSampler(m, s, seed=4)
    x_T = smp.draw_xT((4, 1, 16, 16), "cuda")

    def check(ctl, h=hint):
        got = smp.sample(x_T, h, control=ctl)[0]
        assert torch.equal(got, S.DDPMSampler(m, s, seed=4, use_graph=False).sample(x_T, h, control=ctl)[0])
        return got

    base_opts = dict(scale=0.5, start=0.0, end=0.6, guidance=2.0)
    outs = [check(_opts(**base_opts))]
    key = smp._key
    outs.append(check(_opts(**base_opts), hint2))
    assert smp._key == key                                                  # a new hint: the graphs are reused
    for change in (dict(scale=0.8), dict(guidance=1.5), dict(end=0.9), dict(start=0.3)):
        outs.append(check(_opts(**{**base_opts, **change})))
        assert smp._key != key, change
        key = smp._key
    for i in range(len(outs) - 1):
        assert not torch.equal(outs[i], outs[i + 1]), i
    # two samplers on one model with different scales, interleaved: each graph keeps its own scaled weights alive
    A, B = S.DDPMSampler(m, s, seed=4), S.DDPMSampler(m, s, seed=4)
    oa, ob = _opts(scale=0.5), _opts(scale=1.7)
    a1 = A.sample(x_T, hint, control=oa)[0]
    b1 = B.sample(x_T, hint, control=ob)[0]                                 # replaces the model's scaled copies
    junk = [torch.full_like(t, float("nan")) for ent in E.pinned_scaled(m) for t in ent[1]]
    a2 = A.sample(x_T, hint, control=oa)[0]
    b2 = B.sample(x_T, hint, control=ob)[0]
    assert torch.equal(a1, a2) and torch.equal(b1, b2) and not torch.equal(a1, b1)
    assert torch.equal(a1, S.DDPMSampler(m, s, seed=4, use_graph=False).sample(x_T, hint, control=oa)[0])
    del junk


def _oracle_ddim(fwd_c, fwd_u, ctl, base, ts, x_T):
    """DDIM eta = 0 in float64 from the fp32 tables with eps = eu + w * (ec - eu) inside the window, eu outside."""
    sa = base.sqrt_alpha_cum_prod.double()
    s1m = base.sqrt_one_minus_alpha_cum_prod.double()
    keep = ctl.keep(len(ts))
    xt = x_T.double()
    for k, t in enumerate(ts):
        tt = torch.as_tensor(t).unsqueeze(0)
        eps = fwd_u(xt.float(), tt).double()
        if keep[k]:
            eps = eps + ctl.guidance * (fwd_c(xt.float(), tt).double() - eps)
        x0 = (xt - s1m[t] * eps) / sa[t]
        a_p, s_p = (1.0, 0.0) if k + 1 == len(ts) else (float(sa[ts[k + 1]]), float(s1m[ts[k + 1]]))
        xt = a_p * x0 + s_p * eps
    return xt.float()


@pytest.mark.gpu
@pytest.mark.parametrize("ldm", [False, True])
def test_parity_with_the_oracle(rt, ldm):
    import cn_oracle as O
    S = _mod("sampler")
    ctl = _opts(scale=0.7, start=0.0, end=0.75, guidance=1.5)
    if ldm:
        cfg = syn.TINY_LDM_PARAMS
        m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
        _, hint = inputs("control_oracle_ldm", 2, 4, 8, hint_size=64, p=0.05)
        shape, arch, fwd = (2, 4, 8, 8), O.ldm_arch(cfg), O.controlnet_ldm_forward
    else:
        cfg = syn.TINY_PARAMS
        m = _fill(_mod("models.controlnet").ControlNet(cfg))
        _, hint = inputs("control_oracle", 2, 1, 16)
        shape, arch, fwd = (2, 1, 16, 16), O.base_arch(cfg), O.controlnet_ddpm_forward
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    sd_scaled = {k: (v * ctl.scale if ("_down_zero_convs." in k or "_mid_zero_convs." in k) else v)
                 for k, v in sd.items()}
    base = _base(ldm)
    s = _ddim(base, num_inference_steps=4, eta=0.0)
    ts = s.timesteps()
    assert _bits(ctl.keep(len(ts))) == "TTTF"
    x_T = S.DDPMSampler(m, s, seed=2).draw_xT(shape, "cuda").cpu()
    with torch.no_grad():
        want = _oracle_ddim(lambda a, t: fwd(sd_scaled, cfg, a, t, hint),
                            lambda a, t: O.unet_forward(sd, "trained_unet.", arch, a, t), ctl, base, ts, x_T)
    for mode in _modes(rt):
        rt.set_mode(mode)
        got, _ = S.DDPMSampler(m, s, seed=2).sample(x_T.cuda(), hint.cuda(), control=ctl)
        assert rel_l2(got.cpu(), want) < TRAJ_TOL[mode], mode
