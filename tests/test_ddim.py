"""DDIM sampling (scheduler/ddim_scheduler.py, cnb_ddim_step).

CPU: the timestep schedules, the rejection of bad schedules and the [T, 6] coefficient table against an independent
float64 restatement.  GPU: the fused kernel against a torch-CPU fp32 restatement of its operation order (bit for bit),
its Philox noise and x0 against the DDPM kernel, the DDPM limit (eta = 1, every timestep), parity of the sampled
trajectory with the oracle for the DDPM and the LDM ControlNet, graph replay against the eager loop, sharding,
re-capture and the launch count of the captured step.  The oracle parity and MNIST-size tests also run DPM-Solver++.
"""
import os
import sys

import pytest
import torch

from helpers import (inputs, max_abs, rel_l2, syn, ROOT, TRAJ_TOL, _base, _ddim, _ddim_oracle_loop, _ddim_rows, _dpm,
                     _dpm_oracle_loop, _fill, _hang_guard, _mod, _modes, rt)  # noqa: F401 (fixtures)

sys.path.insert(0, os.path.join(ROOT, "oracle"))

# the oracle parity cases: (the scheduler over a base scheduler, its host oracle loop); the name seeds the inputs
ORACLE_CASES = {"ddim": (lambda base: _ddim(base, num_inference_steps=4, eta=0.0), _ddim_oracle_loop),
                "dpm": (lambda base: _dpm(base, num_inference_steps=4), _dpm_oracle_loop)}


# ---- CPU ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 20, 50, 999, 1000])
def test_timestep_sequences(S):
    T = 1000
    tr = _ddim(num_inference_steps=S).timesteps()
    ld = _ddim(num_inference_steps=S, spacing="leading").timesteps()
    want_tr = (torch.round(T - torch.arange(S, dtype=torch.float64) * (T / S)) - 1).long().tolist()
    assert list(tr) == want_tr and tr[0] == T - 1
    assert list(ld) == [(S - 1 - k) * (T // S) for k in range(S)] and ld[-1] == 0
    for ts in (tr, ld):
        assert len(ts) == S and all(a > b for a, b in zip(ts, ts[1:])) and 0 <= ts[-1]
    if S == T:
        assert tr == ld == tuple(range(T - 1, -1, -1))
    if S == 20:
        assert tr == tuple(range(999, 0, -50)) and ld == tuple(range(950, -1, -50))
    assert _ddim(num_inference_steps=7).timesteps(S) == tr          # steps= overrides the scheduler's own S


def test_bad_schedules_are_rejected():
    CnbError = _mod("runtime").CnbError
    for kw in (dict(num_inference_steps=0), dict(num_inference_steps=1001), dict(num_inference_steps=2.5),
               dict(eta=-0.1), dict(eta=float("nan")), dict(spacing="linspace"), dict(timesteps=[3, 3, 1]),
               dict(timesteps=[1, 2]), dict(timesteps=[1000, 5]), dict(timesteps=[5, -1]), dict(timesteps=[])):
        with pytest.raises(CnbError):
            _ddim(**kw)
    s = _ddim(timesteps=[9, 4, 0])
    assert s.timesteps() == s.timesteps(3) == (9, 4, 0)
    with pytest.raises(CnbError):
        s.timesteps(4)
    s = _ddim()
    s.eta = -1.0                                                      # attributes are re-validated on use
    with pytest.raises(CnbError):
        s.coef_table_host()


@pytest.mark.parametrize("ldm", [False, True])
@pytest.mark.parametrize("S,eta,spacing", [(50, 0.0, "trailing"), (20, 0.5, "leading"), (1, 1.0, "trailing")])
def test_coef_table_matches_the_restated_contract(ldm, S, eta, spacing):
    base = _base(ldm)
    s = _ddim(base, num_inference_steps=S, eta=eta, spacing=spacing)
    ts = s.timesteps()
    tab = s.coef_table_host()
    assert tab.shape == (1000, 6) and tab.dtype == torch.float32
    want = _ddim_rows(base, ts, eta)
    ddpm = base.coef_table_host()
    on = torch.zeros(1000, dtype=torch.bool)
    on[list(ts)] = True
    assert torch.isnan(tab[~on]).all()                                # off-schedule rows poison the output
    for t, row in want.items():
        assert torch.equal(tab[t], torch.tensor(row, dtype=torch.float64).float()), t
        assert torch.equal(tab[t, :2], ddpm[t, :2]), t                # the DDPM table's fp32 values, bit for bit
    assert tab[ts[-1], 2:].tolist() == [1.0, 0.0, 0.0, 0.0]
    if eta == 0.0:
        assert (tab[on, 4:] == 0).all()


@pytest.mark.parametrize("ldm", [False, True])
def test_eta1_at_every_timestep_has_the_ddpm_posterior_sigma(ldm):
    base = _base(ldm)
    tab = _ddim(base, num_inference_steps=1000, eta=1.0).coef_table_host().double()
    ddpm = base.coef_table_host().double()
    assert tab[0, 4] == 0.0 and ddpm[0, 4] == 0.0
    rel = ((tab[1:, 4] - ddpm[1:, 4]) / ddpm[1:, 4]).abs()
    assert float(rel.max()) < 2e-3
    assert torch.equal(tab[1:, 5], ddpm[1:, 5]) and tab[0, 5] == 0.0


# ---- GPU ---------------------------------------------------------------------------------------------------
def _host_ddim(xt, eps, z, row, clip):
    """The kernel's operation order in torch-CPU fp32, one rounding per operation."""
    c = row.float()
    x0 = (xt - c[0] * eps) / c[1]
    x0c = torch.clamp(x0, -1.0, 1.0)
    prev = c[2] * (x0c if clip else x0) + c[3] * eps
    if float(c[5]) != 0.0:
        prev = prev + c[4] * z
    return prev, x0c


@pytest.mark.gpu
def test_kernel_matches_the_host_restatement_bit_for_bit(rt):
    ops = _mod("ops")
    s = _ddim(num_inference_steps=50, eta=0.7)
    ts = s.timesteps()
    tab = s.coef_table_host()
    dtab = s.coef_table("cuda")
    g = torch.Generator().manual_seed(3)
    for n in (4 * 1024, 4 * 257 + 3):
        # scaled up so that clamping to [-1, 1] matters at every row
        xt, eps, z = (3 * torch.randn(n, generator=g) for _ in range(3))
        xc, ec, zc = xt.cuda(), eps.cuda(), z.cuda()
        for t in (ts[0], ts[len(ts) // 2], ts[-1]):
            for clip in (False, True):
                want_p, want_x0 = _host_ddim(xt, eps, z, tab[t], clip)
                p, x0 = ops.ddim_step(xc, ec, dtab[t], z=zc, clip_sample=clip, seed=1, step=2)
                assert torch.equal(p.cpu(), want_p) and torch.equal(x0.cpu(), want_x0), (n, t, clip)
                # out aliasing xt, no x0 output
                buf = xc.clone()
                q, none = ops.ddim_step(buf, ec, dtab[t], z=zc, want_x0=False, clip_sample=clip, out=buf)
                assert none is None and q is buf and torch.equal(buf, p)
        # fused noise at an unaligned global offset, with the tail path
        for off in (0, 6, 4 * 1001 + 1):
            want = ops.philox_normal((n,), "cuda", 9, 4, elem_offset=off).cpu()
            p, _ = ops.ddim_step(xc, ec, dtab[ts[1]], z=None, seed=9, step=4, elem_offset=off)
            assert torch.equal(p.cpu(), _host_ddim(xt, eps, want, tab[ts[1]], False)[0]), (n, off)
            step_dev = torch.tensor([4], dtype=torch.int32, device="cuda")
            q, _ = ops.ddim_step(xc, ec, dtab[ts[1]], z=None, seed=9, step=0, step_dev=step_dev, elem_offset=off)
            assert torch.equal(p, q)


@pytest.mark.gpu
def test_x0_and_the_one_step_ddpm_limit(rt):
    ops = _mod("ops")
    base = _base()
    ddpm = base.coef_table("cuda")
    ddim = _ddim(base, num_inference_steps=1000, eta=1.0).coef_table("cuda")
    g = torch.Generator().manual_seed(5)
    n = 4 * 4096 + 1
    xt, eps, z = (torch.randn(n, generator=g).cuda() for _ in range(3))
    for t in (999, 500, 1, 0):
        p_ddpm, x0_ddpm = ops.sched_step(xt, eps, ddpm[t], z=z)
        p_ddim, x0_ddim = ops.ddim_step(xt, eps, ddim[t], z=z)
        assert torch.equal(x0_ddim, x0_ddpm), t
        assert max_abs(p_ddim.cpu(), p_ddpm.cpu()) < 1e-4, t
        # fused noise: the same Philox stream as the DDPM kernel
        p_ddpm, _ = ops.sched_step(xt, eps, ddpm[t], seed=2, step=t, elem_offset=3)
        p_ddim, _ = ops.ddim_step(xt, eps, ddim[t], seed=2, step=t, elem_offset=3)
        assert max_abs(p_ddim.cpu(), p_ddpm.cpu()) < 1e-4, t


@pytest.mark.gpu
def test_whole_loop_with_every_timestep_and_eta1_is_the_ddpm_loop(rt):
    S = _mod("sampler")
    rt.set_mode("fp32")
    m = _fill(_mod("models.controlnet").ControlNet(syn.TINY_PARAMS))
    x, hint = inputs("ddim_ddpm", 2, 1, 16)
    zs = [syn.det_noise(f"ddim_ddpm:z{k}", tuple(x.shape)) for k in range(5)]
    base = _base()
    want, want0 = S.DDPMSampler(m, base, use_graph=False).sample_eager(x.cuda(), hint.cuda(), steps=5, zs=zs)
    s = _ddim(base, timesteps=[4, 3, 2, 1, 0], eta=1.0)
    got, got0 = S.DDPMSampler(m, s, use_graph=False).sample_eager(x.cuda(), hint.cuda(), zs=zs)
    assert rel_l2(got.cpu(), want.cpu()) < 1e-4 and rel_l2(got0.cpu(), want0.cpu()) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ORACLE_CASES))
def test_ddpm_controlnet_parity_with_the_oracle(rt, case):
    import cn_oracle as O
    S = _mod("sampler")
    sched, oracle_loop = ORACLE_CASES[case]
    cfg = syn.TINY_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    x, hint = inputs(case + "_tiny", 2, 1, 16)
    base = _base()
    s = sched(base)
    with torch.no_grad():
        want = oracle_loop(lambda a, t: O.controlnet_ddpm_forward(sd, cfg, a, t, hint), base, s.timesteps(), x)
    for mode in _modes(rt):
        rt.set_mode(mode)
        got, _ = S.DDPMSampler(m, s, use_graph=True).sample(x.cuda(), hint.cuda())
        assert rel_l2(got.cpu(), want) < TRAJ_TOL[mode], mode


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ORACLE_CASES))
def test_ldm_controlnet_with_vae_decode_parity_with_the_oracle(rt, case):
    import cn_oracle as O
    S = _mod("sampler")
    sched, oracle_loop = ORACLE_CASES[case]
    cfg, vcfg = syn.TINY_LDM_PARAMS, syn.TINY_VAE_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
    vae = _fill(_mod("models.vae").VAE(3, vcfg), seed=1)
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    vsd = {k: v.cpu() for k, v in vae.state_dict().items()}
    x, hint = inputs(case + "_ldm", 2, 4, 8, hint_size=64, p=0.05)
    base = _base(ldm=True)
    s = sched(base)
    with torch.no_grad():
        lat_ref = oracle_loop(lambda a, t: O.controlnet_ldm_forward(sd, cfg, a, t, hint), base, s.timesteps(), x)
        want = (torch.clamp(O.vae_decode(vsd, vcfg, lat_ref), -1., 1.) + 1) / 2
    for mode in _modes(rt):
        rt.set_mode(mode)
        ims, lat = S.LDMSampler(m, s, vae, use_graph=True).sample_images(x.cuda(), hint.cuda())
        assert tuple(ims.shape) == (2, 3, 32, 32)
        assert rel_l2(lat.cpu(), lat_ref) < TRAJ_TOL[mode], mode
        assert rel_l2(ims.cpu(), want) < TRAJ_TOL[mode], mode


def _tiny(rt):
    rt.set_mode("fp32")
    return _fill(_mod("models.controlnet").ControlNet(syn.TINY_PARAMS)), syn.det_hint(4, 16).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_graph_equals_eager_and_shards_reproduce_the_batch(rt, eta):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    s = _ddim(num_inference_steps=5, eta=eta)
    B, per = 4, 16 * 16
    g = S.DDPMSampler(m, s, seed=11, use_graph=True)
    e = S.DDPMSampler(m, s, seed=11, use_graph=False)
    xT = g.draw_xT((B, 1, 16, 16), "cuda")
    a, a0 = g.sample(xT, hint)
    b, b0 = e.sample(xT, hint)
    assert torch.equal(a, b) and torch.equal(a0, b0)
    assert torch.isfinite(a).all()
    x_lo = e.draw_xT((2, 1, 16, 16), "cuda", elem_offset=0)
    x_hi = e.draw_xT((2, 1, 16, 16), "cuda", elem_offset=2 * per)
    c_lo, _ = e.sample(x_lo, hint[:2].contiguous(), elem_offset=0)
    c_hi, _ = e.sample(x_hi, hint[2:].contiguous(), elem_offset=2 * per)
    assert rel_l2(torch.cat([c_lo, c_hi]).cpu(), b.cpu()) < 1e-5
    # through the public data-parallel entry point (one rank)
    d = S.sample_data_parallel(m, s, (B, 1, 16, 16), lambda lo, hi: hint[lo:hi], seed=11)
    assert torch.equal(d, a)


@pytest.mark.gpu
def test_eta0_does_not_depend_on_the_seed(rt):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    s = _ddim(num_inference_steps=6, eta=0.0)
    xT = S.DDPMSampler(m, s, seed=1).draw_xT((4, 1, 16, 16), "cuda")
    a, _ = S.DDPMSampler(m, s, seed=1).sample(xT, hint)
    b, _ = S.DDPMSampler(m, s, seed=2).sample(xT, hint)
    assert torch.equal(a, b)
    c, _ = S.DDPMSampler(m, _ddim(num_inference_steps=6, eta=1.0), seed=2).sample(xT, hint)
    assert not torch.equal(a, c)


@pytest.mark.gpu
def test_one_sampler_recaptures_on_every_change(rt):
    S = _mod("sampler")
    m, hint = _tiny(rt)
    s = _ddim(num_inference_steps=5, eta=0.0)
    smp = S.DDPMSampler(m, s, seed=4)
    xT = smp.draw_xT((4, 1, 16, 16), "cuda")

    def check(steps=None):
        fresh = _ddim(num_inference_steps=s.num_inference_steps, eta=s.eta, spacing=s.spacing,
                      clip_sample=s.clip_sample)
        got, got0 = smp.sample(xT, hint, steps=steps)
        want, want0 = S.DDPMSampler(m, fresh, seed=4).sample(xT, hint, steps=steps)
        assert torch.equal(got, want) and torch.equal(got0, want0)
        return got

    outs = [check()]
    outs.append(check(steps=8))
    s.eta = 1.0
    outs.append(check())
    s.spacing = "leading"
    outs.append(check())
    s.clip_sample = True
    outs.append(check())
    m.load_state_dict(syn.det_state_dict(m.state_dict(), seed=6))
    outs.append(check())
    for i in range(len(outs) - 1):
        assert not torch.equal(outs[i], outs[i + 1]), i
    # and back to DDPM on the same sampler
    smp.scheduler = s.base
    got, _ = smp.sample(xT, hint, steps=5)
    assert torch.equal(got, S.DDPMSampler(m, s.base, seed=4).sample(xT, hint, steps=5)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ddim", "dpm"])
def test_mnist_size_run_and_launch_count(rt, case):
    S = _mod("sampler")
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    m = _fill(_mod("models.controlnet").ControlNet(syn.MNIST_PARAMS))
    hint = syn.det_hint(64, 28).cuda()
    s = _ddim(num_inference_steps=50, eta=1.0) if case == "ddim" else _dpm(num_inference_steps=20, variant="sde")
    g = S.DDPMSampler(m, s, seed=3)
    xT = g.draw_xT((64, 1, 28, 28), "cuda")
    a, a0 = g.sample(xT, hint)
    b, b0 = S.DDPMSampler(m, s, seed=3, use_graph=False).sample(xT, hint)
    assert torch.isfinite(a).all() and torch.isfinite(a0).all()
    assert torch.equal(a, b) and torch.equal(a0, b0)
    d = S.DDPMSampler(m, _base(), seed=3)
    d.sample(xT, hint, steps=2)
    assert g.launches_per_step == d.launches_per_step
