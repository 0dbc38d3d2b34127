"""Whole-path parity (GPU): the drop-in modules on libcnb200 kernels against
  (1) tests/golden/*.npz - outputs of the UNMODIFIED reference (made by oracle/make_golden.py), and
  (2) oracle/cn_oracle.py on freshly seeded inputs,
in both compute modes.  Tolerances are BASELINE.json's: per-step eps rel-L2 <= 1e-4 in fp32 mode, <= 1e-2 in the
tensor-core mode.
"""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from helpers import golden, inputs, max_abs, psnr, rel_l2, syn, ROOT

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(ROOT, "oracle"))

TOL = {"fp32": 1e-4, "f16": 1e-2}
TRAJ_TOL = {"fp32": 5e-4, "f16": 3e-2}


def _mod(name):
    return importlib.import_module("controlnet-pytorch_b200." + name)


@pytest.fixture(scope="module")
def rt():
    r = _mod("runtime")
    r.lib()
    return r


def _fill(model, seed=0):
    model.load_state_dict(syn.det_state_dict(model.state_dict(), seed))
    return model.cuda().eval()


def _modes(rt):
    return ["fp32", "f16"] if rt.lib().cnb_has_tcgen05() else ["fp32"]


@pytest.mark.parametrize("name,cfg,B,ts", [("tiny", syn.TINY_PARAMS, 2, (999, 37, 0)),
                                           ("mnist", syn.MNIST_PARAMS, 2, (999, 500, 0)),
                                           ("cifar", syn.CIFAR_PARAMS, 1, (500,))])
def test_controlnet_ddpm_vs_reference_golden(rt, name, cfg, B, ts):
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    x, hint = inputs(name, B, cfg["im_channels"], cfg["im_size"])
    g = golden(f"controlnet_{name}")
    xc, hc = x.cuda(), hint.cuda()
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            for t in ts:
                eps = m(xc, torch.as_tensor(t).unsqueeze(0).cuda(), hc)
                assert eps.shape == x.shape
                err = rel_l2(eps.cpu(), g[f"eps_{t}"])
                assert err < TOL[mode], (mode, t, err)
            if name == "tiny":
                eps = m(xc, torch.tensor([10, 700]), hc)       # per-sample t, given on the CPU like the tools do
                assert rel_l2(eps.cpu(), g["eps_pers"]) < TOL[mode]
            if name != "cifar":
                sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
                smp = _mod("sampler").DDPMSampler(m, sched, use_graph=False)
                zs = [syn.det_noise(f"{name}:z{k}", tuple(x.shape)) for k in range(3)]
                xt, x0 = smp.sample_eager(xc, hc, steps=3, zs=zs)
                assert rel_l2(xt.cpu(), g["traj3_xt"]) < TRAJ_TOL[mode]
                assert rel_l2(x0.cpu(), g["traj3_x0"]) < TRAJ_TOL[mode]
    assert rt.lib().cnb_tc_error_flag() == 0


# BASELINE.json: "the final x0 matches within a stated PSNR / max-abs bound".  Stated here for configs[0] (MNIST
# ControlNet, batch 16, 50 steps, images in [-1, 1]); measured on a B200 (tests/config1_check.py,
# profiles/r01_config1_check.log): fp32 mode 147 dB / 8.3e-7, tensor-core mode 83 dB / 6.7e-4.
X0_BOUND = {"fp32": dict(psnr_db=120.0, max_abs=1e-5), "f16": dict(psnr_db=65.0, max_abs=5e-3)}


def test_config1_mnist_b16_50step_final_x0_vs_reference_golden(rt):
    """BASELINE.json configs[0]: 50 denoising steps (t = 49 .. 0) at batch 16 with the per-step z injected, against
    the final x_0 / x_{t-1} of the unmodified reference (tests/golden/config1_mnist_b16_50step.npz)."""
    cfg = syn.MNIST_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    x, hint = inputs("config1", 16, 1, 28)
    zs = [syn.det_noise(f"config1:z{k}", tuple(x.shape)) for k in range(50)]
    g = golden("config1_mnist_b16_50step")
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    for mode in _modes(rt):
        rt.set_mode(mode)
        xt, x0 = _mod("sampler").DDPMSampler(m, sched, use_graph=False).sample_eager(x.cuda(), hint.cuda(), steps=50, zs=zs)
        p, a = psnr(x0.cpu(), g["x0"]), max_abs(x0.cpu(), g["x0"])
        assert p > X0_BOUND[mode]["psnr_db"] and a < X0_BOUND[mode]["max_abs"], (mode, p, a)
        assert rel_l2(xt.cpu(), g["xt"]) < TRAJ_TOL[mode]
    assert rt.lib().cnb_tc_error_flag() == 0


def test_controlnet_ldm_vs_reference_golden(rt):
    cfg = syn.TINY_LDM_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
    x, hint = inputs("tiny_ldm", 2, 4, 8, hint_size=64, p=0.05)
    g = golden("controlnet_tiny_ldm")
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            for t in (999, 3):
                eps = m(x.cuda(), torch.as_tensor(t).unsqueeze(0).cuda(), hint.cuda())
                assert rel_l2(eps.cpu(), g[f"eps_{t}"]) < TOL[mode], (mode, t)
            sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(ldm_scheduler=True,
                                                                                  **syn.CELEBHQ_DIFFUSION)
            smp = _mod("sampler").DDPMSampler(m, sched, use_graph=False)
            zs = [syn.det_noise(f"tiny_ldm:z{k}", tuple(x.shape)) for k in range(3)]
            xt, x0 = smp.sample_eager(x.cuda(), hint.cuda(), steps=3, zs=zs)
            assert rel_l2(xt.cpu(), g["traj3_xt"]) < TRAJ_TOL[mode]


def test_unet_vs_reference_golden(rt):
    m = _fill(_mod("models.unet_base").Unet(syn.TINY_PARAMS))
    x, _ = inputs("unet_tiny", 2, 1, 16)
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            eps = m(x.cuda(), torch.as_tensor(123).unsqueeze(0))
        assert rel_l2(eps.cpu(), golden("unet_tiny")["eps_123"]) < TOL[mode]


@pytest.mark.parametrize("name,cfg,sigma", [("tiny", syn.TINY_PARAMS, 80.0), ("mnist", syn.MNIST_PARAMS, 80.0),
                                            ("cifar", syn.CIFAR_PARAMS, 5.0)])
def test_students_vs_reference_golden(rt, name, cfg, sigma):
    B = 2 if name != "cifar" else 1
    cons = _fill(_mod("models.consistency_controlnet_distilled").ConsistencyControlNet(cfg))
    dm = _fill(_mod("models.distribution_matching_controlnet").DistributionMatchingControlNet(cfg))
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            x, hint = inputs("cons_" + name, B, cfg["im_channels"], cfg["im_size"])
            g = golden(f"consistency_{name}")
            xc, hc = x.cuda(), hint.cuda()
            assert rel_l2(cons(xc, torch.full((B,), sigma).cuda(), hc).cpu(), g["x0_max"]) < TOL[mode]
            assert rel_l2(cons(xc, torch.full((B,), 1.7).cuda(), hc).cpu(), g["x0_mid"]) < TOL[mode]
            out = cons(xc, torch.full((B,), 0.001).cuda(), hc)          # boundary: returns x_t itself
            assert out is xc or torch.equal(out, xc)
            x, hint = inputs("dm_" + name, B, cfg["im_channels"], cfg["im_size"])
            g = golden(f"dm_{name}")
            assert rel_l2(dm(x.cuda(), torch.full((B,), 999).cuda(), hint.cuda()).cpu(), g["x0_999"]) < TOL[mode]
            if B == 2:
                assert rel_l2(dm(x.cuda(), torch.tensor([5, 400]).cuda(), hint.cuda()).cpu(), g["x0_pers"]) < TOL[mode]


def test_blocks_callable_standalone_vs_oracle(rt):
    """The public block classes keep the reference's forward(x, t_emb) signatures (NCHW in / NCHW out)."""
    import cn_oracle as O
    ub = _mod("models.unet_base")
    rt.set_mode("fp32")
    torch.manual_seed(0)
    x, temb = torch.randn(2, 16, 8, 8), torch.randn(2, 32)
    d = _fill(ub.DownBlock(16, 32, 32, down_sample=True, num_layers=2))
    sd = {k: v.cpu() for k, v in d.state_dict().items()}
    want = O.down_block(sd, "", x, temb, 2, 8, 4, True, True)
    assert rel_l2(d(x.cuda(), temb.cuda()).cpu(), want) < 1e-5
    mid = _fill(ub.MidBlock(16, 32, 32, num_layers=1))
    sd = {k: v.cpu() for k, v in mid.state_dict().items()}
    assert rel_l2(mid(x.cuda(), temb.cuda()).cpu(), O.mid_block(sd, "", x, temb, 1, 8, 4)) < 1e-5
    up = _fill(ub.UpBlock(32, 16, 32, up_sample=True, num_layers=1))
    sd = {k: v.cpu() for k, v in up.state_dict().items()}
    skip = torch.randn(2, 16, 16, 16)
    assert rel_l2(up(x.cuda(), skip.cuda(), temb.cuda()).cpu(), O.up_block(sd, "", x, skip, temb, 1, 8, 4, True)) < 1e-5


def test_graph_sampler_matches_eager_and_sharding_invariance(rt):
    """CUDA-graph replayed loop == eager loop bit for bit (same kernels, same Philox stream), and two half-batch
    shards with global element offsets reproduce the full-batch result (data-parallel invariance)."""
    cfg = syn.TINY_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    S = _mod("sampler")
    rt.set_mode("fp32")
    B, per = 4, 16 * 16
    hint = syn.det_hint(B, 16).cuda()
    g = S.DDPMSampler(m, sched, seed=11, use_graph=True)
    e = S.DDPMSampler(m, sched, seed=11, use_graph=False)
    xT = g.draw_xT((B, 1, 16, 16), "cuda")
    a, a0 = g.sample(xT, hint, steps=5)
    b, b0 = e.sample(xT, hint, steps=5)
    assert torch.equal(a, b) and torch.equal(a0, b0)
    lo = S.DDPMSampler(m, sched, seed=11, use_graph=False)
    h0, h1 = hint[:2].contiguous(), hint[2:].contiguous()
    x_lo = lo.draw_xT((2, 1, 16, 16), "cuda", elem_offset=0)
    x_hi = lo.draw_xT((2, 1, 16, 16), "cuda", elem_offset=2 * per)
    assert torch.equal(torch.cat([x_lo, x_hi]), xT)
    c_lo, _ = lo.sample(x_lo, h0, steps=5, elem_offset=0)
    c_hi, _ = lo.sample(x_hi, h1, steps=5, elem_offset=2 * per)
    assert rel_l2(torch.cat([c_lo, c_hi]).cpu(), b.cpu()) < 1e-5


def test_hint_cache_and_weight_cache_invalidate(rt):
    cfg = syn.TINY_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    rt.set_mode("fp32")
    x, hint = inputs("tiny", 2, 1, 16)
    xc, hc = x.cuda(), hint.cuda()
    t = torch.tensor([37]).cuda()
    with torch.no_grad():
        e1 = m(xc, t, hc)
        e2 = m(xc, t, hc)                 # cached hint feature
        assert torch.equal(e1, e2)
        m.load_state_dict(syn.det_state_dict(m.state_dict(), seed=5))     # in-place copy bumps version counters
        e3 = m(xc, t, hc)
        assert rel_l2(e3.cpu(), e1.cpu()) > 1e-2
        import cn_oracle as O
        sd = {k: v.cpu() for k, v in m.state_dict().items()}
        want = O.controlnet_ddpm_forward(sd, cfg, x, torch.tensor([37]), hint)
        assert rel_l2(e3.cpu(), want) < 1e-4


def test_vae_vs_reference_golden(rt):
    """models/vae.py decode / encode (SURVEY.md 8f-1) against the reference's outputs: tiny VAE (decoder MidBlock +
    attention UpBlock) and the full-size CelebHQ autoencoder at batch 1."""
    VAE = _mod("models.vae").VAE
    m = _fill(VAE(3, syn.TINY_VAE_PARAMS))
    g = golden("vae_tiny")
    z = syn.det_noise("vae_tiny:z", (2, 4, 8, 8)).cuda()
    x = syn.det_noise("vae_tiny:x", (2, 3, 32, 32)).cuda()
    big = _fill(VAE(3, syn.CELEBHQ_VAE_PARAMS))
    gb = golden("vae_celebhq")
    zb = syn.det_noise("vae_celebhq:z", (1, 4, 32, 32)).cuda()
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            assert rel_l2(m.decode(z).cpu(), g["dec"]) < TOL[mode], mode
            assert rel_l2(m._encode_out(x, rt.get_mode()).cpu(), g["enc_out"]) < TOL[mode], mode
            sample, out = m.encode(x)
            assert tuple(sample.shape) == (2, 4, 8, 8) and tuple(out.shape) == (2, 8, 8, 8)
            img = big.decode(zb)
        assert tuple(img.shape) == (1, 3, 128, 128)
        assert rel_l2(img[:, :, ::4, ::4].cpu(), gb["dec_strided"]) < TOL[mode], mode
    assert rt.lib().cnb_tc_error_flag() == 0


def test_ldm_sampler_with_vae_decode_vs_oracle(rt):
    """tools/sample_ldm_controlnet.py flow on the tiny LDM ControlNet + tiny VAE: injected-noise loop and decode of
    the final latents against the oracle (cn_oracle.ddpm_sample + vae_decode); graph replay == eager with Philox."""
    import cn_oracle as O
    cfg, vcfg = syn.TINY_LDM_PARAMS, syn.TINY_VAE_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=8))
    vae = _fill(_mod("models.vae").VAE(3, vcfg), seed=1)
    sd = {k: v.cpu() for k, v in m.state_dict().items()}
    vsd = {k: v.cpu() for k, v in vae.state_dict().items()}
    x, hint = inputs("ldm_vae", 2, 4, 8, hint_size=64, p=0.05)
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(ldm_scheduler=True, **syn.CELEBHQ_DIFFUSION)
    steps = 4
    zs = [syn.det_noise(f"ldm_vae:z{k}", tuple(x.shape)) for k in range(steps)]
    with torch.no_grad():
        so = O.SchedulerOracle(ldm_scheduler=True, **syn.CELEBHQ_DIFFUSION)
        xt_ref, _ = O.ddpm_sample(lambda a, t, h: O.controlnet_ldm_forward(sd, cfg, a, t, h), so, x, hint, steps, zs)
        want = (torch.clamp(O.vae_decode(vsd, vcfg, xt_ref), -1., 1.) + 1) / 2
    S = _mod("sampler")
    for mode in _modes(rt):
        rt.set_mode(mode)
        smp = S.LDMSampler(m, sched, vae, seed=5, use_graph=False)
        ims, lat = smp.sample_images(x.cuda(), hint.cuda(), steps=steps, zs=zs)
        assert tuple(ims.shape) == (2, 3, 32, 32)
        assert rel_l2(lat.cpu(), xt_ref) < TRAJ_TOL[mode], mode
        assert rel_l2(ims.cpu(), want) < TRAJ_TOL[mode], mode
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    hc = hint.cuda()
    eager = S.LDMSampler(m, sched, vae, seed=5, use_graph=False).sample_images(x.cuda(), hc, steps=steps)[0]
    graph = S.LDMSampler(m, sched, vae, seed=5, use_graph=True, decode_chunk=1).sample_images(x.cuda(), hc, steps=steps)[0]
    assert torch.equal(eager, graph)
    assert rt.lib().cnb_tc_error_flag() == 0


def test_teacher_predictions_vs_reference_golden(rt, tmp_path):
    """Teacher-side inference of the distillation wrappers (SURVEY.md 8f-4) on the GPU kernels: per-sample t, the
    x0 conversion kernel (bit-exact op order), sigma -> timestep lookup."""
    cfg = syn.TINY_PARAMS
    teacher = _mod("models.controlnet").ControlNet(cfg)
    teacher.load_state_dict(syn.det_state_dict(teacher.state_dict(), 3))
    ck = os.path.join(str(tmp_path), "teacher.pth")
    torch.save(teacher.state_dict(), ck)
    dm = _mod("models.distribution_matching_controlnet").DistributionMatchingControlNetDistilled(cfg, ck, device="cuda").cuda().eval()
    cs = _mod("models.consistency_controlnet_distilled").ConsistencyControlNetDistilled(cfg, ck, device="cuda").cuda().eval()
    g = golden("teachers_tiny")
    x, hint = inputs("teacher_tiny", 3, cfg["im_channels"], cfg["im_size"])
    xc, hc = x.cuda(), hint.cuda()
    sig = torch.tensor([60.0, 2.5, 0.05]).cuda()
    assert cs.sigma_to_timestep(sig).cpu().tolist() == g["cs_t"].tolist()
    for mode in _modes(rt):
        rt.set_mode(mode)
        a = dm.get_teacher_prediction(xc, torch.tensor([999, 412, 3]).cuda(), hc)
        b = dm.get_teacher_prediction(xc[:1].contiguous(), torch.tensor(77), hc[:1].contiguous())
        c = cs.get_ddpm_teacher_prediction(xc, sig, hc)
        assert rel_l2(a.cpu(), g["dm_x0"]) < TOL[mode], mode
        assert rel_l2(b.cpu(), g["dm_x0_shared_t"]) < TOL[mode], mode
        assert rel_l2(c.cpu(), g["cs_x0"]) < TOL[mode], mode
    with pytest.raises(ValueError):
        _mod("models.consistency_controlnet_distilled").ConsistencyControlNetDistilled(cfg).get_ddpm_teacher_prediction(xc, sig, hc)
    # the conversion kernel alone is bit-exact against the reference expression
    eps = syn.det_noise("teacher_tiny:eps", tuple(x.shape))
    sch = dm.teacher_scheduler
    t = torch.tensor([5, 500, 998])
    s1 = sch.sqrt_one_minus_alpha_cum_prod[t].reshape(3, 1, 1, 1)
    s2 = sch.sqrt_alpha_cum_prod[t].reshape(3, 1, 1, 1)
    want = torch.clamp((x - s1 * eps) / s2, -1., 1.)
    ops = _mod("ops")
    got = ops.x0_from_eps(xc, eps.cuda(), sch.sqrt_one_minus_alpha_cum_prod.cuda(), sch.sqrt_alpha_cum_prod.cuda(), t.cuda())
    assert torch.equal(got.cpu(), want)


def test_batch_invariance_at_baseline_sizes(rt):
    """Size-independent property at BASELINE.json's full batch sizes: every sample is independent (GroupNorm and
    attention are per sample, t is shared), so row b of a large-batch forward must equal, bit for bit, the forward of
    sample b in a small batch.  MNIST ControlNet at B = 1024 (config 2 shard) against four picked samples, a 128-sample
    shard (the per-rank size on 8 GPUs) and one sample alone; consistency student at B = 4096 (config 4) and DM student
    on CIFAR shapes at B = 2048 (config 5 sweep) against four picked samples, and both students at B = 4096 with one
    scalar sigma / t (a shared time-embedding row at B = 1, per-sample rows at B > 1) against one sample alone."""
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    picks = [0, 1, 517, -1]

    def check(fwd_big, fwd_small, n):
        big = fwd_big()
        assert torch.isfinite(big).all()
        idx = [p % n for p in picks]
        assert torch.equal(big[idx], fwd_small(idx))
        return big

    def draw(B, c, s):
        x = torch.randn(B, c, s, s, device="cuda")
        hint = (torch.rand(B, 1, s, s, device="cuda") < 0.1).float().expand(B, 3, s, s).contiguous()
        return x, hint

    with torch.no_grad():
        cfg = syn.MNIST_PARAMS
        m = _fill(_mod("models.controlnet").ControlNet(cfg))
        B = 1024
        x, hint = draw(B, 1, 28)
        t = torch.tensor([321], device="cuda")
        big = check(lambda: m(x, t, hint), lambda i: m(x[i].contiguous(), t, hint[i].contiguous()), B)
        assert torch.equal(big[128:256], m(x[128:256].contiguous(), t, hint[128:256].contiguous()))
        assert torch.equal(big[517:518], m(x[517:518].contiguous(), t, hint[517:518].contiguous()))
        del m
        cs = _fill(_mod("models.consistency_controlnet_distilled").ConsistencyControlNet(cfg))
        B = 4096
        x, hint = draw(B, 1, 28)
        sig = torch.full((B,), 80.0, device="cuda")
        check(lambda: cs(x, sig, hint), lambda i: cs(x[i].contiguous(), sig[i].contiguous(), hint[i].contiguous()), B)
        one = torch.tensor(80.0, device="cuda")
        big = cs(x, one, hint)
        for b in (0, 2049, B - 1):
            assert torch.equal(big[b:b + 1], cs(x[b:b + 1].contiguous(), one, hint[b:b + 1].contiguous())), b
        del cs
        cfg = syn.CIFAR_PARAMS
        dm = _fill(_mod("models.distribution_matching_controlnet").DistributionMatchingControlNet(cfg))
        B = 2048
        x, hint = draw(B, 3, 32)
        tt = torch.full((B,), 999, device="cuda")
        check(lambda: dm(x, tt, hint), lambda i: dm(x[i].contiguous(), tt[i].contiguous(), hint[i].contiguous()), B)
        B = 4096
        x, hint = draw(B, 3, 32)
        one = torch.tensor(999, device="cuda")
        big = dm(x, one, hint)
        for b in (0, 2049, B - 1):
            assert torch.equal(big[b:b + 1], dm(x[b:b + 1].contiguous(), one, hint[b:b + 1].contiguous())), b
        del dm
        # VAE decoder: the split-statistics GroupNorm picks its number of row ranges from the batch size
        vae = _fill(_mod("models.vae").VAE(3, syn.CELEBHQ_VAE_PARAMS))
        z = torch.randn(40, 4, 32, 32, device="cuda")
        big = vae.decode(z)
        assert torch.equal(big[[0, 39]], vae.decode(z[[0, 39]].contiguous()))
    assert rt.lib().cnb_tc_error_flag() == 0


def test_graphed_students_match_eager(rt):
    """sampler.GraphedStudent: one CUDA graph per input shape, new inputs copied into the static buffers; must equal
    the eager forward bit for bit, also after the inputs change (hint block inside the graph) and at the boundary."""
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    S = _mod("sampler")
    cfg = syn.TINY_PARAMS
    dm = _fill(_mod("models.distribution_matching_controlnet").DistributionMatchingControlNet(cfg))
    cs = _fill(_mod("models.consistency_controlnet_distilled").ConsistencyControlNet(cfg))
    gdm, gcs = S.GraphedStudent(dm), S.GraphedStudent(cs)
    with torch.no_grad():
        for seed in (1, 2, 3):
            x, hint = inputs(f"graphed{seed}", 3, cfg["im_channels"], cfg["im_size"])
            xc, hc = x.cuda(), hint.cuda()
            t = torch.tensor([999, 5, 300 + seed]).cuda()
            assert torch.equal(gdm(xc, t, hc), dm(xc, t, hc))
            sig = torch.tensor([80.0, 1.7, 0.01 * seed]).cuda()
            assert torch.equal(gcs(xc, sig, hc), cs(xc, sig, hc))
        small = torch.full((3,), 1e-3).cuda()
        assert gcs(xc, small, hc) is xc                      # whole-batch early return, like the eager module
    assert rt.lib().cnb_tc_error_flag() == 0


def test_branch_layouts_of_the_step_graph_are_bit_identical(rt):
    """models/_controlnet_common.py lays the ControlNet forward out on four capture streams (trained mids ahead of the
    control join, skip sums and t-embedding rows off the critical path); the eager loop runs it on one stream.  Both
    run the same kernels on the same inputs, so the replayed samples must equal the eager loop bit for bit: MNIST DDPM
    ControlNet, the tiny LDM ControlNet (image-pyramid hints), and a CIFAR-width ControlNet whose conv_in layers share
    the padded fp16 copy of x (built before the fork)."""
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    S = _mod("sampler")
    L = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler
    cases = [
        ("mnist", _fill(_mod("models.controlnet").ControlNet(syn.MNIST_PARAMS)), L(**syn.MNIST_DIFFUSION),
         inputs("branch_mnist", 6, 1, 28)),
        ("tiny_ldm", _fill(_mod("models.controlnet_ldm").ControlNet(4, syn.TINY_LDM_PARAMS, down_sample_factor=8)),
         L(ldm_scheduler=True, **syn.CELEBHQ_DIFFUSION), inputs("branch_ldm", 3, 4, 8, hint_size=64, p=0.05)),
        ("cifar", _fill(_mod("models.controlnet").ControlNet(syn.CIFAR_PARAMS)), L(**syn.MNIST_DIFFUSION),
         inputs("branch_cifar", 3, 3, 32)),
    ]
    for name, m, sched, (x, hint) in cases:
        xc, hc = x.cuda(), hint.cuda()
        eager = S.DDPMSampler(m, sched, seed=11, use_graph=False).sample(xc, hc, steps=3, elem_offset=64)
        got = S.DDPMSampler(m, sched, seed=11, use_graph=True).sample(xc, hc, steps=3, elem_offset=64)
        assert torch.equal(got[0], eager[0]) and torch.equal(got[1], eager[1]), name
        assert torch.isfinite(got[0]).all()
    assert rt.lib().cnb_tc_error_flag() == 0


def test_dropin_shim_runs_the_reference_tool_loop(rt, tmp_path):
    """INTEGRATION.md section 1: the reference tool's import lines and sampling loop (tools/sample_ddpm_controlnet.py
    :9-12, :43-51), run in a fresh interpreter with controlnet-pytorch_b200/dropin first on sys.path, execute on the
    B200 kernels and reproduce the reference's 3-step fixture (tests/dropin_tool_loop.py)."""
    import subprocess
    env = dict(os.environ)
    env["PYTHONSAFEPATH"] = "1"
    env["PYTHONPATH"] = os.path.join(ROOT, "controlnet-pytorch_b200", "dropin")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_tool_loop.py")], env=env, cwd=str(tmp_path),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "dropin tool loop" in r.stdout, r.stdout + r.stderr


def test_sampler_graph_follows_hint_and_weight_updates(rt):
    """ADVICE r1: the captured step bakes in the hint feature and the packed weights.  A hint overwritten IN PLACE, a new
    hint tensor of the same shape, and a load_state_dict after capture must all give what the eager loop gives."""
    cfg = syn.TINY_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    S = _mod("sampler")
    rt.set_mode("fp32")
    B = 4
    g = S.DDPMSampler(m, sched, seed=3, use_graph=True)
    e = S.DDPMSampler(m, sched, seed=3, use_graph=False)
    xT = g.draw_xT((B, 1, 16, 16), "cuda")
    hint = syn.det_hint(B, 16, seed=0).cuda()
    a, _ = g.sample(xT, hint, steps=4)
    assert torch.equal(a, e.sample(xT, hint, steps=4)[0])
    graph0 = g._graph
    hint.copy_(syn.det_hint(B, 16, seed=9, p=0.3).cuda())            # same storage, new contents
    b, _ = g.sample(xT, hint, steps=4)
    assert g._graph is graph0                                          # the graph is re-used ...
    assert torch.equal(b, e.sample(xT, hint, steps=4)[0])              # ... and sees the new hint
    assert not torch.equal(a, b)
    hint2 = syn.det_hint(B, 16, seed=4, p=0.2).cuda()                   # another tensor, caller's buffer freed afterwards
    c, _ = g.sample(xT, hint2.clone(), steps=4)
    assert g._graph is graph0 and torch.equal(c, e.sample(xT, hint2, steps=4)[0])
    m.load_state_dict(syn.det_state_dict(m.state_dict(), seed=5))      # new weights: the graph must be rebuilt
    d, _ = g.sample(xT, hint2, steps=4)
    assert g._graph is not graph0
    assert torch.equal(d, e.sample(xT, hint2, steps=4)[0]) and not torch.equal(c, d)


@pytest.mark.parametrize("cache", ["cat_f16", "tcat", "pad16"])
def test_graph_sampler_follows_the_second_parameter_of_a_cached_weight(rt, cache):
    """Three derived weights are kept on one parameter but built from several: the second 3x3 fused with the residual
    1x1 (`cat_f16`), the concatenated t-embedding rows (`tcat`) and conv_out padded to 16 outputs (`pad16`, taken when
    conv_out reads >= 64 channels, hence the wider LDM).  Changing only the secondary parameter (the 1x1 weight, one
    t-embedding bias, conv_out's bias) in place after capture must rebuild that cache: the re-captured step equals an
    eager step on a fresh copy of the changed model."""
    if not rt.lib().cnb_has_tcgen05():
        pytest.skip("these caches serve the tensor-core mode")
    rt.set_mode("f16")
    S = _mod("sampler")
    L = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler
    if cache == "pad16":
        make = lambda: _mod("models.controlnet_ldm").ControlNet(4, dict(syn.TINY_LDM_PARAMS, conv_out_channels=64),
                                                                down_sample_factor=8)
        sched, (x, hint) = L(ldm_scheduler=True, **syn.CELEBHQ_DIFFUSION), inputs("cache_ldm", 2, 4, 8, hint_size=64)
    else:
        make = lambda: _mod("models.controlnet").ControlNet(syn.TINY_PARAMS)
        sched, (x, hint) = L(**syn.MNIST_DIFFUSION), inputs("cache_tiny", 2, 1, 16)
    m = _fill(make())
    tu = m.trained_unet
    holder, key, prm = {
        "cat_f16": (tu.downs[0].resnet_conv_second[0][2].weight, ("cat_f16",), tu.downs[0].residual_input_conv[0].weight),
        "tcat": (tu.downs[0].t_emb_layers[0][1].weight, ("tcat", True), tu.mids[0].t_emb_layers[0][1].bias),
        "pad16": (tu.conv_out.weight, ("pad16",), tu.conv_out.bias)}[cache]
    xc, hc = x.cuda(), hint.cuda()
    g = S.DDPMSampler(m, sched, seed=11, use_graph=True)
    before = g.sample(xc, hc, steps=2)
    assert key in holder._cnb_pack                                      # the step took the cached route
    with torch.no_grad():
        prm.add_(0.25)
    got = g.sample(xc, hc, steps=2)
    fresh = _fill(make())
    fresh.load_state_dict(m.state_dict())
    want = S.DDPMSampler(fresh, sched, seed=11, use_graph=False).sample(xc, hc, steps=2)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert not torch.equal(got[0], before[0])


def test_cold_cache_graph_sampler(rt):
    """ADVICE r1: the graph sampler's FIRST warm-up runs on cold weight caches, and the captured four-stream step must
    not read packed weights that were still being built.  A fresh model goes straight into the graph sampler and must
    equal the eager loop on a warm copy."""
    cfg = syn.TINY_PARAMS
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    S = _mod("sampler")
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    B = 8
    hint = syn.det_hint(B, 16).cuda()
    cold = _fill(_mod("models.controlnet").ControlNet(cfg))            # no forward has run on this module yet
    g = S.DDPMSampler(cold, sched, seed=2, use_graph=True)
    xT = g.draw_xT((B, 1, 16, 16), "cuda")
    a, _ = g.sample(xT, hint, steps=3)
    warm = _fill(_mod("models.controlnet").ControlNet(cfg))
    b, _ = S.DDPMSampler(warm, sched, seed=2, use_graph=False).sample(xT, hint, steps=3)
    assert torch.equal(a, b)


def test_host_tensors_are_staged_not_computed_on_the_host(rt):
    """A module / inputs still on the host (the reference's own smoke test builds both on the CPU,
    test_distribution_matching.py:36-47) are copied to the device at the public forward; the result comes back on the
    caller's device and equals the all-device call bit for bit."""
    cfg = syn.TINY_PARAMS
    rt.set_mode("fp32")
    DM = _mod("models.distribution_matching_controlnet").DistributionMatchingControlNet
    host = DM(cfg)
    host.load_state_dict(syn.det_state_dict(host.state_dict(), 0))
    x, hint = inputs("tiny", 2, 1, 16)
    t = torch.tensor([7, 900])
    with torch.no_grad():
        y_host = host(x, t, hint)
        assert y_host.device.type == "cpu" and y_host.shape == x.shape
        dev = _fill(DM(cfg))
        y_dev = dev(x.cuda(), t.cuda(), hint.cuda())
        assert torch.equal(y_host, y_dev.cpu())
        y_mixed = dev(x, t, hint)                                       # device module, host inputs
        assert y_mixed.device.type == "cpu" and torch.equal(y_mixed, y_host)
        host.load_state_dict(syn.det_state_dict(host.state_dict(), 3))  # the replica follows the host parameters
        assert not torch.equal(host(x, t, hint), y_host)
    assert next(host.parameters()).device.type == "cpu"


def test_reference_smoke_test_runs_unmodified_on_the_dropins(rt):
    """SURVEY.md section 4 (3): the reference's only test, test_distribution_matching.py, UNMODIFIED, with the drop-in
    packages first on the path: model construction and both forward passes (:36-83) must pass.  Its third section calls
    `distillation_loss` (training, out of scope) and is expected to report a failure, nothing else may."""
    import subprocess
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import install_ref
    ref = install_ref.ref_path()
    if ref is None:
        pytest.skip("no copy of the reference on this box (run oracle/install_ref.py in the build container)")
    env = dict(os.environ)
    env["PYTHONSAFEPATH"] = "1"
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "controlnet-pytorch_b200", "dropin"), ref])
    r = subprocess.run([sys.executable, os.path.join(ref, "test_distribution_matching.py")], env=env, cwd=ref,
                       capture_output=True, text=True, timeout=900)
    out = r.stdout + r.stderr
    assert "✓ Basic model created successfully" in out and "✓ Forward pass successful" in out, out
    assert "✓ Distilled model forward pass successful" in out, out
    assert "Basic model test failed" not in out and "Distilled model test failed" not in out, out
    assert "Parameter counts" in out and "Compatibility test failed" not in out, out


# ---------------------------------------------------------------------------------------------------------------------
# full-size BASELINE configs (fixtures: oracle/make_golden.py::make_fullsize, from the unmodified reference)
# ---------------------------------------------------------------------------------------------------------------------
def test_celebhq_ldm_controlnet_full_size_vs_reference_golden(rt):
    """BASELINE config 3 model: the 190.5 M-parameter CelebHQ LDM ControlNet (config/celebhq.yaml ldm_params, latent
    4 x 32 x 32, hint 3 x 1024 x 1024, down_sample_factor 32) at batch 1, eps at two timesteps, both modes."""
    cfg = syn.CELEBHQ_LDM_PARAMS
    m = _fill(_mod("models.controlnet_ldm").ControlNet(4, cfg, down_sample_factor=32))
    assert sum(p.numel() for p in m.parameters()) == 190_516_868
    x, hint = inputs("celebhq_ldm", 1, 4, 32, hint_size=1024, p=0.05)
    g = golden("controlnet_celebhq_ldm")
    xc, hc = x.cuda(), hint.cuda()
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            for t in (500, 3):
                eps = m(xc, torch.as_tensor(t).unsqueeze(0).cuda(), hc)
                assert torch.isfinite(eps).all()
                assert rel_l2(eps.cpu(), g[f"eps_{t}"]) < TOL[mode], (mode, t, rel_l2(eps.cpu(), g[f"eps_{t}"]))
    assert rt.lib().cnb_tc_error_flag() == 0


def test_celebhq_latent_consistency_student_vs_reference_golden(rt):
    """BASELINE config 4, second shape (SURVEY.md 8d): ConsistencyControlNet(dict(ldm_params, im_channels=4, im_size=32)),
    102.9 M parameters, heads fixed at 4 (head dims 64 .. 192), GroupNorm 8 groups."""
    lat = dict(syn.CELEBHQ_LDM_PARAMS, im_channels=4, im_size=32)
    m = _fill(_mod("models.consistency_controlnet_distilled").ConsistencyControlNet(lat))
    x, hint = inputs("cons_celebhq_latent", 1, 4, 32)
    g = golden("consistency_celebhq_latent")
    for mode in _modes(rt):
        rt.set_mode(mode)
        with torch.no_grad():
            for key, sigma in (("x0_max", 80.0), ("x0_mid", 1.7)):
                out = m(x.cuda(), torch.full((1,), sigma).cuda(), hint.cuda())
                assert rel_l2(out.cpu(), g[key]) < TOL[mode], (mode, key, rel_l2(out.cpu(), g[key]))


def test_consistency_generate_multi_step_vs_reference_golden(rt):
    """ConsistencyControlNetDistilled.generate (consistency_controlnet_distilled.py:375-409), single- and four-step, with
    the x_T / re-noising draws (torch.randn(shape, device) :383, torch.randn_like :398) injected on both sides."""
    mod = _mod("models.consistency_controlnet_distilled")
    cfg = syn.TINY_PARAMS
    w = mod.ConsistencyControlNetDistilled(cfg)
    w.student.load_state_dict(syn.det_state_dict(w.student.state_dict(), 0))
    w = w.cuda().eval()
    hint = syn.det_hint(2, 16).cuda()
    shape = (2, 1, 16, 16)
    g = golden("consistency_generate_tiny")
    for mode in _modes(rt):
        rt.set_mode(mode)
        for steps in (1, 4):
            draws = [syn.det_noise(f"gen{steps}:n{k}", shape).cuda() for k in range(steps)]
            orig_randn, orig_like = torch.randn, torch.randn_like
            torch.randn = lambda *a, **k: draws.pop(0)
            torch.randn_like = lambda *a, **k: draws.pop(0)
            try:
                out = w.generate(hint, shape, num_steps=steps)
            finally:
                torch.randn, torch.randn_like = orig_randn, orig_like
            assert not draws
            err = rel_l2(out.cpu(), g[f"gen_{steps}"])
            assert err < (5e-4 if mode == "fp32" else 3e-2), (mode, steps, err)


def test_config2_long_graph_replay_equals_sharded_run(rt):
    """BASELINE config 2 shape: MNIST ControlNet, batch 1024, 120 graph-replayed timesteps with on-device Philox noise.
    The result is finite, and the job split into four shards (per-rank batch 256, global element offsets) reproduces the
    unsharded samples BIT FOR BIT - what sample_data_parallel + the final all-gather rely on."""
    cfg = syn.MNIST_PARAMS
    m = _fill(_mod("models.controlnet").ControlNet(cfg))
    sched = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    S = _mod("sampler")
    rt.set_mode("f16" if rt.lib().cnb_has_tcgen05() else "fp32")
    B, per, steps = 1024, 28 * 28, 120
    hint = syn.det_hint(B, 28).cuda()
    full = S.DDPMSampler(m, sched, seed=21, use_graph=True)
    xT = full.draw_xT((B, 1, 28, 28), "cuda")
    a, a0 = full.sample(xT, hint, steps=steps)
    assert torch.isfinite(a).all() and torch.isfinite(a0).all()
    assert float(a0.abs().max()) <= 1.0
    part = S.DDPMSampler(m, sched, seed=21, use_graph=True)
    outs = []
    for r in range(4):
        lo, hi = S.shard_bounds(B, 4, r)
        x_r = part.draw_xT((hi - lo, 1, 28, 28), "cuda", elem_offset=lo * per)
        assert torch.equal(x_r, xT[lo:hi])
        outs.append(part.sample(x_r, hint[lo:hi].contiguous(), steps=steps, elem_offset=lo * per)[0])
    assert torch.equal(torch.cat(outs), a)
    assert rt.lib().cnb_tc_error_flag() == 0


def test_f16_mode_activation_range(rt):
    """VERDICT r1 weak #8: the f16 mode keeps the residual stream in fp16.  Two limits, both exercised here by scaling
    conv_in (the residual stream then carries values of that order through every resnet's 1x1 skip path):
      * PRECISION - a 16-bit stream resolves |x| 2^-11: at |x| ~ 1e4 the O(1) output of a GroupNorm'd conv branch is
        below one ulp of the skip path it is added to, so eps parity is only claimed for streams of order <= 1e2
        (DESIGN.md 2); the gate below is the 1e-2 of BASELINE.json at gain 1 and 10, larger gains are printed;
      * RANGE - beyond 65504 the conv epilogue SATURATES (csrc/common.cuh::h2_sat) instead of producing inf, which the
        next GroupNorm would turn into NaN for the whole sample: outputs stay finite at any gain; fp32 mode keeps parity.
    Also: zero-conv weights of order 1e-6 (fp16 subnormals as weights) do not break parity."""
    if not rt.lib().cnb_has_tcgen05():
        pytest.skip("needs the tensor-core mode")
    import cn_oracle as O
    cfg = syn.TINY_PARAMS
    base = syn.det_state_dict(_mod("models.controlnet").ControlNet(cfg).state_dict())
    x, hint = inputs("range", 2, 1, 16)
    t = torch.tensor([300])

    def run(sd, mode):
        m = _mod("models.controlnet").ControlNet(cfg)
        m.load_state_dict(sd)
        m = m.cuda().eval()
        rt.set_mode(mode)
        with torch.no_grad():
            return m(x.cuda(), t.cuda(), hint.cuda()).cpu()

    def scaled(gain, zero_gain=1.0):
        sd = {k: v.clone() for k, v in base.items()}
        for k in sd:
            if k.endswith("conv_in.weight") or k.endswith("conv_in.bias"):
                sd[k] = sd[k] * gain
            if "zero_convs" in k:
                sd[k] = sd[k] * zero_gain
        return sd
    errs = {}
    for gain in (1.0, 10.0, 1e2, 1e3, 3e4, 3e7):
        sd = scaled(gain)
        want = O.controlnet_ddpm_forward(sd, cfg, x, t, hint)
        got = run(sd, "f16")
        assert torch.isfinite(got).all(), gain                 # saturation, never inf / NaN
        errs[gain] = rel_l2(got, want)
    print("f16 eps rel-L2 vs conv_in gain:", {g: f"{e:.2e}" for g, e in errs.items()})
    assert errs[1.0] < 1e-2 and errs[10.0] < 1e-2, errs
    sd = scaled(3e7)
    assert rel_l2(run(sd, "fp32"), O.controlnet_ddpm_forward(sd, cfg, x, t, hint)) < 1e-4
    # lightly trained zero convs: weights of order 1e-6
    sd = scaled(1.0, zero_gain=2e-5)
    want = O.controlnet_ddpm_forward(sd, cfg, x, t, hint)
    got = run(sd, "f16")
    assert rel_l2(got, want) < 1e-2, rel_l2(got, want)
