"""Pins oracle/cn_oracle.py against the reference's own outputs (tests/golden, made by oracle/make_golden.py)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from helpers import REFERENCE, det_sd_for, golden, inputs, max_abs, psnr, rel_l2, syn, ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import cn_oracle as O  # noqa: E402

TOL = 2e-5   # fp32 CPU vs fp32 CPU through a different composition of the same ATen primitives


def _keys_controlnet(cfg, ldm=False, im_channels=None, dsf=8):
    """Build the key->shape template without the reference: use the drop-in modules' own state_dict."""
    pkg = importlib.import_module("controlnet-pytorch_b200")
    if ldm:
        mod = importlib.import_module("controlnet-pytorch_b200.models.controlnet_ldm")
        return mod.ControlNet(im_channels, cfg, down_sample_factor=dsf).state_dict()
    mod = importlib.import_module("controlnet-pytorch_b200.models.controlnet")
    return mod.ControlNet(cfg).state_dict()


@pytest.mark.parametrize("name,cfg,B,ts", [("tiny", syn.TINY_PARAMS, 2, (999, 37, 0)),
                                           ("mnist", syn.MNIST_PARAMS, 2, (999, 500, 0)),
                                           ("cifar", syn.CIFAR_PARAMS, 1, (500,))])
def test_controlnet_ddpm_vs_golden(name, cfg, B, ts):
    sd = syn.det_state_dict(_keys_controlnet(cfg))
    x, hint = inputs(name, B, cfg["im_channels"], cfg["im_size"])
    g = golden(f"controlnet_{name}")
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-9
    with torch.no_grad():
        for t in ts:
            eps = O.controlnet_ddpm_forward(sd, cfg, x, torch.as_tensor(t).unsqueeze(0), hint)
            assert rel_l2(eps, g[f"eps_{t}"]) < TOL
        if name == "tiny":
            eps = O.controlnet_ddpm_forward(sd, cfg, x, torch.tensor([10, 700]), hint)
            assert rel_l2(eps, g["eps_pers"]) < TOL
        if name != "cifar":
            sched = O.SchedulerOracle(**syn.MNIST_DIFFUSION)
            zs = [syn.det_noise(f"{name}:z{k}", tuple(x.shape)) for k in range(3)]
            xt, x0 = O.ddpm_sample(lambda a, t, h: O.controlnet_ddpm_forward(sd, cfg, a, t, h), sched, x, hint, 3, zs)
            assert rel_l2(xt, g["traj3_xt"]) < 5 * TOL
            assert rel_l2(x0, g["traj3_x0"]) < 5 * TOL


def test_config1_mnist_b16_50step_vs_golden():
    """BASELINE.json configs[0] (MNIST ControlNet, batch 16, 50 steps, t = 49 .. 0): the oracle's final x_0 / x_{t-1}
    against the unmodified reference's (tests/golden/config1_mnist_b16_50step.npz, oracle/make_golden.py)."""
    cfg = syn.MNIST_PARAMS
    sd = syn.det_state_dict(_keys_controlnet(cfg))
    x, hint = inputs("config1", 16, cfg["im_channels"], cfg["im_size"])
    g = golden("config1_mnist_b16_50step")
    sched = O.SchedulerOracle(**syn.MNIST_DIFFUSION)
    zs = [syn.det_noise(f"config1:z{k}", tuple(x.shape)) for k in range(50)]
    with torch.no_grad():
        xt, x0 = O.ddpm_sample(lambda a, t, h: O.controlnet_ddpm_forward(sd, cfg, a, t, h), sched, x, hint, 50, zs)
    assert psnr(x0, g["x0"]) > 80.0 and max_abs(x0, g["x0"]) < 1e-3, (psnr(x0, g["x0"]), max_abs(x0, g["x0"]))
    assert rel_l2(xt, g["xt"]) < 1e-4


def test_controlnet_ldm_vs_golden():
    cfg = syn.TINY_LDM_PARAMS
    sd = syn.det_state_dict(_keys_controlnet(cfg, ldm=True, im_channels=4))
    x, hint = inputs("tiny_ldm", 2, 4, 8, hint_size=64, p=0.05)
    g = golden("controlnet_tiny_ldm")
    with torch.no_grad():
        for t in (999, 3):
            eps = O.controlnet_ldm_forward(sd, cfg, x, torch.as_tensor(t).unsqueeze(0), hint)
            assert rel_l2(eps, g[f"eps_{t}"]) < TOL
        sched = O.SchedulerOracle(ldm_scheduler=True, **syn.CELEBHQ_DIFFUSION)
        zs = [syn.det_noise(f"tiny_ldm:z{k}", tuple(x.shape)) for k in range(3)]
        xt, x0 = O.ddpm_sample(lambda a, t, h: O.controlnet_ldm_forward(sd, cfg, a, t, h), sched, x, hint, 3, zs)
        assert rel_l2(xt, g["traj3_xt"]) < 5 * TOL


def test_unet_vs_golden():
    mod = importlib.import_module("controlnet-pytorch_b200.models.unet_base")
    sd = syn.det_state_dict(mod.Unet(syn.TINY_PARAMS).state_dict())
    x, _ = inputs("unet_tiny", 2, 1, 16)
    with torch.no_grad():
        eps = O.unet_forward(sd, "", O.base_arch(syn.TINY_PARAMS), x, torch.as_tensor(123).unsqueeze(0))
    assert rel_l2(eps, golden("unet_tiny")["eps_123"]) < TOL


@pytest.mark.parametrize("name,cfg,sigma", [("tiny", syn.TINY_PARAMS, 80.0), ("mnist", syn.MNIST_PARAMS, 80.0),
                                            ("cifar", syn.CIFAR_PARAMS, 5.0)])
def test_students_vs_golden(name, cfg, sigma):
    B = 2 if name != "cifar" else 1
    cmod = importlib.import_module("controlnet-pytorch_b200.models.consistency_controlnet_distilled")
    dmod = importlib.import_module("controlnet-pytorch_b200.models.distribution_matching_controlnet")
    with torch.no_grad():
        sd = syn.det_state_dict(cmod.ConsistencyControlNet(cfg).state_dict())
        x, hint = inputs("cons_" + name, B, cfg["im_channels"], cfg["im_size"])
        g = golden(f"consistency_{name}")
        assert rel_l2(O.consistency_forward(sd, cfg, x, torch.full((B,), sigma), hint), g["x0_max"]) < TOL
        assert rel_l2(O.consistency_forward(sd, cfg, x, torch.full((B,), 1.7), hint), g["x0_mid"]) < TOL
        assert torch.equal(O.consistency_forward(sd, cfg, x, torch.full((B,), 0.001), hint),
                           torch.from_numpy(g["x0_min"]))
        sd = syn.det_state_dict(dmod.DistributionMatchingControlNet(cfg).state_dict())
        x, hint = inputs("dm_" + name, B, cfg["im_channels"], cfg["im_size"])
        g = golden(f"dm_{name}")
        assert rel_l2(O.dm_forward(sd, cfg, x, torch.full((B,), 999), hint), g["x0_999"]) < TOL
        if B == 2:
            assert rel_l2(O.dm_forward(sd, cfg, x, torch.tensor([5, 400]), hint), g["x0_pers"]) < TOL


@pytest.mark.parametrize("name,kw", [("ddpm", dict(syn.MNIST_DIFFUSION)),
                                     ("ldm", dict(syn.CELEBHQ_DIFFUSION, ldm_scheduler=True))])
def test_scheduler_bit_exact_vs_golden(name, kw):
    g = golden(f"scheduler_{name}")
    s = O.SchedulerOracle(**kw)
    for k in ("betas", "alphas", "alpha_cum_prod", "sqrt_alpha_cum_prod", "sqrt_one_minus_alpha_cum_prod"):
        assert np.array_equal(getattr(s, k).numpy(), g[k]), k
    xt = syn.det_noise("sched:xt", (3, 4, 9, 7))
    eps = syn.det_noise("sched:eps", (3, 4, 9, 7))
    z = syn.det_noise("sched:z", (3, 4, 9, 7))
    for t in (999, 500, 1, 0):
        a, b = s.sample_prev_timestep(xt, eps, t, z)
        assert np.array_equal(a.numpy(), g[f"prev_{t}"]), t
        assert np.array_equal(b.numpy(), g[f"x0_{t}"]), t


@pytest.mark.skipif(REFERENCE is None, reason="needs the reference's modules (CNB_REFERENCE or baseline/_ref)")
def test_oracle_vs_live_reference_default_init():
    """Second pin: default torch init (zero-convs exactly zero) straight from the imported reference."""
    sys.path.insert(0, REFERENCE)
    try:
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]
        from models.controlnet import ControlNet as Ref
        torch.manual_seed(3)
        m = Ref(syn.TINY_PARAMS).eval()
        x, hint = inputs("live", 2, 1, 16)
        with torch.no_grad():
            want = m(x, torch.as_tensor(77).unsqueeze(0), hint)
            got = O.controlnet_ddpm_forward(m.state_dict(), syn.TINY_PARAMS, x, torch.as_tensor(77).unsqueeze(0), hint)
        assert rel_l2(got, want) < TOL
    finally:
        sys.path.remove(REFERENCE)
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.")]:
            del sys.modules[k]


def test_vae_vs_golden():
    """models/vae.py decode / encode (the step after the LDM sampling loop) against the reference's outputs."""
    cfg = syn.TINY_VAE_PARAMS
    sd = det_sd_for(lambda: importlib.import_module("controlnet-pytorch_b200.models.vae").VAE(3, cfg), "vae_tiny")
    g = golden("vae_tiny")
    with torch.no_grad():
        dec = O.vae_decode(sd, cfg, syn.det_noise("vae_tiny:z", (2, 4, 8, 8)))
        sample, enc = O.vae_encode(sd, cfg, syn.det_noise("vae_tiny:x", (2, 3, 32, 32)),
                                   noise=syn.det_noise("vae_tiny:n", (2, 4, 8, 8)))
    assert rel_l2(dec, g["dec"]) < 2e-6
    assert rel_l2(enc, g["enc_out"]) < 2e-6
    assert rel_l2(sample, g["enc_sample"]) < 2e-6


def test_vae_celebhq_decode_vs_golden():
    """Full-size CelebHQ autoencoder (config/celebhq.yaml:27-38) decode at batch 1: strided image sample + moments."""
    cfg = syn.CELEBHQ_VAE_PARAMS
    sd = det_sd_for(lambda: importlib.import_module("controlnet-pytorch_b200.models.vae").VAE(3, cfg), "vae_celebhq")
    g = golden("vae_celebhq")
    with torch.no_grad():
        img = O.vae_decode(sd, cfg, syn.det_noise("vae_celebhq:z", (1, 4, 32, 32)))
    assert tuple(img.shape) == (1, 3, 128, 128)
    assert rel_l2(img[:, :, ::4, ::4], g["dec_strided"]) < 5e-6
    assert abs(float(img.double().pow(2).sum()) / float(g["dec_sqsum"]) - 1) < 1e-5


def _teacher_wrappers(tmp_path):
    """Product wrappers (CPU parameter holders) built from a det_state_dict ControlNet checkpoint, as make_golden does."""
    cfg = syn.TINY_PARAMS
    CN = importlib.import_module("controlnet-pytorch_b200.models.controlnet").ControlNet
    teacher = CN(cfg)
    teacher.load_state_dict(syn.det_state_dict(teacher.state_dict(), 3))
    ck = os.path.join(str(tmp_path), "teacher.pth")
    torch.save(teacher.state_dict(), ck)
    dm = importlib.import_module("controlnet-pytorch_b200.models.distribution_matching_controlnet")
    cs = importlib.import_module("controlnet-pytorch_b200.models.consistency_controlnet_distilled")
    return (cfg, dm.DistributionMatchingControlNetDistilled(cfg, ck, device=torch.device("cpu")),
            cs.ConsistencyControlNetDistilled(cfg, ck, device=torch.device("cpu")))


def test_teacher_predictions_vs_golden(tmp_path):
    """get_teacher_prediction / get_ddpm_teacher_prediction / sigma_to_timestep (SURVEY.md 8f-4)."""
    cfg, dm, cs = _teacher_wrappers(tmp_path)
    g = golden("teachers_tiny")
    x, hint = inputs("teacher_tiny", 3, cfg["im_channels"], cfg["im_size"])
    so = O.SchedulerOracle(**syn.MNIST_DIFFUSION)
    sig = torch.tensor([60.0, 2.5, 0.05])
    with torch.no_grad():
        a = O.teacher_x0(dm.state_dict(), cfg, so, x, torch.tensor([999, 412, 3]), hint, prefix="teacher.")
        b = O.teacher_x0(dm.state_dict(), cfg, so, x[:1], torch.tensor(77), hint[:1], prefix="teacher.")
        t = O.sigma_to_timestep(so, sig)
        c = O.teacher_x0(cs.state_dict(), cfg, so, x, t, hint, prefix="ddpm_teacher.")
    assert rel_l2(a, g["dm_x0"]) < TOL and rel_l2(b, g["dm_x0_shared_t"]) < TOL
    assert t.tolist() == g["cs_t"].tolist()
    assert cs.sigma_to_timestep(sig).tolist() == g["cs_t"].tolist()     # host-side table lookup of the product class
    assert rel_l2(c, g["cs_x0"]) < TOL
