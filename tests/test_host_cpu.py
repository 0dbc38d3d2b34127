"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/cnb200.h declares, the drop-in
modules reproduce the reference's state_dict layout, host-side scheduler tables are bit-identical to the reference's,
the product path fails loudly on CPU tensors, and the data-parallel sharding / gather logic works under a
world_size-2 gloo group."""
import ctypes
import importlib
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

import helpers as H
from helpers import GOLDEN, REFERENCE, ROOT, golden, syn


def _mod(name):
    return importlib.import_module("controlnet-pytorch_b200." + name)


def test_library_exports_every_declared_symbol():
    rt = _mod("runtime")
    lib = rt.lib()
    with open(os.path.join(ROOT, "include", "cnb200.h")) as f:
        declared = sorted(set(re.findall(r"\b(cnb_[A-Za-z0-9_]+)\s*\(", f.read())))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(lib, name), name
    assert set(declared) == set(rt.EXPORTS), set(declared) ^ set(rt.EXPORTS)
    assert lib.cnb_abi_version() == 1
    assert lib.cnb_sizeof_conv_params() == ctypes.sizeof(rt.ConvParams)


def test_state_dict_layout_matches_reference_manifest():
    """Key names and shapes of every drop-in module == the reference's (manifest written by oracle/make_golden.py)."""
    with open(os.path.join(GOLDEN, "state_dict_manifest.json")) as f:
        man = json.load(f)
    cn, cnl = _mod("models.controlnet"), _mod("models.controlnet_ldm")
    ub, uc = _mod("models.unet_base"), _mod("models.unet_cond_base")
    cs, dm = _mod("models.consistency_controlnet_distilled"), _mod("models.distribution_matching_controlnet")
    built = {
        "controlnet_mnist": cn.ControlNet(syn.MNIST_PARAMS),
        "unet_mnist": ub.Unet(syn.MNIST_PARAMS),
        "unet_mnist_noup": ub.Unet(syn.MNIST_PARAMS, use_up=False),
        "controlnet_ldm_tiny": cnl.ControlNet(4, syn.TINY_LDM_PARAMS, down_sample_factor=8),
        "unet_ldm_tiny": uc.Unet(4, syn.TINY_LDM_PARAMS),
        "consistency_mnist": cs.ConsistencyControlNet(syn.MNIST_PARAMS),
        "dm_mnist": dm.DistributionMatchingControlNet(syn.MNIST_PARAMS),
        "consistency_distilled_tiny": cs.ConsistencyControlNetDistilled(syn.TINY_PARAMS),
        "dm_distilled_tiny": dm.DistributionMatchingControlNetDistilled(syn.TINY_PARAMS, "missing.pth", device=None),
    }
    for tag, mod in built.items():
        mine = {k: list(v.shape) for k, v in mod.state_dict().items()}
        assert list(mine.keys()) == list(man[tag].keys()), tag          # same keys in the same order
        assert mine == man[tag], tag
    assert not hasattr(built["unet_mnist_noup"], "ups") and not hasattr(built["unet_mnist_noup"], "conv_out")
    n = sum(p.numel() for p in built["controlnet_mnist"].parameters())
    assert n == 20070545                                                  # SURVEY.md Appendix E
    with open(os.path.join(GOLDEN, "state_dict_manifest_vae.json")) as f:
        man = json.load(f)
    vae = _mod("models.vae")
    for tag, mod in (("vae_tiny", vae.VAE(3, syn.TINY_VAE_PARAMS)), ("vae_celebhq", vae.VAE(3, syn.CELEBHQ_VAE_PARAMS))):
        mine = {k: list(v.shape) for k, v in mod.state_dict().items()}
        assert list(mine.keys()) == list(man[tag].keys()), tag
        assert mine == man[tag], tag


def test_default_init_is_seed_identical_to_reference_when_present():
    """torch.manual_seed(7) + ControlNet(TINY) gives the tensors the reference's class gives.  Without the reference
    the comparison is with the regression pin of the parent's drop-ins (tests/helpers.py: expected)."""
    cn = _mod("models.controlnet")
    torch.manual_seed(7)
    mine = cn.ControlNet(syn.TINY_PARAMS).state_dict()
    want, against = H.expected("init", H.init_digests)
    assert H.digest(mine) == want["controlnet_tiny_seed7"], against
    # the zero convolutions really are zero at init (controlnet.py:7-10)
    assert float(mine["control_copy_unet_down_zero_convs.0.weight"].abs().sum()) == 0.0


def test_checkpoint_round_trip_and_prefix_split(tmp_path):
    """ControlNet(model_ckpt=...) accepts a raw U-Net checkpoint or a full ControlNet one (controlnet.py:27-65)."""
    cn, ub = _mod("models.controlnet"), _mod("models.unet_base")
    cfg = syn.TINY_PARAMS
    unet_sd = syn.det_state_dict(ub.Unet(cfg).state_dict(), seed=3)
    p1 = str(tmp_path / "ddpm.pth")
    torch.save(unet_sd, p1)
    m = cn.ControlNet(cfg, model_ckpt=p1, device="cpu")
    assert torch.equal(m.trained_unet.conv_in.weight, unet_sd["conv_in.weight"])
    assert torch.equal(m.control_copy_unet.downs[0].resnet_conv_first[0][2].weight,
                       unet_sd["downs.0.resnet_conv_first.0.2.weight"])
    full = syn.det_state_dict(m.state_dict(), seed=4)
    p2 = str(tmp_path / "controlnet.pth")
    torch.save(full, p2)
    m2 = cn.ControlNet(cfg, model_ckpt=p2, device="cpu")
    for k, v in m2.state_dict().items():
        assert torch.equal(v, full[k]), k
    # ckpt is ignored unless BOTH model_ckpt and device are given (controlnet.py:27)
    m3 = cn.ControlNet(cfg, model_ckpt="does_not_exist.pth", device=None)
    assert float(m3.control_copy_unet_mid_zero_convs[0].weight.abs().sum()) == 0.0


@pytest.mark.parametrize("name,kw", [("ddpm", dict(syn.MNIST_DIFFUSION)),
                                     ("ldm", dict(syn.CELEBHQ_DIFFUSION, ldm_scheduler=True))])
def test_scheduler_tables_bit_identical(name, kw):
    s = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**kw)
    g = golden(f"scheduler_{name}")
    for k in ("betas", "alphas", "alpha_cum_prod", "sqrt_alpha_cum_prod", "sqrt_one_minus_alpha_cum_prod"):
        assert np.array_equal(getattr(s, k).numpy(), g[k]), k
    tab = s.coef_table_host()
    assert tab.shape == (1000, 6) and float(tab[0, 5]) == 0.0 and float(tab[1, 5]) == 1.0
    t = 500   # sigma_t restated from linear_noise_scheduler.py:68-70 with 0-d tensor ops
    var = (1 - s.alpha_cum_prod[t - 1]) / (1.0 - s.alpha_cum_prod[t]) * s.betas[t]
    assert float(tab[t, 4]) == float(var ** 0.5)
    assert float(tab[t, 1]) == float(torch.sqrt(s.alpha_cum_prod[t]))


def test_product_path_has_no_cpu_fallback():
    rt = _mod("runtime")
    m = _mod("models.controlnet").ControlNet(syn.TINY_PARAMS)
    with pytest.raises(rt.CnbError):
        m(torch.zeros(1, 1, 16, 16), torch.tensor([3]), torch.zeros(1, 3, 16, 16))
    s = _mod("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    with pytest.raises(rt.CnbError):
        s.sample_prev_timestep(torch.zeros(1, 1, 4, 4), torch.zeros(1, 1, 4, 4), torch.as_tensor(5))
    with pytest.raises(AssertionError):                      # same config asserts as unet_base.py:308-310
        bad = dict(syn.TINY_PARAMS, mid_channels=[32, 64, 64])
        _mod("models.unet_base").Unet(bad)
    # nothing under the product package imports the oracle
    pkg = os.path.join(ROOT, "controlnet-pytorch_b200")
    for dp, _, fs in os.walk(pkg):
        for fn in fs:
            if fn.endswith(".py"):
                src = open(os.path.join(dp, fn)).read()
                assert "cn_oracle" not in src and "import oracle" not in src, fn


def test_shard_bounds_partition():
    S = _mod("sampler")
    for total in (1, 7, 16, 1024, 1025):
        for world in (1, 2, 3, 8):
            b = [S.shard_bounds(total, world, r) for r in range(world)]
            assert b[0][0] == 0 and b[-1][1] == total
            assert all(b[i][1] == b[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, world, port, total, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        S = importlib.import_module("controlnet-pytorch_b200.sampler")
        lo, hi = S.shard_bounds(total, world, rank)
        full = torch.arange(total * 6, dtype=torch.float32).reshape(total, 1, 2, 3)
        out = S.gather_shards(full[lo:hi].clone(), total)
        q.put((rank, bool(torch.equal(out, full))))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("total", [8, 7])
def test_gather_shards_gloo_world2(total):
    """The only collective of the job (final sample all-gather), equal and ragged shards, on a 2-rank gloo group."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000) + total
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, total, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]


def _dropin_env(extra_path=()):
    env = dict(os.environ)
    env["PYTHONSAFEPATH"] = "1"           # keep the cwd (a reference checkout has its own `models`) off sys.path
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "controlnet-pytorch_b200", "dropin"), *extra_path])
    return env


def test_dropin_shim_serves_the_reference_import_lines(tmp_path):
    """INTEGRATION.md section 1: with controlnet-pytorch_b200/dropin first on sys.path the reference's import lines
    (`from models.controlnet import ControlNet`, ...) resolve to the B200 classes."""
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_tool_loop.py"), "--check-imports"],
                       env=_dropin_env(), cwd=str(tmp_path), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dropin imports ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.skipif(REFERENCE is None or not os.path.isdir(os.path.join(REFERENCE, "tools")),
                    reason="needs a reference checkout (CNB_REFERENCE)")
def test_reference_tools_import_the_dropins_and_keep_their_other_modules():
    """The unmodified tools/sample_*.py, run from the reference checkout, get the B200 models / scheduler while
    dataset.*, scheduler.consistency_scheduler and models.discriminator still come from the reference."""
    import subprocess
    code = (
        "import tools.sample_ddpm_controlnet as t, tools.sample_ldm_controlnet as l\n"
        "import tools.sample_consistency_controlnet_distilled as c\n"
        "import tools.sample_distribution_matching_controlnet_distilled as d\n"
        "import scheduler.consistency_scheduler as cs, models.discriminator as md\n"
        "P = 'controlnet-pytorch_b200.'\n"
        "assert t.ControlNet.__module__ == P + 'models.controlnet'\n"
        "assert t.LinearNoiseScheduler.__module__ == P + 'scheduler.linear_noise_scheduler'\n"
        "assert l.ControlNet.__module__ == P + 'models.controlnet_ldm' and l.VAE.__module__ == P + 'models.vae'\n"
        "assert c.ConsistencyControlNetDistilled.__module__ == P + 'models.consistency_controlnet_distilled'\n"
        "assert d.DistributionMatchingControlNetDistilled.__module__ == P + 'models.distribution_matching_controlnet'\n"
        f"assert cs.__file__.startswith({REFERENCE + os.sep!r}) and md.__file__.startswith({REFERENCE + os.sep!r})\n"
        "assert t.MnistDataset.__module__ == 'dataset.mnist_dataset'\n"
        "print('tools ok')\n")
    r = subprocess.run([sys.executable, "-c", code], env=_dropin_env([REFERENCE]), cwd=REFERENCE,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "tools ok" in r.stdout, r.stdout + r.stderr


def test_checkpoints_written_by_the_reference_load_the_way_the_tools_load_them(tmp_path):
    """The construction / checkpoint sequences of tools/sample_ddpm_controlnet.py:80-92,
    tools/sample_consistency_controlnet_distilled.py:30-49 and
    tools/sample_distribution_matching_controlnet_distilled.py:33-54, fed with files written by the REFERENCE classes:
    every tensor of the resulting B200 module equals the reference module built the same way.  Without the reference
    the drop-in classes write the files and both their modules and the loaded ones are compared with the regression
    pins of the parent's drop-ins (tests/helpers.py: expected)."""
    cfg = syn.TINY_PARAMS
    if REFERENCE is not None:
        paths, want = H.on_reference(lambda get: H.write_tool_checkpoints(get, tmp_path))
        against = "reference"
    else:
        paths, written = H.write_tool_checkpoints(_mod, tmp_path)
        want, against = H.expected("tool_checkpoints", None)
        assert written == want, against
    ddpm, ctrl, cons, dmck = paths["ddpm"], paths["ctrl"], paths["cons"], paths["dm"]
    dev = torch.device("cpu")
    torch.manual_seed(20)
    cn = _mod("models.controlnet").ControlNet(cfg, model_ckpt=ddpm, device=dev).to(dev)
    cn.load_state_dict(torch.load(ctrl, map_location=dev))
    torch.manual_seed(21)       # same seed as the reference construction: the unloaded tensors (hint blocks) match too
    mc = _mod("models.consistency_controlnet_distilled").ConsistencyControlNetDistilled(cfg, ddpm, device=dev).to(dev)
    mc.student.load_state_dict(torch.load(cons, map_location=dev, weights_only=False)["model_state_dict"])
    torch.manual_seed(22)
    md = _mod("models.distribution_matching_controlnet").DistributionMatchingControlNetDistilled(cfg, ctrl, device=dev).to(dev)
    md.student.load_state_dict(torch.load(dmck, map_location=dev, weights_only=False)["model_state_dict"])
    for tag, mine in (("cn", cn.state_dict()), ("cons", mc.state_dict()), ("dm", md.state_dict())):
        assert H.digest(mine) == want[tag], (tag, against)


def test_every_dropin_class_initialises_seed_identically_to_the_reference():
    """torch.manual_seed(s) + constructor gives the same tensors under the same keys as the reference class, for every
    module on the path (layers are created in the reference's order, so the default initialisers draw the same numbers).
    Without the reference: the regression pins of the parent's drop-ins (tests/helpers.py: expected)."""
    want, against = H.expected("init", H.init_digests)
    mine = H.init_digests(_mod)
    for name in want:
        assert mine[name] == want[name], (name, against)


def test_public_surface_matches_the_reference_signatures():
    """Every public class / function of the reference's hot-path modules exists in the drop-in module, and the
    inference-side methods take the reference's parameters (names, order, defaults); extra trailing keyword
    parameters (`z=`, `step_index=`) are allowed.  Without the reference the recorded surface is the parent's drop-in
    surface (re-exported duplicates such as blocks.get_time_embedding included), so there the extras are pinned too."""
    ref, against = H.expected("public_surface", H.public_surface)
    checked = 0
    for m, entries in ref.items():
        mod = _mod(m)
        for name, want in entries.items():
            mine = getattr(mod, name, None)
            assert mine is not None, (m, name, against)
            for meth, w in (want.items() if isinstance(want, dict) else [(None, want)]):
                got = H.signature(mine if meth is None else getattr(mine, meth))
                assert got[:len(w)] == w, (m, name, meth, w, got, against)
                checked += 1
    assert checked >= 40


def test_host_side_helpers_are_bit_identical_to_the_reference():
    """add_noise (linear_noise_scheduler.py:25-47), the EDM scalings (consistency_controlnet_distilled.py:45-74) and the
    Karras schedule (:175-196) are plain host tensor expressions in both implementations: bit-identical on the CPU.
    Without the reference: the regression pins of the parent's drop-ins (tests/helpers.py: expected)."""
    want, against = H.expected("host_helpers", H.host_helper_digests)
    mine = H.host_helper_digests(_mod)
    assert len(mine) == len(want)
    for i, (a, b) in enumerate(zip(mine, want)):
        assert a == b, (i, against)


@pytest.mark.parametrize("locked", [True, False])
def test_model_locked_and_get_params_match_the_reference(locked):
    """`model_locked` freezes the same parameters and `get_params()` (controlnet.py:140-156, controlnet_ldm.py) returns
    the same parameters in the same order as the reference.  Without the reference: the regression pins of the parent's
    drop-ins (tests/helpers.py: expected)."""
    want, against = H.expected("locked_params", lambda get: {str(lk): H.locked_params(get, lk) for lk in (True, False)})
    assert H.locked_params(_mod, locked) == want[str(locked)], against
