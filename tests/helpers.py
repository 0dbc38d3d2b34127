"""Shared helpers for the parity tests (model builders over a flat state_dict, metrics, host-side parity checks)."""
import hashlib
import importlib
import importlib.util
import inspect
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
syn = importlib.import_module("controlnet-pytorch_b200.utils.synthetic")
GOLDEN = os.path.join(ROOT, "tests", "golden")
_spec = importlib.util.spec_from_file_location("install_ref", os.path.join(ROOT, "oracle", "install_ref.py"))
install_ref = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(install_ref)

# where the reference's own modules can be imported from (oracle/install_ref.py: its checkout, else the copy under
# baseline/_ref), else None
REFERENCE = install_ref.ref_path()


def rel_l2(a, b):
    a = torch.as_tensor(a).double().flatten()
    b = torch.as_tensor(b).double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def psnr(a, b, peak_to_peak=2.0):
    """PSNR in dB of images in [-1, 1] (peak-to-peak 2, as written by the sampling tools before the [0, 1] map)."""
    a = torch.as_tensor(a).double().flatten()
    b = torch.as_tensor(b).double().flatten()
    mse = float(((a - b) ** 2).mean())
    return float("inf") if mse == 0.0 else 10.0 * float(np.log10(peak_to_peak ** 2 / mse))


def max_abs(a, b):
    return float((torch.as_tensor(a).double() - torch.as_tensor(b).double()).abs().max())


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def inputs(name, B, C, S, hint_size=None, p=0.1):
    return syn.det_noise(name + ":x", (B, C, S, S)), syn.det_hint(B, hint_size or S, p=p)


_SD_CACHE = {}


def det_sd_for(module_factory, tag, seed=0):
    """state_dict with deterministic weights for a freshly built (CPU) module; cached per tag."""
    if tag not in _SD_CACHE:
        m = module_factory()
        _SD_CACHE[tag] = syn.det_state_dict(m.state_dict(), seed)
    return _SD_CACHE[tag]


# ---------------------------------------------------------------------------------------------------------------------
# Host-side parity checks.  Each function below takes `get(name)`, which returns the module `name` ("models.controlnet",
# ...) of one implementation, so the drop-ins and the reference run the same code.  With the reference importable
# (REFERENCE) the tests compare the drop-ins with it directly.  Without it they compare with tests/golden/
# regression_pins.json (tests/record_regression_pins.py): these are NOT reference data, they were recorded from the
# drop-ins of the parent commit 70d0cc0 because no copy of the reference was at hand, so they only catch changes of the
# drop-ins' own behaviour since then.
# ---------------------------------------------------------------------------------------------------------------------
PINS = os.path.join(GOLDEN, "regression_pins.json")


def _purge():
    for k in [k for k in sys.modules if k.split(".")[0] in ("models", "scheduler")]:
        del sys.modules[k]


def on_reference(fn):
    """fn(get) with `get` importing the reference's own modules (REFERENCE first on sys.path)."""
    sys.path.insert(0, REFERENCE)
    try:
        _purge()
        return fn(importlib.import_module)
    finally:
        sys.path.remove(REFERENCE)
        _purge()


def expected(key, fn):
    """(what the reference gives for fn, "reference") when it is importable, else (the regression pin `key`, a label
    naming the torch version the pins were recorded with: the default initialisers' bytes depend on it)."""
    if REFERENCE is not None:
        return on_reference(fn), "reference"
    with open(PINS) as f:
        pins = json.load(f)
    return pins[key], f"regression pins of 70d0cc0's drop-ins (torch {pins['_torch']}; running {torch.__version__})"


def digest(tensors):
    """SHA-256 over the names, dtypes, shapes and bytes of an ordered tensor dict (equal digests <=> torch.equal
    tensors under the same keys in the same order)."""
    h = hashlib.sha256()
    for k, v in tensors.items():
        v = v.detach().cpu().contiguous()
        h.update(f"{k}|{v.dtype}|{tuple(v.shape)}|".encode())
        h.update(v.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


INIT_SPECS = [("models.controlnet_ldm", "ControlNet", (4, syn.TINY_LDM_PARAMS), dict(down_sample_factor=8)),
              ("models.vae", "VAE", (3, syn.TINY_VAE_PARAMS), {}),
              ("models.unet_base", "Unet", (syn.TINY_PARAMS,), {}),
              ("models.unet_cond_base", "Unet", (4, syn.TINY_LDM_PARAMS), {}),
              ("models.consistency_controlnet_distilled", "ConsistencyControlNet", (syn.TINY_PARAMS,), {}),
              ("models.consistency_controlnet_distilled", "ConsistencyControlNetDistilled", (syn.TINY_PARAMS,), {}),
              ("models.distribution_matching_controlnet", "DistributionMatchingControlNet", (syn.TINY_PARAMS,), {}),
              ("models.controlnet", "ControlNet", (syn.MNIST_PARAMS,), {})]


def init_digests(get):
    """torch.manual_seed(s) + constructor with default init: tiny ControlNet at seed 7, then every INIT_SPECS class at
    seed 100 + i."""
    torch.manual_seed(7)
    out = {"controlnet_tiny_seed7": digest(get("models.controlnet").ControlNet(syn.TINY_PARAMS).state_dict())}
    for i, (mod, cls, a, k) in enumerate(INIT_SPECS):
        torch.manual_seed(100 + i)
        out[f"{mod}.{cls}"] = digest(getattr(get(mod), cls)(*a, **k).state_dict())
    return out


def write_tool_checkpoints(get, d):
    """The checkpoint files the training tools write for tools/sample_ddpm_controlnet.py:80-92,
    tools/sample_consistency_controlnet_distilled.py:30-49 and tools/sample_distribution_matching_controlnet_distilled.py
    :33-54, built with the classes of `get`; returns (paths, digests of the modules built the tools' way)."""
    cfg = syn.TINY_PARAMS
    p = {k: os.path.join(str(d), k + ".pth") for k in ("ddpm", "ctrl", "cons", "dm")}
    torch.manual_seed(11)
    torch.save(get("models.unet_base").Unet(cfg).state_dict(), p["ddpm"])
    torch.manual_seed(20)
    cn = get("models.controlnet").ControlNet(cfg, model_ckpt=p["ddpm"], device=torch.device("cpu"))
    cn.load_state_dict(syn.det_state_dict(cn.state_dict(), seed=5))
    torch.save(cn.state_dict(), p["ctrl"])
    torch.manual_seed(21)
    cons = get("models.consistency_controlnet_distilled").ConsistencyControlNetDistilled(cfg, p["ddpm"],
                                                                                         device=torch.device("cpu"))
    torch.save({"model_state_dict": syn.det_state_dict(cons.student.state_dict(), seed=6)}, p["cons"])
    cons.student.load_state_dict(torch.load(p["cons"], weights_only=False)["model_state_dict"])
    torch.manual_seed(22)
    dm = get("models.distribution_matching_controlnet").DistributionMatchingControlNetDistilled(
        cfg, p["ctrl"], device=torch.device("cpu"))
    torch.save({"model_state_dict": syn.det_state_dict(dm.student.state_dict(), seed=7)}, p["dm"])
    dm.student.load_state_dict(torch.load(p["dm"], weights_only=False)["model_state_dict"])
    return p, {"cn": digest(cn.state_dict()), "cons": digest(cons.state_dict()), "dm": digest(dm.state_dict())}


SURFACE_MODULES = ["models.unet_base", "models.blocks", "models.unet_cond_base", "models.controlnet",
                   "models.controlnet_ldm", "models.consistency_controlnet_distilled",
                   "models.distribution_matching_controlnet", "models.vae", "scheduler.linear_noise_scheduler"]
SURFACE_METHODS = ("__init__", "forward", "encode", "decode", "generate", "sample_prev_timestep", "add_noise",
                   "get_params", "get_teacher_prediction", "get_ddpm_teacher_prediction", "sigma_to_timestep",
                   "get_noise_schedule", "c_skip", "c_out", "c_in", "c_noise")


def signature(f):
    return [[p.name, repr(p.default)] for p in inspect.signature(f).parameters.values()]


def public_surface(get, reexports=False):
    """{module: {public class / function defined there: its signature, or {method: signature}}}.  `reexports` also
    takes the names a module imports from another SURFACE_MODULES module: the drop-ins re-export some of the
    reference's duplicate definitions (blocks.get_time_embedding is unet_base's), which only the reference defines
    in place."""
    out = {}
    for m in SURFACE_MODULES:
        mod, entries = get(m), {}
        for name, obj in vars(mod).items():
            home = str(getattr(obj, "__module__", ""))
            if name.startswith("_") or not any(home.endswith(o) for o in (SURFACE_MODULES if reexports else [m])):
                continue
            if inspect.isclass(obj):
                entries[name] = {meth: signature(getattr(obj, meth)) for meth in SURFACE_METHODS if meth in vars(obj)}
            elif inspect.isfunction(obj):
                entries[name] = signature(obj)
        out[m] = entries
    return out


def host_helper_digests(get):
    """add_noise (linear_noise_scheduler.py:25-47), the EDM scalings (consistency_controlnet_distilled.py:45-74) and the
    Karras schedule (:175-196): plain host tensor expressions."""
    s = get("scheduler.linear_noise_scheduler").LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    g = torch.Generator().manual_seed(0)
    x, n = torch.randn(4, 1, 8, 8, generator=g), torch.randn(4, 1, 8, 8, generator=g)
    t, sig = torch.tensor([0, 5, 500, 999]), torch.tensor([0.002, 1.7, 80.0])
    cc = get("models.consistency_controlnet_distilled")
    cm, cd = cc.ConsistencyControlNet(syn.TINY_PARAMS), cc.ConsistencyControlNetDistilled(syn.TINY_PARAMS)
    vals = [s.add_noise(x, n, t), cm.c_skip(sig), cm.c_out(sig), cm.c_in(sig), cm.c_noise(sig),
            cd.get_noise_schedule(10, device=torch.device("cpu"))]
    return [digest({"v": v}) for v in vals]


def locked_params(get, locked):
    """Digest of (name, requires_grad) of every parameter under `model_locked` and of the names get_params() returns,
    in order (controlnet.py:140-156, controlnet_ldm.py), for the DDPM and the LDM ControlNet."""
    def describe(m):
        names = {id(p): n for n, p in m.named_parameters()}
        d = [[[n, p.requires_grad] for n, p in m.named_parameters()], [names[id(p)] for p in m.get_params()]]
        return hashlib.sha256(json.dumps(d).encode()).hexdigest()
    return [describe(get("models.controlnet").ControlNet(syn.TINY_PARAMS, model_locked=locked)),
            describe(get("models.controlnet_ldm").ControlNet(4, syn.TINY_LDM_PARAMS, model_locked=locked,
                                                             down_sample_factor=8))]
