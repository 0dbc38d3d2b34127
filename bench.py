"""bench.py - headline benchmark of the ControlNet denoising hot path (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 2|3|4|5]
                    [--scaling strong|weak] [--mode f16|fp32] [--dump-outputs DIR]

Workload : MNIST DDPM ControlNet (config/mnist.yaml model_params), synthetic random-init weights, x_T ~ N(0,1),
           Canny-like hints (Bernoulli 0.1 in {0,1}, 3 identical channels), GLOBAL batch 1024 (BASELINE config 2).
Step     : ONE denoising timestep over the rank's shard = ControlNet forward (eps) + fused sample_prev_timestep, replayed
           from a CUDA graph (t, scheduler coefficients and Philox step are read on the device).
Metric   : samples/s of full 1000-step sampling = global_batch / (1000 * seconds_per_step), max over ranks.
Multi-GPU: one process per GPU (torchrun); the global batch of 1024 is SHARDED (1024 / N per rank, "scaling": "strong"),
           no collective inside the loop, one NCCL all-gather of the final samples (inside the timed `e2e` region).
           `weak` (N > 1) is a second, labelled record with 1024 samples per GPU.
The line also carries `e2e` (the whole job through the public API sampler.sample_data_parallel: pinned-host x_T + hint
shard H2D, all 1000 timesteps, all-gather, D2H of the gathered samples - all inside the timed region), `roofline`
(dominant kernel, timed live with CUDA events), `cpu_baseline` / `torch_cuda_reference` (the reference's own modules on
the box's host cores / on the same GPU through stock PyTorch) and `clocks` (nvidia-smi under load).
`--impl reference` times the reference's own modules (baseline/_ref, installed by oracle/install_ref.py) on the CPU.
`--config 3|4|5` run the other BASELINE configs (CelebHQ LDM + VAE decode; consistency students; CIFAR DM sweep).
`--dump-outputs DIR` writes what the timed step computed in its last replay, the (x_{t-1}, x0) pair a caller of
sampler.DDPMSampler.sample receives, as DIR/xt.npy and DIR/x0.npy (float32, the whole global batch, or a fixed seeded
sample of its rows above 64 MB in all).  Weights, hints, x_T and the Philox noise are all seeded, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True          # the tree may be read-only: nothing of this run is cached in it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
METRIC = "controlnet_ddpm_samples_per_sec"
UNIT = "samples/s"
STEPS_PER_SAMPLE = 1000
FLOP_PER_SAMPLE_STEP = 3.878e9          # BASELINE.md section 2 (MNIST ControlNet, 2*MAC convention)
DUMP_LIMIT_BYTES = 63 * 10 ** 6          # --dump-outputs: under 64 MB in all, .npy headers included


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tf=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                    tf_burst=float(p["bf16_tflops"]), src="measured")
    except Exception:
        return dict(hbm=6650.0, tf=1400.0, tf_burst=1590.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self, t0, t1):
        rows = [r for (ts, r) in self.rows if t0 <= ts <= t1 + 0.15] or [r for (_, r) in self.rows]
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_problem(batch, device, seed_offset=0):
    import torch
    syn = importlib.import_module("controlnet-pytorch_b200.utils.synthetic")
    cn = importlib.import_module("controlnet-pytorch_b200.models.controlnet")
    sch = importlib.import_module("controlnet-pytorch_b200.scheduler.linear_noise_scheduler")
    cfg = syn.MNIST_PARAMS
    model = cn.ControlNet(cfg)
    model.load_state_dict(syn.det_state_dict(model.state_dict()))
    model = model.to(device).eval()
    sched = sch.LinearNoiseScheduler(**syn.MNIST_DIFFUSION)
    g = torch.Generator().manual_seed(1234 + seed_offset)
    hint_host = (torch.rand(batch, 1, 28, 28, generator=g) < 0.1).float().repeat(1, 3, 1, 1).contiguous()
    return cfg, model, sched, hint_host


# ------------------------------------------------------------------------------------------------------------
# roofline: instrumented eager step, CUDA events around every libcnb200 launch on the launching stream
# ------------------------------------------------------------------------------------------------------------
def k_heads(a, k):
    return a[1] if len(a) > 1 else k.get("heads", 1)


LAST_ORDINALS = []      # (process-wide launch ordinal, family, shape) of the launches kernel_breakdown timed last


def kernel_breakdown(model, sched, x, hint, n_steps=2):
    import torch
    ops = importlib.import_module("controlnet-pytorch_b200.ops")
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    rec = []
    orig = {k: getattr(ops, k) for k in ("conv", "groupnorm", "attention", "sched_step")}

    rtm = importlib.import_module("controlnet-pytorch_b200.runtime")
    count = rtm.lib().cnb_launch_count

    def timed(name, meta_fn, fn):
        def w(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            first = int(count())                    # ordinal of this call's first libcnb200 launch in the process
            e0.record()
            out = fn(*a, **k)
            e1.record()
            meta = meta_fn(out, a, k)
            meta["ordinal"] = first
            rec.append((name, meta, e0, e1))
            return out
        return w

    def conv_meta(out, a, k):
        x_, w_, kind, cout = a[0], a[1], a[2], a[3]
        B, H, W, ldi = x_.shape
        cin = k.get("cin") or (ldi - k.get("in_coff", 0))
        ntaps = w_.shape[-2] if w_.dim() == 3 else 4
        if k.get("phase") is not None:
            OH, OW = H, W
        else:
            OH, OW = ops.out_size(kind, H), ops.out_size(kind, W)
        fam = "conv_tc" if (cin % 4 == 0 and cin > 4 and cout % 16 == 0) else "conv_small"
        x2 = k.get("x2")
        cin2 = x2.shape[3] if x2 is not None else 0
        flops = 2.0 * B * OH * OW * (ntaps * cin + cin2) * cout
        res = k.get("residual")
        byts = (B * H * W * cin * x_.element_size() + out.shape[0] * out.shape[1] * out.shape[2] * cout * out.element_size()
                + (res.numel() * res.element_size() if res is not None else 0)
                + (x2.numel() * x2.element_size() if x2 is not None else 0) + w_.numel() * x_.element_size())
        shape = f"{kind or 'convT'} {cin}{'+%d' % cin2 if cin2 else ''}->{cout} @{H}x{W}"
        return dict(fam=fam, flops=flops, bytes=byts, shape=shape)

    ops.conv = timed("conv", conv_meta, orig["conv"])
    ops.groupnorm = timed("groupnorm", lambda o, a, k: dict(
        fam="groupnorm", flops=0.0, bytes=float(a[0].numel() * a[0].element_size() + o.numel() * o.element_size()),
        shape=f"C={a[0].shape[3]} @{a[0].shape[1]}x{a[0].shape[2]}"), orig["groupnorm"])
    ops.attention = timed("attention", lambda o, a, k: dict(
        fam="attention", bytes=float(a[0].numel() * a[0].element_size() + o.numel() * o.element_size()),
        flops=4.0 * a[0].shape[0] * (a[0].shape[1] * a[0].shape[2]) ** 2 * (a[0].shape[3] // 3),
        scores=float(a[0].shape[0]) * k_heads(a, k) * (a[0].shape[1] * a[0].shape[2]) ** 2,
        shape=f"L={a[0].shape[1] * a[0].shape[2]} E={a[0].shape[3] // 3} heads={k_heads(a, k)}"), orig["attention"])
    ops.sched_step = timed("sched_step", lambda o, a, k: dict(fam="sched_step", flops=0.0, bytes=16.0 * a[0].numel(),
                                                              shape="step"), orig["sched_step"])
    try:
        smp = S.DDPMSampler(model, sched, seed=3, use_graph=False)
        smp.sample_eager(x, hint, steps=1)          # warm caches
        rec.clear()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # the eager step is enqueued BEHIND a spinning kernel, so that every (event, launch, event) triple is already in
        # the stream when the GPU reaches it: the per-launch times are device time, not the host's launch gaps (which at
        # small per-rank batches, with N processes sharing the host, were longer than the kernels)
        torch.cuda.synchronize()
        torch.cuda._sleep(int(3e8))
        t0.record()
        smp.sample_eager(x, hint, steps=n_steps)
        t1.record()
        torch.cuda.synchronize()
    finally:
        for k_, v in orig.items():
            setattr(ops, k_, v)
    fams = {}
    LAST_ORDINALS.clear()
    for name, meta, e0, e1 in rec:
        LAST_ORDINALS.append((meta["ordinal"], meta["fam"], meta.get("shape", "?")))
        ms = e0.elapsed_time(e1)
        f = fams.setdefault(meta["fam"], dict(ms=0.0, flops=0.0, bytes=0.0, launches=0, shapes={}))
        f["ms"] += ms
        f["flops"] += meta["flops"]
        f["bytes"] += meta["bytes"]
        f["launches"] += 1
        sh = f["shapes"].setdefault(meta.get("shape", "?"), dict(ms=0.0, flops=0.0, bytes=0.0, scores=0.0, launches=0))
        sh["ms"] += ms
        sh["flops"] += meta["flops"]
        sh["bytes"] += meta["bytes"]
        sh["scores"] += meta.get("scores", 0.0)
        sh["launches"] += 1
    for f in fams.values():
        for k_ in ("ms", "flops", "bytes"):
            f[k_] /= n_steps
        f["launches"] //= n_steps
        for sh in f["shapes"].values():                     # per step, like the family totals they are compared with
            for k_ in ("ms", "flops", "bytes", "scores"):
                sh[k_] /= n_steps
            sh["launches"] = max(1, sh["launches"] // n_steps)
    return fams, t0.elapsed_time(t1) / n_steps


def _ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of named kernel instances, read from the
    committed summary of this round's `ncu --set full` captures (profiles/ncu_traffic.json: {"family|shape|batch": bytes});
    absent entries report null - nothing is hard-coded here."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return {k: float(v) for k, v in json.load(f).items() if not k.startswith("_")}
    except Exception:
        return {}


MUFU_PEAK_TSCORES = 148 * 16 * 1.965e9 / 1e12      # one ex2 per attention score, 16 MUFU lanes per SM per clock


def make_roofline(fams, step_ms, batch):
    """Roofline of the dominant kernel: the (family, layer shape) with the largest share of the step; achieved =
    algorithmic FLOPs (or bytes) per launch / average launch duration (CUDA events on the launching stream)."""
    pk = _peaks()
    traffic = _ncu_traffic()
    total = sum(f["ms"] for f in fams.values()) or 1.0
    dom = max(fams, key=lambda k_: fams[k_]["ms"])
    shape, sh = max(fams[dom]["shapes"].items(), key=lambda kv: kv[1]["ms"])
    n = sh["launches"]
    sec = sh["ms"] * 1e-3 / n                      # average launch duration
    rt = importlib.import_module("controlnet-pytorch_b200.runtime")
    attn_name = "attention kernel"
    if dom == "attention":                                  # shape label: "L=784 E=64 heads=4"
        kv = dict(t.split("=") for t in shape.split())
        attn_name = rt.attention_kernel_name(int(kv["L"]), int(kv["E"]) // int(kv["heads"]))
    kernel_names = {"conv_tc": "conv_tma_kernel (tcgen05 + TMA)", "conv_small": "conv_small_*_kernel",
                    "groupnorm": "groupnorm_*_kernel", "attention": attn_name, "sched_step": "sched_step_kernel"}
    if dom in ("conv_tc", "attention"):
        ach = sh["flops"] / n / sec / 1e12
        r = {"bound": "tensor", "achieved": round(ach, 2), "peak": pk["tf"], "unit": "TFLOP/s",
             "frac": round(ach / pk["tf"], 4)}
    else:
        ach = sh["bytes"] / n / sec / 1e9
        r = {"bound": "hbm", "achieved": round(ach, 1), "peak": pk["hbm"], "unit": "GB/s", "frac": round(ach / pk["hbm"], 4)}
    r.update({"traffic": traffic.get(f"{dom}|{shape}|{batch}"), "kernel": kernel_names.get(dom, dom), "shape": shape,
              "avg_launch_us": round(sec * 1e6, 1), "algorithmic_per_launch": {"flops": sh["flops"] / n, "bytes": sh["bytes"] / n},
              "share_of_step": round(sh["ms"] / sum(x["ms"] for f in fams.values() for x in f["shapes"].values()), 3),
              "family_share_of_step": round(fams[dom]["ms"] / total, 3),
              "peak_source": pk["src"] + (" (sustained bf16 dense)" if r["bound"] == "tensor" else " (copy)"),
              "launches_per_step": fams[dom]["launches"]})
    if dom == "attention":
        ts = sh["scores"] / n / sec / 1e12
        r["note"] = ("attention at head dim <= 64 is bound by the exponential (one MUFU ex2 per score), not by the tensor "
                     "pipe: see `xu` and DESIGN.md 4.2")
        r["xu"] = {"achieved": round(ts, 3), "peak": round(MUFU_PEAK_TSCORES, 3), "unit": "Tscore/s",
                   "frac": round(ts / MUFU_PEAK_TSCORES, 3)}

    # every family against its own roofline (BASELINE metric: conv tensor-pipe % of peak, fused norm kernels as a fraction
    # of HBM bandwidth): the TIME-WEIGHTED fraction of the whole family, its dominant shape, and its WORST shape among
    # those that take at least 2 % of the step
    def shape_line(fam_, shape_, sh_):
        sec_ = sh_["ms"] * 1e-3 / sh_["launches"]
        share = round(sh_["ms"] / total, 4)
        if fam_ in ("conv_tc", "attention"):
            a_ = sh_["flops"] / sh_["launches"] / sec_ / 1e12
            return {"shape": shape_, "bound": "tensor", "achieved": round(a_, 1), "peak": pk["tf"], "unit": "TFLOP/s",
                    "frac": round(a_ / pk["tf"], 3), "avg_launch_us": round(sec_ * 1e6, 1), "share_of_step": share,
                    "launches": sh_["launches"], "traffic": traffic.get(f"{fam_}|{shape_}|{batch}")}
        a_ = sh_["bytes"] / sh_["launches"] / sec_ / 1e9
        return {"shape": shape_, "bound": "hbm", "achieved": round(a_, 1), "peak": pk["hbm"], "unit": "GB/s",
                "frac": round(a_ / pk["hbm"], 3), "avg_launch_us": round(sec_ * 1e6, 1), "share_of_step": share,
                "launches": sh_["launches"], "traffic": traffic.get(f"{fam_}|{shape_}|{batch}")}
    by_family = {}
    for fam_ in ("conv_tc", "attention", "groupnorm"):
        if fam_ not in fams:
            continue
        f = fams[fam_]
        lines = [shape_line(fam_, s_, v_) for s_, v_ in sorted(f["shapes"].items(), key=lambda kv: -kv[1]["ms"])]
        big = [l_ for l_ in lines if l_["share_of_step"] >= 0.02] or lines[:1]
        if os.environ.get("CNB_BENCH_SHAPES"):               # full per-shape table, one JSON line per family
            with open(os.environ["CNB_BENCH_SHAPES"], "a") as fh:
                fh.write(json.dumps({"family": fam_, "batch": batch, "shapes": lines}) + "\n")
        s_ = f["ms"] * 1e-3
        if fam_ == "groupnorm":
            tw = {"achieved": round(f["bytes"] / s_ / 1e9, 1), "peak": pk["hbm"], "unit": "GB/s",
                  "frac": round(f["bytes"] / s_ / 1e9 / pk["hbm"], 3)}
        else:
            tw = {"achieved": round(f["flops"] / s_ / 1e12, 1), "peak": pk["tf"], "unit": "TFLOP/s",
                  "frac": round(f["flops"] / s_ / 1e12 / pk["tf"], 3)}
        by_family[fam_] = {"time_weighted": tw, "dominant": lines[0], "worst_ge_2pct": min(big, key=lambda l_: l_["frac"]),
                           "family_share_of_step": round(f["ms"] / total, 3), "launches_per_step": f["launches"]}
    r["by_family"] = by_family
    fam_out = {}
    for k_, v in fams.items():
        s_ = v["ms"] * 1e-3
        fam_out[k_] = {"ms": round(v["ms"], 3), "launches": v["launches"],
                       "TFLOP/s": round(v["flops"] / s_ / 1e12, 2) if v["flops"] else None,
                       "GB/s": round(v["bytes"] / s_ / 1e9, 1)}
    return r, fam_out


# ------------------------------------------------------------------------------------------------------------
# CPU / stock-PyTorch legs: the REFERENCE's own modules (baseline/_ref, oracle/install_ref.py); the oracle port only if
# no copy of the reference travelled to this box
# ------------------------------------------------------------------------------------------------------------
def _reference_path():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import install_ref
        return install_ref.ref_path()
    except Exception:
        return None


def reference_modules():
    """(ControlNet class, LinearNoiseScheduler class) of the UNMODIFIED reference, or None."""
    path = _reference_path()
    if path is None:
        return None
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k in ("models", "scheduler") or
             k.startswith("models.") or k.startswith("scheduler.")}
    sys.path.insert(0, path)
    try:
        cn = importlib.import_module("models.controlnet").ControlNet
        sc = importlib.import_module("scheduler.linear_noise_scheduler").LinearNoiseScheduler
        return cn, sc, path
    except Exception:
        return None
    finally:
        sys.path.remove(path)
        for k in [k for k in sys.modules if k in ("models", "scheduler") or k.startswith("models.") or
                  k.startswith("scheduler.")]:
            sys.modules.pop(k)
        sys.modules.update(saved)


def reference_problem(batch, device="cpu"):
    """The reference ControlNet + scheduler with the bench weights, and one timestep of tools/sample_ddpm_controlnet.py's
    loop (:43-51): eps = model(xt, t(1,), hint); xt = scheduler.sample_prev_timestep(xt, eps, t)[0]."""
    import torch
    syn = importlib.import_module("controlnet-pytorch_b200.utils.synthetic")
    mods = reference_modules()
    cfg = syn.MNIST_PARAMS
    g = torch.Generator().manual_seed(99)
    state = {"x": torch.randn(batch, 1, 28, 28, generator=g).to(device), "t": 999}
    hint = (torch.rand(batch, 1, 28, 28, generator=g) < 0.1).float().repeat(1, 3, 1, 1).to(device)
    if mods is not None:
        RefCN, RefSched, path = mods
        model = RefCN(cfg)
        model.load_state_dict(syn.det_state_dict(model.state_dict()))
        model = model.to(device).eval()
        sched = RefSched(**syn.MNIST_DIFFUSION)

        def step():
            with torch.no_grad():
                t = state["t"]
                eps = model(state["x"], torch.as_tensor(t).unsqueeze(0).to(device), hint)
                state["x"], _ = sched.sample_prev_timestep(state["x"], eps, torch.as_tensor(t).to(device))
                state["t"] = t - 1 if t > 1 else 999
        return step, "reference", "the reference's models/controlnet.py + scheduler/linear_noise_scheduler.py (%s)" % (
            "baseline/_ref" if path.endswith("_ref") else path)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cn_oracle as O
    cn = importlib.import_module("controlnet-pytorch_b200.models.controlnet")
    sd = syn.det_state_dict(cn.ControlNet(cfg).state_dict())
    so = O.SchedulerOracle(**syn.MNIST_DIFFUSION)

    def step():
        with torch.no_grad():
            t = state["t"]
            eps = O.controlnet_ddpm_forward(sd, cfg, state["x"], torch.tensor([t]), hint)
            z = torch.randn(state["x"].shape)
            state["x"], _ = so.sample_prev_timestep(state["x"], eps, t, z)
            state["t"] = t - 1 if t > 1 else 999
    return step, "port", "oracle/cn_oracle.py (the reference is absent on this box)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    batch = args.ref_batch
    step, kind, what = reference_problem(batch)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = batch / (dt * STEPS_PER_SAMPLE)
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 5), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "mnist_ddpm_controlnet_1000step", "global_batch": 1024, "batch_per_step": batch,
                       "timesteps_per_sample": STEPS_PER_SAMPLE,
                       "step": "one denoising timestep on the CPU (a bounded sample of the batch-1024 job: %d samples per "
                               "step, which saturates the host cores)" % batch},
            "cpu_baseline": {"value": round(val, 5), "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": f"{args.steps} timesteps x batch {batch}: {what}, torch CPU fp32"},
            "e2e": {"value": round(val, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def torch_cuda_reference(batch, dev, steps=3):
    """The reference's own modules on THIS GPU through stock PyTorch (cuDNN / cuBLAS; nn.MultiheadAttention takes its
    fused SDPA path in eval + no_grad): ms per timestep with TF32 off and on.  None if the reference did not travel."""
    import torch
    if reference_modules() is None:
        return None
    out = {"batch": batch, "what": "reference models/controlnet.py ControlNet + LinearNoiseScheduler.sample_prev_timestep "
                                   "on cuda through stock PyTorch %s" % torch.__version__}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.benchmark = True
            step, kind, _ = reference_problem(batch, device=dev)
            if kind != "reference":
                return None
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": round(ms, 2), "samples_per_s": round(batch / (ms * 1e-3 * STEPS_PER_SAMPLE), 3)}
            del step
            torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["error"] = f"{type(e).__name__}: {e}"[:200]
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return out


# ------------------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------------------
def _setup_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local, dev


def _timed_replay(smp, steps, warmup, world, dev):
    """W untimed replays, then exactly K timed ones between barrier + synchronize; max over ranks (ms per step)."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    smp.replay_steps(max(warmup, 3), reset=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    smp.replay_steps(steps, reset=False)
    e1.record()
    barrier()
    w1 = time.time()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps, w0, w1


def dump_outputs(smp, total, world, rank, out_dir):
    """Write the sampler's state after the last timed replay (x_{t-1} and the x0 prediction of that step, gathered over
    the ranks) as float32 .npy files; above DUMP_LIMIT_BYTES a fixed seeded sample of the batch rows is kept."""
    import numpy as np
    import torch
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    outs = {"xt": smp.xt, "x0": smp.x0}
    if world > 1:
        outs = {k: S.gather_shards(v, total) for k, v in outs.items()}
    if rank != 0:
        return
    row_bytes = sum(v[0].numel() * 4 for v in outs.values())
    keep = None
    if total * row_bytes > DUMP_LIMIT_BYTES:
        g = torch.Generator().manual_seed(0)
        keep = torch.randperm(total, generator=g)[: DUMP_LIMIT_BYTES // row_bytes].sort().values.to(smp.xt.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in outs.items():
        v = v if keep is None else v.index_select(0, keep)
        np.save(os.path.join(out_dir, name + ".npy"), v.float().cpu().numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    rt = importlib.import_module("controlnet-pytorch_b200.runtime")
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    # stdout carries exactly one JSON line: anything libraries print there (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    world, rank, local, dev = _setup_dist()
    rt.lib()
    rt.set_mode(args.mode)
    eng = importlib.import_module("controlnet-pytorch_b200.models._engine")
    # arithmetic type of the tensor-core mode: fp16 operands (fp32 accumulate) once GroupNorm / the activation stream emit fp16
    dtype_name = "f32" if args.mode == "fp32" else ("f16" if eng._F16_ENABLED else "tf32")
    G = args.batch                                           # GLOBAL batch of the job
    strong = args.scaling == "strong"
    per = 28 * 28
    # one job, identical at every N: hints and x_T are functions of the GLOBAL sample index
    cfg, model, sched, hint_host_all = build_problem(G if strong else G * world, dev)
    if strong:
        lo, hi = S.shard_bounds(G, world, rank)
    else:
        lo, hi = rank * G, (rank + 1) * G
    B = hi - lo                                              # this rank's shard
    total = G if strong else G * world
    smp = S.DDPMSampler(model, sched, seed=5, use_graph=True)
    hint = hint_host_all[lo:hi].to(dev)
    x_T = smp.draw_xT((B, 1, 28, 28), dev, elem_offset=lo * per)

    # ---- device-resident throughput: K graph replays of the captured timestep ---------------------------
    with torch.no_grad():
        smp._capture(x_T, hint, STEPS_PER_SAMPLE, lo * per)
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
        time.sleep(0.3)
    ms_per_step, w0, w1 = _timed_replay(smp, args.steps, args.warmup, world, dev)
    if rank == 0:
        clk.stop()
    if args.dump_outputs:
        dump_outputs(smp, total, world, rank, args.dump_outputs)
    value = total / (ms_per_step * 1e-3 * STEPS_PER_SAMPLE)
    launches = smp.launches_per_step * args.steps

    # ---- the other scaling mode as a second, labelled record (N > 1 only; at N = 1 they are the same job) -----
    other = None
    if world > 1 and not args.no_other:
        B2 = G if strong else S.shard_bounds(G, world, rank)[1] - S.shard_bounds(G, world, rank)[0]
        g2 = torch.Generator().manual_seed(4321 + rank)
        hint2 = (torch.rand(B2, 1, 28, 28, generator=g2) < 0.1).float().repeat(1, 3, 1, 1).to(dev)
        smp_o = S.DDPMSampler(model, sched, seed=7, use_graph=True)
        with torch.no_grad():
            smp_o._capture(smp_o.draw_xT((B2, 1, 28, 28), dev, elem_offset=rank * B2 * per), hint2, STEPS_PER_SAMPLE,
                           rank * B2 * per)
        ms2, _, _ = _timed_replay(smp_o, args.steps, args.warmup, world, dev)
        tot2 = B2 * world if strong else G
        other = {"scaling": "weak" if strong else "strong", "batch_per_gpu": B2, "global_batch": tot2,
                 "ms_per_step": round(ms2, 4), "value": round(tot2 / (ms2 * 1e-3 * STEPS_PER_SAMPLE), 3), "unit": UNIT}
        del smp_o, hint2

    # ---- end to end: the WHOLE job through the public API, host buffers in and out ------------------------------
    #   rank r: pinned-host x_T / hint shard -> device, all timesteps of its shard (graph replay), one NCCL all-gather of
    #   the final samples, rank 0 copies the gathered batch back to pinned host memory.  Everything is inside the timed
    #   region; the time is the max over ranks.  (tools/sample_ddpm_controlnet.py:21-51 as one sharded job.)
    k_e2e = args.e2e_steps
    gx = torch.Generator().manual_seed(777)
    xh_all = torch.randn(total, 1, 28, 28, generator=gx)
    xh = xh_all[lo:hi].contiguous().pin_memory()
    hh = hint_host_all[lo:hi].contiguous().pin_memory()
    out_h = torch.empty(total, 1, 28, 28).pin_memory() if rank == 0 else None
    smp2 = S.DDPMSampler(model, sched, seed=6, use_graph=True)
    xd = torch.empty((B, 1, 28, 28), device=dev)
    hd = torch.empty((B, 3, 28, 28), device=dev)

    def job():
        def hint_fn(a, b):
            hd.copy_(hh, non_blocking=True)
            return hd

        def x_fn(a, b):
            xd.copy_(xh, non_blocking=True)
            return xd
        full = S.sample_data_parallel(model, sched, (total, 1, 28, 28), hint_fn, steps=k_e2e, sampler=smp2, x_T_fn=x_fn,
                                      gather=True) if strong else smp2.sample(x_fn(lo, hi), hint_fn(lo, hi), steps=k_e2e,
                                                                              elem_offset=lo * per)[0]
        if rank == 0:
            out_h[: full.shape[0]].copy_(full, non_blocking=True)
        return full

    with torch.no_grad():
        job()                                                # capture + warm (also warms NCCL's all-gather)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        job()
        e1.record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
    ms2 = torch.tensor([max(e0.elapsed_time(e1), (t1 - t0) * 1e3)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_s = float(ms2.item()) * 1e-3 * (STEPS_PER_SAMPLE / k_e2e)
    e2e = {"value": round(total / e2e_s, 3), "unit": UNIT,
           "h2d_bytes_per_step": int((xh.numel() + hh.numel()) * 4 / k_e2e),
           "d2h_bytes_per_step": int(total * per * 4 / k_e2e) if rank == 0 else 0,
           "timesteps_run": k_e2e, "job_seconds": round(float(ms2.item()) * 1e-3, 3),
           "note": ("sampler.sample_data_parallel(global batch %d over %d rank(s), steps=%d): per rank pinned-host x_T + hint "
                    "shard H2D, %d timesteps (graph replay), %s, rank 0 D2H of all %d samples - all inside the timed "
                    "region, max over ranks%s" % (
                        total, world, k_e2e, k_e2e,
                        "one NCCL all_gather_into_tensor of the final samples" if (world > 1 and strong) else "no collective",
                        total, "" if k_e2e == STEPS_PER_SAMPLE else "; scaled to 1000 timesteps/sample"))}

    # ---- the reference TOOL's own loop on the drop-in classes (tools/sample_ddpm_controlnet.py:43-51), rank 0 -------------
    #   per step: model(xt, t(1,), hints) + scheduler.sample_prev_timestep(xt, eps, t) with the reference's default noise
    #   (torch.randn on the CPU generator + H2D copy, linear_noise_scheduler.py:71) - what a user gets by only swapping
    #   the imports (INTEGRATION.md 1), without the graph-replayed sampler
    e2e_dropin = None
    if rank == 0 and not args.no_dropin:
        k_d = max(5, min(args.steps, 20))
        with torch.no_grad():
            xt = xh.to(dev)
            for i in reversed(range(STEPS_PER_SAMPLE - 2, STEPS_PER_SAMPLE)):          # warm
                eps_ = model(xt, torch.as_tensor(i).unsqueeze(0).to(dev), hint)
                xt, _ = sched.sample_prev_timestep(xt, eps_, torch.as_tensor(i).to(dev))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in reversed(range(STEPS_PER_SAMPLE - 2 - k_d, STEPS_PER_SAMPLE - 2)):
                eps_ = model(xt, torch.as_tensor(i).unsqueeze(0).to(dev), hint)
                xt, _ = sched.sample_prev_timestep(xt, eps_, torch.as_tensor(i).to(dev))
            torch.cuda.synchronize()
            dt_d = (time.perf_counter() - t0) / k_d
        e2e_dropin = {"value": round(B / (dt_d * STEPS_PER_SAMPLE), 3), "unit": UNIT, "ms_per_step": round(dt_d * 1e3, 3),
                      "batch": B, "timesteps_run": k_d,
                      "note": "reference tool loop on the drop-in ControlNet + LinearNoiseScheduler of this rank's shard (eager "
                              "launches, CPU torch.randn + H2D per step, as tools/sample_ddpm_controlnet.py:43-51), wall clock"}

    # ---- roofline of the dominant kernel family + CPU / stock-PyTorch baselines (rank 0) ------------------------
    roofline, fam = None, None
    cpu_baseline, tcr = None, None
    if rank == 0:
        with torch.no_grad():
            fams, eager_ms = kernel_breakdown(model, sched, x_T, hint, n_steps=2)
        roofline, fam = make_roofline(fams, eager_ms, B)
        if world == 1 and not args.no_cpu:
            del smp2, smp
            torch.cuda.empty_cache()
            tcr = torch_cuda_reference(G, dev)
            torch.set_num_threads(os.cpu_count() or 1)
            nb, ns = args.cpu_batch, args.cpu_steps
            step, kind, what = reference_problem(nb)
            step()
            t0 = time.perf_counter()
            for _ in range(ns):
                step()
            dt = (time.perf_counter() - t0) / ns
            cpu_baseline = {"value": round(nb / (dt * STEPS_PER_SAMPLE), 5), "unit": UNIT,
                            "cores": torch.get_num_threads(), "kind": kind,
                            "sample": f"{ns} timesteps x batch {nb} of the same workload ({what}, torch CPU fp32, "
                                      f"{os.cpu_count()} host CPUs), {dt * 1e3:.0f} ms/timestep"}
    if world > 1:
        dist.barrier()
    if rank == 0:
        flop_step = FLOP_PER_SAMPLE_STEP - 0.178e9           # the t-independent hint block is cached, not run per step
        line = {"metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": dtype_name, "data": "synthetic",
                "config": {"workload": "mnist_ddpm_controlnet_1000step", "batch_per_gpu": B, "global_batch": total,
                           "timesteps_per_sample": STEPS_PER_SAMPLE,
                           "step": "one denoising timestep of this rank's shard: ControlNet eps + fused sample_prev_timestep "
                                   "(CUDA graph replay; control encoder, trained encoder + first mid, skip sums and t-embedding rows as parallel graph branches)",
                           "parallelism": f"dp{world}: global batch {total} sharded {B}/rank, no collective in the loop, one "
                                          "all-gather of the final samples (timed in e2e)",
                           "l2": "inputs larger than L2 at %d samples/rank: ~%.1f GB of activations per step vs 126 MB L2" % (
                               B, B * 2.98e6 * 4 * 2 / 1e9) if B >= 64 else
                                 "activations of a %d-sample shard (%.0f MB / step) do not exceed L2: the step is "
                                 "launch-latency bound, not bandwidth bound" % (B, B * 2.98e6 * 2 / 1e6),
                           "sample_steps_per_sec": round(total / (ms_per_step * 1e-3), 1),
                           "model_tflops": round(total * flop_step / (ms_per_step * 1e-3) / 1e12, 2),
                           "flop_per_sample_step": flop_step},
                "e2e": e2e, "e2e_dropin": e2e_dropin, "gpu_launches": int(launches), "launches_per_step": int(launches // args.steps),
                "roofline": roofline, "kernel_families": fam, "cpu_baseline": cpu_baseline,
                "torch_cuda_reference": tcr, "clocks": clk.summary(w0, w1)}
        if other is not None:
            line[other["scaling"]] = other
    if world > 1:
        dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json configs[] index + 1")
    ap.add_argument("--batch", type=int, default=None, help="GLOBAL batch (strong) / per-GPU batch (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--mode", default="f16", choices=["f16", "fp32", "tf32"])
    ap.add_argument("--e2e-steps", type=int, default=STEPS_PER_SAMPLE, help="timesteps of the end-to-end job (1000 = the job)")
    ap.add_argument("--ref-batch", type=int, default=64)
    ap.add_argument("--cpu-batch", type=int, default=64)
    ap.add_argument("--cpu-steps", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-other", action="store_true", help="skip the second (weak / strong) record at N > 1")
    ap.add_argument("--no-dropin", action="store_true", help="skip the reference-tool-loop measurement (e2e_dropin)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (config 2, --impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.config != 2 or args.impl != "b200"):
        ap.error("--dump-outputs is implemented for the config 2 run of --impl b200")
    if args.mode == "tf32":
        args.mode = "f16"
    if args.config != 2:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import bench_configs
        return bench_configs.run(args)
    if args.batch is None:
        args.batch = 1024
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
