"""Image-to-image and inpainting on the MNIST ControlNet (bench.py's model and hints), on one GPU:

  * step time of the captured img2img step graph with and without a mask (DDIM S = 50, strength 0.5), CUDA events
    over --replays replays, the two alternated for --rounds rounds, and launches_per_step of each;
  * wall time of the whole job through sampler.sample_data_parallel, DDIM S = 50 at strength 0.5 and 1.0 with a
    mask, the first call (capture included) and the second (replay only);
  * cnb_inpaint_blend alone at 64, 128 and 192 Mi elements (C = 4, a broadcast soft mask, so every element is
    blended; Philox noise), CUDA events over 20 launches, against the 12 B + 4 / C B per element it moves.

    python tests/img2img_bench.py --out DIR [--batches 1024,128] [--replays 200] [--rounds 3]

Writes DIR/img2img_bench.json with the card name and power limit read by nvidia-smi in the same run, and prints it.
Not collected by pytest (no test_ prefix).
"""
import argparse
import importlib
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from ddim_bench import gpu_info, step_times   # noqa: E402


def blend_alone(torch, ops, dev, n_mi):
    C, HW = 4, 64 * 64
    B = n_mi * (1 << 20) // (C * HW)
    x = torch.randn((B, C, 64, 64), device=dev)
    x_ref = torch.randn_like(x)
    mask = torch.full((B, 1, 64, 64), 0.5, device=dev)
    levels = torch.tensor([[0.8, 0.6]], device=dev)
    for _ in range(3):
        ops.inpaint_blend(x, x_ref, mask, levels, seed=1, noise_step=1 << 40)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        ops.inpaint_blend(x, x_ref, mask, levels, seed=1, noise_step=1 << 40)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = x.numel() * (12 + 4 / C)
    return {"elements": x.numel(), "ms": round(ms, 4), "bytes": int(nbytes), "GB_per_s": round(nbytes / ms / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", default="1024,128")
    ap.add_argument("--replays", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--mode", default="f16", choices=["f16", "fp32"])
    args = ap.parse_args()
    import torch
    import bench as BN
    rt = importlib.import_module("controlnet-pytorch_b200.runtime")
    ops = importlib.import_module("controlnet-pytorch_b200.ops")
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    DDIM = importlib.import_module("controlnet-pytorch_b200.scheduler.ddim_scheduler").DDIMScheduler
    if not torch.cuda.is_available():
        raise SystemExit("img2img_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rt.lib()
    rt.set_mode(args.mode)
    report = {"gpu": gpu_info(), "mode": args.mode, "replays": args.replays, "rounds": args.rounds, "batches": []}
    for B in (int(b) for b in args.batches.split(",")):
        _, model, ddpm, hint_host = BN.build_problem(B, dev)
        hint = hint_host.to(dev)
        x_ref = torch.tanh(torch.randn((B, 1, 28, 28), generator=torch.Generator().manual_seed(0))).to(dev)
        mask = torch.zeros((B, 1, 28, 28), device=dev)
        mask[:, :, 7:21, 7:21] = 1.0
        sch = DDIM(ddpm, 50)
        smps = {"no_mask": S.DDPMSampler(model, sch, seed=5), "mask": S.DDPMSampler(model, sch, seed=5)}
        with torch.no_grad():
            smps["no_mask"].img2img(x_ref, hint, strength=0.5)
            smps["mask"].img2img(x_ref, hint, strength=0.5, mask=mask)
            times = step_times(torch, smps, args.replays, args.rounds)
        rec = {"batch": B, "step_ms": {k: [round(v, 4) for v in ts] for k, ts in times.items()},
               "step_ms_median": {k: round(statistics.median(ts), 4) for k, ts in times.items()},
               "launches_per_step": {k: smp.launches_per_step for k, smp in smps.items()}, "job": {}}
        del smps

        def hint_fn(lo, hi):
            return hint_host[lo:hi].to(dev, non_blocking=False)

        for strength in (0.5, 1.0):
            smp = S.DDPMSampler(model, sch, seed=5)
            walls = []
            for _ in range(2):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = S.sample_data_parallel(model, sch, (B, 1, 28, 28), hint_fn, seed=5, sampler=smp,
                                             x_ref_fn=lambda lo, hi: x_ref[lo:hi], mask_fn=lambda lo, hi: mask[lo:hi],
                                             strength=strength)
                torch.cuda.synchronize()
                walls.append(time.perf_counter() - w0)
            rec["job"][f"ddim_S50_strength{strength}"] = {
                "steps_run": smp._nsteps, "first_call_s": round(walls[0], 4), "second_call_s": round(walls[1], 4),
                "finite": bool(torch.isfinite(out).all())}
            del smp, out
        report["batches"].append(rec)
        del model
        torch.cuda.empty_cache()
    report["blend_alone"] = [blend_alone(torch, ops, dev, n) for n in (64, 128, 192)]
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "img2img_bench.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
