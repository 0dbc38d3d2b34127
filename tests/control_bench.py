"""Control strength on the MNIST ControlNet (bench.py's model and hints), on one GPU:

  * step time of three captured DDIM (S = 50) step graphs: the default ControlNet step, the guided step
    (ControlOptions(guidance=3)) and the plain U-Net step (ControlOptions(scale=0), which sends every step to the
    frozen U-Net alone), CUDA events over --replays replays, the three alternated for --rounds rounds;
  * launches per step of each, and the peak memory the capture and replays of each add to what was allocated before
    (the weight caches of all three are built first, so none of them is counted);
  * wall time of a DDIM S = 50 job through sampler.sample_data_parallel with the control window (0, 0.5) against the
    default job, the second call of each (the step graphs already captured).

    python tests/control_bench.py --out DIR [--batches 1024,128] [--replays 200] [--rounds 3]

Writes DIR/control_bench.json with the card name and power limit read by nvidia-smi in the same run, and prints it.
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
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    DDIM = importlib.import_module("controlnet-pytorch_b200.scheduler.ddim_scheduler").DDIMScheduler
    if not torch.cuda.is_available():
        raise SystemExit("control_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rt.lib()
    rt.set_mode(args.mode)
    report = {"gpu": gpu_info(), "mode": args.mode, "replays": args.replays, "rounds": args.rounds,
              "celebhq_ldm_B256": "not measured", "batches": []}
    variants = {"controlnet": None, "guided_w3": S.ControlOptions(guidance=3.0),
                "plain_unet": S.ControlOptions(scale=0.0)}
    for B in (int(b) for b in args.batches.split(",")):
        _, model, ddpm, hint_host = BN.build_problem(B, dev)
        hint = hint_host.to(dev)
        sch = DDIM(ddpm, 50)
        smps, peak, launches = {}, {}, {}
        with torch.no_grad():
            for ctl in variants.values():                 # weight caches built before any memory is counted
                S.DDPMSampler(model, sch, seed=5).sample(hint.new_zeros((B, 1, 28, 28)), hint, control=ctl)
            torch.cuda.synchronize()
            for name, ctl in variants.items():
                smp = S.DDPMSampler(model, sch, seed=5)
                x_T = smp.draw_xT((B, 1, 28, 28), dev)
                torch.cuda.synchronize()
                before = torch.cuda.memory_allocated(dev)
                torch.cuda.reset_peak_memory_stats(dev)
                # the capture and five replays alone, without the output copies of a whole sample() call
                smp._prepare(x_T, hint, 0, smp._plan(x_T, hint, None, 0, control=ctl))
                smp.replay_steps(5, reset=True)
                torch.cuda.synchronize()
                peak[name] = torch.cuda.max_memory_allocated(dev) - before
                launches[name] = smp.launches_per_step if smp._keep is None or smp._keep[0] else \
                    smp.plain_launches_per_step
                smps[name] = smp
            times = step_times(torch, smps, args.replays, args.rounds)
        rec = {"batch": B, "step_ms": {k: [round(v, 4) for v in ts] for k, ts in times.items()},
               "step_ms_median": {k: round(statistics.median(ts), 4) for k, ts in times.items()},
               "launches_per_step": launches, "peak_mem_added_MiB": {k: round(v / 2 ** 20, 1) for k, v in peak.items()},
               "job": {}}
        del smps

        def hint_fn(lo, hi):
            return hint_host[lo:hi].to(dev, non_blocking=False)

        for name, ctl in (("default", None), ("window_0_0.5", S.ControlOptions(start=0.0, end=0.5))):
            smp = S.DDPMSampler(model, sch, seed=5)
            walls = []
            for _ in range(2):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = S.sample_data_parallel(model, sch, (B, 1, 28, 28), hint_fn, seed=5, sampler=smp, control=ctl)
                torch.cuda.synchronize()
                walls.append(time.perf_counter() - w0)
            rec["job"][f"ddim_S50_{name}"] = {"first_call_s": round(walls[0], 4), "second_call_s": round(walls[1], 4),
                                              "finite": bool(torch.isfinite(out).all())}
            del smp, out
        report["batches"].append(rec)
        del model
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "control_bench.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
