"""DDIM against DDPM on the MNIST ControlNet (bench.py's model and hints), on one GPU:

  * step time of the captured step graph, CUDA events over --replays replays, the samplers alternated for --rounds
    rounds (DDPM, DDIM eta = 0, DDIM eta = 1), and launches_per_step of each;
  * wall time of the whole job through sampler.sample_data_parallel: DDIM at S = 20 and 50 against DDPM at 1000 steps,
    the first call (capture of the step graph included) and the second (replay only).  Hints go host -> device inside
    the timed call.

    python tests/ddim_bench.py --out DIR [--batches 1024,128] [--replays 200] [--rounds 3]

Writes DIR/ddim_bench.json with the card name and power limit read by nvidia-smi in the same run, and prints it.
Not collected by pytest (no test_ prefix).
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def step_times(torch, samplers, replays, rounds):
    """ms per replayed step of every sampler, one entry per round; the samplers take turns within a round."""
    res = {k: [] for k in samplers}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        for name, smp in samplers.items():
            smp.replay_steps(5, reset=True)
            torch.cuda.synchronize()
            e0.record()
            smp.replay_steps(replays, reset=False)
            e1.record()
            torch.cuda.synchronize()
            res[name].append(e0.elapsed_time(e1) / replays)
    return res


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
        raise SystemExit("ddim_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rt.lib()
    rt.set_mode(args.mode)
    report = {"gpu": gpu_info(), "mode": args.mode, "replays": args.replays, "rounds": args.rounds, "batches": []}
    for B in (int(b) for b in args.batches.split(",")):
        _, model, ddpm, hint_host = BN.build_problem(B, dev)
        hint = hint_host.to(dev)
        scheds = {"ddpm": ddpm, "ddim50_eta0": DDIM(ddpm, 50, eta=0.0), "ddim50_eta1": DDIM(ddpm, 50, eta=1.0)}
        smps = {k: S.DDPMSampler(model, s, seed=5) for k, s in scheds.items()}
        with torch.no_grad():
            for smp in smps.values():
                x_T = smp.draw_xT((B, 1, 28, 28), dev)
                smp._capture(x_T, hint, None, 0)
            times = step_times(torch, smps, args.replays, args.rounds)
        rec = {"batch": B, "step_ms": {k: [round(v, 4) for v in ts] for k, ts in times.items()},
               "step_ms_median": {k: round(statistics.median(ts), 4) for k, ts in times.items()},
               "launches_per_step": {k: smp.launches_per_step for k, smp in smps.items()}, "job": {}}
        del smps

        def hint_fn(lo, hi):
            return hint_host[lo:hi].to(dev, non_blocking=False)

        for name, sch, steps in (("ddim_S20_eta0", DDIM(ddpm, 20), 20), ("ddim_S50_eta0", DDIM(ddpm, 50), 50),
                                 ("ddpm_1000", ddpm, 1000)):
            smp = S.DDPMSampler(model, sch, seed=5)
            walls = []
            for _ in range(2):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = S.sample_data_parallel(model, sch, (B, 1, 28, 28), hint_fn, steps=steps, seed=5, sampler=smp)
                torch.cuda.synchronize()
                walls.append(time.perf_counter() - w0)
            rec["job"][name] = {"steps": steps, "first_call_s": round(walls[0], 4), "second_call_s": round(walls[1], 4),
                                "finite": bool(torch.isfinite(out).all())}
            del smp, out
        report["batches"].append(rec)
        del model
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "ddim_bench.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
