"""DPM-Solver++(2M) against DDIM on the MNIST ControlNet (bench.py's model and hints), on one GPU:

  * step time of the captured step graph, CUDA events over --replays replays, the samplers alternated for --rounds
    rounds (DDIM eta = 0, 2M "ode", 2M "sde", all at S = 20), and launches_per_step of each;
  * wall time of the whole job through sampler.sample_data_parallel: 2M at S = 10 and 20 against DDIM (eta = 0) at
    S = 20 and 50, the first call (capture of the step graph included) and the second (replay only).  Hints go
    host -> device inside the timed call;
  * distance from the ODE solution: rel-L2 of the final samples of DDIM (eta = 0) and 2M "ode" at S = 5, 10, 20 and 50
    against a DDIM S = 1000, eta = 0 run from the same x_T, at batch --err-batch, in fp32 and in f16 mode.  With the
    synthetic weights of bench.py this measures the solver's error, not image quality.

    python tests/dpm_solver_bench.py --out DIR [--batches 1024,128] [--replays 200] [--rounds 3] [--err-batch 128]

Writes DIR/dpm_solver_bench.json with the card name and power limit read by nvidia-smi in the same run, and prints it.
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
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from ddim_bench import gpu_info, step_times  # noqa: E402


def solver_errors(torch, S, model, ddpm, hint, B, dev, DDIM, DPM):
    """rel-L2 of the final samples of each solver against DDIM S = 1000, eta = 0 from the same x_T."""
    ref_smp = S.DDPMSampler(model, DDIM(ddpm, 1000), seed=5)
    x_T = ref_smp.draw_xT((B, 1, 28, 28), dev)
    ref, _ = ref_smp.sample(x_T, hint)
    del ref_smp
    out = {}
    for steps in (5, 10, 20, 50):
        for name, sch in (("ddim_eta0", DDIM(ddpm, steps)), ("dpm2m_ode", DPM(ddpm, steps))):
            got, _ = S.DDPMSampler(model, sch, seed=5).sample(x_T, hint)
            out.setdefault(name, {})[steps] = float((got - ref).norm() / ref.norm())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batches", default="1024,128")
    ap.add_argument("--replays", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--err-batch", type=int, default=128)
    ap.add_argument("--mode", default="f16", choices=["f16", "fp32"])
    args = ap.parse_args()
    import torch
    import bench as BN
    rt = importlib.import_module("controlnet-pytorch_b200.runtime")
    S = importlib.import_module("controlnet-pytorch_b200.sampler")
    DDIM = importlib.import_module("controlnet-pytorch_b200.scheduler.ddim_scheduler").DDIMScheduler
    DPM = importlib.import_module("controlnet-pytorch_b200.scheduler.dpm_solver_scheduler").DPMSolverMultistepScheduler
    if not torch.cuda.is_available():
        raise SystemExit("dpm_solver_bench.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    rt.lib()
    rt.set_mode(args.mode)
    report = {"gpu": gpu_info(), "mode": args.mode, "replays": args.replays, "rounds": args.rounds, "batches": []}
    for B in (int(b) for b in args.batches.split(",")):
        _, model, ddpm, hint_host = BN.build_problem(B, dev)
        hint = hint_host.to(dev)
        scheds = {"ddim20_eta0": DDIM(ddpm, 20), "dpm2m20_ode": DPM(ddpm, 20),
                  "dpm2m20_sde": DPM(ddpm, 20, variant="sde")}
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

        for name, sch in (("dpm2m_S10_ode", DPM(ddpm, 10)), ("dpm2m_S20_ode", DPM(ddpm, 20)),
                          ("ddim_S20_eta0", DDIM(ddpm, 20)), ("ddim_S50_eta0", DDIM(ddpm, 50))):
            smp = S.DDPMSampler(model, sch, seed=5)
            walls = []
            for _ in range(2):
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                out = S.sample_data_parallel(model, sch, (B, 1, 28, 28), hint_fn, seed=5, sampler=smp)
                torch.cuda.synchronize()
                walls.append(time.perf_counter() - w0)
            rec["job"][name] = {"steps": sch.num_inference_steps, "first_call_s": round(walls[0], 4),
                                "second_call_s": round(walls[1], 4), "finite": bool(torch.isfinite(out).all())}
            del smp, out
        report["batches"].append(rec)
        del model
        torch.cuda.empty_cache()
    B = args.err_batch
    _, model, ddpm, hint_host = BN.build_problem(B, dev)
    report["solver_error"] = {"note": "rel-L2 of the final samples against DDIM S = 1000, eta = 0 from the same x_T; "
                                      "synthetic weights, so this is the solver's error, not image quality",
                              "batch": B}
    with torch.no_grad():
        for mode in ("fp32", "f16"):
            rt.set_mode(mode)
            report["solver_error"][mode] = solver_errors(torch, S, model, ddpm, hint_host.to(dev), B, dev, DDIM, DPM)
    rt.set_mode(args.mode)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "dpm_solver_bench.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
