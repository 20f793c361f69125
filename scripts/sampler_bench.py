#!/usr/bin/env python
"""Time per step and per image of each sampler at bench.py's default workload shapes (configs[1]: SD1.5-shape UNet,
512x512, 1 image, CFG 7.5, fp16, CUDA-graph replay).

    python scripts/sampler_bench.py --out DIR [--reps 3]

For LMS and the Euler, Euler-ancestral and DPM-Solver++(2M) samplers it reports
  * ms per step: CUDA-event time over graph replays of whole schedules;
  * ms per image at that sampler's step count (30 for LMS / Euler / Euler a, 20 for DPM++ 2M -- common settings, not
    a statement about image quality per step);
  * native launches per step (PwWSampler.native_launches_per_step);
  * the step tail's kernel time, from a torch.profiler run of its own: the kernels one eager step launches that a bare
    UNet forward on a ready fp16 channels-last input does not (the scale / cat / cast / layout copy before the UNet and
    the CFG combine / update after it), counted per kernel name;
  * the card's name and power limit, read in the same run.
Writes DIR/sampler_bench.json and prints it.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import paint_with_words_sd_b200 as P  # noqa: E402
from paint_with_words_sd_b200.pipeline import PwWSampler  # noqa: E402
from paint_with_words_sd_b200.scheduler import (DPMSolverMultistepScheduler, EulerAncestralDiscreteScheduler,  # noqa: E402
                                                EulerDiscreteScheduler, LMSDiscreteScheduler)
from paint_with_words_sd_b200.synthetic import RandomTextEncoder, SimpleWordTokenizer  # noqa: E402
from paint_with_words_sd_b200.unet import build_unet  # noqa: E402

SD = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
SAMPLERS = [("lms", LMSDiscreteScheduler, 30), ("euler", EulerDiscreteScheduler, 30),
            ("euler_a", EulerAncestralDiscreteScheduler, 30), ("dpmpp_2m", DPMSolverMultistepScheduler, 20)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # noqa: BLE001
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})"}


def kernel_counts(fn, reps):
    """{kernel name: (launches per call, total us per call)} of `fn` under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    agg = collections.defaultdict(lambda: [0, 0.0])
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
            agg[ev.name][0] += 1
            agg[ev.name][1] += ev.device_time_total
    return {k: (n / reps, t / reps) for k, (n, t) in agg.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3, help="whole schedules timed per sampler")
    ap.add_argument("--out", required=True, help="directory for sampler_bench.json")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sampler_bench.py measures on the GPU"
    dev = torch.device("cuda", 0)
    cfg = bench.CONFIGS[2]
    unet = build_unet(bench.unet_config(cfg["unet"]), seed=0, dtype=torch.float16, device=dev)
    P.patch_unet(unet)
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(cfg["text_dim"]).to(dev)
    wf = bench.make_weight_function(cfg["coef"])
    result = {"workload": f"{cfg['tag']}: {cfg['what']} (the LMS row is bench.py's workload)", "card": card(),
              "samplers": {}}
    for name, cls, steps in SAMPLERS:
        sch = cls(**SD)
        sch.set_timesteps(steps)
        conds, unconds, lat0, extra = bench.build_images(cfg, dev, [0], tok, enc, sch)
        with torch.no_grad():
            s = PwWSampler(unet, sch, conds, unconds, lat0, wf, bench.GUIDANCE, extra_input=extra, use_graph=True,
                           noise_seeds=[0])
            s.run()                                               # capture + warm-up schedule
            times = []
            for _ in range(args.reps):
                s.restart(lat0)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                s.run()
                b.record()
                torch.cuda.synchronize()
                times.append(a.elapsed_time(b))
            assert torch.isfinite(s.latents).all()
            ms_image = sorted(times)[len(times) // 2]
            # step tail from an eager profile: kernels of one step minus those of a bare UNet forward
            e = PwWSampler(unet, sch, conds, unconds, lat0, wf, bench.GUIDANCE, extra_input=extra, use_graph=False,
                           noise_seeds=[0])

            def eager_step():
                e.restart(lat0)
                e.step()
            x_in = torch.zeros((2,) + tuple(s._unet_in.shape[1:]) if hasattr(s, "_unet_in") else
                               (2, unet.in_channels, lat0.shape[2], lat0.shape[3]), dtype=torch.float16, device=dev)
            x_in = x_in.contiguous(memory_format=torch.channels_last)
            e.step(); e.restart(lat0)                              # the K/V cache and workspaces are set up
            t_in = torch.tensor([500.0], device=dev)
            bare = lambda: unet(x_in, t_in, encoder_hidden_states=e._ctx)   # noqa: E731
            bare(); eager_step()
            ks, ku = kernel_counts(eager_step, 5), kernel_counts(bare, 5)
            tail = {}
            for k, (n, t) in ks.items():
                nu = ku.get(k, (0.0, 0.0))[0]
                if n - nu > 0.5:
                    tail[k[:90]] = {"launches": round(n - nu, 2), "us": round(t / n * (n - nu), 2)}
        result["samplers"][name] = {
            "steps": steps, "ms_per_image": round(ms_image, 3), "ms_per_step": round(ms_image / steps, 4),
            "native_launches_per_step": s.native_launches_per_step,
            "step_tail_kernel_us": round(sum(v["us"] for v in tail.values()), 2),
            "step_tail_launches": round(sum(v["launches"] for v in tail.values()), 2), "step_tail_kernels": tail,
            "schedule_ms_all_reps": [round(t, 3) for t in times]}
        print(name, json.dumps({k: v for k, v in result["samplers"][name].items() if k != "step_tail_kernels"}),
              flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sampler_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
