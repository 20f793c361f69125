#!/usr/bin/env python
"""bench.py -- UNet steps/sec of the Paint-with-Words denoising loop on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] -- aurora_1 colour map, SD1.5-shaped UNet (seeded random
weights; no checkpoints exist offline), 512x512, 30-step LMS schedule, CFG 7.5, fp16, runner.py's weight
function 0.4*w*log(1+sigma)*qk.max().  One "step" = one denoising step of one image: the cond+uncond UNet
forwards (run here as one batch-2 forward), the CFG combine and the LMS update (paint_with_words.py:471-506).
N GPUs = N independent images, one per rank (weak scaling); weights are replicated with one NCCL broadcast at
init and nothing is exchanged per step.

One JSON line on stdout (rank 0):
  value      steps/s over all ranks, inputs resident in HBM, CUDA-graph replay, CUDA-event time, max over ranks
  e2e        the same steps driven from HOST buffers: every step H2D-copies latents, text context and the four
             weight maps from pinned memory, runs the step, and D2H-reads the new latents (sync per step)
  roofline   the dominant kernel of the path -- pww_xattn_fused_f16 (ONE launch: statistic + bias + softmax + PV) at
             N=4096 (C=320, 8 heads) -- timed live with CUDA events as a graph of back-to-back launches over rotating
             buffers larger than L2, at the batch this workload launches it with (cond+uncond); `batched` repeats it
             with 16 images per launch; `dense_pair` times the round-1 two-launch path on the same inputs
  reference_gpu_eager   comparison only: the reference's loop and inj_forward op sequence as eager fp16 PyTorch on this GPU
  cpu_baseline  the oracle port of the reference loop on this box's host cores (rank 0, N=1 only), bounded sample
--impl reference: only that CPU loop (the reference is pure Python/torch; its CPU path is what is timed).
--dump-outputs DIR: after the timed steps, write the latents the last timed step left (what PwWSampler.run returns)
as DIR/latents.npy (float32; DIR/latents_rank<r>.npy per rank when N > 1).  Inputs are seeded, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from paint_with_words_sd_b200 import sharding  # noqa: E402
from paint_with_words_sd_b200.conditioning import _encode_text_color_inputs  # noqa: E402
from paint_with_words_sd_b200.scheduler import LMSDiscreteScheduler  # noqa: E402
from paint_with_words_sd_b200.synthetic import RandomTextEncoder, SimpleWordTokenizer  # noqa: E402
from paint_with_words_sd_b200.unet import UNetConfig, build_unet  # noqa: E402
from tests.fixtures import SETTINGS, color_map_image  # noqa: E402

METRIC = "unet_steps_per_sec_512sq_cfg"
UNIT = "steps/s"
SIZE, SCHEDULE_STEPS, GUIDANCE = 512, 30, 7.5


def weight_function(w, sigma, qk):          # runner.py:104
    return 0.4 * w * math.log(1 + sigma) * qk.max()


def workload_config(n_gpus: int, cfg_id: int = 2, images_per_gpu: int = 1) -> dict:
    cfg = CONFIGS[cfg_id]
    size = cfg["size"]
    total = cfg["total_images"] or n_gpus
    return {"workload": f"{cfg['tag']}: {cfg['what']}; weight_function {cfg['coef']}*w*log(1+sigma)*qk.max()",
            "images_per_gpu": images_per_gpu, "unet_batch": 2 * images_per_gpu, "global_images": total,
            "latent": [4, size // 8, size // 8], "tokens": 77,
            "parallelism": f"image-sharded x{n_gpus}, weights replicated (1 broadcast), no per-step collective",
            "l2_policy": "inputs larger than L2: each step streams the fp16 UNet weights (1.7 GB; L2 is 126 MB)"}


# BASELINE.json configs (1-based, BASELINE.md section 4 numbering).  The driver runs the default (2 = configs[1], the
# configuration the metric is quoted on); `--config N` measures the others with the same machinery
# (scripts/bench_configs.sh fills BASELINE.md's table from them).  "weak": one image per GPU; "strong": a fixed set of
# images sharded over the GPUs (image i -> rank i mod G).
CONFIGS = {
    1: dict(tag="configs[0]", what="runner.py cat/dog colour map, SD1.5-shape UNet 256x256, 10-step LMS, CFG 7.5 "
                                  "(the reference runs this one on the CPU)",
            unet="sd15", size=256, sched_steps=10, maps=["cat_dog"], coef=0.4, text_dim=768, total_images=None),
    2: dict(tag="configs[1]", what="aurora_1 colour map, SD1.5-shape UNet 512x512, 30-step LMS, CFG 7.5, fp16",
            unet="sd15", size=512, sched_steps=30, maps=["aurora"], coef=0.4, text_dim=768, total_images=None),
    3: dict(tag="configs[2]", what="4 colour maps x 2 seeds = 8 images (16 forward items), SD1.5-shape 512x512, 30 steps, "
                                  "image-sharded",
            unet="sd15", size=512, sched_steps=30, maps=["aurora", "cat_dog", "aurora/flip", "cat_dog/flip"], coef=0.4,
            text_dim=768, total_images=8),
    4: dict(tag="configs[3]", what="paint_with_words_inpaint: SD1.5-inpainting-shape UNet (9 input channels) 512x512, "
                                  "moon_mask, 50 steps, weight 0.15",
            unet="sd15_inpaint", size=512, sched_steps=50, maps=["aurora"], coef=0.15, text_dim=768, total_images=None,
            inpaint=True),
    5: dict(tag="configs[4]", what="SD2.1-shape UNet (d=64, ctx 1024, linear proj) 768x768, 50 steps, 5-region colour "
                                  "context with regional seeding, 8 images (16 forward items), image-sharded",
            unet="sd21", size=768, sched_steps=50, maps=["aurora"], coef=0.4, text_dim=1024, total_images=8,
            region_seeds=True),
}


def make_weight_function(coef: float):
    def wf(w, sigma, qk):                   # runner.py:94,104 (0.4) / runner_inpaint.py:72,87 (0.15)
        return coef * w * math.log(1 + sigma) * qk.max()
    return wf


def unet_config(name: str):
    return {"sd15": UNetConfig.sd15, "sd15_inpaint": UNetConfig.sd15_inpaint, "sd21": UNetConfig.sd21}[name]()


def build_images(cfg: dict, device, image_ids, tok, enc, sch):
    """Conditioning + initial latents of the images this rank owns.  Returns (conds, unconds, latents [m,4,h,w],
    extra_input or None)."""
    from PIL import Image as _Image
    from paint_with_words_sd_b200.pipeline import initial_latents
    size = cfg["size"]
    conds, unconds, lats, extras = [], [], [], []
    for i in image_ids:
        spec = cfg["maps"][i % len(cfg["maps"])]
        name, flip = (spec.split("/") + [""])[:2]
        seed = i // len(cfg["maps"]) if cfg["total_images"] else i
        img = color_map_image(name, size)
        if flip:
            img = img.transpose(_Image.FLIP_LEFT_RIGHT)
        ctx = dict(SETTINGS[name]["ctx"])
        if cfg.get("region_seeds"):                      # runner.py:61-72 style: ",seed" on one region
            key = list(ctx.keys())[-1]
            ctx[key] = ctx[key] + ",2077"
        extra_seeds, separated, cond, uncond = _encode_text_color_inputs(enc, tok, device, img, ctx,
                                                                         SETTINGS[name]["prompt"], "")
        lat = initial_latents((1, 4, size // 8, size // 8), seed, extra_seeds, separated) * sch.init_noise_sigma
        conds.append(cond); unconds.append(uncond); lats.append(lat)
        if cfg.get("inpaint"):                           # paint_with_words_inpaint.py:230-250: cat[latents, mask, masked latents]
            import torch.nn.functional as F_
            from tests.fixtures import moon_mask_image
            m = torch.from_numpy(np.array(moon_mask_image(size)).astype(np.float32) / 255.0)[None, None]
            m = F_.interpolate((m > 0.5).float(), size=(size // 8, size // 8), mode="nearest")
            masked = torch.randn(1, 4, size // 8, size // 8, generator=torch.manual_seed(1000 + seed)) * 0.18215 * (1 - m)
            extras.append(torch.cat([m, masked], 1))
    extra = torch.cat(extras, 0).to(device) if extras else None
    return conds, unconds, torch.cat(lats, 0).to(device), extra


def ncu_traffic(key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of the
    one-launch kernel (profiles/r02_xattn_traffic.json, written by scripts/ncu_summary.py); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_xattn_traffic.json")) as f:
            return float(json.load(f)[key]["traffic_bytes"])
    except Exception:
        return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the reference loop)
# ------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Threads the CPU arm may really use: the affinity mask, capped by the cgroup CPU quota (a container that shows 128
    logical CPUs but is allowed 16 cores' worth of time runs a 128-thread GEMM far slower than a 16-thread one)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2: "<quota> <period>" or "max <period>"
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(math.ceil(int(quota) / int(period)))))
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                quota = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = int(f.read())
            if quota > 0:
                n = min(n, max(1, int(math.ceil(quota / period))))
        except Exception:
            pass
    return max(1, n)


def cpu_reference(max_timed_steps: int, warmup: int, budget_s: float):
    """Timed oracle loop on the host cores: same UNet weights (seed 0, fp32), same conditioning, same schedule."""
    from oracle import loop as oracle_loop
    # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every host core it CAN use, whatever launched it
    torch.set_num_threads(host_threads())
    torch.manual_seed(0)
    unet = build_unet(UNetConfig.sd15(), seed=0, dtype=torch.float32, device="cpu")
    oracle_loop.patch_with_oracle(unet)
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(768)
    s = SETTINGS["aurora"]
    _, _, cond, uncond = _encode_text_color_inputs(enc, tok, "cpu", color_map_image("aurora", SIZE), dict(s["ctx"]),
                                                   s["prompt"], "")
    sch = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    sch.set_timesteps(SCHEDULE_STEPS)
    lat = torch.randn(1, 4, SIZE // 8, SIZE // 8, generator=torch.manual_seed(0)) * sch.init_noise_sigma
    stamps = [time.perf_counter()]
    state = {"n": 0}

    class _Stop(Exception):
        pass

    def on_step(i):
        stamps.append(time.perf_counter())
        done = len(stamps) - 1
        per = (stamps[-1] - stamps[0]) / done
        timed = done - warmup
        if timed >= max_timed_steps or (timed >= 1 and (stamps[-1] - stamps[0]) + per > budget_s):
            raise _Stop

    try:
        oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat, weight_function, GUIDANCE, on_step=on_step)
    except _Stop:
        pass
    done = len(stamps) - 1
    w = min(warmup, done - 1)
    timed = done - w
    dt = stamps[-1] - stamps[w]
    return {"steps": timed, "warmup": w, "seconds": dt, "steps_per_s": timed / dt, "cores": torch.get_num_threads()}


def run_reference_arm(args, rank: int):
    if rank != 0:
        return
    r = cpu_reference(max_timed_steps=max(1, args.steps), warmup=min(args.warmup, 1), budget_s=150.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["steps_per_s"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": 1e3 / r["steps_per_s"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": r["steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                             "sample": f"{r['steps']} denoising steps (2 UNet forwards each, oracle port of "
                                       f"inj_forward patched in) of the same 512x512 workload, fp32, "
                                       f"{r['seconds']:.1f} s; bounded to ~150 s"},
            "e2e": {"value": r["steps_per_s"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------
# kernel roofline (live, CUDA events)
# ------------------------------------------------------------------------------------------------
def region_weight_map(N: int, T: int = 77, regions: int = 5, seed: int = 0) -> torch.Tensor:
    """A dense [N, T] fp32 weight map with the structure the reference's builder produces (paint_with_words.py:247-276):
    `regions` painted regions, each a contiguous band of pixels with its own strength and soft edge, each attached to
    1-3 prompt tokens.  Used where no golden map of that resolution exists (kernel timing only)."""
    g = torch.Generator().manual_seed(seed)
    w = torch.zeros(N, T)
    edges = torch.linspace(0, N, regions + 1).long().tolist()
    tok = 5
    for r in range(regions):
        col = torch.zeros(N)
        lo, hi = edges[r], edges[r + 1]
        col[lo:hi] = float(torch.rand(1, generator=g) * 1.8 + 0.2)
        if hi - lo > 8:
            col[lo:lo + 4] *= torch.linspace(0.2, 0.8, 4)      # bilinear-resize style soft edge
        ntok = 1 + r % 3
        for t in range(tok, tok + ntok):
            w[:, t] = col
        tok += ntok + 1
    return w


def golden_weight_map(N: int):
    """The real aurora_1 map at this resolution when the golden fixtures hold it (SD1.5 512x512 levels), else None."""
    key = {4096: "aurora_512_w8", 1024: "aurora_512_w16", 256: "aurora_512_w32", 64: "aurora_512_w64"}.get(N)
    if key is None:
        return None
    return torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "mask_builder.npz"))[key])


def xattn_roofline(device, B: int, biased: int, N=4096, H=8, D=40, T=77, target_mb=192, iters=64, reps=5,
                   dense_pair: bool = False):
    """Average duration of ONE pww_xattn_fused_f16 launch over a CUDA graph of back-to-back launches that cycle through
    enough distinct buffer sets to exceed L2 (so Q / packed maps / O really come from / go to HBM).  Maps: the golden
    aurora_1 map of that resolution (or a region-structured synthetic one), packed by conditioning.pack_weight_map.
    dense_pair=True additionally times pww_xattn_stats_f16 + pww_xattn_fwd_f16 on the dense fp32 form of the same maps."""
    from paint_with_words_sd_b200 import _native
    from paint_with_words_sd_b200.conditioning import pack_weight_map
    L = _native.lib()
    C = H * D
    per_set = B * N * C * 2 * 2 + biased * N * 64
    nsets = max(2, int(math.ceil(target_mb * 1e6 / per_set)))
    g = torch.Generator(device="cpu").manual_seed(0)
    qs = [(torch.randn(B, N, C, generator=g) * 0.5).half().to(device) for _ in range(nsets)]
    outs = [torch.empty(B, N, C, dtype=torch.float16, device=device) for _ in range(nsets)]
    k = (torch.randn(B, T, C, generator=g) * 0.5).half().to(device)
    v = (torch.randn(B, T, C, generator=g) * 0.5).half().to(device)
    base = golden_weight_map(N)
    if base is None:
        base = region_weight_map(N, T)
    dense = torch.stack([base] * max(1, biased), 0).contiguous()
    mp0, ci0 = pack_weight_map(dense)
    mps = [mp0.to(device).clone() for _ in range(nsets)]
    ci = ci0.to(device)
    idx = torch.tensor(list(range(biased)) + [-1] * (B - biased), dtype=torch.int32, device=device)
    stats = torch.zeros(B, dtype=torch.float32, device=device)
    gs = torch.full((1,), 0.4 * math.log(1 + 7.0), dtype=torch.float32, device=device)
    fws = torch.zeros(L.pww_xattn_fused_workspace_bytes(), dtype=torch.uint8, device=device)
    scale = D ** -0.5

    def launch_fused(i, stream):
        q, o, mp = qs[i % nsets], outs[i % nsets], mps[i % nsets]
        rc = L.pww_xattn_fused_f16(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B, H, N, T, D, q.stride(0),
                                   q.stride(1), k.stride(0), k.stride(1), o.stride(0), o.stride(1),
                                   mp.data_ptr() if biased else None, mp.stride(0), mp.shape[0],
                                   ci.data_ptr() if biased else None, idx.data_ptr() if biased else None, 0,
                                   gs.data_ptr(), scale, stats.data_ptr(), fws.data_ptr(), fws.numel(), stream)
        _native.check(rc, "fused")

    def timed(fn):
        s = torch.cuda.Stream(device=device)
        with torch.cuda.stream(s):
            for i in range(3):
                fn(i, s.cuda_stream)
        s.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            for i in range(iters):
                fn(i, torch.cuda.current_stream(device).cuda_stream)
        best = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(device)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize(device)
            best.append(e0.elapsed_time(e1) * 1e3 / iters)     # us per launch
        return float(np.median(best))

    t_fused = timed(launch_fused)
    qkvo = B * (2 * N * C * 2 + 2 * T * C * 2)
    res = {"us_op": t_fused, "alg_bytes": qkvo + biased * (N * 64 + 80), "alg_bytes_dense_map": qkvo + biased * N * T * 4,
           "sets": nsets, "iters": iters}
    if dense_pair and biased:
        ws = [dense.to(device).clone() for _ in range(min(nsets, 8))]
        ws_bytes = L.pww_xattn_workspace_bytes(B, H, N, T, D)
        work = torch.zeros(ws_bytes, dtype=torch.uint8, device=device)

        def launch_stats(i, stream):
            q = qs[i % nsets]
            rc = L.pww_xattn_stats_f16(q.data_ptr(), k.data_ptr(), B, H, N, T, D, q.stride(0), q.stride(1), k.stride(0),
                                       k.stride(1), 0, idx.data_ptr(), stats.data_ptr(), work.data_ptr(), ws_bytes, stream)
            _native.check(rc, "stats")

        def launch_fwd(i, stream):
            q, o, w = qs[i % nsets], outs[i % nsets], ws[i % len(ws)]
            rc = L.pww_xattn_fwd_f16(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), B, H, N, T, D, q.stride(0),
                                     q.stride(1), k.stride(0), k.stride(1), o.stride(0), o.stride(1), w.data_ptr(),
                                     w.stride(0), idx.data_ptr(), stats.data_ptr(), gs.data_ptr(), scale, stream)
            _native.check(rc, "fwd")

        res["us_dense_stats"], res["us_dense_fwd"] = timed(launch_stats), timed(launch_fwd)
    return res


def eager_torch_xattn_us(device, N=4096, H=8, D=40, T=77, iters=20, dtype=torch.float16):
    """Comparison only (SURVEY 8d: "time the reference path on the B200"): the op sequence of the reference's
    inj_forward between to_q/to_k/to_v and to_out (paint_with_words.py:83-118) as eager PyTorch on this device, for
    one conditional call (bias = 0.4*w*log(1+sigma)*qk.max()) plus one unconditional call -- the work one B=2 launch
    pair (pww_xattn_stats_f16 + pww_xattn_fwd_f16) of this repo does.  Returns microseconds per cond+uncond pair."""
    C = H * D
    g = torch.Generator(device="cpu").manual_seed(0)
    q = (torch.randn(1, N, C, generator=g) * 0.5).to(device=device, dtype=dtype)
    k = (torch.randn(1, T, C, generator=g) * 0.5).to(device=device, dtype=dtype)
    v = (torch.randn(1, T, C, generator=g) * 0.5).to(device=device, dtype=dtype)
    w = (torch.rand(N, T, generator=g) > 0.8).float().to(device)
    sigma = torch.tensor(7.0)
    scale = D ** -0.5

    def heads_to_batch(x):
        b, n, _ = x.shape
        return x.reshape(b, n, H, D).permute(0, 2, 1, 3).reshape(b * H, n, D)

    def call(biased):
        qh, kh, vh = heads_to_batch(q), heads_to_batch(k), heads_to_batch(v)
        s = torch.matmul(qh, kh.transpose(-1, -2))
        bias = 0.4 * w * math.log(1 + float(sigma)) * s.max() if biased else 0.0
        p = ((s + bias) * scale).softmax(dim=-1).to(dtype)
        o = torch.matmul(p, vh)
        return o.reshape(1, H, N, D).permute(0, 2, 1, 3).reshape(1, N, C)

    for _ in range(3):
        call(True); call(False)
    if device.type != "cuda":
        t0 = time.perf_counter()
        for _ in range(iters):
            call(True); call(False)
        return (time.perf_counter() - t0) * 1e6 / iters
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(device)
    e0.record()
    for _ in range(iters):
        call(True); call(False)
    e1.record()
    torch.cuda.synchronize(device)
    return e0.elapsed_time(e1) * 1e3 / iters


def reference_gpu_eager(device, steps: int, warmup: int):
    """Comparison only (BASELINE.md section 3, "the real bar"; SURVEY 8d last line): the REFERENCE's control flow and op
    sequence as eager fp16 PyTorch on this GPU -- two batch-1 UNet forwards per step (paint_with_words.py:483-499),
    inj_forward's op sequence under torch.autocast (paint_with_words.py:60-125: three projections, heads->batch copies,
    QK^T, weight function with qk.max(), bias add, softmax, PV, batch->heads copy, to_out), the host-side sigma lookup
    with its `.nonzero().item()` sync (paint_with_words.py:473) and the stock PyTorch UNet route (no fused ops, no
    CUDA graph, no K/V caching).  Same UNet weights (seed 0), same conditioning, same schedule as the b200 arm.
    Returns steps/s (CUDA events).  Patches CrossAttention.__call__ class-wide; the caller re-patches afterwards."""
    from oracle import loop as oracle_loop
    from paint_with_words_sd_b200 import fused_ops
    from paint_with_words_sd_b200.unet import CrossAttention

    @torch.autocast("cuda")
    def eager_inj_forward(self, hidden_states, context=None, mask=None):
        as_dict = isinstance(context, dict)
        ctx = hidden_states if context is None else (context["CONTEXT_TENSOR"] if as_dict else context)
        q, k, v = (self.reshape_heads_to_batch_dim(t) for t in (self.to_q(hidden_states), self.to_k(ctx), self.to_v(ctx)))
        scores = torch.matmul(q, k.transpose(-1, -2))
        bias = 0.0
        if as_dict:
            bias = context["WEIGHT_FUNCTION"](context[f"CROSS_ATTENTION_WEIGHT_{scores.shape[-2]}"], context["SIGMA"], scores)
        probs = ((scores + bias) * self.scale).softmax(dim=-1)
        out = self.reshape_batch_dim_to_heads(torch.matmul(probs, v))
        return self.to_out[1](self.to_out[0](out))

    unet = build_unet(UNetConfig.sd15(), seed=0, dtype=torch.float16, device=device)
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(768).to(device)
    st = SETTINGS["aurora"]
    _, _, cond, uncond = _encode_text_color_inputs(enc, tok, device, color_map_image("aurora", SIZE), dict(st["ctx"]),
                                                   st["prompt"], "")
    cond.pop("CROSS_ATTENTION_WEIGHT_ORIG", None)        # (kept on the host by this repo; all four keys hit at 512x512)
    sch = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    sch.set_timesteps(SCHEDULE_STEPS)
    lat = (torch.randn(1, 4, SIZE // 8, SIZE // 8, generator=torch.manual_seed(0)) * sch.init_noise_sigma).to(device)
    old_call, old_enabled = CrossAttention.__dict__.get("__call__"), fused_ops.ENABLED
    CrossAttention.__call__ = eager_inj_forward
    fused_ops.ENABLED = False
    events = []

    def on_step(i):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        events.append(e)

    try:
        n = min(SCHEDULE_STEPS, warmup + steps)
        with torch.autocast("cuda"):
            oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat, weight_function, GUIDANCE,
                                               max_steps=n, on_step=on_step)
        torch.cuda.synchronize(device)
    finally:
        fused_ops.ENABLED = old_enabled
        if old_call is None:
            del CrossAttention.__call__
        else:
            CrossAttention.__call__ = old_call
    w = min(warmup, len(events) - 2)
    ms = events[w].elapsed_time(events[-1])
    timed = len(events) - 1 - w
    return {"steps_per_s": timed / (ms / 1e3), "steps": timed, "warmup": w + 1, "ms_per_step": ms / timed}


# ------------------------------------------------------------------------------------------------
# main arm
# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _claim_stdout():
    """Keep stdout for the ONE JSON line: route everything else written to fd 1 (NCCL's version banner, library
    chatter) to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def dump_outputs(out_dir: str, arrays: dict, rank: int, world: int):
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), t.detach().float().cpu().numpy())


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=27)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--quick", action="store_true", help="timed region only (for ncu launch lists): no e2e/roofline/cpu legs")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS),
                    help="BASELINE.json config (1-based); 2 = configs[1], the one the metric is quoted on (default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the latents of the last timed step to DIR/latents.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the b200 arm")
    cfg = CONFIGS[args.config]
    rank, local_rank, world = sharding.env_world()
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); use --impl reference for the CPU arm")
    args.warmup = max(args.warmup, 3)
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    # NCCL chatter goes to stderr through _claim_stdout(); NCCL_DEBUG is left to the caller (the driver reads INFO lines)
    sharding.init_distributed("nccl")
    import torch.distributed as dist
    import paint_with_words_sd_b200 as P
    from paint_with_words_sd_b200 import _native, attention
    from paint_with_words_sd_b200.pipeline import PwWSampler

    torch.backends.cudnn.benchmark = True
    # weights: rank 0 builds the seeded replica, everyone else receives it in one broadcast
    ucfg = unet_config(cfg["unet"])
    if rank == 0:
        unet = build_unet(ucfg, seed=0, dtype=torch.float16, device=device)
    else:
        with torch.device(device):
            unet = P.unet.UNet2DConditionModel(ucfg).half().eval().requires_grad_(False)
    bcast_bytes = sharding.broadcast_module_weights(unet, src=0)
    unet = unet.to(memory_format=torch.channels_last)
    P.patch_unet(unet)

    SCHED = cfg["sched_steps"]
    wf = weight_function if args.config == 2 else make_weight_function(cfg["coef"])
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(cfg["text_dim"]).to(device)
    sch = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    sch.set_timesteps(SCHED)
    if cfg["total_images"]:
        if cfg["total_images"] % world:
            raise SystemExit(f"--config {args.config} shards {cfg['total_images']} images: --gpus must divide it")
        image_ids = sharding.shard_images(cfg["total_images"], rank, world)
    else:
        image_ids = [rank]
    conds, unconds, lat0, extra = build_images(cfg, device, image_ids, tok, enc, sch)
    m_img = len(image_ids)
    total_images = cfg["total_images"] or world
    sampler = PwWSampler(unet, sch, conds, unconds, lat0, wf, GUIDANCE, extra_input=extra, use_graph=not args.no_graph)

    def run_steps(n, per_step=None):
        done = 0
        while done < n:
            if sampler._step_no >= SCHED:
                sampler.restart(lat0)
            if per_step is not None:
                per_step()
            else:
                sampler.step()
            done += 1

    def sync_all():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(device)

    def timed_region(n, per_step=None):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.cuda.nvtx.range_push("pww_timed")
        run_steps(n, per_step)
        torch.cuda.nvtx.range_pop()
        e1.record()
        torch.cuda.synchronize(device)
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    with torch.no_grad():
        run_steps(args.warmup)
        launches_before = _native.launch_count
        with ClockSampler(local_rank) as clk:
            ms = timed_region(args.steps)
        clocks = clk.summary()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"latents": sampler.latents}, rank, world)
        per_step_launches = sampler.native_launches_per_step
        if per_step_launches is None:
            per_step_launches = (_native.launch_count - launches_before) // max(1, args.steps)
        value = total_images * args.steps / (ms / 1e3)        # one step = one denoising step of ONE image

        if args.quick:
            if rank == 0:
                emit({"metric": METRIC, "value": value, "unit": UNIT, "ms_per_step": ms / args.steps,
                      "steps": args.steps, "quick": True})
            return
        # ---- e2e: host buffers in, host buffer out, every step ----
        dev_in = sampler.device_inputs()
        pinned = {k: t.detach().to("cpu").pin_memory() for k, t in dev_in.items()}
        lat_host = pinned["latents"]
        h2d = sum(t.numel() * t.element_size() for t in pinned.values())
        d2h = lat_host.numel() * lat_host.element_size()

        def e2e_step():
            sampler.stage_from_host(pinned)
            sampler.step()
            lat_host.copy_(sampler.latents, non_blocking=True)
            torch.cuda.current_stream(device).synchronize()

        sampler.restart(lat0)
        lat_host.copy_(lat0)
        run_steps(3, e2e_step)
        ms_e2e = timed_region(args.steps, e2e_step)
        e2e_value = total_images * args.steps / (ms_e2e / 1e3)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if cfg["total_images"] else "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic", "config": workload_config(world, args.config, m_img),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(per_step_launches) * args.steps,
            "impl": "b200"}
    line["config"]["self_attn"] = attention.SELF_ATTN_IMPL
    line["config"]["cuda_graph"] = not args.no_graph
    line["config"]["weights_broadcast_bytes"] = bcast_bytes

    if rank == 0:
        peak, peak_src = measured_peaks()
        try:
            r2 = xattn_roofline(device, B=2, biased=1, dense_pair=True)
            r16 = xattn_roofline(device, B=16, biased=8, iters=32, dense_pair=True)
            ach = r2["alg_bytes"] / (r2["us_op"] * 1e-6) / 1e9
            ach16 = r16["alg_bytes"] / (r16["us_op"] * 1e-6) / 1e9
            line["roofline"] = {
                "kernel": "pww_xattn_fused_f16 (one launch: statistic + packed-map bias + softmax + PV) N=4096 C=320 H=8 "
                          "T=77, B=2 (cond+uncond) as launched by this workload",
                "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": ncu_traffic("B2_fused"),
                "peak_source": peak_src, "us_per_launch": r2["us_op"], "alg_bytes_per_launch": r2["alg_bytes"],
                "alg_bytes_note": "SURVEY 8d formula with the PACKED map (64 B per pixel + 80 B index) instead of the "
                                  "dense fp32 map (308 B per pixel); alg_bytes_dense_map is the round-1 figure",
                "alg_bytes_dense_map": r2["alg_bytes_dense_map"],
                "frac_with_dense_map_bytes": r2["alg_bytes_dense_map"] / (r2["us_op"] * 1e-6) / 1e9 / peak,
                "op_frac": ach / peak,          # the op IS this one launch (round 1: stats launch + forward launch)
                "dense_pair": {"us_stats": r2.get("us_dense_stats"), "us_fwd": r2.get("us_dense_fwd"),
                               "note": "round-1 path (pww_xattn_stats_f16 + pww_xattn_fwd_f16, dense fp32 map), same inputs"},
                "batched": {"B": 16, "biased": 8, "us_per_launch": r16["us_op"], "achieved": ach16, "frac": ach16 / peak,
                            "alg_bytes_per_launch": r16["alg_bytes"], "traffic": ncu_traffic("B16_fused"),
                            "alg_bytes_dense_map": r16["alg_bytes_dense_map"],
                            "frac_with_dense_map_bytes": r16["alg_bytes_dense_map"] / (r16["us_op"] * 1e-6) / 1e9 / peak,
                            "op_frac": ach16 / peak,
                            "dense_pair": {"us_stats": r16.get("us_dense_stats"), "us_fwd": r16.get("us_dense_fwd")}},
                "method": "CUDA events around a CUDA graph of back-to-back launches cycling through buffer sets > L2"}
        except Exception as e:  # keep the headline even if the micro-bench fails
            line["roofline"] = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None,
                                "traffic": None, "error": repr(e)}
        try:    # comparison only: the reference's eager op sequence on this GPU, same shapes, cond + uncond call
            us = eager_torch_xattn_us(device)
            line["roofline"]["eager_torch_fp16"] = {
                "us_per_cond_uncond_pair": us,
                "note": "reference inj_forward op sequence (heads->batch copies, QK^T, max, bias add, softmax, PV) as eager "
                        "PyTorch fp16 on this GPU at N=4096 C=320; compare with us_per_launch"}
        except Exception as e:
            line["roofline"]["eager_torch_fp16"] = {"error": repr(e)}
        try:    # comparison only: the reference's loop as eager fp16 PyTorch on this GPU (same weights/inputs/schedule)
            if args.config != 2:
                raise RuntimeError("measured for the default config only")
            rg = reference_gpu_eager(device, steps=args.steps, warmup=3)
            P.patch_unet(unet)
            line["reference_gpu_eager"] = {
                "value": rg["steps_per_s"], "unit": UNIT, "steps": rg["steps"], "warmup": rg["warmup"],
                "ms_per_step": rg["ms_per_step"], "dtype": "f16 (torch.autocast)",
                "what": "reference control flow on this B200: 2 batch-1 eager UNet forwards/step, inj_forward op sequence "
                        "(paint_with_words.py:60-125) under autocast, stock PyTorch ops, no graph / caching / fused kernels",
                "speedup_value": value / total_images / rg["steps_per_s"],
                "speedup_e2e": e2e_value / total_images / rg["steps_per_s"]}
        except Exception as e:
            line["reference_gpu_eager"] = {"value": None, "error": repr(e)}
        if world == 1 and not args.no_cpu_baseline and args.config == 2:
            try:
                r = cpu_reference(max_timed_steps=2, warmup=0, budget_s=45.0)
                line["cpu_baseline"] = {"value": r["steps_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                        "sample": f"{r['steps']} denoising step(s) of the same 512x512 workload through "
                                                  f"the oracle port of the reference loop, fp32, {r['seconds']:.1f} s"}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                        "sample": "failed: " + repr(e)}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
