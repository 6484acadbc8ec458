#!/usr/bin/env python
"""Cost of the training precisions, kernel by kernel: the fused training step (nerf/fused_train.py) at 2048 rays, 64 coarse + 64
fine samples, perturb + sigma noise, for each --precisions entry, with the variants alternated round by round in one process.

Prints one JSON line: the card and its power limit, per precision the step time of every round (CUDA events around --steps
steps, after --warmup steps) and, from a separate torch.profiler pass, the mean device time per step of the training forward
(render_kernel), the dX chain (chain_kernel) and the weight-gradient GEMMs (dw_kernel), plus the record bytes per step."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "4d-facial-avatars_b200"))

KERNELS = {"forward (SAVE)": "render_kernel", "chain": "chain_kernel", "dw": "dw_kernel"}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = ""
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precisions", default="fast,exact,exact_grad")
    ap.add_argument("--rays", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--profile-steps", type=int, default=3)
    a = ap.parse_args()
    import nerface_oracle as O
    import nerf
    from nerf import fused_train

    dev = torch.device("cuda", 0)
    H = W = 512
    fr = O.synthetic_frame(0, H, W)
    ro, rd = nerf.get_ray_bundle(H, W, fr["intrinsics"], fr["pose"].to(dev))
    ro, rd = ro.reshape(-1, 3), rd.reshape(-1, 3)
    bg = fr["bg"].reshape(-1, 3).to(dev)
    tgt = torch.rand(H * W, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    expr = fr["expr"].to(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    batches = [torch.randint(0, H * W, (a.rays,), device=dev, generator=g) for _ in range(a.steps + a.warmup)]
    precs = a.precisions.split(",")
    trainers = {}
    for p in precs:
        mk = lambda: nerf.models.ConditionalBlendshapePaperNeRFModel(  # noqa: E731
            num_encoding_fn_xyz=10, num_encoding_fn_dir=4, include_input_xyz=True, include_input_dir=False)
        mc, mf = mk(), mk()
        mc.load_state_dict(O.random_init_params(100))
        mf.load_state_dict(O.random_init_params(101))
        trainers[p] = fused_train.FusedTrainer(mc.to(dev), mf.to(dev), n_latent=16, lr=5e-4, num_coarse=64, num_fine=64, perturb=True,
                                               noise_std=0.1, near=0.2, far=0.8, latent_reg=0.005, precision=p)

    def step(p, sel):
        trainers[p].step(ro[sel], rd[sel], tgt[sel], expr, 3, background=bg[sel])

    ms = {p: [] for p in precs}
    for _ in range(a.rounds):
        for p in precs:
            for i in range(a.warmup):
                step(p, batches[i])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(a.warmup, a.warmup + a.steps):
                step(p, batches[i])
            e1.record()
            torch.cuda.synchronize()
            ms[p].append(e0.elapsed_time(e1) / a.steps)

    kern = {}
    from torch.profiler import ProfilerActivity, profile
    for p in precs:
        step(p, batches[0])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(a.profile_steps):
                step(p, batches[i])
            torch.cuda.synchronize()
        tot = {k: 0.0 for k in KERNELS}
        for ev in prof.key_averages():
            for k, pat in KERNELS.items():
                if pat in ev.key:
                    tot[k] += ev.device_time_total / 1e3  # us -> ms
        kern[p] = {k: v / a.profile_steps for k, v in tot.items()}

    tiles = (a.rays // 2) * 3  # units of two rays x (1 coarse + 2 fine tiles) at 64c + 64f
    rec = {p: tiles * (2 if p == "exact_grad" else 1) * (1 << 20) for p in precs}
    print(json.dumps({"card (name, power limit, max SM clock)": card(), "rays": a.rays, "samples": "64c+64f, perturb + noise 0.1",
                      "ms_per_step_by_round": ms,
                      "ms_per_step_median": {p: sorted(v)[len(v) // 2] for p, v in ms.items()},
                      "ms_per_step_spread": {p: max(v) - min(v) for p, v in ms.items()},
                      "kernel_ms_per_step": kern, "record_bytes_per_step": rec}), flush=True)


if __name__ == "__main__":
    main()
