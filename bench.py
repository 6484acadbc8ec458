#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: rays/sec at 512x512 with 64 coarse + 128 fine samples per ray.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
    python bench.py --impl reference ...                       (the reference algorithm on the host cores)
    python bench.py ... --dump-outputs DIR                     (also write the last timed step's outputs to DIR/<name>.npy)

Headline (`value`, `e2e`, `roofline`): one step = one full 512x512 frame per GPU (BASELINE config 2; with N GPUs config 5:
N concurrent frames with different expression codes, all-gathered into one [N,512,512,3] video tensor) => weak scaling,
value = N*H*W*K / time.  Synthetic per-frame pose / expression / latent / background, random-init weights (SURVEY.md §8d).

`value`  : inputs already resident in HBM; per step nfb_set_frame + the fused render kernel (+ NCCL all-gather
           when N>1), timed with CUDA events per step (L2 flushed between steps, outside the events).
`e2e`    : the same frame through the C-ABI host entry nfb_render_frame_host: pinned host expression / latent /
           background in, 11 floats per ray out, copies inside the timed region (N>1: the same all-gather as `value`).
`roofline`: dominant kernel = the render kernel; achieved = algorithmic FLOP per launch (1,100,032 FLOP per MLP evaluation x
           (2*Nc+Nf) evaluations per ray x rays) / its CUDA-event time; peak from MEASURED_PEAKS.json.
`cpu_baseline`: the reference algorithm (oracle/nerface_oracle.py, the bit-exact port of its run_one_iter_of_nerf) on the host
           cores for a 64x64 crop.

Sub-records in the same JSON line (SURVEY.md §8e, the split `north_star` names):
`rows`, `rows_1024`: ONE frame (512x512 64c+128f; 1024x1024 128c+256f = BASELINE config 4) sharded by pixel rows over the
           N ranks (NfbRays.row_begin), one NCCL all-gather of the packed 11-float output tiles per frame => strong scaling.
`train`  : BASELINE config 3: 2048-ray batches (64c+64f, perturb + noise) sharded over the N ranks, one flat FP32 gradient
           all-reduce, Adam — per-iteration time incl. loss, backward, collective, optimizer and weight re-pack.
Each carries ms_per_step (max over ranks), the single-GPU time of the same work measured in the same run (`t1_ms`),
efficiency_vs_1gpu = t1 / (N * tN) and the time spent in the collective.
"""
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
sys.path.insert(0, os.path.join(ROOT, "oracle"))

NEAR, FAR = 0.2, 0.8
ALGO_FLOP_PER_EVAL = 1100032
NAMES = ["rgb_coarse", "disp_coarse", "acc_coarse", "rgb_fine", "disp_fine", "acc_fine", "w_last"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("NFB_PRECISION", "fast"), choices=["fast", "exact"])
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--num-coarse", type=int, default=64)
    ap.add_argument("--num-fine", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only: skip rows / train / exact / stress records")
    ap.add_argument("--extras", default="all", help="comma list out of rows,rows_1024,train,single (exact / stress); default all")
    ap.add_argument("--train-impl", default=os.environ.get("NFB_TRAIN_IMPL", "fused"), choices=["fused", "dropin"])
    ap.add_argument("--no-train-graph", action="store_true", help="fused training step launch by launch instead of one CUDA graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy, "
                    "float32: rank 0's 7 per-ray outputs and, with N>1 GPUs, the all-gathered [N,H*W,3] video (--impl ours only)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        pw = sorted(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = max((float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w": pw[len(pw) // 2] if pw else None}


# ------------------------------------------------------------------------------------------------
# the reference algorithm on the host cores (cpu_baseline / --impl reference)
def reference_frame_crop(frame_index, H, W, crop, nc, nf, threads):
    """(run, rays): the reference algorithm (oracle/nerface_oracle.py) on a crop x crop centre block of the synthetic frame."""
    import nerface_oracle as O
    torch.set_num_threads(threads)
    fr = O.synthetic_frame(frame_index, H, W)
    pc, pf = O.random_init_params(100), O.random_init_params(101)
    r0, c0 = (H - crop) // 2, (W - crop) // 2
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    ro, rd = ro[r0:r0 + crop, c0:c0 + crop].contiguous(), rd[r0:r0 + crop, c0:c0 + crop].contiguous()
    bg = fr["bg"][r0:r0 + crop, c0:c0 + crop].reshape(-1, 3)
    s = O.Sampling(nc, nf, False, 0.0, False, 65536)

    def run():
        with torch.no_grad():
            return O.run_one_iter(ro, rd, pc, pf if nf > 0 else None, s, NEAR, FAR, fr["expr"], fr["latent"], bg, "validation")
    return run, crop * crop


def pick_threads(H, W, nc, nf):
    """torch's intra-op pool does not scale to a 100+-core host on these small GEMMs (oversubscription makes it
    10-30x slower), so time a 16x16 crop at a few pool sizes and keep the fastest; that count is reported."""
    cores = os.cpu_count() or 1
    best = (None, 1e30)
    for th in sorted({cores, 64, 32, 16, 8}):
        if th > cores:
            continue
        run, _ = reference_frame_crop(0, H, W, 16, nc, nf, th)
        run()
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (th, dt)
    return best[0]


CPU_SAMPLE = "oracle/nerface_oracle.py (bit-exact port of the reference, torch CPU FP32)"


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = pick_threads(a.height, a.width, a.num_coarse, a.num_fine)
    run, rays = reference_frame_crop(0, a.height, a.width, 64, a.num_coarse, a.num_fine, cores)
    for _ in range(max(1, min(a.warmup, 1))):
        run()
    times = []
    for _ in range(a.steps):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    value = rays * a.steps / total
    line = {"impl": "reference", "metric": "rays/sec at 512x512 (64c+128f samples)", "value": value, "unit": "rays/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"person_1-shaped eval {a.height}x{a.width}, {a.num_coarse}c+{a.num_fine}f, 76-dim expr + 32-dim latent",
                       "sample": "64x64 centre crop of the frame per step"},
            "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "host_cores": os.cpu_count(),
                             "sample": CPU_SAMPLE + " on a 64x64 crop per step"},
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, v, n, video=None):
    """The outputs of one render_camera call as out_dir/<name>.npy (float32, [n] or [n,3]) and, when given, the all-gathered
    [N,n,3] video as video.npy.  Past DUMP_LIMIT_BYTES in all, a fixed seeded sample of rays (the same for every frame of the
    video) is written instead, with their indices in ray_index.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    per_ray = 4 * sum(v[k][:1].numel() for k in NAMES) + (4 * video.shape[0] * video.shape[2] if video is not None else 0)
    budget = DUMP_LIMIT_BYTES - 4096  # room for the .npy headers
    idx = None
    if per_ray * n > budget:
        keep = budget // (per_ray + 8)
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        np.save(os.path.join(out_dir, "ray_index.npy"), idx.double().numpy())
        idx = idx.to(v[NAMES[0]].device)
    for k in NAMES:
        t = v[k] if idx is None else v[k].index_select(0, idx)
        np.save(os.path.join(out_dir, k + ".npy"), t.float().cpu().numpy())
    if video is not None:
        t = video if idx is None else video.index_select(1, idx)
        np.save(os.path.join(out_dir, "video.npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------
class Ctx:
    pass


def make_models(nerf, O, dev, stress=False):
    mk = lambda: nerf.models.ConditionalBlendshapePaperNeRFModel(  # noqa: E731
        num_encoding_fn_xyz=10, num_encoding_fn_dir=4, include_input_xyz=True, include_input_dir=False)
    mc, mf = mk(), mk()
    mc.load_state_dict(O.random_init_params(100, stress))
    mf.load_state_dict(O.random_init_params(101, stress))
    return mc.to(dev), mf.to(dev)


def sync_all(c):
    torch.cuda.synchronize()
    if c.world > 1:
        c.dist.barrier()
        torch.cuda.synchronize()


def max_over_ranks(c, x):
    t = torch.tensor([x], device=c.dev, dtype=torch.float64)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return float(t[0])


def bench_rows(c, H, W, nc, nf, steps, warmup, precision):
    """ONE frame sharded by pixel rows (SURVEY.md §8e): rank r renders rows [r*H/N, (r+1)*H/N) with in-kernel ray generation
    (NfbRays.row_begin) and the packed [11, rows*W] output tiles are all-gathered (NCCL) into [N, 11, rows*W] on every rank."""
    from nerf import parallel
    O, eng, dev, world, rank = c.O, c.eng, c.dev, c.world, c.rank
    if H % world:
        return {"unavailable": f"{H} rows do not split evenly over {world} ranks"}
    fr = O.synthetic_frame(0, H, W)
    expr, latent = fr["expr"].to(dev), fr["latent"].to(dev)
    bg = fr["bg"].reshape(-1, 3).to(dev).contiguous()
    begin, rows = parallel.shard_rows(H, world, rank)
    n, nl = H * W, rows * W
    local = torch.empty((11, nl), device=dev)
    gathered = torch.empty((world, 11, nl), device=dev)
    full = torch.empty((11, n), device=dev)
    bg_local = bg[begin * W:(begin + rows) * W].contiguous()

    def step_full():
        eng.set_frame(expr, latent)
        eng.render_camera(fr["pose"], fr["intrinsics"], H, W, 0, H, NEAR, FAR, nc, nf, background=bg, out=full, precision=precision)

    def step_sharded(ev=None):
        eng.set_frame(expr, latent)
        eng.render_camera(fr["pose"], fr["intrinsics"], H, W, begin, rows, NEAR, FAR, nc, nf, background=bg_local, out=local,
                          precision=precision)
        if ev is not None:
            ev.record()
        if world > 1:
            c.dist.all_gather_into_tensor(gathered.view(-1), local.view(-1))

    def run(fn, k, with_mid=False):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(k)]
        sync_all(c)
        for i in range(k):
            c.flush.fill_(float(i))
            evs[i][0].record()
            if with_mid:
                fn(evs[i][1])
            else:
                fn()
            evs[i][2].record()
        sync_all(c)
        tot = sum(e[0].elapsed_time(e[2]) for e in evs) / k
        coll = sum(e[1].elapsed_time(e[2]) for e in evs) / k if with_mid else 0.0
        return tot, coll

    n1 = max(2, min(steps, 3 if n > 512 * 512 else 5))
    step_full()
    t1, _ = run(step_full, n1)  # the whole frame on ONE GPU (every rank does it; rank 0's time is reported)
    for _ in range(max(1, warmup)):
        step_sharded()
    tn, coll = run(step_sharded, steps, with_mid=True)
    tn_max = max_over_ranks(c, tn)
    identical = None
    if world > 1:  # the sharded frame must be the single-GPU frame bit for bit
        asm = gathered.permute(1, 0, 2).reshape(11, n)
        # rgb rows are [n,3] inside the packed tile: compare per output through the same views render_camera hands out
        ok = True
        for name, lo, hi, ch in (("rgb_coarse", 0, 3, 3), ("disp_coarse", 3, 4, 1), ("acc_coarse", 4, 5, 1), ("rgb_fine", 5, 8, 3),
                                 ("disp_fine", 8, 9, 1), ("acc_fine", 9, 10, 1), ("w_last", 10, 11, 1)):
            f = full.view(-1)[lo * n:hi * n].view(n, ch)
            parts = [gathered[r].reshape(-1)[lo * nl:hi * nl].view(nl, ch) for r in range(world)]
            ok = ok and bool(torch.equal(f, torch.cat(parts, dim=0)))
        del asm
        identical = ok
    rec = {"workload": f"ONE {H}x{W} frame, {nc}c+{nf}f, rows sharded over {world} GPU(s), all-gather of packed 11-float tiles",
           "scaling": "strong", "ms_per_step": tn_max, "rays_per_s": n / (tn_max * 1e-3), "t1_ms": t1,
           "efficiency_vs_1gpu": t1 / (world * tn_max), "collective_ms": coll if world > 1 else 0.0,
           "gather_bytes_per_rank": 11 * nl * 4, "bit_identical_to_1gpu": identical, "steps": steps,
           "roofline_frac_1gpu": n * (2 * nc + nf) * ALGO_FLOP_PER_EVAL / (t1 * 1e-3) / 1e12 / c.peak}
    return rec


def bench_train(c, steps, warmup, impl, rays=2048, nc=64, nf=64, graph=True):
    """BASELINE config 3 (shipped YAML train block): 2048 rays of one 512x512 frame per iteration, 64c+64f, perturb + sigma
    noise 0.1, loss = mse(rgb_c) + mse(rgb_f) + 0.005*|latent|, Adam lr 5e-4 with the YAML's LR decay; with N ranks the batch is
    sharded (2048/N rays per rank) and ONE flat FP32 gradient bucket is all-reduced per iteration."""
    import nerf
    from nerf import parallel
    O, dev, world, rank = c.O, c.dev, c.world, c.rank
    if rays % world:
        return {"unavailable": f"{rays} rays do not split evenly over {world} ranks"}
    H = W = 512
    fr = O.synthetic_frame(0, H, W)
    ro, rd = nerf.get_ray_bundle(H, W, fr["intrinsics"], fr["pose"].to(dev))
    ro, rd = ro.reshape(-1, 3).contiguous(), rd.reshape(-1, 3).contiguous()
    bg = fr["bg"].reshape(-1, 3).to(dev).contiguous()
    target_img = torch.rand(H * W, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    expr = fr["expr"].to(dev)
    g = torch.Generator(device=dev).manual_seed(7)
    n_it = 2 * (steps + warmup) + 4
    idx = [torch.randint(0, H * W, (rays,), device=dev, generator=g) for _ in range(n_it)]
    launches_before = c.eng.launch_count()

    if impl == "fused":
        from nerf import fused_train
        mc, mf = make_models(nerf, O, dev)
        tr = fused_train.FusedTrainer(mc, mf, n_latent=16, lr=5e-4, lr_decay_steps=250000, lr_decay_factor=0.1,
                                      num_coarse=nc, num_fine=nf, perturb=True, noise_std=0.1, near=NEAR, far=FAR,
                                      latent_reg=0.005)

        captured = {"shard": None}

        def step(i, shard, ev=None):
            w, r = (world, rank) if shard else (1, 0)
            per = rays // w
            sel = idx[i][r * per:(r + 1) * per]
            if graph and not captured.get("failed"):  # the whole iteration (incl. the all-reduce) is ONE graph replay; re-captured when the shard size changes
                if captured["shard"] != shard:
                    try:
                        tr.capture(per, has_background=True, world=w, n_total=rays)
                        captured["shard"] = shard
                    except Exception as e:  # same on every rank: fall back to launch-by-launch steps and say so in the record
                        captured["failed"] = repr(e)[:200]
                        return step(i, shard, ev)
                if ev is not None:
                    ev[0].record()
                    ev[1].record()
                return tr.step_graph(ro[sel], rd[sel], target_img[sel], expr, 3, background=bg[sel])
            return tr.step(ro[sel], rd[sel], target_img[sel], expr, latent_index=3, background=bg[sel],
                           world=w, n_total=rays, events=ev)
    else:
        mc, mf = make_models(nerf, O, dev)
        latent_codes = torch.zeros(16, 32, device=dev, requires_grad=True)
        params = [p for k, p in list(mc.named_parameters()) + list(mf.named_parameters()) if not k.startswith("layers_dir.3")]
        opt = torch.optim.Adam(params + [latent_codes], lr=5e-4)
        blk = dict(num_coarse=nc, num_fine=nf, perturb=True, lindisp=False, radiance_field_noise_std=0.1, white_background=False,
                   chunksize=2048)
        cfg = nerf.CfgNode(dict(nerf=dict(use_viewdirs=True, train=blk), dataset=dict(no_ndc=True, near=NEAR, far=FAR)))

        def step(i, shard, ev=None):
            w, r = (world, rank) if shard else (1, 0)
            per = rays // w
            sel = idx[i][r * per:(r + 1) * per]
            out = nerf.run_one_iter_of_nerf(H, W, fr["intrinsics"], mc, mf, ro[sel], rd[sel], cfg, mode="train", expressions=expr,
                                            background_prior=bg[sel], latent_code=latent_codes[3])
            tgt = target_img[sel]
            loss = ((out[0] - tgt) ** 2).mean() + ((out[3] - tgt) ** 2).mean() + 0.005 * latent_codes[3].norm()
            opt.zero_grad(set_to_none=True)
            loss.backward()
            if ev is not None:
                ev[0].record()
            if w > 1:
                parallel.allreduce_gradients(params + [latent_codes], average=True)
            if ev is not None:
                ev[1].record()
            opt.step()
            return loss

    def run(k, first, shard):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(k)]
        sync_all(c)
        for j in range(k):
            evs[j][0].record()
            last = step(first + j, shard, evs[j][1:3])
            evs[j][3].record()
        sync_all(c)
        tot = sum(e[0].elapsed_time(e[3]) for e in evs) / k
        coll = sum(e[1].elapsed_time(e[2]) for e in evs) / k
        return tot, coll, float(last.sum())

    k = 0
    for j in range(max(3, warmup)):  # single-GPU warm-up (packs, allocations)
        step(k, False); k += 1  # noqa: E702
    t1, _, loss1 = run(max(5, min(steps, 20)), k, False)
    k += max(5, min(steps, 20))
    rec = {"workload": f"{rays} rays/iter of one 512x512 frame, {nc}c+{nf}f, perturb + noise 0.1, mse x2 + latent reg, Adam",
           "impl": impl + (" + CUDA graph (one replay per iteration, all-reduce inside)" if (impl == "fused" and graph) else ""),
           "scaling": "strong", "t1_ms": t1, "rays_per_s_1gpu": rays / (t1 * 1e-3)}
    if world > 1:
        for j in range(max(3, warmup)):
            step(k, True); k += 1  # noqa: E702
        tn, coll, lossn = run(max(5, min(steps, 20)), k, True)
        tn_max = max_over_ranks(c, tn)
        rec.update({"ms_per_step": tn_max, "rays_per_s": rays / (tn_max * 1e-3), "efficiency_vs_1gpu": t1 / (world * tn_max),
                    "collective_ms": None if (impl == "fused" and graph) else coll, "rays_per_rank": rays // world, "loss_last": lossn})
    else:
        rec.update({"ms_per_step": t1, "rays_per_s": rays / (t1 * 1e-3), "efficiency_vs_1gpu": 1.0, "collective_ms": 0.0,
                    "rays_per_rank": rays, "loss_last": loss1})
    flop = 3 * ALGO_FLOP_PER_EVAL * (2 * nc + nf) * rays
    rec["roofline_frac"] = flop / (rec["ms_per_step"] * 1e-3) / 1e12 / c.peak / world
    rec["gpu_launches_total"] = c.eng.launch_count() - launches_before
    if impl == "fused" and graph and captured.get("failed"):
        rec["impl"] = impl + " (launch by launch: graph capture failed)"
        rec["graph_capture_error"] = captured["failed"]
    return rec


def stress_psnr(c, precision):
    """Fast-mode accuracy where it is hardest (SURVEY.md §8d): opaque-stress weights, two image rows against the oracle."""
    import nerf
    O, eng, dev = c.O, c.eng, c.dev
    H = W = 512
    fr = O.synthetic_frame(0, H, W)
    mc, mf = make_models(nerf, O, dev, stress=True)
    eng.sync_weights(mc, mf)
    eng.set_frame(fr["expr"].to(dev), fr["latent"].to(dev))
    r0, rows = H // 2, 2
    bg = fr["bg"].reshape(-1, 3)[r0 * W:(r0 + rows) * W].contiguous()
    out = {}
    for prec in ("fast", "exact"):
        v = eng.render_camera(fr["pose"], fr["intrinsics"], H, W, r0, rows, NEAR, FAR, 64, 128, background=bg.to(dev), precision=prec)
        torch.cuda.synchronize()
        out[prec] = {k: v[k].cpu().clone() for k in NAMES}
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    with torch.no_grad():
        ref = O.run_one_iter(ro[r0:r0 + rows], rd[r0:r0 + rows], O.random_init_params(100, True), O.random_init_params(101, True),
                             O.Sampling(64, 128, False, 0.0, False, 65536), NEAR, FAR, fr["expr"], fr["latent"], bg, "validation")
    res = {}
    for prec in ("fast", "exact"):
        mse = float(((out[prec]["rgb_fine"].reshape(ref[3].shape) - ref[3]) ** 2).mean())
        res[prec] = {"psnr_rgb_fine_db": 99.0 if mse == 0 else min(99.0, -10.0 * math.log10(mse)),
                     "max_abs_rgb": float((out[prec]["rgb_fine"].reshape(ref[3].shape) - ref[3]).abs().max()),
                     "max_abs_disp": float((out[prec]["disp_fine"].reshape(ref[4].shape) - ref[4]).abs().max())}
    res["rays"] = rows * W
    res["min_w_last"] = float(ref[6].min())
    return res


def main():
    a = parse()
    if a.impl == "reference":
        return reference_arm(a)

    sys.path.insert(0, os.path.join(ROOT, "4d-facial-avatars_b200"))
    import nerface_oracle as O
    import nerf
    from nerf import _engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    H, W, nc, nf = a.height, a.width, a.num_coarse, a.num_fine
    n = H * W
    pk, pk_src = peaks()

    mc, mf = make_models(nerf, O, dev)
    eng = _engine.renderer_for(dev)
    eng.sync_weights(mc, mf)
    c = Ctx()
    c.O, c.eng, c.dev, c.world, c.rank, c.dist, c.peak = O, eng, dev, world, rank, dist, pk["bf16_tflops"]
    c.flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)  # > 126 MB L2

    # synthetic frames: frame f on rank r uses generator seed 42 + (f*world + r)
    n_frames = a.steps + a.warmup
    frames = [O.synthetic_frame(f * world + rank, H, W) for f in range(min(n_frames, 4))]
    dev_frames = [dict(expr=fr["expr"].to(dev), latent=fr["latent"].to(dev), bg=fr["bg"].reshape(-1, 3).to(dev).contiguous())
                  for fr in frames]
    host_frames = [dict(expr=fr["expr"].pin_memory(), latent=fr["latent"].pin_memory(),
                        bg=fr["bg"].reshape(-1, 3).contiguous().pin_memory()) for fr in frames]
    out_buf = torch.empty((11, n), device=dev)
    out_host = torch.empty((11 * n,), dtype=torch.float32).pin_memory()
    video = torch.empty((world, n, 3), device=dev) if world > 1 else None
    rgb_stage = torch.empty((n, 3), device=dev) if world > 1 else None
    last_out = {}

    def step_resident(i, ev=None):
        fr, d = frames[i % len(frames)], dev_frames[i % len(frames)]
        eng.set_frame(d["expr"], d["latent"])
        if ev:
            ev[0].record()
        v = eng.render_camera(fr["pose"], fr["intrinsics"], H, W, 0, H, NEAR, FAR, nc, nf, background=d["bg"], out=out_buf,
                              precision=a.precision)
        if ev:
            ev[1].record()
        if world > 1:
            dist.all_gather_into_tensor(video.view(-1), v["rgb_fine"].reshape(-1))
        last_out["v"] = v
        return v

    def step_host(i):
        fr, hst = frames[i % len(frames)], host_frames[i % len(frames)]
        eng.render_frame_host(fr["pose"], fr["intrinsics"], H, W, 0, H, NEAR, FAR, hst["expr"], hst["latent"], hst["bg"],
                              nc, nf, out_host, precision=a.precision)
        if world > 1:  # the same collective as `value`: the frame's rgb_fine (already back on the host) joins the video tensor
            rgb_stage.copy_(out_host[5 * n:8 * n].view(n, 3), non_blocking=True)
            dist.all_gather_into_tensor(video.view(-1), rgb_stage.view(-1))

    def timed(fn, steps, kernel_events=False):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kevs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sync_all(c)
        wall0 = time.perf_counter()
        for i in range(steps):
            c.flush.fill_(float(i))  # L2 flush, outside the timed events
            evs[i][0].record()
            if kernel_events:
                fn(a.warmup + i, kevs[i])
            else:
                fn(a.warmup + i)
            evs[i][1].record()
        sync_all(c)
        wall = time.perf_counter() - wall0
        ms = sum(s.elapsed_time(e) for s, e in evs)
        kms = sum(s.elapsed_time(e) for s, e in kevs) if kernel_events else None
        return max_over_ranks(c, ms), kms, wall

    for i in range(max(a.warmup, 3)):
        step_resident(i)
        step_host(i)
    sync_all(c)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = eng.launch_count()
    ms_total, kernel_ms, wall = timed(step_resident, a.steps, kernel_events=True)
    launches = eng.launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs and rank == 0:
        torch.cuda.synchronize()
        dump_outputs(a.dump_outputs, last_out["v"], n, video)
    ms_e2e, _, _ = timed(lambda i: step_host(i), a.steps)

    # ---- in-run parity (rank 0): two image rows of the last rendered frame against the oracle
    parity = psnr = None
    if rank == 0:
        last = (a.warmup + a.steps - 1) % len(frames)
        fr, dfr = frames[last], dev_frames[last]
        eng.set_frame(dfr["expr"], dfr["latent"])  # no collective here: only rank 0 runs the parity check
        v = eng.render_camera(fr["pose"], fr["intrinsics"], H, W, 0, H, NEAR, FAR, nc, nf, background=dfr["bg"], out=out_buf,
                              precision=a.precision)
        torch.cuda.synchronize()
        ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
        rows = slice(H // 2, H // 2 + 2)
        s = O.Sampling(nc, nf, False, 0.0, False, 65536)
        with torch.no_grad():
            ref = O.run_one_iter(ro[rows], rd[rows], O.random_init_params(100), O.random_init_params(101), s, NEAR, FAR,
                                 fr["expr"], fr["latent"], fr["bg"][rows].reshape(-1, 3), "validation")
        sl = slice((H // 2) * W, (H // 2 + 2) * W)
        parity = max(float((v[k][sl].cpu().reshape(r.shape) - r).abs().max()) for k, r in zip(NAMES, ref))
        mse = float(((v["rgb_fine"][sl].cpu().reshape(ref[3].shape) - ref[3]) ** 2).mean())
        psnr = 99.0 if mse == 0 else min(99.0, -10.0 * math.log10(mse))

    # ---- sub-records (collectives inside: every rank takes part)
    extras = {}
    want = (lambda k: a.extras == "all" or k in a.extras.split(","))  # noqa: E731
    if not a.no_extras:
        if want("rows"):
            extras["rows"] = bench_rows(c, 512, 512, 64, 128, a.steps, a.warmup, a.precision)
        if want("rows_1024"):
            extras["rows_1024"] = bench_rows(c, 1024, 1024, 128, 256, max(3, min(a.steps, 5)), 1, a.precision)
        if want("train"):
            try:
                extras["train"] = bench_train(c, a.steps, a.warmup, a.train_impl, graph=not a.no_train_graph)
            except Exception as e:  # a training-path failure must not take the headline down
                extras["train"] = {"unavailable": repr(e)[:300]}
                if world > 1:
                    raise
        eng.sync_weights(mc, mf)
        if rank == 0 and world == 1 and want("single"):
            # exact mode (FP16 hi+lo x3) on the headline workload: the mode that holds 1e-4 on trained-like weights
            for _ in range(2):
                step_resident(0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            fr, d = frames[0], dev_frames[0]
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                eng.render_camera(fr["pose"], fr["intrinsics"], H, W, 0, H, NEAR, FAR, nc, nf, background=d["bg"], out=out_buf,
                                  precision="exact")
            e1.record()
            torch.cuda.synchronize()
            extras["exact_mode_rays_per_s"] = 3 * n / (e0.elapsed_time(e1) * 1e-3)
            extras["stress"] = stress_psnr(c, a.precision)
            eng.sync_weights(mc, mf)

    if rank == 0:
        rays_total = n * world * a.steps
        value = rays_total / (ms_total * 1e-3)
        e2e_value = rays_total / (ms_e2e * 1e-3)
        evals_per_ray = 2 * nc + nf
        flop_per_launch = n * evals_per_ray * ALGO_FLOP_PER_EVAL
        k_ms = kernel_ms / a.steps
        achieved = flop_per_launch / (k_ms * 1e-3) / 1e12
        peak = pk["bf16_tflops"]
        # dram bytes per launch of the dominant kernel, from the committed `ncu --set full` capture of THIS kernel build
        kinfo = eng.kernel_info(a.precision) if hasattr(eng, "kernel_info") else {}
        kernel_name = kinfo.get("name", "nfb::v6::render2_kernel" if a.precision == "fast" else "nfb::render_kernel")
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", kinfo.get("ncu_json", "r1b_render_kernel_ncu.json"))
        if os.path.exists(tpath) and (H, W, nc, nf) == (512, 512, 64, 128):
            with open(tpath) as f:
                tj = json.load(f)
            if tj.get("block_size") in (None, kinfo.get("block_size")):
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), os.path.basename(tpath)

        cpu = None
        if not a.no_cpu_baseline:
            cores = pick_threads(H, W, nc, nf)
            run, crays = reference_frame_crop(0, H, W, 64, nc, nf, cores)
            run()
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                run()
                ts.append(time.perf_counter() - t0)
            cpu = {"value": crays / (sorted(ts)[1]), "unit": "rays/s", "cores": cores, "host_cores": os.cpu_count(),
                   "sample": CPU_SAMPLE + ", best of 8/16/32/64/all intra-op threads, 64x64 centre crop, median of 3"}
        line = {
            "metric": "rays/sec at 512x512 (64c+128f samples)", "value": value, "unit": "rays/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands / f32 accumulate (tcgen05)" if a.precision == "fast" else "f16 hi+lo split x3 / f32 accumulate (tcgen05)",
            "data": "synthetic",
            "config": {"workload": f"person_1-shaped eval: {H}x{W}, {nc} coarse + {nf} fine samples/ray, 76-dim expr + 32-dim latent, "
                                   f"one frame per GPU per step", "precision": a.precision, "parallelism": f"frame-per-gpu x{world}",
                       "l2": "flushed between timed steps (256 MB write outside the events)",
                       "parity_max_abs_vs_oracle": parity, "psnr_rgb_fine_db": psnr, "parity_rays": 2 * W,
                       "wall_s_timed_region": wall},
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": (76 + 32 + 3 * n) * 4,
                    "d2h_bytes_per_step": 11 * n * 4, "ms_per_step": ms_e2e / a.steps},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "frac_of_sustained": achieved / pk.get("bf16_tflops_sustained", peak), "peak_source": pk_src,
                         "kernel": kernel_name, "kernel_ms": k_ms, "flop_per_launch": flop_per_launch, "traffic": traffic,
                         "traffic_unit": "bytes of DRAM read+write per launch (ncu --set full" + (f", profiles/{traffic_src})" if traffic_src else "; no capture of this build)")},
            "cpu_baseline": cpu, "clocks": clocks,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
