#!/usr/bin/env python
"""Drive the reference's two command-line programs UNMODIFIED on the B200 render path (SURVEY.md §8b, §8f rank 1):

    train_transformed_rays.py  (callers of the path: :336-352 train, :488-504 in-loop validation, optimizer :391-399)
    eval_transformed_rays.py   (:449-467, plus its normal-map / PNG tail)

through 4d-facial-avatars_b200/run_reference_script.py, which only puts this repository's drop-in `nerf` package first on
sys.path (and, under torchrun, shards run_one_iter_of_nerf over the ranks — nerf/parallel.py).  The script bodies come from the
reference tree (the byte-for-byte copy oracle/stage_reference.py stages into oracle/_ref); the dataset is synthetic
(tools/make_synthetic_dataset.py); the YAML is the shipped paper-model config with only paths and iteration counts replaced.

    python tools/run_reference_clis.py --out gpurun_out/cli --gpus 1 --iters 40
    python tools/run_reference_clis.py --out gpurun_out/cli8 --gpus 8 --iters 40

Writes <out>/train_g<N>.log, <out>/eval_g<N>.log and a one-line JSON summary per program (iterations/s, seconds per image).
The unedited eval loop reads pose/expression 100 and the direction bundle of frame 240+i, so with 244 synthetic test frames it
renders 4 images and then ends with the reference's own IndexError at i = 4 (SURVEY.md §8b) — that exit is expected."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "cli"))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--test-frames", type=int, default=244)
    ap.add_argument("--port", type=int, default=29547)
    a = ap.parse_args()
    import ref_loader
    import make_synthetic_dataset as M
    train_py, eval_py = ref_loader.script_path("train_transformed_rays.py"), ref_loader.script_path("eval_transformed_rays.py")
    yml = ref_loader.script_path(os.path.join("config", "dave", "dave_dvp_lcode_fixed_bg_512_paper_model.yml"))
    if not train_py or not os.path.exists(train_py):
        sys.exit("no reference tree: run oracle/stage_reference.py --ref PATH_TO_REFERENCE_CHECKOUT first")
    out = os.path.abspath(a.out)
    data, logs = os.path.join(out, "data"), os.path.join(out, "logs")
    os.makedirs(out, exist_ok=True)
    if not os.path.exists(os.path.join(data, "transforms_test.json")):
        print(M.write_dataset(data, a.size, 12, 2, a.test_frames), flush=True)  # >= 11 train frames: the eval script reads latent code idx_map[10]
    cfg = open(yml).read()
    exp_id = f"synthetic_g{a.gpus}"
    subs = {r"^(\s*id:).*$": rf"\1 {exp_id}", r"^(\s*logdir:).*$": rf"\1 {logs}", r"^(\s*basedir:).*$": rf"\1 {data}",
            r"^(\s*train_iters:).*$": rf"\1 {a.iters}", r"^(\s*validate_every:).*$": rf"\1 {max(1, a.iters // 2)}",
            r"^(\s*save_every:).*$": rf"\1 {a.iters - 1}", r"^(\s*print_every:).*$": r"\1 10", r"^(\s*half_res:).*$": r"\1 False"}
    for pat, rep in subs.items():
        cfg, k = re.subn(pat, rep, cfg, count=1, flags=re.M)
        assert k == 1, pat
    cfg_path = os.path.join(out, f"{exp_id}.yml")
    open(cfg_path, "w").write(cfg)
    launcher = os.path.join(ROOT, "4d-facial-avatars_b200", "run_reference_script.py")
    prefix = [sys.executable]
    if a.gpus > 1:
        prefix += ["-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={a.gpus}", "--master-addr", "127.0.0.1",
                   "--master-port", str(a.port)]
    env = dict(os.environ, MPLBACKEND="Agg")
    summary = {"gpus": a.gpus, "size": a.size}

    def run(name, args, ok_codes=(0,)):
        log = os.path.join(out, f"{name}_g{a.gpus}.log")
        t0 = time.time()
        with open(log, "w") as f:
            rc = subprocess.run(prefix + [launcher] + args, stdout=f, stderr=subprocess.STDOUT, env=env, cwd=out).returncode
        dt = time.time() - t0
        text = open(log).read()
        print(f"[{name}] rc={rc} {dt:.1f}s -> {log}", flush=True)
        print("\n".join(text.strip().splitlines()[-6:]), flush=True)
        return rc, dt, text

    rc, dt, text = run("train", [train_py, "--config", cfg_path])
    its = re.findall(r"\[TRAIN\] Iter: (\d+) Loss: ([0-9.e+-]+)", text)
    summary["train"] = {"rc": rc, "wall_s": dt, "iters": a.iters, "printed": its[-3:], "validated": text.count("[VAL]")}
    ckpt = os.path.join(logs, exp_id, "checkpoint" + str(a.iters - 1).zfill(5) + ".ckpt")
    summary["train"]["checkpoint"] = os.path.exists(ckpt)
    if os.path.exists(ckpt):
        rc, dt, text = run("eval", [eval_py, "--config", cfg_path, "--checkpoint", ckpt, "--savedir", os.path.join(out, f"renders_g{a.gpus}")])
        per = re.findall(r"Avg time per image: ([0-9.e+-]+)", text)
        pngs = [f for f in os.listdir(os.path.join(out, f"renders_g{a.gpus}")) if f.endswith(".png")] if os.path.isdir(os.path.join(out, f"renders_g{a.gpus}")) else []
        summary["eval"] = {"rc": rc, "wall_s": dt, "avg_s_per_image": [float(p) for p in per], "images_written": len(pngs),
                           "ended_with_reference_IndexError": "IndexError" in text}
    print(json.dumps(summary), flush=True)
    with open(os.path.join(out, f"summary_g{a.gpus}.json"), "w") as f:
        json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
