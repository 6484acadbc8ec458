"""Golden data for the tests that compare this project with the UNMODIFIED reference, so that they run from this repository
alone: it executes the reference (read-only) once and writes what each test compares against to tests/golden/reference_checks/.

  oracle_cases.npz      test_oracle_vs_reference_cpu.py: rays, ablation directions, recorded torch.rand / torch.randn draws and
                        the outputs of run_one_iter_of_nerf on six configurations outside the eight golden cases
  backward.npz          test_backward_reference_cpu.py: draws, outputs and loss of the training-mode forward, and the reference
                        autograd's gradients — the latent gradient and every tensor of at most GRAD_FULL entries (biases,
                        fc_alpha, fc_rgb) in full, each larger one as its max |g|, its sum of squares and a seeded sample of
                        GRAD_SAMPLES entries (the full set is 3 x 1.1 M floats)
  helpers.json          test_dropin_helpers_cpu.py: ray bundles, positional encodings, minibatches, metrics and the model class's
                        forward (digests: the test compares bit for bit), its state_dict layout, the CfgNode tree of the shipped
                        paper-model config
  dataset.json          test_dataset_cpu.py: digests of every member load_flame_data returns on the synthetic dataset
  products.json         test_post_gpu.py: digests of cast_to_image / torch_normal_map / cast_to_disparity_image bytes, computed
                        with torch CPU ("cpu") and with torch CUDA ("cuda"; the two back ends round the normal map differently)

    python oracle/make_golden_reference_checks.py --ref PATH_TO_REFERENCE_CHECKOUT                  (everything but "cuda")
    python oracle/make_golden_reference_checks.py --ref oracle/_ref --cuda-products   (on a GPU: adds "cuda" to products.json;
                                                                                        oracle/stage_reference.py stages oracle/_ref)
"""
import argparse
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import make_golden as MG  # noqa: E402
import nerface_oracle as O  # noqa: E402
import ref_loader  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_checks")
GRAD_FULL, GRAD_SAMPLES = 256, 128

# ---- shared with the tests: case tables and the digests they compare

# name: (H, W, Sampling(nc, nf, perturb, noise_std, white_bkgd, chunksize), mode, use_bg, use_fine, stress, ablation)
ORACLE_CASES = {
    "min_coarse_3c5f": (3, 4, O.Sampling(3, 5, False, 0.0, False, 65536), "validation", True, True, True, False),
    "one_fine_sample": (2, 5, O.Sampling(64, 1, False, 0.0, False, 65536), "validation", True, True, False, False),
    "ragged_chunks_train": (5, 3, O.Sampling(16, 8, True, 0.2, False, 7), "train", True, True, True, False),
    "perturb_only_white_nobg": (4, 4, O.Sampling(40, 72, True, 0.0, True, 65536), "validation", False, True, True, False),
    "noise_only_coarse_only": (4, 3, O.Sampling(24, 0, False, 0.3, False, 5), "train", True, False, False, False),
    # chunk size divides the ray count: with a ragged last chunk the reference itself raises (every chunk takes the FIRST chunk's
    # ablation directions, train_utils.py:82 — the quirk the oracle and the kernels reproduce)
    "ablation_all_stochastic": (3, 5, O.Sampling(32, 48, True, 0.1, False, 5), "validation", True, True, True, True),
}
BACKWARD_CASES = {"random_init": (False, False, True), "opaque_stress": (True, False, True), "opaque_stress_white_nobg": (True, True, False)}
RAY_BUNDLE_CASES = [(7, 5, [1200.0, 1250.0, 0.5, 0.5]), (4, 9, [-900.0, 910.0, 0.48, 0.53]), (16, 16, [333.3, -444.4, 0.1, 0.9])]
PE_CASES = [(10, True, True), (4, False, True), (6, True, False), (1, False, True), (0, True, True)]
MODEL_KW = dict(num_layers=8, hidden_size=256, skip_connect_every=3, num_encoding_fn_xyz=10, num_encoding_fn_dir=4,
                include_input_xyz=True, include_input_dir=False, use_viewdirs=True, include_expression=True, latent_code_dim=32)
MODEL_SEED = 11
LOADER_CALLS = [dict(half_res=False, testskip=1, test=True), dict(half_res=True, testskip=1), dict(half_res=False, testskip=2)]
PRODUCT_SIZES = (64, 512)


def pose_for(seed):
    g = torch.Generator().manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
    p = torch.eye(4)
    p[:3, :3] = q
    p[:3, 3] = torch.randn(3, generator=g) * 0.3
    return p


def grad_sample_index(numel, k):
    """Flat indices of the stored entries of parameter k's gradient: all of them up to GRAD_FULL, else a seeded sample."""
    if numel <= GRAD_FULL:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(1000 + k))[:GRAD_SAMPLES].sort().values


def product_inputs(H):
    gen = torch.Generator().manual_seed(H)
    d = torch.rand(H, H, generator=gen) * 4 + 1
    w = torch.rand(H, H, generator=gen) ** 3
    c = torch.rand(H, H, 3, generator=gen) * 1.2 - 0.1
    intr = np.array([1200.0 * H / 512, 1150.0 * H / 512, 0.52, 0.47])
    return c, d, w, intr


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def array_digest(a):
    a = np.asarray(a)
    return {"shape": list(a.shape), "dtype": str(a.dtype), "sha256": sha256(a)}


def describe(x):
    """What test_dataset_cpu compares of one member load_flame_data returns: tensors by shape and FP32 values, the [H, W, focal]
    list by value, lists of index arrays element by element."""
    if torch.is_tensor(x):
        return {"shape": list(x.shape), "sha256": sha256(x.float().numpy())}
    if isinstance(x, list) and len(x) == 3 and not isinstance(x[0], np.ndarray):
        return {"H": int(x[0]), "W": int(x[1]), "focal": [float(v) for v in np.asarray(x[2]).ravel()]}
    if isinstance(x, list):
        return {"arrays": [{"shape": list(np.shape(p)), "dtype": str(np.asarray(p).dtype), "sha256": sha256(np.asarray(p))} for p in x]}
    assert x is None, type(x)
    return None


def split_draws(draws, s, n_rays):
    """Recorded draws back into the per-chunk order the reference made them in (train_utils.py:69-76, 105-119)."""
    it = iter(draws)
    noises = []
    for _ in range(0, n_rays, s.chunksize):
        nz = O.Noise()
        if s.perturb:
            nz.t_rand = next(it)
        if s.noise_std > 0:
            nz.n_c = next(it)
        if s.num_fine > 0:
            if s.perturb:
                nz.u = next(it)
            if s.noise_std > 0:
                nz.n_f = next(it)
        noises.append(nz)
    assert next(it, None) is None, "the reference drew more random tensors than the oracle's model of it consumes"
    return noises


# ---- generation (needs the reference)

def oracle_cases(ref):
    save = {}
    near, far = 0.2, 0.8
    for ci0, (name, (H, W, s, mode, use_bg, use_fine, stress, ablation)) in enumerate(ORACLE_CASES.items()):
        ci = 200 + ci0
        pc = O.random_init_params(300 + ci, stress)
        pf = O.random_init_params(400 + ci, stress) if use_fine else None
        fr = O.synthetic_frame(ci, H, W)
        ro, rd = ref.get_ray_bundle(H, W, np.array(fr["intrinsics"]), fr["pose"][:3, :4])
        save[f"{name}/ro"], save[f"{name}/rd"] = ro.numpy(), rd.numpy()
        if mode == "train":
            ro, rd = ro.reshape(-1, 3).clone(), rd.reshape(-1, 3).clone()
        bg = fr["bg"].reshape(-1, 3) if use_bg else None
        rd_abl = None
        if ablation:
            fr2 = O.synthetic_frame(ci + 50, H, W)
            _, rd_abl = ref.get_ray_bundle(H, W, np.array(fr2["intrinsics"]), fr2["pose"][:3, :4])
            save[f"{name}/rd_ablation"] = rd_abl.numpy()
        mc = ref_loader.build_model(ref, pc)
        mf = ref_loader.build_model(ref, pf) if use_fine else None
        cfg = ref_loader.make_cfg(ref, s.num_coarse, s.num_fine, s.perturb, s.noise_std, s.white_bkgd, s.chunksize, mode, near, far)
        torch.manual_seed(4321 + ci)
        with torch.no_grad(), MG.Recorder() as rec:
            want = ref.run_one_iter_of_nerf(H, W, fr["intrinsics"], mc, mf, ro.clone(), rd.clone(), cfg, mode=mode,
                                            encode_position_fn=ref.get_embedding_function(10, True, True),
                                            encode_direction_fn=ref.get_embedding_function(4, False, True),
                                            expressions=fr["expr"], background_prior=bg, latent_code=fr["latent"],
                                            ray_directions_ablation=rd_abl)
        split_draws([t for _, t in rec.draws], s, H * W)
        save[f"{name}/n_draws"] = np.array(len(rec.draws))
        for j, (_, t) in enumerate(rec.draws):
            save[f"{name}/draw{j}"] = t.numpy()
        save[f"{name}/arity"] = np.array(len(want))
        for i, t in enumerate(want):
            if t is not None:
                save[f"{name}/out{i}"] = t.numpy()
    return save


def backward_cases(ref):
    import torch_reference as TR
    save = {}
    orig_relu = torch.nn.functional.relu
    # `sigma_a[:, -1] += 1e-6` (volume_rendering_utils.py:53) writes into F.relu's output in place, which torch >= 2 refuses to
    # differentiate through: the one patch BASELINE.md §4 names for gradient baselines — F.relu returns a copy, same values.
    torch.nn.functional.relu = lambda x, *a, **k: orig_relu(x).clone()
    try:
        for name, (stress, white, use_bg) in BACKWARD_CASES.items():
            H, W, nc, nf, near, far = 2, 5, 64, 64, 0.2, 0.8
            fr = O.synthetic_frame(31, H, W)
            pc, pf = O.random_init_params(100, stress), O.random_init_params(101, stress)
            ro, rd = ref.get_ray_bundle(H, W, np.array(fr["intrinsics"]), fr["pose"][:3, :4])
            ro, rd = ro.reshape(-1, 3).clone(), rd.reshape(-1, 3).clone()
            bg = fr["bg"].reshape(-1, 3) if use_bg else None
            target = torch.rand(ro.shape[0], 3, generator=torch.Generator().manual_seed(5))
            mc, mf = ref_loader.build_model(ref, pc), ref_loader.build_model(ref, pf)
            lat = fr["latent"].clone().requires_grad_(True)
            cfg = ref_loader.make_cfg(ref, nc, nf, True, 0.1, white, 2048, "train", near, far)
            torch.manual_seed(77)
            with MG.Recorder() as rec:
                out = ref.run_one_iter_of_nerf(H, W, fr["intrinsics"], mc, mf, ro.clone(), rd.clone(), cfg, mode="train",
                                               encode_position_fn=ref.get_embedding_function(10, True, True),
                                               encode_direction_fn=ref.get_embedding_function(4, False, True),
                                               expressions=fr["expr"], background_prior=bg, latent_code=lat)
            loss = torch.nn.functional.mse_loss(out[0][..., :3], target) + torch.nn.functional.mse_loss(out[3][..., :3], target)
            loss.backward()
            save[f"{name}/ro"], save[f"{name}/rd"] = ro.numpy(), rd.numpy()
            for j, (_, t) in enumerate(rec.draws):
                save[f"{name}/draw{j}"] = t.numpy()
            for i, t in enumerate(out):
                save[f"{name}/out{i}"] = t.detach().numpy()
            save[f"{name}/loss"] = np.array(float(loss.detach()), dtype=np.float32)
            save[f"{name}/grad_latent"] = lat.grad.numpy()
            # [coarse, fine] x PARAM_ORDER; NaN where the reference leaves the gradient None.  The stored entries of every
            # gradient, in that order, concatenated into one array
            max_abs = np.full((2, len(TR.PARAM_ORDER)), np.nan, dtype=np.float32)
            sum_sq = np.full((2, len(TR.PARAM_ORDER)), np.nan, dtype=np.float64)
            sample = []
            for m_i, model in enumerate((mc, mf)):
                named = dict(model.named_parameters())
                for k, pname in enumerate(TR.PARAM_ORDER):
                    g = named[pname].grad
                    if g is None:
                        continue
                    flat = g.reshape(-1)
                    max_abs[m_i, k] = float(flat.abs().max())
                    sum_sq[m_i, k] = float((flat.double() ** 2).sum())
                    sample.append(flat[grad_sample_index(flat.numel(), k)].numpy())
            save[f"{name}/grad_max_abs"], save[f"{name}/grad_sum_sq"] = max_abs, sum_sq
            save[f"{name}/grad_sample"] = np.concatenate(sample)
    finally:
        torch.nn.functional.relu = orig_relu
    return save


def helpers(ref):
    import yaml
    save = {}
    for H, W, intr in RAY_BUNDLE_CASES:
        ro, rd = ref.get_ray_bundle(H, W, np.array(intr), pose_for(H * 100 + W)[:3, :4])
        save[f"ray_bundle/{H}x{W}/ro"], save[f"ray_bundle/{H}x{W}/rd"] = ro.numpy(), rd.numpy()
    for n_freq, include_input, log_sampling in PE_CASES:
        x = torch.randn(37, 3, generator=torch.Generator().manual_seed(n_freq)) * 3.0
        key = f"pe/{n_freq}/{int(include_input)}/{int(log_sampling)}"
        pe = ref.positional_encoding(x, n_freq, include_input, log_sampling)
        assert torch.equal(ref.get_embedding_function(n_freq, include_input, log_sampling)(x), pe)  # the tests check both on one array
        save[key] = pe.numpy()
    a, b = torch.arange(5, dtype=torch.float32), torch.arange(3, dtype=torch.float32) * 2.0
    for i, t in enumerate(ref.meshgrid_xy(a, b)):
        save[f"meshgrid/{i}"] = t.numpy()
    x = torch.randn(23, 4, generator=torch.Generator().manual_seed(3))
    for cs in (1, 7, 23, 100):
        mb = ref.get_minibatches(x, chunksize=cs)
        save[f"minibatches/{cs}/n"] = np.array(len(mb))
        for i, t in enumerate(mb):
            save[f"minibatches/{cs}/{i}"] = t.numpy()
    y = torch.randn(23, 4, generator=torch.Generator().manual_seed(4))
    save["img2mse"] = ref.img2mse(x, y).numpy()
    save["mse2psnr"] = np.array([ref.mse2psnr(m) for m in (0.0, 1e-5, 0.0123, 1.0)], dtype=np.float64)
    m = ref.models.ConditionalBlendshapePaperNeRFModel(**MODEL_KW)
    m.load_state_dict(O.random_init_params(MODEL_SEED), strict=True)
    g = torch.Generator().manual_seed(12)
    x = torch.randn(19, m.dim_xyz + m.dim_dir, generator=g)
    expr, lat = torch.randn(76, generator=g), torch.randn(32, generator=g)
    with torch.no_grad():
        save["model/forward"] = m(x, expr, lat).numpy()

    path = ref_loader.script_path(os.path.join("config", "dave", "dave_dvp_lcode_fixed_bg_512_paper_model.yml"))
    with open(path) as f:
        raw = yaml.load(f, Loader=yaml.FullLoader)
    cfg = ref.CfgNode(raw)
    leaves = []

    def walk(node, trail):
        for k in node.keys():
            v = getattr(node, k)
            if isinstance(v, dict):
                walk(v, trail + [k])
            else:
                leaves.append([trail + [k], type(v).__name__, v])
    walk(cfg, [])
    meta = {"state_dict": [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()],
            "attributes": {n: getattr(m, n) for n in ("dim_xyz", "dim_dir", "dim_expression", "dim_latent_code", "use_viewdirs")},
            "n_parameters": sum(p.numel() for p in m.parameters()),
            "config": raw, "config_leaves": leaves, "config_dump": yaml.safe_load(cfg.dump())}
    return save, meta


def dataset(ref):
    import cv2
    import make_synthetic_dataset
    sys.modules["imageio"].imread = lambda p: cv2.imread(p, cv2.IMREAD_UNCHANGED)[..., ::-1]
    with tempfile.TemporaryDirectory() as d:
        make_synthetic_dataset.write_dataset(d, 32, 3, 1, 4)
        return {"calls": [{"kwargs": kw, "members": [describe(x) for x in ref.load_flame_data(d, **kw)]} for kw in LOADER_CALLS]}


def products(device="cpu"):
    """The reference's post-render bytes on product_inputs, with the torch back end of `device`."""
    ev = ref_loader.load_eval_script()
    res = {}
    for H in PRODUCT_SIZES:
        c, d, w, intr = (t.to(device) if torch.is_tensor(t) else t for t in product_inputs(H))
        n = ev.torch_normal_map(d.clone(), intr, w.clone(), clean=True).cpu().numpy().astype("uint8")
        res[str(H)] = {name: {"shape": list(a.shape), "sha256": sha256(a)} for name, a in
                       (("rgb", np.asarray(ev.cast_to_image(c, "blender"))), ("normals", n), ("disparity", ev.cast_to_disparity_image(d)))}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True, help="root of the reference checkout (the directory holding nerface_code/)")
    ap.add_argument("--cuda-products", action="store_true", help="only add the torch-CUDA digests to products.json (needs a GPU)")
    a = ap.parse_args()
    assert torch.get_float32_matmul_precision() == "highest"
    ref_loader.CANDIDATES[:] = [os.path.abspath(a.ref)]
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    ref = ref_loader.load_reference()
    assert ref is not None, f"no reference package under {a.ref}"
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, "products.json")
    if a.cuda_products:
        with open(path) as f:
            digests = json.load(f)
        digests["cuda"] = products("cuda")
        with open(path, "w") as f:
            json.dump(digests, f, indent=1)
            f.write("\n")
        print(json.dumps(digests["cuda"], indent=1))
        return
    np.savez_compressed(os.path.join(OUT, "oracle_cases.npz"), **oracle_cases(ref))
    np.savez_compressed(os.path.join(OUT, "backward.npz"), **backward_cases(ref))
    save, meta = helpers(ref)
    meta["values"] = {k: v.tolist() for k, v in save.items() if k.endswith("/n") or k == "mse2psnr"}
    meta["arrays"] = {k: array_digest(v) for k, v in save.items() if k not in meta["values"]}
    digests = {"cpu": products("cpu")}
    if os.path.exists(path):  # keep the torch-CUDA digests, which only a GPU can make
        with open(path) as f:
            digests["cuda"] = json.load(f).get("cuda")
    for name, obj in (("helpers.json", meta), ("dataset.json", dataset(ref)), ("products.json", digests)):
        with open(os.path.join(OUT, name), "w") as f:
            json.dump(obj, f, indent=1)
            f.write("\n")
    for f in sorted(os.listdir(OUT)):
        print(f"{f:20s} {os.path.getsize(os.path.join(OUT, f)):>8d} bytes")


if __name__ == "__main__":
    main()
