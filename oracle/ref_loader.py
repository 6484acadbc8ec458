"""Import the UNMODIFIED reference `nerf` package (test / baseline infrastructure only — never from the product).

Looks for the reference tree in oracle/_ref (the byte-for-byte copy staged by oracle/stage_reference.py; a script may point
CANDIDATES elsewhere).  The package is loaded under the alias
`nerf_reference`, so it never collides with this repository's drop-in package, which is importable as `nerf`.

Hot-path-unused dependencies that are absent from the image (SURVEY.md §8c: pytorch3d, torchsearchsorted, imageio) get
empty stand-in modules.  `relu_clone=True` applies the one patch BASELINE.md §4 names for gradient baselines on
torch >= 2: F.relu returns a clone, because `sigma_a[:, -1] += 1e-6` (volume_rendering_utils.py:53) otherwise trips
autograd's in-place check.  Mathematically identical."""
import importlib.util
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CANDIDATES = [os.path.join(ROOT, "oracle", "_ref")]
NP = os.path.join("nerface_code", "nerf-pytorch")


def reference_root():
    for c in CANDIDATES:
        if os.path.isfile(os.path.join(c, NP, "nerf", "train_utils.py")):
            return c
    return None


def script_path(name):
    """Absolute path of train_transformed_rays.py / eval_transformed_rays.py / a config YAML in the reference tree."""
    r = reference_root()
    return os.path.join(r, NP, name) if r else None


def load_reference(relu_clone=False):
    """Returns the reference package (module `nerf_reference`) or None when no reference tree is reachable."""
    if "nerf_reference" in sys.modules:
        return sys.modules["nerf_reference"]
    root = reference_root()
    if root is None:
        return None
    for name in ("pytorch3d", "pytorch3d.transforms", "torchsearchsorted", "imageio"):
        sys.modules.setdefault(name, types.ModuleType(name))
    if relu_clone:
        import torch
        orig = torch.nn.functional.relu
        if not getattr(orig, "_nfb_clone", False):
            def relu(x, *a, **k):
                return orig(x).clone()
            relu._nfb_clone = True
            torch.nn.functional.relu = relu
    pkg_dir = os.path.join(root, NP, "nerf")
    spec = importlib.util.spec_from_file_location("nerf_reference", os.path.join(pkg_dir, "__init__.py"),
                                                  submodule_search_locations=[pkg_dir])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["nerf_reference"] = mod
    try:
        spec.loader.exec_module(mod)
    except Exception:
        del sys.modules["nerf_reference"]
        raise
    mod.__nfb_root__ = root
    return mod


def make_cfg(ref, num_coarse, num_fine, perturb, noise_std, white_bkgd, chunksize, mode, near, far):
    blk = dict(num_coarse=num_coarse, num_fine=num_fine, perturb=perturb, lindisp=False, radiance_field_noise_std=noise_std,
               white_background=white_bkgd, chunksize=chunksize)
    return ref.CfgNode(dict(nerf={"use_viewdirs": True, mode: blk}, dataset=dict(no_ndc=True, near=near, far=far)))


def build_model(ref, params, device="cpu"):
    m = ref.models.ConditionalBlendshapePaperNeRFModel(
        num_encoding_fn_xyz=10, num_encoding_fn_dir=4, include_input_xyz=True, include_input_dir=False,
        use_viewdirs=True, include_expression=True, latent_code_dim=32)
    m.load_state_dict(params)
    return m.to(device)


def reference_renderer(ref, frame, params_c, params_f, H, W, rows, cols, nc, nf, device="cpu", chunksize=65536):
    """Closure running the reference's run_one_iter_of_nerf (validation mode, deterministic) on the pixel block
    rows x cols (slices) of the synthetic frame `frame` (nerface_oracle.synthetic_frame).  Returns (fn, n_rays)."""
    import torch
    mc = build_model(ref, params_c, device)
    mf = build_model(ref, params_f, device) if nf > 0 else None
    cfg = make_cfg(ref, nc, nf, False, 0.0, False, chunksize, "validation", 0.2, 0.8)
    pose = frame["pose"].to(device)
    import numpy as np
    ro, rd = ref.get_ray_bundle(H, W, np.array(frame["intrinsics"]), pose[:3, :4])
    ro, rd = ro[rows, cols].contiguous(), rd[rows, cols].contiguous()
    bg = frame["bg"].to(device)[rows, cols].reshape(-1, 3).contiguous()
    expr, latent = frame["expr"].to(device), frame["latent"].to(device)
    enc_xyz = ref.get_embedding_function(num_encoding_functions=10, include_input=True, log_sampling=True)
    enc_dir = ref.get_embedding_function(num_encoding_functions=4, include_input=False, log_sampling=True)
    h, w = ro.shape[0], ro.shape[1]

    def run():
        with torch.no_grad():
            return ref.run_one_iter_of_nerf(h, w, frame["intrinsics"], mc, mf, ro, rd, cfg, mode="validation",
                                            encode_position_fn=enc_xyz, encode_direction_fn=enc_dir, expressions=expr,
                                            background_prior=bg, latent_code=latent)
    return run, h * w


def load_eval_script(name="eval_transformed_rays.py"):
    """The reference's eval script as a module WITHOUT running main(): gives tests the unmodified post-render functions
    (torch_normal_map :84-119, cast_to_image :184-192, cast_to_disparity_image :195-198).  matplotlib / imageio get inert
    stand-ins when absent; `from nerf import ...` inside the script resolves to the reference package for the import only."""
    key = "nerf_reference_eval_script"
    if key in sys.modules:
        return sys.modules[key]
    ref = load_reference()
    path = script_path(name)
    if ref is None or not path or not os.path.exists(path):
        return None

    class _Anything:
        def __call__(self, *a, **k):
            return self

        def __getattr__(self, n):
            return self
    try:
        import matplotlib  # noqa: F401
        import matplotlib.pyplot  # noqa: F401
    except ImportError:
        anything = _Anything()

        def _attr(n):
            if n.startswith("__"):
                raise AttributeError(n)
            return anything
        mpl, plt = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
        mpl.__getattr__ = _attr
        plt.__getattr__ = _attr
        mpl.pyplot = plt
        sys.modules["matplotlib"], sys.modules["matplotlib.pyplot"] = mpl, plt
    saved = sys.modules.get("nerf")
    sys.modules["nerf"] = ref
    try:
        spec = importlib.util.spec_from_file_location(key, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)  # top level only defines functions; main() is behind __name__ == "__main__"
    finally:
        if saved is not None:
            sys.modules["nerf"] = saved
        else:
            del sys.modules["nerf"]
    sys.modules[key] = mod
    return mod
