"""Stage the UNMODIFIED reference files of the hot path (golden-data and tooling infrastructure, not product).

This recipe copies — byte for byte, nothing edited — the reference's `nerf` package, the two CLI scripts that call the
path and the shipped paper-model YAML from a reference checkout into `oracle/_ref/` (git-ignored: reference sources never
enter this repository's history; the directory can be carried to a GPU machine together with a copy of the tree).  It is
the offline "install" of a reference that has no setup.py.  Users of the staged copy (through oracle/ref_loader.py):

  * run_reference_script.py (tools/run_reference_clis.py): the unmodified train_transformed_rays.py /
    eval_transformed_rays.py with this repo's drop-in `nerf` package first on sys.path;
  * oracle/make_golden_reference_checks.py --ref oracle/_ref --cuda-products: the reference's post-render functions on a GPU.

    python oracle/stage_reference.py --ref PATH_TO_REFERENCE_CHECKOUT

Run it by hand where the reference tree is present; the build does not run it, and no test needs the staged copy (the tests
compare with golden data made by oracle/make_golden_reference_checks.py).
"""
import argparse
import hashlib
import json
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DEST = os.path.join(ROOT, "oracle", "_ref")
NP = os.path.join("nerface_code", "nerf-pytorch")
FILES = [os.path.join(NP, "nerf", f) for f in (
    "__init__.py", "cfgnode.py", "load_blender.py", "load_flame.py", "load_llff.py", "models.py", "nerf_helpers.py",
    "train_utils.py", "volume_rendering_utils.py")] + [
    os.path.join(NP, "train_transformed_rays.py"), os.path.join(NP, "eval_transformed_rays.py"),
    os.path.join(NP, "config", "dave", "dave_dvp_lcode_fixed_bg_512_paper_model.yml")]


def stage(ref_root, dest=DEST):
    """Copy FILES from ref_root to dest (same relative paths) + MANIFEST.json with their sha256.  Returns dest, or None
    when the reference tree is absent."""
    if not os.path.isdir(os.path.join(ref_root, NP)):
        return None
    manifest = {}
    for rel in FILES:
        src, dst = os.path.join(ref_root, rel), os.path.join(dest, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(src, dst)
        with open(dst, "rb") as f:
            manifest[rel] = hashlib.sha256(f.read()).hexdigest()
    with open(os.path.join(dest, "MANIFEST.json"), "w") as f:
        json.dump({"source": ref_root, "files": manifest}, f, indent=1)
    return dest


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True, help="root of the reference checkout (the directory holding nerface_code/)")
    a = ap.parse_args()
    d = stage(a.ref)
    print(d if d else f"{a.ref} not found: nothing staged")
