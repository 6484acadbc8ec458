"""Golden vectors for the post-render products (SURVEY.md §8f rank 4), produced by the UNMODIFIED reference functions of
eval_transformed_rays.py — torch_normal_map (:84-119), cast_to_image (:184-192), cast_to_disparity_image (:195-198) — on the
disparity / weights / colours the oracle renders for a synthetic 64x64 frame with opaque-stress weights (so the disparity map
has structure and w_last crosses the 0.22 cleaning threshold).  Needs the copy oracle/stage_reference.py stages into oracle/_ref.

    python oracle/make_golden_products.py        ->  tests/golden_products/frame_products_64.npz
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import nerface_oracle as O  # noqa: E402
import ref_loader  # noqa: E402


def main():
    ev = ref_loader.load_eval_script()
    H = W = 64
    fr = O.synthetic_frame(21, H, W)
    pc, pf = O.random_init_params(100, True), O.random_init_params(101, True)
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    with torch.no_grad():
        out = O.run_one_iter(ro, rd, pc, pf, O.Sampling(64, 128, False, 0.0, False, 65536), 0.2, 0.8, fr["expr"], fr["latent"],
                             fr["bg"].reshape(-1, 3), "validation")
    rgb, disp, w_last = out[3].contiguous(), out[4].contiguous(), out[6].contiguous()
    focal = np.array(fr["intrinsics"])
    normals = ev.torch_normal_map(disp.clone(), focal, w_last.clone(), clean=True).numpy().astype("uint8")
    normals_noclean = ev.torch_normal_map(disp.clone(), focal, None, clean=True).numpy().astype("uint8")
    rgb_u8 = ev.cast_to_image(rgb[..., :3], "blender")
    disp_u8 = ev.cast_to_disparity_image(disp)
    dst = os.path.join(os.path.dirname(HERE), "tests", "golden_products")
    os.makedirs(dst, exist_ok=True)
    np.savez_compressed(os.path.join(dst, "frame_products_64.npz"), rgb=rgb.numpy(), disp=disp.numpy(), w_last=w_last.numpy(),
                        intrinsics=focal, normals_u8=normals, normals_noclean_u8=normals_noclean, rgb_u8=np.asarray(rgb_u8), disp_u8=disp_u8)
    print("wrote", dst, normals.shape, rgb_u8.shape, disp_u8.shape, "w_last > 0.22:", float((w_last > 0.22).float().mean()),
          "normal bytes min/max", normals.min(), normals.max())


if __name__ == "__main__":
    main()
