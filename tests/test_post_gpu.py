"""The steps either side of the render path on the device (SURVEY.md §8f ranks 3, 4): the training-ray sampler against
np.random.choice itself, and the post-render 8-bit products against golden vectors made by the reference's own functions
(oracle/make_golden_products.py) — bit-exact indices, bit-exact bytes."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden_products", "frame_products_64.npz")


@pytest.fixture(scope="module")
def env(built_lib):
    import nerf
    from nerf import ray_sampler
    return nerf, ray_sampler, torch.device("cuda", 0)


def numpy_choice_with_recorded_draws(n_pix, size, p, seed):
    """np.random.choice(n_pix, size, replace=False, p=p) twice from the same seed: once for real (the expected indices), once
    re-enacting RandomState.choice's loop with explicit np.random.rand calls to record the uniform draws it consumes."""
    np.random.seed(seed)
    expected = np.random.choice(n_pix, size=size, replace=False, p=p)
    np.random.seed(seed)
    draws, found, pp = [], np.zeros(0, dtype=np.int64), p.copy()
    while found.size < size:
        x = np.random.rand(size - found.size)
        draws.append(x)
        if found.size:
            pp[found] = 0
        cdf = np.cumsum(pp)
        cdf /= cdf[-1]
        new = cdf.searchsorted(x, side="right")
        _, first = np.unique(new, return_index=True)
        first.sort()
        found = np.concatenate((found, new.take(first)))
    assert np.array_equal(found, expected)  # the re-enactment IS numpy's algorithm
    return expected, draws


@pytest.mark.parametrize("H,W,bbox,size,seed", [(512, 512, (150, 400, 128, 380), 2048, 42), (128, 128, (20, 100, 30, 90), 2048, 7),
                                                 (96, 160, (0, 96, 0, 160), 777, 3), (64, 64, (10, 14, 12, 15), 2048, 5)])
def test_ray_sampler_matches_numpy_choice(env, H, W, bbox, size, seed):
    """Same draws -> same indices as np.random.choice, in the same order (the 64x64 case needs many rounds: half the pixels are
    drawn from a 12-pixel box with 90 % weight each... the duplicates are many).  Gathers use the reference's transposed indexing."""
    nerf, ray_sampler, dev = env
    smp = ray_sampler.RaySampler(H, W, [bbox], p=0.9, size=size, device=dev)
    _, flat = ray_sampler.importance_map(H, W, bbox, 0.9)
    expected, draws = numpy_choice_with_recorded_draws(H * W, size, flat, seed)
    g = torch.Generator().manual_seed(seed)
    image, bg = torch.rand(H, W, 3, generator=g), torch.rand(H, W, 3, generator=g)
    import nerface_oracle as O
    fr = O.synthetic_frame(seed, H, W)
    d = torch.from_numpy(np.concatenate(draws)).to(dev)
    out = smp.sample(0, draws=d, pose=fr["pose"], intrinsics=fr["intrinsics"], image=image, background=bg, max_rounds=64)
    torch.cuda.synchronize()
    st = out["state"].cpu().tolist()
    assert st[0] == size and st[1] == len(draws) and st[2] == sum(x.size for x in draws), (st, len(draws))
    got = out["indices"].cpu().numpy()
    assert np.array_equal(got, expected)
    # train_transformed_rays.py:303-331: coords[k] = (k % H, k // H); rays, target, background gathered at that pixel
    rows, cols = expected % H, expected // H
    assert np.array_equal(out["pixel_rc"].cpu().numpy(), np.stack((rows, cols), axis=1))
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    if H == W:  # the reference indexes [k % H, k // H] into [H, W] arrays: in range for every k only when H >= W ... square here
        assert torch.equal(out["ray_directions"].cpu(), rd[rows, cols]) and torch.equal(out["ray_origins"].cpu(), ro[rows, cols])
        assert torch.equal(out["target"].cpu(), image[rows, cols]) and torch.equal(out["background"].cpu(), bg[rows, cols])


def test_ray_sampler_numpy_lockstep_and_device_rng(env):
    """numpy_lockstep: the global numpy stream advances exactly as the reference's np.random.choice call would, so the rest of an
    unmodified script stays on its seeded trajectory.  Device-RNG mode: distinct, in-range, box-weighted."""
    nerf, ray_sampler, dev = env
    H = W = 256
    bbox = (60, 200, 80, 180)
    smp = ray_sampler.RaySampler(H, W, [bbox], size=2048, device=dev)
    _, flat = ray_sampler.importance_map(H, W, bbox, 0.9)
    np.random.seed(11)
    expected = np.random.choice(H * W, size=2048, replace=False, p=flat)
    after_ref = np.random.rand()
    np.random.seed(11)
    out = smp.sample(0, numpy_lockstep=True)
    after_ours = np.random.rand()
    assert np.array_equal(out["indices"].cpu().numpy(), expected) and after_ours == after_ref
    out = smp.sample(0)
    idx = out["indices"].cpu().numpy()
    assert int(out["state"][0]) == 2048 and len(set(idx.tolist())) == 2048 and idx.min() >= 0 and idx.max() < H * W
    inside = ((idx // W >= bbox[0]) & (idx // W < bbox[1]) & (idx % W >= bbox[2]) & (idx % W < bbox[3])).mean()
    area = (bbox[1] - bbox[0]) * (bbox[3] - bbox[2]) / (H * W)
    expect_inside = 0.9 * area / (0.9 * area + 0.1 * (1 - area))
    assert abs(inside - expect_inside) < 0.05


def test_frame_products_match_the_reference_functions(env):
    """cast_to_image / torch_normal_map(clean=True) / cast_to_disparity_image bytes against the reference functions' outputs on the
    same FP32 inputs: with NFB_PRODUCTS_LIKE_TORCH_CPU against the functions run with CPU torch, in full at 64x64 (golden_products)
    and as digests of the whole frame at 64x64 and 512x512; in the default mode against the functions run with torch CUDA on a
    B200 (what the unmodified eval script computes on a GPU), as digests at 64x64 and 512x512 (golden/reference_checks/products.json,
    oracle/make_golden_reference_checks.py)."""
    import json
    import sys

    nerf, ray_sampler, dev = env
    g = np.load(GOLD)
    rgb, disp, w_last = (torch.from_numpy(g[k]).to(dev) for k in ("rgb", "disp", "w_last"))
    rgb_u8, normals_u8, disp_u8 = ray_sampler.frame_products(rgb, disp, w_last, list(g["intrinsics"]), want_disparity=True, like_torch_cpu=True)
    _, normals_nc, _ = ray_sampler.frame_products(rgb, disp, None, list(g["intrinsics"]), like_torch_cpu=True)
    torch.cuda.synchronize()
    for name, got, ref in (("rgb", rgb_u8, g["rgb_u8"]), ("normals", normals_u8, g["normals_u8"]), ("disparity", disp_u8, g["disp_u8"]),
                           ("normals, no cleaning", normals_nc, g["normals_noclean_u8"])):
        got = got.cpu().numpy()
        assert got.shape == ref.shape and got.dtype == np.uint8, name
        bad = int((got != ref).sum())
        assert bad == 0, (name, bad, int(np.abs(got.astype(int) - ref.astype(int)).max()))
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import make_golden_reference_checks as G
    with open(os.path.join(G.OUT, "products.json")) as f:
        digests = json.load(f)
    for H in G.PRODUCT_SIZES:
        c, d, w, intr = (t.to(dev) if torch.is_tensor(t) else t for t in G.product_inputs(H))
        for backend, like_cpu in (("cpu", True), ("cuda", False)):
            got = ray_sampler.frame_products(c, d, w, list(intr), want_disparity=True, like_torch_cpu=like_cpu)
            for name, t in zip(("rgb", "normals", "disparity"), got):
                t, want = t.cpu().numpy(), digests[backend][str(H)][name]
                assert t.dtype == np.uint8 and list(t.shape) == want["shape"] and G.sha256(t) == want["sha256"], (backend, H, name)
