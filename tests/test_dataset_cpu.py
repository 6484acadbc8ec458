"""The dataset layout either side of the render path (SURVEY.md §8f): tools/make_synthetic_dataset.py writes what the
reference's scripts read, nerf.load_flame_data (the drop-in for nerf/load_flame.py:40-211) reads it back.  CPU only."""
import importlib.util
import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _writer():
    spec = importlib.util.spec_from_file_location("make_synthetic_dataset", os.path.join(ROOT, "tools", "make_synthetic_dataset.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_round_trip_through_load_flame_data(tmp_path, built_lib):
    import nerf
    info = _writer().write_dataset(str(tmp_path), size=16, n_train=3, n_val=2, n_test=4, seed=7)
    for name in ("transforms_train.json", "transforms_val.json", "transforms_test.json", "index_map.npy", os.path.join("bg", "00050.png")):
        assert os.path.exists(tmp_path / name), name
    imgs, poses, render_poses, hwk, i_split, exprs, frontal, bboxs = nerf.load_flame_data(str(tmp_path), half_res=False, testskip=1)
    n = 3 + 2 + 4
    assert imgs.shape == (n, 16, 16, 3) and imgs.dtype == torch.float32 and 0.0 <= float(imgs.min()) and float(imgs.max()) <= 1.0
    assert poses.shape == (n, 4, 4) and exprs.shape == (n, 76) and bboxs.shape == (n, 4) and bboxs.dtype == torch.int32
    assert [len(s) for s in i_split] == [3, 2, 4] and i_split[2][0] == 5
    H, W, intr = hwk
    assert (H, W) == (16, 16) and np.allclose(intr, info["intrinsics"])
    meta = json.load(open(tmp_path / "transforms_train.json"))
    f0 = meta["frames"][0]
    assert np.allclose(poses[0].numpy(), np.array(f0["transform_matrix"], dtype=np.float32))
    assert np.allclose(exprs[0].numpy(), np.array(f0["expression"], dtype=np.float32))
    # bbox: relative (row_lo, row_hi, col_lo, col_hi) scaled by H, H, W, W and floored, as the reference does
    assert bboxs[0].tolist() == [int(np.floor(f0["bbox"][0] * H)), int(np.floor(f0["bbox"][1] * H)),
                                 int(np.floor(f0["bbox"][2] * W)), int(np.floor(f0["bbox"][3] * W))]
    # the rotation block is orthonormal and the camera sits at distance 0.5
    r = poses[:, :3, :3]
    assert torch.allclose(r @ r.transpose(1, 2), torch.eye(3).expand(n, 3, 3), atol=1e-5)
    assert torch.allclose(poses[:, :3, 3].norm(dim=1), torch.full((n,), 0.5), atol=1e-6)
    # test=True: the test split only (images included, as the reference returns them)
    imgs_t, poses_t, _, hwk_t, i_t, exprs_t, _, _ = nerf.load_flame_data(str(tmp_path), test=True)
    assert imgs_t.shape == (4, 16, 16, 3) and poses_t.shape == (4, 4, 4) and exprs_t.shape == (4, 76) and hwk_t[:2] == [16, 16]
    # half resolution halves the focal lengths and the images
    imgs_h, _, _, hwk_h, _, _, _, _ = nerf.load_flame_data(str(tmp_path), half_res=True)
    assert imgs_h.shape == (n, 8, 8, 3) and np.allclose(hwk_h[2][:2], np.array(info["intrinsics"][:2]) * 0.5)


def test_loader_matches_the_reference_loader(tmp_path, built_lib):
    """nerf.load_flame_data against the UNMODIFIED reference loader (nerf/load_flame.py:40-211) on the same synthetic dataset:
    every returned member equal, for the train and the test-only call, with and without half_res.  The reference loader's
    members are stored as digests of their values in tests/golden/reference_checks/dataset.json
    (oracle/make_golden_reference_checks.py)."""
    import sys

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import make_golden_reference_checks as G
    import nerf
    with open(os.path.join(G.OUT, "dataset.json")) as f:
        gold = json.load(f)["calls"]
    _writer().write_dataset(str(tmp_path), 32, 3, 1, 4)
    assert [c["kwargs"] for c in gold] == G.LOADER_CALLS
    for call in gold:
        got = nerf.load_flame_data(str(tmp_path), **call["kwargs"])
        assert len(got) == len(call["members"]) == 8
        for i, (want, y) in enumerate(zip(call["members"], got)):
            assert G.describe(y) == want, (call["kwargs"], i)
