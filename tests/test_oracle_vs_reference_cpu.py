"""The oracle against the UNMODIFIED reference on configurations the golden fixtures do not hold: the smallest sample counts the
kernels accept, a single fine sample, ragged chunk sizes, perturbation without noise, white background without a background
image, the direction-ablation input with every stochastic option on.  Every output must be bit-identical — the same statement
oracle/make_golden.py prints for the eight committed cases.

What the reference computed (rays, the torch.rand / torch.randn draws it made, its outputs) is stored in
tests/golden/reference_checks/oracle_cases.npz by oracle/make_golden_reference_checks.py.  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

import nerface_oracle as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import make_golden_reference_checks as G  # noqa: E402

CASES = G.ORACLE_CASES


@pytest.fixture(scope="module")
def gold():
    assert torch.get_float32_matmul_precision() == "highest"
    return np.load(os.path.join(G.OUT, "oracle_cases.npz"))


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_is_bit_identical_to_the_live_reference(gold, name):
    H, W, s, mode, use_bg, use_fine, stress, ablation = CASES[name]
    g = lambda k: torch.from_numpy(gold[f"{name}/{k}"])  # noqa: E731
    ci = 200 + list(CASES).index(name)
    near, far = 0.2, 0.8
    pc = O.random_init_params(300 + ci, stress)
    pf = O.random_init_params(400 + ci, stress) if use_fine else None
    fr = O.synthetic_frame(ci, H, W)
    ro, rd = g("ro"), g("rd")
    o_ro, o_rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    assert torch.equal(ro, o_ro) and torch.equal(rd, o_rd)
    if mode == "train":  # the trainer passes flat gathered rays (train_transformed_rays.py:320-326)
        ro, rd = ro.reshape(-1, 3).clone(), rd.reshape(-1, 3).clone()
    bg = fr["bg"].reshape(-1, 3) if use_bg else None
    rd_abl = g("rd_ablation") if ablation else None
    # the recorded draws, split back into the per-chunk order the reference made them in (train_utils.py:69-76, 105-119)
    noises = G.split_draws([g(f"draw{j}") for j in range(int(gold[f"{name}/n_draws"]))], s, H * W)
    with torch.no_grad():
        got = O.run_one_iter(ro, rd, pc, pf, s, near, far, fr["expr"], fr["latent"], bg, mode, noise_per_chunk=noises,
                             rd_ablation=rd_abl)
    assert len(got) == int(gold[f"{name}/arity"])
    for i, b in enumerate(got):
        key = f"{name}/out{i}"
        assert (key not in gold) == (b is None), i
        if b is not None:
            a = g(f"out{i}")
            assert a.shape == b.shape, (i, a.shape, b.shape)
            assert torch.equal(a, b), (name, i, float((a - b).abs().max()))
