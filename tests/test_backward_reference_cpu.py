"""Pins the floating-point reference of the fused backward kernels (tests/torch_reference.py: render_at_depths, what
tests/test_backward_gpu.py compares the CUDA gradients with) to the UNMODIFIED reference's own autograd: the training loss of
train_transformed_rays.py:355-389 (mse of the coarse and the fine colour against the target) back-propagated through the
reference's run_one_iter_of_nerf (mode "train", perturbation and sigma noise on, background image) and through render_at_depths at
the depths the reference sampled; parameter gradients of both networks and the latent-code gradient must agree to FP32 rounding.

So the chain for SURVEY.md §8 row a11 is: CUDA backward  <->  torch_reference (GPU tests)  <->  reference autograd (this file).
The reference's rays, draws, outputs, loss and gradients are stored in tests/golden/reference_checks/backward.npz by
oracle/make_golden_reference_checks.py: the latent gradient and the small parameter gradients in full, each larger one as its
largest magnitude, its sum of squares and a seeded sample of entries.  CPU only."""
import math
import os
import sys

import numpy as np
import pytest
import torch

import nerface_oracle as O
import torch_reference as TR

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import make_golden_reference_checks as G  # noqa: E402


@pytest.mark.parametrize("name", list(G.BACKWARD_CASES))
def test_torch_reference_gradients_equal_reference_autograd(name, monkeypatch):
    stress, white, use_bg = G.BACKWARD_CASES[name]
    gold = np.load(os.path.join(G.OUT, "backward.npz"))
    g = lambda k: torch.from_numpy(gold[f"{name}/{k}"])  # noqa: E731
    # the reference's gradients were taken with F.relu returning a copy (`sigma_a[:, -1] += 1e-6`, volume_rendering_utils.py:53,
    # writes into its output in place, which torch >= 2 refuses to differentiate through; BASELINE.md §4): same values, same gradients
    orig_relu = torch.nn.functional.relu
    monkeypatch.setattr(torch.nn.functional, "relu", lambda x, *a, **k: orig_relu(x).clone())
    H, W, nc, nf, near, far = 2, 5, 64, 64, 0.2, 0.8
    s = O.Sampling(nc, nf, True, 0.1, white, 2048)
    fr = O.synthetic_frame(31, H, W)
    pc, pf = O.random_init_params(100, stress), O.random_init_params(101, stress)
    ro, rd = g("ro"), g("rd")
    o_ro, o_rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    assert torch.equal(ro, o_ro.reshape(-1, 3)) and torch.equal(rd, o_rd.reshape(-1, 3))
    n = ro.shape[0]
    bg = fr["bg"].reshape(-1, 3) if use_bg else None
    target = torch.rand(n, 3, generator=torch.Generator().manual_seed(5))
    out = [g(f"out{i}") for i in range(7)]
    loss_ref = float(gold[f"{name}/loss"])
    # rand[N,Nc], randn[N,Nc], rand[N,Nf], randn[N,Nc+Nf] (train_utils.py:69-76, 105-119)
    draws = [g(f"draw{j}") for j in range(4)]
    assert f"{name}/draw4" not in gold
    noise = O.Noise(t_rand=draws[0], n_c=draws[1], u=draws[2], n_f=draws[3])

    # ---- the depths the reference sampled (the oracle reproduces the forward bit for bit, test_oracle_vs_reference_cpu.py)
    rays = torch.cat((ro, rd, near * torch.ones_like(rd[:, :1]), far * torch.ones_like(rd[:, :1])), dim=-1)
    ex = {}
    with torch.no_grad():
        o_out = O.render_chunk(rays, pc, pf, s, fr["expr"], fr["latent"], bg, noise, extras=ex)
    for a, b in zip(out, o_out):
        assert torch.equal(a, b)

    # ---- the backward tests' floating-point reference at those depths
    lc = {k: v.clone().requires_grad_(True) for k, v in pc.items()}
    lf = {k: v.clone().requires_grad_(True) for k, v in pf.items()}
    lat = fr["latent"].clone().requires_grad_(True)
    got = TR.render_at_depths(rays, lc, lf, fr["expr"], lat, ex["z_coarse"], ex["z_fine"], near, far, 0.1,
                              {"n_c": noise.n_c, "n_f": noise.n_f}, white, bg, None)
    for i in (0, 1, 2, 3, 4, 5, 6):
        assert float((got[i].detach() - out[i]).abs().max()) <= 2e-6 * max(1.0, float(out[i].abs().max())), i
    loss = torch.nn.functional.mse_loss(got[0], target) + torch.nn.functional.mse_loss(got[3], target)
    assert abs(float(loss.detach()) - loss_ref) <= 1e-7
    loss.backward()

    def close(a, b, what, scale=None):
        scale = max(float(b.abs().max()), 1e-12) if scale is None else scale
        assert float((a - b).abs().max()) <= 2e-5 * scale, (what, float((a - b).abs().max()), scale)

    # max |g_ours - g_ref| <= 2e-5 max|g_ref| over every entry implies it on the stored entries, for the largest magnitudes and,
    # summed over the n entries, |  ||g_ours|| - ||g_ref||  | <= sqrt(n) 2e-5 max|g_ref|
    max_abs, sum_sq, stored = gold[f"{name}/grad_max_abs"], gold[f"{name}/grad_sum_sq"], torch.from_numpy(gold[f"{name}/grad_sample"])
    n_checked, at = 0, 0
    for m_i, (leaves, tag) in enumerate(((lc, "coarse"), (lf, "fine"))):
        for k, pname in enumerate(TR.PARAM_ORDER):
            grad = leaves[pname].grad
            if pname.startswith("layers_dir.3"):  # built by the reference model but never used by its forward (models.py:257)
                assert np.isnan(max_abs[m_i, k]) and grad is None
                continue
            assert not np.isnan(max_abs[m_i, k]) and grad is not None, (tag, pname)
            flat, scale = grad.reshape(-1), max(float(max_abs[m_i, k]), 1e-12)
            idx = G.grad_sample_index(flat.numel(), k)
            close(flat[idx], stored[at:at + idx.numel()], (tag, pname, "entries"), scale)
            at += idx.numel()
            assert abs(float(flat.abs().max()) - float(max_abs[m_i, k])) <= 2e-5 * scale, (tag, pname, "max")
            norm, norm_ref = math.sqrt(float((flat.double() ** 2).sum())), math.sqrt(float(sum_sq[m_i, k]))
            assert abs(norm - norm_ref) <= 2e-5 * scale * math.sqrt(flat.numel()), (tag, pname, "norm", norm, norm_ref)
            n_checked += 1
    assert n_checked == 2 * 24 and at == stored.numel()
    lat_ref = g("grad_latent")
    close(lat.grad, lat_ref, "latent")
    assert float(lat_ref.abs().max()) > 0


@pytest.mark.parametrize("white,use_bg", [(False, True), (True, False)], ids=["bg", "white_nobg"])
def test_masked_reference_reproduces_unmasked_gradients(white, use_bg):
    """render_at_depths(masks=...) with the ReLU decisions a > 0 of an unmasked run gives, in FP64, the unmasked run's outputs and
    gradients exactly: the masked reference the GPU tests evaluate with the kernel's own decisions differs from the plain one only
    where those decisions differ."""
    torch.manual_seed(0)
    n, nc, nf, near, far = 5, 16, 24, 0.2, 0.8
    fr = O.synthetic_frame(7, 1, n)
    ro, rd = (t.reshape(-1, 3).double() for t in O.ray_bundle(1, n, fr["intrinsics"], fr["pose"]))
    rays = torch.cat((ro, rd, torch.full((n, 1), near, dtype=torch.float64), torch.full((n, 1), far, dtype=torch.float64)), dim=-1)
    z_c = near + (far - near) * torch.sort(torch.rand(n, nc, dtype=torch.float64), dim=-1).values
    z_f = torch.sort(torch.cat((z_c, near + (far - near) * torch.rand(n, nf, dtype=torch.float64)), dim=-1), dim=-1).values
    noise = {"n_c": torch.randn(n, nc, dtype=torch.float64), "n_f": torch.randn(n, nc + nf, dtype=torch.float64)}
    bg = fr["bg"].reshape(-1, 3).double() if use_bg else None
    dir_z = torch.rand(n, dtype=torch.float64) * 2.0 - 1.0
    expr = fr["expr"].double()
    params = [{k: v.double() for k, v in O.random_init_params(seed).items()} for seed in (100, 101)]

    def run(masks):
        lc, lf = ({k: v.clone().requires_grad_(True) for k, v in p.items()} for p in params)
        lat = fr["latent"].double().requires_grad_(True)
        taps = {}
        out = TR.render_at_depths(rays, lc, lf, expr, lat, z_c, z_f, near, far, 0.1, noise, white, bg, dir_z, taps, masks)
        gen = torch.Generator().manual_seed(3)
        torch.autograd.backward(out, [torch.randn(o.shape, generator=gen, dtype=torch.float64) for o in out])
        grads = [leaves[k].grad for leaves in (lc, lf) for k in TR.PARAM_ORDER] + [lat.grad]
        return [o.detach() for o in out], grads, taps

    out, grads, taps = run(None)
    masks = {key: [taps[key][f"a{i}"].detach() > 0 for i in range(9)] for key in ("coarse", "fine")}
    assert all(bool(m.any()) and not bool(m.all()) for ms in masks.values() for m in ms)
    m_out, m_grads, m_taps = run(masks)
    for a, b in zip(out, m_out):
        assert torch.equal(a, b)
    for k, a, b in zip([f"coarse {k}" for k in TR.PARAM_ORDER] + [f"fine {k}" for k in TR.PARAM_ORDER] + ["latent"], grads, m_grads):
        assert (a is None) == (b is None), k
        if a is not None:
            assert a.dtype == torch.float64 and torch.equal(a, b), k
    for key in ("coarse", "fine"):
        for i in range(9):
            assert torch.equal(taps[key][f"a{i}"].grad, m_taps[key][f"a{i}"].grad), (key, i)
        assert torch.equal(taps[key]["raw"].grad, m_taps[key]["raw"].grad), key
