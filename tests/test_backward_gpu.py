"""Fused backward (csrc/nfb_train.cu) stage by stage against a plain-PyTorch FP32 restatement on the same device
(tests/torch_reference.py, TF32 off), evaluated at the depths the fused forward sampled:

  saved state   : colours / ReLU inputs of sigma, FP16 activation images, ReLU masks      (forward, SAVE variant)
  composite bwd : dL/d(rgb_raw, sigma_raw) per sample
  chain         : dL/d(pre-activation) of every layer, as stored in the tile records
  dW + finalize : parameter and latent-code gradients in the reference's layout

Tolerances are relative to the largest reference magnitude of the tensor compared (FP16 operands, FP32 accumulate)."""
import ctypes as C

import numpy as np
import pytest
import torch

import nerface_oracle as O
import torch_reference as TR

pytestmark = pytest.mark.gpu

REC = dict(pe=(0, 64), ped=(16384 + 6 * 65536 + 3 * 32768, 32), mask=16384 + 6 * 65536 + 3 * 32768 + 8192)
REC["dy0"] = REC["mask"] + 9 * 128 * 32
REC["dy6"] = REC["dy0"] + 6 * 65536
REC["draw"] = REC["dy6"] + 3 * 32768


def x_off(layer):
    return 16384 + layer * 65536 if layer < 6 else 16384 + 6 * 65536 + (layer - 6) * 32768


def dy_off(layer):
    return REC["dy0"] + layer * 65536 if layer < 6 else REC["dy6"] + (layer - 6) * 32768


class _DevArr:
    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, data=(int(ptr), False), version=2)


def dev_tensor(ptr, shape, typestr="<f4"):
    return torch.as_tensor(_DevArr(ptr, shape, typestr), device="cuda")


def decode_image(records_i16, off, rows):
    """records_i16: [tiles, 2^19] int16 view of the records.  Returns FP32 [tiles, 128, rows] (sample row, feature)."""
    k = torch.arange(rows).view(-1, 1)
    r = torch.arange(128).view(1, -1)
    byte = off + (r >> 6) * rows * 128 + k * 128 + ((((r & 63) >> 3) ^ (k & 7)) << 4) + (r & 7) * 2
    idx = (byte // 2).to(records_i16.device)
    img = records_i16[:, idx.reshape(-1)].reshape(records_i16.shape[0], rows, 128)
    return img.view(torch.float16).float().transpose(1, 2).contiguous()


def rel_err(got, ref):
    return float((got - ref).abs().max()) / (float(ref.abs().max()) + 1e-30)


class Ctx:
    pass


@pytest.fixture(scope="module", params=[(48, 64, 64, False), (33, 64, 128, True)], ids=["48r_64c64f", "33r_64c128f_stress"])
def ctx(request, built_lib):
    import nerf
    from nerf import _engine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    n, nc, nf, stress = request.param
    dev = torch.device("cuda", 0)
    c = Ctx()
    c.n, c.nc, c.nf = n, nc, nf
    fr = O.synthetic_frame(21, 6, 8)
    ro, rd = O.ray_bundle(6, 8, fr["intrinsics"], fr["pose"])
    ro, rd = ro.reshape(-1, 3)[:n].contiguous(), rd.reshape(-1, 3)[:n].contiguous()
    if n > 48:
        raise ValueError
    bg = fr["bg"].reshape(-1, 3)[:n].contiguous()
    s = O.Sampling(nc, nf, True, 0.1, False, 2048)
    noise = O.draw_noise(n, s, torch.Generator().manual_seed(77))
    models = []
    for seed in (100, 101):
        m = nerf.models.ConditionalBlendshapePaperNeRFModel(num_encoding_fn_xyz=10, num_encoding_fn_dir=4,
                                                            include_input_xyz=True, include_input_dir=False)
        m.load_state_dict(O.random_init_params(seed, stress))
        models.append(m.to(dev))
    mc, mf = models
    eng = _engine.renderer_for(dev)
    eng.sync_weights(mc, mf)
    expr, latent = fr["expr"].to(dev), fr["latent"].to(dev)
    eng.set_frame(expr, latent)
    nz = dict(t_rand=noise.t_rand.to(dev), n_c=noise.n_c.to(dev), u=noise.u.to(dev), n_f=noise.n_f.to(dev))
    out = eng.render(ro.to(dev), rd.to(dev), 0.2, 0.8, nc, nf, perturb=True, noise_std=0.1, background=bg.to(dev), noise=nz,
                     precision="exact", train=True)
    torch.cuda.synchronize()
    d = eng.train_debug()
    c.dbg = d
    c.R = d.rays_per_unit
    c.tc, c.tf = d.tiles_coarse, d.tiles_fine
    c.tpu = c.tc + c.tf
    S = nc + nf
    c.z_c = dev_tensor(d.z_coarse, (n, nc)).clone()
    c.z_f = dev_tensor(d.z_fine, (n, S)).clone()
    c.raw_c = dev_tensor(d.raw_coarse, (n, nc, 4)).clone()
    c.raw_f = dev_tensor(d.raw_fine, (n, S, 4)).clone()
    c.out = out

    # ---- torch reference at the same depths
    pc = {k: v.detach().clone().requires_grad_(True) for k, v in mc.named_parameters()}
    pf = {k: v.detach().clone().requires_grad_(True) for k, v in mf.named_parameters()}
    lat = latent.clone().requires_grad_(True)
    rays = torch.cat((ro, rd, torch.full((n, 1), 0.2), torch.full((n, 1), 0.8)), dim=-1).to(dev)
    taps = {}
    ref = TR.render_at_depths(rays, pc, pf, expr, lat, c.z_c, c.z_f, 0.2, 0.8, 0.1, nz, False, bg.to(dev), None, taps)
    g = torch.Generator().manual_seed(5)
    target = torch.rand(n, 3, generator=g).to(dev)
    c.gouts = [None] * 7
    loss = ((ref[0] - target) ** 2).mean() + ((ref[3] - target) ** 2).mean() \
        + 0.3 * ref[1].mean() + 0.2 * ref[2].mean() + 0.1 * ref[4].mean() + 0.2 * ref[5].mean() + 0.5 * ref[6].mean()
    outs_for_grad = [r for r in ref]
    c.gouts = [gg.detach() for gg in torch.autograd.grad(loss, outs_for_grad, retain_graph=True)]
    loss.backward()
    c.ref, c.taps, c.pc, c.pf, c.lat = ref, taps, pc, pf, lat
    c.mc, c.mf, c.eng = mc, mf, eng

    # ---- fused backward with the same output gradients
    params_c = [dict(mc.named_parameters())[k] for k in TR.PARAM_ORDER]
    params_f = [dict(mf.named_parameters())[k] for k in TR.PARAM_ORDER]
    c.grads_c, c.grads_f, c.glat = eng.backward(c.gouts, params_c, params_f)
    torch.cuda.synchronize()
    n_tiles = int(d.n_tiles)
    c.records = dev_tensor(d.records, (n_tiles, d.record_bytes // 2), "<i2")
    c.d_raw = dev_tensor(d.d_raw, (n_tiles, 128, 4))
    c.scale = dev_tensor(d.scale, (2,)).cpu()
    c.n_tiles = n_tiles

    # ---- (ray, sample) -> (tile, row) maps per pass
    def rowmap(pas):
        Sx = S if pas else nc
        gi = torch.arange(n).view(-1, 1).expand(n, Sx)
        ii = torch.arange(Sx).view(1, -1).expand(n, Sx)
        unit, rr = gi // c.R, gi % c.R
        prow = rr * Sx + ii
        tile = unit * c.tpu + (c.tc if pas else 0) + prow // 128
        return tile.reshape(-1).to(dev), (prow % 128).reshape(-1).to(dev)
    c.map = [rowmap(0), rowmap(1)]
    return c


def test_forward_outputs_match_reference(ctx):
    names = ["rgb_coarse", "disp_coarse", "acc_coarse", "rgb_fine", "disp_fine", "acc_fine", "w_last"]
    for nme, r in zip(names, ctx.ref):
        assert float((ctx.out[nme] - r.detach()).abs().max()) < 2e-3, nme


def test_saved_colours_and_sigma(ctx):
    for pas, raw in ((0, ctx.raw_c), (1, ctx.raw_f)):
        t = ctx.taps["fine" if pas else "coarse"]["raw"].detach()
        col = torch.sigmoid(t[..., :3])
        assert float((raw[:, :-1, :3] - col[:, :-1]).abs().max()) < 2e-4  # last sample holds the background colour


def test_saved_activation_images(ctx):
    worst = 0.0
    for pas, key in ((0, "coarse"), (1, "fine")):
        tile, row = ctx.map[pas]
        tp = ctx.taps[key]
        for layer, name in [(i, f"h{i}") for i in range(6)] + [(6, "g0"), (7, "g1"), (8, "g2")]:
            img = decode_image(ctx.records, x_off(layer), 256 if layer < 6 else 128)
            got = img[tile, row]
            ref = tp[name].detach()
            err = float((got - ref).abs().max())
            tol = 2e-3 * float(ref.abs().max()) + 1e-5
            worst = max(worst, err / (float(ref.abs().max()) + 1e-30))
            assert err <= tol, (key, name, err, float(ref.abs().max()))
        pe = decode_image(ctx.records, REC["pe"][0], 64)[tile, row]
        assert float((pe[:, :63] - tp["pe"].detach()).abs().max()) < 2e-3
        assert float(pe[:, 63].abs().max()) == 0.0
        ped = decode_image(ctx.records, REC["ped"][0], 32)[tile, row]
        assert float((ped[:, :24] - tp["ped"].detach()).abs().max()) < 2e-3
    print(f"activation images: worst relative error {worst:.2e}")


def _mask_bits(ctx):
    rec8 = ctx.records.view(torch.uint8).reshape(ctx.n_tiles, -1)
    return rec8[:, REC["mask"]:REC["mask"] + 9 * 128 * 32].contiguous().view(torch.int32).reshape(ctx.n_tiles, 9, 128, 8)


def _layer_mask(masks, tile, row, layer):
    width = 256 if layer < 6 else 128
    m = masks[tile, layer, row]  # [rows, 8]
    return ((m.unsqueeze(-1) >> torch.arange(32, device=m.device)) & 1).reshape(m.shape[0], 256)[:, :width].bool()


def test_relu_masks(ctx):
    masks = _mask_bits(ctx)
    flips = 0
    for pas, key in ((0, "coarse"), (1, "fine")):
        tile, row = ctx.map[pas]
        tp = ctx.taps[key]
        for layer in range(9):
            bits = _layer_mask(masks, tile, row, layer)
            a = tp[f"a{layer}"].detach()
            decided = a.abs() > 1e-4 * a.abs().max()  # FP association may flip the sign of a near-zero pre-activation
            assert bool(((bits == (a > 0)) | ~decided).all()), (key, layer)
            flips += int((bits != (a > 0)).sum())
    print(f"ReLU masks: {flips} sign flips at near-zero pre-activations")


def test_composite_backward(ctx):
    for pas, key in ((0, "coarse"), (1, "fine")):
        tile, row = ctx.map[pas]
        got = ctx.d_raw[tile, row]
        ref = ctx.taps[key]["raw"].grad.reshape(-1, 4)
        e = rel_err(got, ref)
        print(f"d raw {key}: rel {e:.2e}, max |ref| {float(ref.abs().max()):.3e}")
        assert e < 5e-4, (key, e)
    # rows that belong to no sample stay zero
    used = torch.zeros(ctx.n_tiles, 128, dtype=torch.bool, device=ctx.d_raw.device)
    for pas in (0, 1):
        used[ctx.map[pas][0], ctx.map[pas][1]] = True
    assert float(ctx.d_raw[~used].abs().max() if (~used).any() else 0.0) == 0.0


def test_chain_gradients(ctx):
    """dL/d(pre-activation) per layer.  A sample row in which some ReLU decision differs from the reference's
    (pre-activation within FP32 rounding of zero, see test_relu_masks) legitimately differs from there on down the
    chain; such rows (a handful out of thousands) are excluded here and covered by the parameter-gradient tolerance."""
    scale = float(ctx.scale[0])
    masks = _mask_bits(ctx)
    worst = 0.0
    for pas, key in ((0, "coarse"), (1, "fine")):
        tile, row = ctx.map[pas]
        tp = ctx.taps[key]
        row_ok = torch.ones(tile.shape[0], dtype=torch.bool, device=tile.device)
        for layer in range(9):
            row_ok &= (_layer_mask(masks, tile, row, layer) == (tp[f"a{layer}"].detach() > 0)).all(dim=1)
        assert int((~row_ok).sum()) <= max(8, tile.shape[0] // 500)
        for layer in range(8, -1, -1):
            img = decode_image(ctx.records, dy_off(layer), 256 if layer < 6 else 128)
            got = img[tile, row] / scale
            ref = tp[f"a{layer}"].grad
            e = float((got - ref)[row_ok].abs().max()) / (float(ref.abs().max()) + 1e-30)
            worst = max(worst, e)
            print(f"dY{layer} {key}: rel {e:.2e} (max |ref| {float(ref.abs().max()):.3e}, {int((~row_ok).sum())} rows excluded)")
            assert e < 5e-3, (key, layer, e)
    print(f"chain: worst relative error {worst:.2e}, loss scale {scale:.3g}")


def test_parameter_gradients(ctx):
    worst = 0.0
    for grads, ref_p, tag in ((ctx.grads_c, ctx.pc, "coarse"), (ctx.grads_f, ctx.pf, "fine")):
        for k, g in zip(TR.PARAM_ORDER, grads):
            if k.startswith("layers_dir.3"):
                assert g is None and ref_p[k].grad is None
                continue
            ref = ref_p[k].grad
            err = float((g - ref).abs().max())
            scale = float(ref.abs().max()) + 1e-12
            worst = max(worst, err / scale)
            print(f"{tag} {k}: rel {err / scale:.2e}")
            assert err <= 1e-2 * scale + 1e-9, (tag, k, err, scale)  # FP16 operands (2^-11 each) + rare ReLU flips
    e = rel_err(ctx.glat, ctx.lat.grad)
    print(f"latent: rel {e:.2e}; worst parameter rel {worst:.2e}")
    assert e < 1e-2
