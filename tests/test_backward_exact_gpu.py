"""Exact-gradient training (NFB_PREC_EXACT_GRAD): the exact forward that also keeps the lo halves of every activation, and the
backward whose dX chain and weight-gradient GEMMs multiply hi+lo operands (csrc/nfb_train.cu, EXACT variants).  Checked against
the exact mode it extends (forward bit for bit), the FP32 layer probe (lo halves), and a plain-PyTorch FP32 reference
(tests/torch_reference.py, TF32 off) at the depths the fused forward sampled."""
import pytest
import torch

import nerface_oracle as O
import torch_reference as TR
from test_backward_gpu import REC, decode_image, dev_tensor, dy_off, rel_err, x_off

pytestmark = pytest.mark.gpu

REC_LO = 1 << 20            # nfb_layout.h kRecLo
NAMES = ["rgb_coarse", "disp_coarse", "acc_coarse", "rgb_fine", "disp_fine", "acc_fine", "w_last"]


class Ctx:
    pass


def _models(nerf, dev, stress):
    out = []
    for seed in (100, 101):
        m = nerf.models.ConditionalBlendshapePaperNeRFModel(num_encoding_fn_xyz=10, num_encoding_fn_dir=4,
                                                            include_input_xyz=True, include_input_dir=False)
        m.load_state_dict(O.random_init_params(seed, stress))
        out.append(m.to(dev))
    return out


def _mask_bits(records_i16, n_tiles):
    rec8 = records_i16.view(torch.uint8).reshape(n_tiles, -1)
    return rec8[:, REC["mask"]:REC["mask"] + 9 * 128 * 32].contiguous().view(torch.int32).reshape(n_tiles, 9, 128, 8)


def _layer_mask(masks, tile, row, layer):
    width = 256 if layer < 6 else 128
    m = masks[tile, layer, row]
    return ((m.unsqueeze(-1) >> torch.arange(32, device=m.device)) & 1).reshape(m.shape[0], 256)[:, :width].bool()


def _hi_lo(records, off, rows):
    return decode_image(records, off, rows) + decode_image(records, REC_LO + off, rows)


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
    ro, rd = ro.reshape(-1, 3)[:n].contiguous().to(dev), rd.reshape(-1, 3)[:n].contiguous().to(dev)
    bg = fr["bg"].reshape(-1, 3)[:n].contiguous().to(dev)
    s = O.Sampling(nc, nf, True, 0.1, False, 2048)
    noise = O.draw_noise(n, s, torch.Generator().manual_seed(77))
    mc, mf = _models(nerf, dev, stress)
    eng = _engine.renderer_for(dev)
    eng.sync_weights(mc, mf)
    expr, latent = fr["expr"].to(dev), fr["latent"].to(dev)
    eng.set_frame(expr, latent)
    nz = dict(t_rand=noise.t_rand.to(dev), n_c=noise.n_c.to(dev), u=noise.u.to(dev), n_f=noise.n_f.to(dev))
    kw = dict(perturb=True, noise_std=0.1, background=bg, noise=nz)

    def render(prec, **more):  # other tests may have packed other weights into the device's renderer in between
        eng.invalidate()
        eng.sync_weights(mc, mf)
        eng.set_frame(expr, latent)
        return eng.render(ro, rd, 0.2, 0.8, nc, nf, precision=prec, **kw, **more)
    c.render = render

    # ---- exact-mode training forward: outputs and the forward-written part of its records
    out_exact = c.render("exact", train=True)
    torch.cuda.synchronize()
    d = eng.train_debug()
    assert d.record_bytes == 1 << 20
    c.rec_exact = dev_tensor(d.records, (int(d.n_tiles), d.record_bytes // 2), "<i2").clone()
    c.out_exact = {k: v.clone() for k, v in out_exact.items() if k in NAMES}

    # ---- exact-gradient training forward + backward
    out = c.render("exact_grad", train=True)
    torch.cuda.synchronize()
    d = eng.train_debug()
    c.dbg = d
    c.R = d.rays_per_unit
    c.tc, c.tf = d.tiles_coarse, d.tiles_fine
    c.tpu = c.tc + c.tf
    S = nc + nf
    c.z_c = dev_tensor(d.z_coarse, (n, nc)).clone()
    c.z_f = dev_tensor(d.z_fine, (n, S)).clone()
    c.out = {k: v.clone() for k, v in out.items() if k in NAMES}

    # ---- torch reference at the same depths
    pc = {k: v.detach().clone().requires_grad_(True) for k, v in mc.named_parameters()}
    pf = {k: v.detach().clone().requires_grad_(True) for k, v in mf.named_parameters()}
    lat = latent.clone().requires_grad_(True)
    rays = torch.cat((ro, rd, torch.full((n, 1), 0.2, device=dev), torch.full((n, 1), 0.8, device=dev)), dim=-1)
    taps = {}
    ref = TR.render_at_depths(rays, pc, pf, expr, lat, c.z_c, c.z_f, 0.2, 0.8, 0.1, nz, False, bg, None, taps)
    target = torch.rand(n, 3, generator=torch.Generator().manual_seed(5)).to(dev)

    def loss_of(r):
        return ((r[0] - target) ** 2).mean() + ((r[3] - target) ** 2).mean() \
            + 0.3 * r[1].mean() + 0.2 * r[2].mean() + 0.1 * r[4].mean() + 0.2 * r[5].mean() + 0.5 * r[6].mean()
    c.loss_of = loss_of
    loss = loss_of(ref)
    c.gouts = [gg.detach() for gg in torch.autograd.grad(loss, list(ref), retain_graph=True)]
    loss.backward()
    c.ref, c.taps, c.pc, c.pf, c.lat = ref, taps, pc, pf, lat
    c.mc, c.mf, c.eng, c.expr, c.latent, c.rays, c.nz, c.bg = mc, mf, eng, expr, latent, rays, nz, bg

    # ---- fused backward with the same output gradients
    params_c = [dict(mc.named_parameters())[k] for k in TR.PARAM_ORDER]
    params_f = [dict(mf.named_parameters())[k] for k in TR.PARAM_ORDER]
    c.params_c, c.params_f = params_c, params_f
    c.grads_c, c.grads_f, c.glat = eng.backward(c.gouts, params_c, params_f)
    torch.cuda.synchronize()
    c.n_tiles = int(d.n_tiles)
    assert d.record_bytes == 2 << 20
    c.records = dev_tensor(d.records, (c.n_tiles, d.record_bytes // 2), "<i2").clone()
    c.scale = dev_tensor(d.scale, (2,)).cpu()

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


def test_forward_is_exact_mode_bit_for_bit(ctx):
    """Training and evaluation outputs equal exact mode's; the hi MiB holds, byte for byte, what an exact training forward writes
    (PE, h0..h5, g0..g2, PEd, ReLU masks)."""
    for k in NAMES:
        assert torch.equal(ctx.out[k], ctx.out_exact[k]), k
    ev_x = ctx.render("exact")
    ev_g = ctx.render("exact_grad")
    for k in NAMES:
        assert torch.equal(ev_x[k], ev_g[k]), k
    hi = ctx.records[:, :REC["mask"] // 2]
    assert torch.equal(hi, ctx.rec_exact[:, :REC["mask"] // 2])
    # masks: words 0..3 of every layer, words 4..7 of the 256-wide layers 0..5 (the others are never written)
    m_g, m_x = _mask_bits(ctx.records, ctx.n_tiles), _mask_bits(ctx.rec_exact, ctx.n_tiles)
    assert torch.equal(m_g[:, :, :, :4], m_x[:, :, :, :4])
    assert torch.equal(m_g[:, :6, :, 4:], m_x[:, :6, :, 4:])


def test_lo_halves_complete_the_fp32_activations(ctx):
    """hi + lo of every activation image of the first coarse tile equals the FP32 layer probe to <= 2^-21 |x| + 2^-24."""
    worst = 0.0
    for step in range(-1, 9):
        probe = ctx.render("exact_grad", act_step=step)["act"]
        torch.cuda.synchronize()
        width = 64 if step < 0 else (256 if step < 6 else 128)
        off = REC["pe"][0] if step < 0 else x_off(step)
        got = _hi_lo(ctx.records[:1], off, width)[0]           # tile 0 = the first 128 coarse rows
        ref = probe[:, :width]
        if step < 0:
            got, ref = got[:, :63], ref[:, :63]
        err = (got - ref).abs()
        tol = 2.0 ** -21 * ref.abs() + 2.0 ** -24
        worst = max(worst, float((err / (ref.abs() + 2.0 ** -3)).max()))
        assert bool((err <= tol).all()), (step, float(err.max()), float((err - tol).max()))
    print(f"hi + lo vs FP32 probe: worst relative error {worst:.2e}")


def test_lo_direction_encoding(ctx):
    tile, row = ctx.map[0]
    ped = _hi_lo(ctx.records, REC["ped"][0], 32)[tile, row]
    ref = ctx.taps["coarse"]["ped"].detach()
    assert float((ped[:, :24] - ref).abs().max()) <= 2.0 ** -21 * float(ref.abs().max()) + 2.0 ** -24
    assert float(ped[:, 24:].abs().max()) == 0.0


def test_chain_gradients_exact(ctx):
    """dY images (hi + lo) / loss scale vs the reference's pre-activation gradients, on rows whose ReLU masks agree with the
    reference (as test_backward_gpu.test_chain_gradients): <= 5e-5 of the largest reference entry (FP16 single operands: 5e-3,
    measured up to 9e-4).  Measured on a B200: 1.1e-5 to 1.7e-5 over two runs.  What is left is not the operand split (~2^-21): the d raw that
    enters the chain already differs from the reference's by up to 1.6e-6 of its largest entry (FP32 compositing of forward
    outputs that differ in the last bits), and a layer's largest gradient is a sum with cancellation that magnifies it."""
    scale = float(ctx.scale[0])
    masks = _mask_bits(ctx.records, ctx.n_tiles)
    worst = 0.0
    for pas, key in ((0, "coarse"), (1, "fine")):
        tile, row = ctx.map[pas]
        tp = ctx.taps[key]
        row_ok = torch.ones(tile.shape[0], dtype=torch.bool, device=tile.device)
        for layer in range(9):
            row_ok &= (_layer_mask(masks, tile, row, layer) == (tp[f"a{layer}"].detach() > 0)).all(dim=1)
        assert int((~row_ok).sum()) <= max(8, tile.shape[0] // 500)
        for layer in range(8, -1, -1):
            got = _hi_lo(ctx.records, dy_off(layer), 256 if layer < 6 else 128)[tile, row] / scale
            ref = tp[f"a{layer}"].grad
            e = float((got - ref)[row_ok].abs().max()) / (float(ref.abs().max()) + 1e-30)
            worst = max(worst, e)
            print(f"dY{layer} {key}: rel {e:.2e} ({int((~row_ok).sum())} rows excluded)")
            assert e <= 5e-5, (key, layer, e)
    print(f"exact chain: worst relative error {worst:.2e}, loss scale {scale:.3g}")


def _masked_reference(ctx):
    """The FP32 reference with the kernel's ReLU decisions (decoded from the records) in place of a > 0, so that a
    pre-activation within rounding of zero cannot stand in for arithmetic error.  Returns (grads_c, grads_f, d latent)."""
    masks = _mask_bits(ctx.records, ctx.n_tiles)
    pc = {k: v.detach().clone().requires_grad_(True) for k, v in ctx.mc.named_parameters()}
    pf = {k: v.detach().clone().requires_grad_(True) for k, v in ctx.mf.named_parameters()}
    lat = ctx.latent.clone().requires_grad_(True)
    m = {key: [_layer_mask(masks, *ctx.map[pas], layer) for layer in range(9)] for pas, key in ((0, "coarse"), (1, "fine"))}
    outs = TR.render_at_depths(ctx.rays, pc, pf, ctx.expr, lat, ctx.z_c, ctx.z_f, 0.2, 0.8, 0.1, ctx.nz, False, ctx.bg, None,
                               masks=m)
    torch.autograd.backward(outs, ctx.gouts)
    return [pc[k].grad for k in TR.PARAM_ORDER], [pf[k].grad for k in TR.PARAM_ORDER], lat.grad


def test_parameter_gradients_exact(ctx):
    """All 48 used parameter tensors and the latent code against the masked FP32 reference: <= 1e-4 max|ref| + 1e-9.  The
    worst error against the unmasked reference (test_backward_gpu's comparison) is printed and stays within its 1e-2."""
    rc, rf, rlat = _masked_reference(ctx)
    worst, worst_unmasked = 0.0, 0.0
    for grads, refs, plain, tag in ((ctx.grads_c, rc, ctx.pc, "coarse"), (ctx.grads_f, rf, ctx.pf, "fine")):
        for k, g, ref in zip(TR.PARAM_ORDER, grads, refs):
            if k.startswith("layers_dir.3"):
                assert g is None and ref is None
                continue
            scale = float(ref.abs().max()) + 1e-12
            err = float((g - ref).abs().max())
            worst = max(worst, err / scale)
            u = plain[k].grad
            worst_unmasked = max(worst_unmasked, float((g - u).abs().max()) / (float(u.abs().max()) + 1e-12))
            print(f"{tag} {k}: rel {err / scale:.2e}")
            assert err <= 1e-4 * scale + 1e-9, (tag, k, err, scale)
    e = rel_err(ctx.glat, rlat)
    print(f"latent: rel {e:.2e}; worst parameter rel {worst:.2e} (masked reference), {worst_unmasked:.2e} (unmasked reference)")
    assert float((ctx.glat - rlat).abs().max()) <= 1e-4 * float(rlat.abs().max()) + 1e-9
    assert worst_unmasked <= 1e-2 and rel_err(ctx.glat, ctx.lat.grad) <= 1e-2


def _batches(dev, n):
    H = W = 32
    fr = O.synthetic_frame(2, H, W)
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    g = torch.Generator().manual_seed(3)
    tgt = torch.rand(H * W, 3, generator=g).to(dev)
    sel = torch.randperm(H * W, generator=g)[:n].to(dev)
    return fr, ro.reshape(-1, 3).to(dev), rd.reshape(-1, 3).to(dev), fr["bg"].reshape(-1, 3).to(dev), tgt, sel


def test_chunked_training_matches_one_launch(built_lib, monkeypatch):
    """NFB_TRAIN_MEM_MB=48: a 160-ray 64c+64f batch (240 tiles = 480 MiB of 2 MiB records) runs in chunks with their own loss
    scales; in this mode the gradients agree with the one-launch path to 3e-5 of each tensor's largest entry (FP16: 3e-3).
    Measured on a B200: 1.2e-5, the FP32 accumulation order of the weight-gradient atomics (which differs between one launch and
    ten chunks) on tensors whose largest entry is a sum with cancellation."""
    import nerf
    from nerf import _engine
    dev = torch.device("cuda", 0)
    fr, ro, rd, bg, tgt, sel = _batches(dev, 160)
    expr = fr["expr"].to(dev)
    blk = dict(num_coarse=64, num_fine=64, perturb=True, lindisp=False, radiance_field_noise_std=0.1, white_background=False, chunksize=64)
    cfg = nerf.CfgNode(dict(nerf=dict(use_viewdirs=True, train=blk), dataset=dict(no_ndc=True, near=0.2, far=0.8)))
    prev = _engine.get_precision()
    nerf.set_precision("exact_grad")
    results = []
    try:
        for budget in (None, "48"):
            if budget:
                monkeypatch.setenv("NFB_TRAIN_MEM_MB", budget)
            mc, mf = _models(nerf, dev, False)
            lat = torch.full((32,), 0.01, device=dev, requires_grad=True)
            torch.manual_seed(9)
            eng = _engine.renderer_for(dev)
            l0 = eng.launch_count()
            out = nerf.run_one_iter_of_nerf(32, 32, fr["intrinsics"], mc, mf, ro[sel], rd[sel], cfg, mode="train", expressions=expr,
                                            background_prior=bg[sel], latent_code=lat)
            loss = ((out[0] - tgt[sel]) ** 2).mean() + ((out[3] - tgt[sel]) ** 2).mean() + out[6].mean() * 0.1
            loss.backward()
            torch.cuda.synchronize()
            results.append(([o.detach().clone() for o in out],
                            [p.grad.clone() for p in list(mc.parameters()) + list(mf.parameters()) if p.grad is not None] + [lat.grad.clone()],
                            eng.launch_count() - l0))
    finally:
        nerf.set_precision(prev)
        monkeypatch.delenv("NFB_TRAIN_MEM_MB", raising=False)
    (o1, g1, n1), (o2, g2, n2) = results
    assert n2 > n1 + 10
    for a, b in zip(o1, o2):
        assert float((a - b).abs().max()) < 1e-5   # the evaluation kernel renders what the training forward renders
    rel = [float((a - b).abs().max()) / max(float(a.abs().max()), 1e-12) for a, b in zip(g1, g2)]
    print(f"chunked vs one launch (exact gradients): relative difference per tensor {['%.1e' % e for e in rel]}")
    assert max(rel) <= 3e-5, rel


def test_fused_trainer_exact_grad(built_lib):
    """FusedTrainer(precision="exact_grad"): the captured graph step follows the eager fused step (losses to 2e-6, parameters
    after one step to 1e-6), and the drop-in run_one_iter_of_nerf + loss.backward() gives Renderer.backward's gradients."""
    import nerf
    from nerf import _engine, fused_train
    dev = torch.device("cuda", 0)
    steps, n, lat = 3, 64, 2
    H = W = 32
    fr = O.synthetic_frame(2, H, W)
    ro, rd = O.ray_bundle(H, W, fr["intrinsics"], fr["pose"])
    ro, rd = ro.reshape(-1, 3).to(dev), rd.reshape(-1, 3).to(dev)
    bg = fr["bg"].reshape(-1, 3).to(dev)
    g = torch.Generator().manual_seed(3)
    tgt = torch.rand(H * W, 3, generator=g).to(dev)
    idx = [torch.randperm(H * W, generator=g)[:n].to(dev) for _ in range(steps)]
    expr = fr["expr"].to(dev)

    def mk():
        mc, mf = _models(nerf, dev, False)
        return fused_train.FusedTrainer(mc, mf, n_latent=8, lr=5e-4, lr_decay_steps=250.0, lr_decay_factor=0.1, num_coarse=64,
                                        num_fine=64, perturb=False, noise_std=0.0, precision="exact_grad")
    ta, tb = mk(), mk()
    tb.capture(n)
    eng = _engine.renderer_for(dev)
    for i in range(steps):
        sel = idx[i]
        la = ta.step(ro[sel], rd[sel], tgt[sel], expr, lat, background=bg[sel]).clone()
        tb._own_engine()
        lb = tb.step_graph(ro[sel], rd[sel], tgt[sel], expr, lat, background=bg[sel]).clone()
        torch.cuda.synchronize()
        assert float((la - lb).abs().max()) < 2e-6, (i, la, lb)
        if i == 0:
            assert float((ta.params - tb.params).abs().max()) <= 1e-6

    # drop-in path vs Renderer.backward, same kernels in the same mode
    blk = dict(num_coarse=64, num_fine=64, perturb=False, lindisp=False, radiance_field_noise_std=0.0, white_background=False, chunksize=2048)
    cfg = nerf.CfgNode(dict(nerf=dict(use_viewdirs=True, train=blk), dataset=dict(no_ndc=True, near=0.2, far=0.8)))
    sel = idx[0]
    mc, mf = _models(nerf, dev, False)
    latent = torch.full((32,), 0.01, device=dev)
    prev = _engine.get_precision()
    nerf.set_precision("exact_grad")
    try:
        lt = latent.clone().requires_grad_(True)
        out = nerf.run_one_iter_of_nerf(H, W, fr["intrinsics"], mc, mf, ro[sel], rd[sel], cfg, mode="train", expressions=expr,
                                        background_prior=bg[sel], latent_code=lt)
        loss = ((out[0] - tgt[sel]) ** 2).mean() + ((out[3] - tgt[sel]) ** 2).mean()
        loss.backward()
    finally:
        nerf.set_precision(prev)
    drop = [dict(m.named_parameters())[k].grad for m in (mc, mf) for k in TR.PARAM_ORDER] + [lt.grad]
    eng.sync_weights(mc, mf)
    eng.set_frame(expr, latent)
    o = eng.render(ro[sel], rd[sel], 0.2, 0.8, 64, 64, background=bg[sel], precision="exact_grad", train=True)
    gc_ = 2.0 * (o["rgb_coarse"] - tgt[sel]) / (3 * n)
    gf_ = 2.0 * (o["rgb_fine"] - tgt[sel]) / (3 * n)
    pc = [dict(mc.named_parameters())[k] for k in TR.PARAM_ORDER]
    pf = [dict(mf.named_parameters())[k] for k in TR.PARAM_ORDER]
    gc, gf, glat = eng.backward((gc_, None, None, gf_, None, None, None), pc, pf)
    torch.cuda.synchronize()
    for k, a, b in zip(TR.PARAM_ORDER * 2 + ["latent"], drop, gc + gf + [glat]):
        assert (a is None) == (b is None), k
        if a is not None:
            assert float((a - b).abs().max()) <= 1e-5 * max(float(a.abs().max()), 1e-12), k
