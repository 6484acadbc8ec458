"""The fused backward (csrc/nfb_train.cu: compositing backward, dX chain, weight-gradient GEMMs, finalize) against an FP64
reference (tests/torch_reference.py with the kernel's own ReLU decisions) across the shapes, tile layouts, compositing options
and precision modes the training path supports:

  - the shipped iteration (2048 rays, 64c+64f: ~7 units per forward / chain CTA, ~171 tiles per weight-gradient CTA), and a
    batch whose last persistent iteration leaves one CTA of a chain cluster empty;
  - partial tiles (padding rows in one or both passes), two coarse tiles per unit, one ray per unit, S = 512, a pass shorter
    than one tile, coarse-only training, one to three rays;
  - no background, a white background, deterministic depths, ablation directions;
  - fast, exact and exact_grad precision;
  - the chunked re-run of the training forward at shapes where its per-ray pointer strides differ.

Per case and mode: the ReLU masks agree with the reference's own decisions, d raw / dY / parameter and latent gradients are
within the mode's gate of the largest reference entry, every row that belongs to no sample carries an exactly-zero gradient,
and the training forward renders what the evaluation forward renders, bit for bit.  The reference runs in ray blocks on the
GPU (output gradients and ReLU masks are per ray, so the block sums are the full gradients)."""
import pytest
import torch

import nerface_oracle as O
import torch_reference as TR
from test_backward_exact_gpu import NAMES, REC_LO, _layer_mask, _mask_bits, _models
from test_backward_gpu import decode_image, dev_tensor, dy_off

pytestmark = pytest.mark.gpu

NEAR, FAR = 0.2, 0.8
BLOCK = 256            # rays per reference block (a multiple of every rays-per-unit)
ONE_LAUNCH_MB = "16384"  # records budget that keeps every one-launch case in one launch (prod exact_grad: 6 GiB)
DEFAULTS = dict(perturb=True, noise_std=0.1, bg=True, white=False, dir_z=False)

# Relative to max|ref| of each tensor: parameters and latent (+ 1e-9 absolute), dY0..dY5, dY6..dY8 (direction branch), d raw.
# Worst measured on a B200 (1000 W power limit), per mode:
#   exact_grad: parameters 1.5e-4 (prod), latent 4.5e-5 (prod), dY0..5 < 1e-5, dY6..8 1.9e-4 (determ), d raw 1.2e-5.
#     Two effects the FP32 reference of test_backward_exact_gpu cannot see, both measured against it and against the exact
#     FP64 sum of the kernel's own records:
#     - the forward composites in FP32 as the reference project does: alpha = 1 - exp(-sigma delta) carries an absolute error of
#       ~2^-24, relative ~2^-24 / (sigma delta), which reaches 1e-4 in every sample weight where sigma delta ~ 1e-3 (deterministic
#       depths, no sigma noise, 512 samples).  d colour and so dY6..8 and the direction-branch parameters inherit it; the kernel
#       agrees with an FP32 reference there to ~1e-6, and the FP32 reference differs from FP64 by the same 1e-4.
#     - the weight-gradient kernel sums a CTA's tiles in its FP32 accumulator: against the FP64 sum of dY^T X of its own
#       records it is off by 3.5e-5 / 7e-5 / 1.45e-4 at 512 / 1024 / 2048 rays (64c+64f), growing linearly with the tiles per
#       CTA, and no single tile accounts for the difference (a dropped tile would).
#   exact (FP16 backward): parameters 6.8e-4, dY 9.5e-4, d raw 2e-6.
#   fast (FP16 forward and backward): parameters 6.8e-4, latent 4.5e-4, dY 1.0e-3, d raw 4.5e-5 -- all under half their gates.
GATES = {"exact_grad": (3e-4, 5e-5, 4e-4, 5e-4), "exact": (1e-2, 5e-3, 5e-3, 5e-4), "fast": (1e-2, 5e-3, 5e-3, 5e-4)}
# A ReLU decision may differ from the FP64 reference's only where |a| is within MASK_DECIDED of the layer's max|a|, and in at
# most MASK_FLIP_ROWS of the rows (at least 8).  FP16 operands in the fast forward move a pre-activation by up to ~2^-11 of
# the largest term: measured, flips at |a| <= 3.6e-4 max|a| in 15-17 % of the rows (exact modes: 1.3e-6, 0.1 %).
MASK_DECIDED = {"exact_grad": 1e-4, "exact": 1e-4, "fast": 1e-3}
MASK_FLIP_ROWS = {"exact_grad": 1 / 500, "exact": 1 / 500, "fast": 1 / 4}

# id: rays (None: 2 * (2 * SMs + 37) - 1), coarse, fine, options, modes
CASES = {
    "prod": (2048, 64, 64, {}, ("fast", "exact", "exact_grad")),
    "mixed": (None, 64, 128, {}, ("exact_grad",)),
    "100c60f": (13, 100, 60, {}, ("exact_grad", "fast")),
    "128c64f": (13, 128, 64, {}, ("exact_grad",)),
    "200c300f": (9, 200, 300, {}, ("exact_grad", "exact")),
    "256c256f": (5, 256, 256, {}, ("exact_grad",)),
    "40c24f": (17, 40, 24, {}, ("exact_grad",)),
    "coarse": (48, 64, 0, {}, ("exact_grad", "fast")),
    "coarse3": (5, 3, 0, dict(perturb=False), ("exact_grad",)),
    "tiny1": (1, 64, 64, {}, ("exact_grad",)),
    "tiny2": (2, 64, 64, {}, ("exact_grad",)),
    "tiny3": (3, 64, 64, {}, ("exact_grad",)),
    "no_bg": (33, 64, 64, dict(bg=False), ("exact_grad", "exact")),
    "white_bg": (33, 64, 64, dict(white=True), ("exact_grad",)),
    "white_nobg": (33, 64, 64, dict(white=True, bg=False), ("exact_grad",)),
    "determ": (33, 64, 64, dict(perturb=False, noise_std=0.0), ("exact_grad",)),
    "ablation": (33, 64, 64, dict(dir_z=True), ("exact_grad",)),
}


class _Case:
    """Seeded inputs of one case on cuda:0 and a render call that re-packs the weights first (the renderer is shared)."""

    def __init__(self, n, nc, nf, opts):
        import nerf
        from nerf import _engine
        self.dev = dev = torch.device("cuda", 0)
        self.o = o = dict(DEFAULTS, **opts)
        self.n, self.nc, self.nf = n, nc, nf
        fr = O.synthetic_frame(21, 48, 48)
        ro, rd = O.ray_bundle(48, 48, fr["intrinsics"], fr["pose"])
        assert n <= 48 * 48
        self.ro, self.rd = ro.reshape(-1, 3)[:n].contiguous().to(dev), rd.reshape(-1, 3)[:n].contiguous().to(dev)
        self.bg = fr["bg"].reshape(-1, 3)[:n].contiguous().to(dev) if o["bg"] else None
        g = torch.Generator().manual_seed(77)
        noise = O.draw_noise(n, O.Sampling(nc, nf, o["perturb"], o["noise_std"], o["white"], 2048), g)
        self.nz = {k: getattr(noise, k).to(dev) for k in ("t_rand", "n_c", "u", "n_f") if getattr(noise, k) is not None}
        self.dir_z = (torch.rand(n, generator=g) * 2.0 - 1.0).to(dev) if o["dir_z"] else None
        self.mc, self.mf = _models(nerf, dev, False)
        if nf == 0:
            self.mf = None
        self.expr, self.latent = fr["expr"].to(dev), fr["latent"].to(dev)
        self.eng = _engine.renderer_for(dev)
        self.params_c = [dict(self.mc.named_parameters())[k] for k in TR.PARAM_ORDER]
        self.params_f = [dict(self.mf.named_parameters())[k] for k in TR.PARAM_ORDER] if nf else None

    def render(self, prec, train):
        eng, o = self.eng, self.o
        eng.invalidate()
        eng.sync_weights(self.mc, self.mf)
        eng.set_frame(self.expr, self.latent)
        out = eng.render(self.ro, self.rd, NEAR, FAR, self.nc, self.nf, perturb=o["perturb"], noise_std=o["noise_std"],
                         white_bkgd=o["white"], background=self.bg, dir_z=self.dir_z, noise=self.nz, precision=prec, train=train)
        return {k: v for k, v in out.items() if k in NAMES}

    def out_grads(self, out):
        """d loss / d output (FP32) of a loss over all seven outputs (the existing backward fixtures' loss) at `out`."""
        r = {k: v.detach().double().requires_grad_(True) for k, v in out.items()}
        tgt = torch.rand(self.n, 3, generator=torch.Generator().manual_seed(5)).to(self.dev, torch.float64)
        loss = ((r["rgb_coarse"] - tgt) ** 2).mean() + 0.3 * r["disp_coarse"].mean() + 0.2 * r["acc_coarse"].mean() \
            + 0.5 * r["w_last"].mean()
        if self.nf:
            loss = loss + ((r["rgb_fine"] - tgt) ** 2).mean() + 0.1 * r["disp_fine"].mean() + 0.2 * r["acc_fine"].mean()
        keys = [k for k in NAMES if k in r]
        grads = dict(zip(keys, torch.autograd.grad(loss, [r[k] for k in keys])))
        return [grads[k].float().contiguous() if k in grads else None for k in NAMES]

    def layout(self):
        """(rays per unit, coarse tiles, fine tiles) the host picks for this shape (nfb_api.cu render_impl)."""
        S = self.nc + self.nf
        R = 2 if 2 * S <= 512 else 1
        return R, (R * self.nc + 127) // 128, (R * S + 127) // 128 if self.nf else 0


def _rowmap(b0, b1, S, R, tpu, base, dev):
    """(tile, row) of every (ray, sample) of rays [b0, b1) of one pass, ray-major like the reference's rows."""
    gi = torch.arange(b0, b1, device=dev).view(-1, 1).expand(b1 - b0, S)
    ii = torch.arange(S, device=dev).view(1, -1).expand(b1 - b0, S)
    unit, rr = gi // R, gi % R
    prow = rr * S + ii
    return (unit * tpu + base + prow // 128).reshape(-1), (prow % 128).reshape(-1)


def _mode_cases():
    return [pytest.param(name, mode, id=f"{name}-{mode}") for name, c in CASES.items() for mode in c[4]]


@pytest.mark.parametrize("name,mode", _mode_cases())
def test_backward_matches_fp64_reference(name, mode, built_lib, monkeypatch):
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    n, nc, nf, opts, _ = CASES[name]
    if n is None:
        n = 2 * (2 * torch.cuda.get_device_properties(0).multi_processor_count + 37) - 1
    monkeypatch.setenv("NFB_TRAIN_MEM_MB", ONE_LAUNCH_MB)  # a busy GPU must not turn a one-launch case into a chunked one
    c = _Case(n, nc, nf, opts)
    dev, eng, S = c.dev, c.eng, nc + nf
    passes = ((0, "coarse"), (1, "fine")) if nf else ((0, "coarse"),)
    g_par, g_dy, g_dy_dir, g_draw = GATES[mode]
    fails = []

    # ---- forward: evaluation, then training (same mode, same noise)
    out_eval = c.render(mode, train=False)
    out = c.render(mode, train=True)
    torch.cuda.synchronize()
    for k in out:
        if not torch.equal(out[k], out_eval[k]):
            fails.append(f"training forward {k} differs from the evaluation forward by {float((out[k] - out_eval[k]).abs().max()):.3e}")
    d = eng.train_debug()
    R, tc, tf = d.rays_per_unit, d.tiles_coarse, d.tiles_fine
    assert (R, tc, tf) == c.layout()
    tpu = tc + tf
    n_units = (n + R - 1) // R
    n_tiles = int(d.n_tiles)
    assert n_tiles == n_units * tpu
    assert d.record_bytes == (2 << 20 if mode == "exact_grad" else 1 << 20)
    z_c = dev_tensor(d.z_coarse, (n, nc)).double()
    z_f = dev_tensor(d.z_fine, (n, S)).double() if nf else None
    raw_k = {"coarse": dev_tensor(d.raw_coarse, (n, nc, 4)).clone()}   # (colour, ReLU input of sigma) the forward saved
    if nf:
        raw_k["fine"] = dev_tensor(d.raw_fine, (n, S, 4)).clone()

    # ---- fused backward with output gradients of a loss over all seven outputs
    gouts = c.out_grads(out)
    grads_c, grads_f, glat = eng.backward(gouts, c.params_c, c.params_f)
    torch.cuda.synchronize()
    records = dev_tensor(d.records, (n_tiles, d.record_bytes // 2), "<i2")
    d_raw = dev_tensor(d.d_raw, (n_tiles, 128, 4))
    scale = float(dev_tensor(d.scale, (2,))[0])
    masks = _mask_bits(records, n_tiles)
    if not nf:
        assert grads_f is None
        assert float(dev_tensor(d.acc_fine, (d.acc_floats,)).abs().max()) == 0.0  # no fine weight gradient is accumulated

    def dy_image(tiles, layer):
        img = decode_image(tiles, dy_off(layer), 256 if layer < 6 else 128)
        return img + decode_image(tiles, REC_LO + dy_off(layer), 256 if layer < 6 else 128) if mode == "exact_grad" else img

    # ---- FP64 reference with the kernel's ReLU decisions, ray block by ray block
    f64 = dict(dtype=torch.float64)
    pc = {k: v.detach().to(**f64).requires_grad_(True) for k, v in c.mc.named_parameters()}
    pf = {k: v.detach().to(**f64).requires_grad_(True) for k, v in c.mf.named_parameters()} if nf else None
    lat = c.latent.to(**f64).requires_grad_(True)
    expr = c.expr.to(**f64)
    rays = torch.cat((c.ro, c.rd, torch.full((n, 1), NEAR, device=dev), torch.full((n, 1), FAR, device=dev)), dim=-1).to(**f64)
    nz = {k: c.nz[k].to(**f64) for k in ("n_c", "n_f") if k in c.nz}
    bg = c.bg.to(**f64) if c.bg is not None else None
    dir_z = c.dir_z.to(**f64) if c.dir_z is not None else None
    g64 = [g.to(**f64) if g is not None else None for g in gouts]
    err = {}   # key -> [max |got - ref|, max |ref|]

    def track(key, e, r):
        cur = err.setdefault(key, [0.0, 0.0])
        cur[0], cur[1] = max(cur[0], e), max(cur[1], r)

    flip_rows = {key: 0 for _, key in passes}
    sigma_flips = {key: 0 for _, key in passes}
    for b0 in range(0, n, BLOCK):
        b1 = min(n, b0 + BLOCK)
        t0, t1 = (b0 // R) * tpu, ((b1 + R - 1) // R) * tpu   # the block's whole units, including an invalid last ray
        maps = {key: _rowmap(b0, b1, nc if pas == 0 else S, R, tpu, tc if pas else 0, dev) for pas, key in passes}
        m = {key: [_layer_mask(masks, *maps[key], layer) for layer in range(9)] for _, key in passes}
        taps = {}
        sl = slice(b0, b1)
        ref = TR.render_at_depths(rays[sl], pc, pf, expr, lat, z_c[sl], z_f[sl] if nf else None, NEAR, FAR, c.o["noise_std"],
                                  {k: v[sl] for k, v in nz.items()}, c.o["white"], bg[sl] if bg is not None else None,
                                  dir_z[sl] if dir_z is not None else None, taps, m)
        used = [(o, g[sl]) for o, g in zip(ref, g64) if o is not None]
        torch.autograd.backward([o for o, _ in used], [g for _, g in used])
        dys = [dy_image(records[t0:t1], layer) for layer in range(9)]
        row_used = torch.zeros(t1 - t0, 128, dtype=torch.bool, device=dev)
        for pas, key in passes:
            tile, row = maps[key]
            row_used[tile - t0, row] = True
            tp = taps[key]
            # 1. the kernel's ReLU decisions vs the reference's own a > 0
            bad = torch.zeros(tile.shape[0], dtype=torch.bool, device=dev)
            for layer in range(9):
                a = tp[f"a{layer}"].detach()
                diff = m[key][layer] != (a > 0)
                bad |= diff.any(dim=1)
                track(f"|a| {key} {layer}", float(a.abs()[diff].max()) if bool(diff.any()) else 0.0, float(a.abs().max()))
            flip_rows[key] += int(bad.sum())
            # the sigma ReLU: a sample whose ReLU input lies on the other side of zero than the reference's has d sigma = 0 on one
            # side only (alpha ~ 0 either way, so no other sample notices); such samples are counted, not compared
            sig_in = tp["raw"].detach()[..., 3]
            if c.o["noise_std"] > 0.0:
                sig_in = sig_in + nz["n_c" if pas == 0 else "n_f"][sl] * c.o["noise_std"]
            ok = (raw_k[key][sl].reshape(-1, 4)[:, 3] > 0) == (sig_in.reshape(-1) > 0)
            sigma_flips[key] += int((~ok).sum())
            # 2. d raw per sample
            r = tp["raw"].grad.reshape(-1, 4)[ok]
            track(f"d raw {key}", float((d_raw[tile, row][ok].double() - r).abs().max()), float(r.abs().max()))
            # 3. dY of every layer (the reference follows the kernel's masks, so every row compares)
            for layer in range(9):
                r = tp[f"a{layer}"].grad[ok]
                got = dys[layer][tile - t0, row][ok].double() / scale
                track(f"dY{layer} {key}", float((got - r).abs().max()), float(r.abs().max()))
        # rows that belong to no sample (padding rows, the invalid second ray of a last unit): exactly zero gradient
        if bool((~row_used).any()):
            if float(d_raw[t0:t1][~row_used].abs().max()) != 0.0:
                fails.append(f"d raw of rays [{b0}, {b1}): non-zero on rows that belong to no sample")
            for layer in range(9):
                if float(dys[layer][~row_used].abs().max()) != 0.0:
                    fails.append(f"dY{layer} of rays [{b0}, {b1}): non-zero on rows that belong to no sample")
        del taps, ref, used, dys

    # ---- checks
    worst = {"mask": 0.0, "d raw": 0.0, "dY": 0.0, "param": 0.0}
    for key, (e, r) in err.items():
        rel = e / (r + 1e-300)
        if key.startswith("|a|"):
            worst["mask"] = max(worst["mask"], rel)
            if rel > MASK_DECIDED[mode]:
                fails.append(f"ReLU mask {key[4:]} differs from the reference at |a| = {rel:.2e} max|a|")
        elif key.startswith("d raw"):
            worst["d raw"] = max(worst["d raw"], rel)
            if not rel <= g_draw:
                fails.append(f"{key}: {rel:.2e} > {g_draw:.0e}")
        else:
            worst["dY"] = max(worst["dY"], rel)
            gate = g_dy if int(key[2]) < 6 else g_dy_dir
            if not rel <= gate:
                fails.append(f"{key}: {rel:.2e} > {gate:.0e}")
    for pas, key in passes:
        rows = n * (nc if pas == 0 else S)
        if flip_rows[key] > max(8, int(rows * MASK_FLIP_ROWS[mode])):
            fails.append(f"{flip_rows[key]} of {rows} {key} rows have a ReLU decision unlike the reference's")
        if sigma_flips[key] > max(8, rows // 500):
            fails.append(f"{sigma_flips[key]} of {rows} {key} samples have a sigma ReLU decision unlike the reference's")
    for grads, ref_p, tag in ((grads_c, pc, "coarse"), (grads_f, pf, "fine"))[:len(passes)]:
        for k, g in zip(TR.PARAM_ORDER, grads):
            r = ref_p[k].grad
            if k.startswith("layers_dir.3"):
                if g is not None or r is not None:
                    fails.append(f"{tag} {k}: gradient of an unused parameter")
                continue
            e, s = float((g.double() - r).abs().max()), float(r.abs().max())
            worst["param"] = max(worst["param"], e / (s + 1e-300))
            if not e <= g_par * s + 1e-9:
                fails.append(f"{tag} {k}: {e / s:.2e} > {g_par:.0e}")
    e, s = float((glat.double() - lat.grad).abs().max()), float(lat.grad.abs().max())
    worst["latent"] = e / (s + 1e-300)
    if not e <= g_par * s + 1e-9:
        fails.append(f"latent: {e / s:.2e} > {g_par:.0e}")
    print(f"\n{name} {mode}: {n} rays, {nc}c+{nf}f, R={R}, {tc}+{tf} tiles/unit, {n_units} units | worst rel: params "
          f"{worst['param']:.2e}, latent {worst['latent']:.2e}, dY {worst['dY']:.2e}, d raw {worst['d raw']:.2e} | ReLU flips: "
          f"{flip_rows} rows, largest flipped |a| {worst['mask']:.1e} max|a|; sigma flips {sigma_flips}")
    assert not fails, "\n".join(fails)


# id: rays, coarse, fine, options, records budget in MB (mode exact_grad: 2 MiB records)
CHUNKED = {
    "100c60f": (41, 100, 60, dict(dir_z=True), 60),   # 5 tiles/unit, 6 units = 12 rays a chunk: 12 + 12 + 12 + 5
    "200c300f": (17, 200, 300, {}, 48),              # 6 tiles/unit, 1 ray a unit, 4 units a chunk: 4 x 4 + 1
    "64c0f": (41, 64, 0, {}, 12),                    # 1 tile/unit, 6 units = 12 rays a chunk: 12 + 12 + 12 + 5
}


@pytest.mark.parametrize("name", list(CHUNKED))
def test_chunked_backward_matches_one_launch(name, built_lib, monkeypatch):
    """A records budget too small for the batch makes the backward re-run the training forward chunk by chunk, each with the
    per-ray pointers (rays, directions, background, depth and sigma noise) advanced to the chunk's first ray.  In exact_grad
    mode its gradients agree with the one-launch backward's to 3e-5 of each tensor's largest entry, its outputs (rendered by
    the evaluation kernel) with the training forward's to 1e-5: as at 64c+64f (test_backward_exact_gpu), but at shapes where
    the coarse, fine and per-sample strides differ and the last chunk is ragged."""
    n, nc, nf, opts, budget = CHUNKED[name]
    c = _Case(n, nc, nf, opts)
    R, tc, tf = c.layout()
    units = budget // 2 // (tc + tf) & ~1
    chunk_rays = max(units, 2) * R
    chunks = (n + chunk_rays - 1) // chunk_rays
    assert chunks >= 4 and n % chunk_rays != 0
    results = []
    gouts = None
    for mb in (ONE_LAUNCH_MB, str(budget)):
        monkeypatch.setenv("NFB_TRAIN_MEM_MB", mb)
        out = c.render("exact_grad", train=True)
        if gouts is None:
            gouts = c.out_grads(out)
        l0 = c.eng.launch_count()
        gc, gf, glat = c.eng.backward(gouts, c.params_c, c.params_f)
        torch.cuda.synchronize()
        grads = [g for g in gc + (gf or []) if g is not None] + [glat]
        results.append((out, grads, c.eng.launch_count() - l0))
    (o1, g1, l1), (o2, g2, l2) = results
    # one launch: compositing backward, loss scale, chain, weight gradients, then finalize (2); chunked: the training forward
    # and those four per chunk, then finalize
    assert l1 == 6 and l2 == 5 * chunks + 2, (l1, l2, chunks)
    for k in o1:
        assert float((o1[k] - o2[k]).abs().max()) < 1e-5, k
    rel = [float((a - b).abs().max()) / max(float(a.abs().max()), 1e-12) for a, b in zip(g1, g2)]
    print(f"\nchunked {name} ({chunks} chunks of {chunk_rays} rays) vs one launch: worst relative difference {max(rel):.2e}")
    assert max(rel) <= 3e-5, rel
