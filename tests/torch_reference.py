"""Plain-PyTorch restatement of one training forward/backward of the render path AT GIVEN sample depths — test
infrastructure only (the floating-point reference for the fused backward kernels; runs on whatever device and in whatever
floating-point type its inputs have: FP32 or FP64).  Follows train_utils.py:36-162, volume_rendering_utils.py:7-75, models.py:236-261; resampled depths carry no
gradient (`z_samples.detach()`, train_utils.py:124)."""
import torch

PARAM_ORDER = ([f"layers_xyz.{i}.{k}" for i in range(6) for k in ("weight", "bias")]
               + ["fc_feat.weight", "fc_feat.bias", "fc_alpha.weight", "fc_alpha.bias"]
               + [f"layers_dir.{i}.{k}" for i in range(4) for k in ("weight", "bias")]
               + ["fc_rgb.weight", "fc_rgb.bias"])


def _posenc(x, n_freq, include_input):
    parts = [x] if include_input else []
    for k in range(n_freq):
        parts += [torch.sin(x * float(2 ** k)), torch.cos(x * float(2 ** k))]
    return torch.cat(parts, dim=-1)


def _mlp(p, x, expr, latent, taps=None, masks=None):
    """taps (dict): receives the post-activation outputs h0..h5, g0..g2 and the pre-activations a0..a8 (retain_grad).
    masks: None, or the nine ReLU decisions ([rows, width] bool, layers a0..a8) to apply in place of a > 0."""
    F = torch.nn.functional
    xyz, dirs = x[..., :63], x[..., 63:]
    rows = xyz.shape[0]
    cond = torch.cat(((expr * 1 / 3).reshape(1, -1).expand(rows, -1), latent.reshape(1, -1).expand(rows, -1)), dim=1)
    initial = torch.cat((xyz, cond), dim=1)

    def act(a, name_pre, name_post):
        if taps is not None:
            a.retain_grad()
            taps[name_pre] = a
        h = F.relu(a) if masks is None else a * masks[int(name_pre[1:])]
        if taps is not None:
            taps[name_post] = h
        return h

    h = initial
    for i in range(6):
        h = act(F.linear(torch.cat((initial, h), dim=-1) if i == 3 else h, p[f"layers_xyz.{i}.weight"], p[f"layers_xyz.{i}.bias"]),
                f"a{i}", f"h{i}")
    feat = F.linear(h, p["fc_feat.weight"], p["fc_feat.bias"])
    sigma = F.linear(feat, p["fc_alpha.weight"], p["fc_alpha.bias"])
    g = act(F.linear(torch.cat((feat, dirs), dim=-1), p["layers_dir.0.weight"], p["layers_dir.0.bias"]), "a6", "g0")
    g = act(F.linear(g, p["layers_dir.1.weight"], p["layers_dir.1.bias"]), "a7", "g1")
    g = act(F.linear(g, p["layers_dir.2.weight"], p["layers_dir.2.bias"]), "a8", "g2")
    if taps is not None:
        taps["pe"] = xyz
        taps["ped"] = dirs
    return torch.cat((F.linear(g, p["fc_rgb.weight"], p["fc_rgb.bias"]), sigma), dim=-1)


def _composite(raw, z, rd, noise_std, noise, white_bkgd, bg):
    n, s = z.shape
    delta = torch.cat((z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)), dim=-1) * rd.norm(p=2, dim=-1, keepdim=True)
    col = torch.sigmoid(raw[..., :3])
    if bg is not None:
        col = torch.cat((col[:, :-1], bg[:, None, :]), dim=1)
    sig_in = raw[..., 3]
    if noise_std > 0.0:
        sig_in = sig_in + noise * noise_std
    last = torch.zeros(s, device=z.device, dtype=z.dtype)
    last[-1] = 1e-6
    sigma = torch.relu(sig_in) + last
    alpha = 1.0 - torch.exp(-sigma * delta)
    trans = torch.cumprod(1.0 - alpha + 1e-10, dim=-1)
    trans = torch.cat((torch.ones_like(trans[:, :1]), trans[:, :-1]), dim=-1)
    w = alpha * trans
    rgb = (w[..., None] * col).sum(dim=-2)
    depth = (w * z).sum(dim=-1)
    acc = w.sum(dim=-1)
    disp = 1.0 / torch.max(1e-10 * torch.ones_like(depth), depth / acc)
    if white_bkgd:
        rgb = rgb + (1.0 - acc[..., None])
    return rgb, disp, acc, w


def _pass(p, z, rays, dir_cols, expr, latent, noise_std, noise, white_bkgd, bg, taps=None, masks=None):
    ro, rd = rays[:, :3], rays[:, 3:6]
    n, s = z.shape
    pts = ro[:, None, :] + rd[:, None, :] * z[:, :, None]
    x = torch.cat((_posenc(pts.reshape(-1, 3), 10, True), _posenc(dir_cols[:, None, :].expand(n, s, 3).reshape(-1, 3), 4, False)), dim=-1)
    raw = _mlp(p, x, expr, latent, taps, masks).reshape(n, s, 4)
    if taps is not None:
        raw.retain_grad()
        taps["raw"] = raw
    return _composite(raw, z, rd, noise_std, noise, white_bkgd, bg)


def render_at_depths(rays, params_c, params_f, expr, latent, z_c, z_f, near, far, noise_std=0.0, noise=None,
                     white_bkgd=False, bg=None, dir_z=None, taps=None, masks=None):
    """rays [N,8]; params_*: dict name -> tensor (requires_grad leaves).  Returns the 7-tuple as differentiable tensors.
    `taps` (dict): receives per-pass intermediate tensors under "coarse"/"fine".  `masks` (dict): per pass ("coarse"/"fine")
    the nine [N*S, width] ReLU decisions to use instead of a > 0 (rows ray-major: ray i, sample j at i*S + j)."""
    dir_cols = torch.cat((dir_z.reshape(-1, 1) if dir_z is not None else rays[:, 5:6],
                          torch.full_like(rays[:, :1], near), torch.full_like(rays[:, :1], far)), dim=-1)
    nz = noise or {}
    mk = masks or {}
    tc = taps.setdefault("coarse", {}) if taps is not None else None
    rgb_c, disp_c, acc_c, w = _pass(params_c, z_c, rays, dir_cols, expr, latent, noise_std, nz.get("n_c"), white_bkgd, bg, tc,
                                    mk.get("coarse"))
    outs = [rgb_c, disp_c, acc_c, None, None, None, w[:, -1]]
    if params_f is not None:
        tf = taps.setdefault("fine", {}) if taps is not None else None
        rgb_f, disp_f, acc_f, w = _pass(params_f, z_f, rays, dir_cols, expr, latent, noise_std, nz.get("n_f"), white_bkgd, bg, tf,
                                        mk.get("fine"))
        outs[3:7] = [rgb_f, disp_f, acc_f, w[:, -1]]
    return outs
