"""The small tensor helpers of the drop-in `nerf` package (nerf/nerf_helpers.py) that the reference's unmodified scripts call on
the host side of the boundary, against the reference's own functions on CPU: same values bit for bit, same shapes, same
chunking.  What the reference returned is stored in tests/golden/reference_checks/helpers.json (arrays as digests of their
bytes) by oracle/make_golden_reference_checks.py; CPU only."""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import make_golden_reference_checks as G  # noqa: E402


class Gold:
    def __init__(self):
        with open(os.path.join(G.OUT, "helpers.json")) as f:
            self.meta = json.load(f)

    def equal(self, key, t):
        """t is bit for bit the array the reference returned under `key` (same shape, dtype and bytes)."""
        return self.meta["arrays"][key] == G.array_digest(t.detach().numpy())


@pytest.fixture(scope="module")
def both(built_lib):
    sys.path.insert(0, os.path.join(ROOT, "4d-facial-avatars_b200"))
    import nerf
    return nerf, Gold()


@pytest.mark.parametrize("H,W,intr", G.RAY_BUNDLE_CASES)
def test_get_ray_bundle(both, H, W, intr):
    nerf, ref = both
    pose = G.pose_for(H * 100 + W)
    got = nerf.get_ray_bundle(H, W, intr, pose)
    got34 = nerf.get_ray_bundle(H, W, np.array(intr), pose[:3, :4])
    for key, b, c in zip(("ro", "rd"), got, got34):
        assert b.shape == (H, W, 3) and ref.equal(f"ray_bundle/{H}x{W}/{key}", b) and torch.equal(b, c)


@pytest.mark.parametrize("n_freq,include_input,log_sampling", G.PE_CASES)
def test_positional_encoding_and_embedding_function(both, n_freq, include_input, log_sampling):
    nerf, ref = both
    x = torch.randn(37, 3, generator=torch.Generator().manual_seed(n_freq)) * 3.0
    key = f"pe/{n_freq}/{int(include_input)}/{int(log_sampling)}"  # the reference's embedding function returns the same
    assert ref.equal(key, nerf.positional_encoding(x, n_freq, include_input, log_sampling))
    f = nerf.get_embedding_function(n_freq, include_input, log_sampling)
    assert ref.equal(key, f(x))


def test_meshgrid_minibatches_and_metrics(both):
    nerf, ref = both
    a, b = torch.arange(5, dtype=torch.float32), torch.arange(3, dtype=torch.float32) * 2.0
    got = nerf.meshgrid_xy(a, b)
    assert len(got) == 2 and "meshgrid/2" not in ref.meta["arrays"]
    for i, v in enumerate(got):
        assert ref.equal(f"meshgrid/{i}", v)
    x = torch.randn(23, 4, generator=torch.Generator().manual_seed(3))
    for cs in (1, 7, 23, 100):
        g = nerf.get_minibatches(x, chunksize=cs)
        assert len(g) == ref.meta["values"][f"minibatches/{cs}/n"] and all(ref.equal(f"minibatches/{cs}/{i}", q) for i, q in enumerate(g))
    y = torch.randn(23, 4, generator=torch.Generator().manual_seed(4))
    assert ref.equal("img2mse", nerf.img2mse(x, y))
    for m, want in zip((0.0, 1e-5, 0.0123, 1.0), ref.meta["values"]["mse2psnr"]):
        assert want == nerf.mse2psnr(m)


def test_cfgnode_on_the_shipped_yaml(both):
    """The scripts build `CfgNode(yaml.load(...))`, read nested attributes and write `cfg.dump()` next to the checkpoints
    (train_transformed_rays.py:46-50, 126-128): same tree, same leaves, a dump that loads back to the same dict."""
    import yaml
    nerf, ref = both
    raw = ref.meta["config"]
    b = nerf.CfgNode(raw)
    leaves = {}

    def walk(y, trail):
        for k in y.keys():
            v = getattr(y, k)
            if isinstance(v, dict):
                assert isinstance(v, nerf.CfgNode), trail + [k]
                walk(v, trail + [k])
            else:
                leaves[tuple(trail + [k])] = (type(v).__name__, v)

    walk(b, [])
    # the reference's CfgNode on the same dict: the same tree and the same leaves, of the same types
    assert leaves == {tuple(trail): (tname, v) for trail, tname, v in ref.meta["config_leaves"]}
    assert b.nerf.train.num_coarse == 64 and b.nerf.validation.num_fine == 64 and b.dataset.no_ndc is True
    assert yaml.safe_load(b.dump()) == ref.meta["config_dump"] == raw
    with pytest.raises(AttributeError):
        b.nerf.no_such_option


def test_model_class_against_the_reference_class(both):
    """ConditionalBlendshapePaperNeRFModel built with the keyword arguments the scripts pass (train_transformed_rays.py:150-176):
    same state_dict keys / shapes / dtypes, a reference checkpoint loads into the drop-in and back (strict), the torch forward of
    the drop-in (not the hot path) returns the reference module's values bit for bit, and the attributes the scripts and the
    renderer read are the same."""
    import nerface_oracle as O
    nerf, ref = both
    m = nerf.models.ConditionalBlendshapePaperNeRFModel(**G.MODEL_KW)
    # the reference model's state_dict layout; the checkpoint below loaded into the reference model strictly
    assert [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()] == ref.meta["state_dict"]
    m.load_state_dict(O.random_init_params(G.MODEL_SEED), strict=True)
    for name in ("dim_xyz", "dim_dir", "dim_expression", "dim_latent_code", "use_viewdirs"):
        assert getattr(m, name) == ref.meta["attributes"][name], name
    g = torch.Generator().manual_seed(12)
    x = torch.randn(19, m.dim_xyz + m.dim_dir, generator=g)
    expr, lat = torch.randn(76, generator=g), torch.randn(32, generator=g)
    with torch.no_grad():
        assert ref.equal("model/forward", m(x, expr, lat))
    assert sum(p.numel() for p in m.parameters()) == ref.meta["n_parameters"]
