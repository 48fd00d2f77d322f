"""NeRF field variant on the GPU (csrc/nerf.cu behind neddf_b200.NeRF) against goldens recorded from the REAL
reference (tests/golden/make_nerf_golden.py) and the oracle restatement: per-sample field outputs with explicit
samples and with the fused ray geometry, render_rays through NeRFRender with the recorded uniforms, the image path."""
import numpy as np
import pytest
import torch

from oracle import neddf_oracle as orc
from tests.helpers import PARITY_TOL, nerr
from tests.test_nerf_oracle import NerfCase

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def build(c: NerfCase):
    import neddf_b200
    render = neddf_b200.NeRFRender(network_config=dict(c.net_cfg), **c.render_cfg)
    sd = {}
    for tag in ("fine", "coarse"):
        pre = f"w_{tag}." if f"w_{tag}.layers.0.weight" in c.z else "w_fine."
        for k, v in c.z.items():
            if k.startswith(pre):
                sd[f"network_{tag}." + k[len(pre):]] = torch.from_numpy(v)
    missing = render.load_state_dict(sd)
    assert not missing.missing_keys and not missing.unexpected_keys, missing  # the reference's state_dict layout
    render.to(DEV)
    render.set_iter(c.iter)
    cam = neddf_b200.Camera.from_matrix(neddf_b200.PinholeCalib(c.z["cam_calib"]), c.z["cam_R"], c.z["cam_T"]).to(DEV)
    cam.update_transform()
    return render, cam


@pytest.mark.parametrize("name", ["relu", "tanhexp"])
def test_nerf_field_matches_reference(name):
    import neddf_b200
    c = NerfCase(name)
    render, _ = build(c)
    d, o = orc.make_rays(c.t("uv"), c.cam)
    radius = neddf_b200.ray.CONE_RAY_RADIUS if c.rc.sampling_type == "cone" else 0.0
    for tag, net, dists in (("coarse", render.network_coarse, orc.coarse_dists(c.rc, c.t("u_coarse"))),
                            ("fine", render.network_fine, c.t("dists_fine"))):
        pos, dd, var = orc.make_samples(c.rc, d, o, dists)
        with torch.no_grad():
            out = net(neddf_b200.Sampling(pos.to(DEV), dd.contiguous().to(DEV), var.to(DEV)))
            fused = net.forward_rays(d.to(DEV), o.to(DEV), dists.to(DEV), c.rc.sampling_type, radius)
        for k in ("density", "color"):
            ref = c.z[f"field_{tag}_{k}"]
            assert out[k].shape == ref.shape
            assert nerr(out[k].cpu().numpy(), ref) < PARITY_TOL, (tag, k)
            assert nerr(fused[k].cpu().numpy(), ref) < PARITY_TOL, (tag, k, "fused geometry")


@pytest.mark.parametrize("name", ["relu", "tanhexp"])
def test_nerf_render_rays_matches_reference(name):
    c = NerfCase(name)
    render, cam = build(c)
    with torch.no_grad():
        out = render.render_rays(c.t("uv").to(DEV), cam, uniforms=(c.t("u_coarse").to(DEV), c.t("u_fine").to(DEV)))
    ref_keys = sorted(k[4:] for k in c.z if k.startswith("out_"))
    assert sorted(out.keys()) == ref_keys  # no penalty keys for this variant (nerf_render.py:149-187)
    for k in ref_keys:
        tol = 1e-3 if k.startswith("weight") else PARITY_TOL  # same bounds as the NeDDF render test
        assert nerr(out[k].cpu().numpy(), c.z["out_" + k]) < tol, k


def test_nerf_image_path_and_ragged_tiles():
    """render_image through the NeRF kernel (sample counts that are not multiples of the 64-sample tile) against
    the oracle field on the same samples; training-mode calls are refused."""
    import neddf_b200
    c = NerfCase("relu")
    render, cam = build(c)
    img = render.render_image(40, 30, cam, ["color", "depth", "transmittance"], 1, 333)
    assert img["color"].shape == (30, 40, 3) and bool(torch.isfinite(img["color"]).all())
    net = render.network_fine
    g = torch.Generator().manual_seed(5)
    for n in (1, 63, 65, 1000):
        pos = (torch.rand(1, n, 3, generator=g) * 2 - 1)
        dd = torch.nn.functional.normalize(torch.randn(1, n, 3, generator=g), dim=-1)
        var = torch.rand(1, n, 3, generator=g) * 1e-3
        with torch.no_grad():
            out = net(neddf_b200.Sampling(pos.to(DEV), dd.to(DEV), var.to(DEV)))
            ref = orc.nerf_forward(c.params("fine"), c.nc, c.alpha, pos, dd, var)
        for k in ("density", "color"):
            a, r = out[k].cpu().numpy(), ref[k].numpy()
            assert np.abs(a - r).max() <= PARITY_TOL * max(np.abs(r).max(), 1.0), (n, k)
    with pytest.raises(NotImplementedError):
        render.render_rays(c.t("uv").to(DEV), cam)  # autograd enabled, trainable parameters
