"""(child process of tests/test_zzz_nerf_train_gpu.py - run as `python -m tests.nerf_train_gpu_child <check> <case>`)

NeRF variant, training backward on the GPU (the training kernel of csrc/nerf.cu + neddf_wgrad behind neddf_b200.NeRF with
training_kernels=True) against the REAL reference's autograd gradients (tests/golden/make_nerf_train_golden.py).

STATUS - read before trusting a green or red mark here: this kernel was written after the round's GPU budget was
spent.  Its tile program is validated on the CPU (tests/test_nerf_train_emul.py: 256 OS threads per CTA, the same
fixtures, AddressSanitizer / UBSan / ThreadSanitizer, the autograd glue over a fake library), but these tests have never
run on hardware.  They are therefore NON-STRICT expected failures: an XPASS in the driver's log is the first hardware
run succeeding, an XFAIL is a finding for the next round; neither hides behind the rest of the suite, and the feature
stays opt-in (NeRF.training_kernels) either way."""
import sys

import numpy as np
import torch

from oracle import neddf_oracle as orc
from tests.helpers import assert_parity, nerr
from tests.test_nerf_train_emul import TrainCase

DEV = torch.device("cuda:0")


def build(c: TrainCase):
    import neddf_b200
    render = neddf_b200.NeRFRender(network_config=dict(c.net_cfg), **c.render_cfg)
    sd = {}
    for tag in ("fine", "coarse"):
        pre = f"w_{tag}." if (tag == "fine" or c.separate) else "w_fine."
        for k, v in c.z.items():
            if k.startswith(pre):
                sd[f"network_{tag}." + k[len(pre):]] = torch.from_numpy(v)
    render.load_state_dict(sd)
    render.to(DEV)
    render.set_iter(c.iter)
    for net in (render.network_coarse, render.network_fine):
        net.training_kernels = True
    cam = neddf_b200.Camera.from_matrix(neddf_b200.PinholeCalib(c.z["cam_calib"]), c.z["cam_R"], c.z["cam_T"]).to(DEV)
    cam.update_transform()
    return render, cam


def check_grads(c: TrainCase, render, tol):
    kinked = c.nc.activation_type != "tanhExp"
    checked = 0
    for k, p in render.named_parameters():
        if ("grad_" + k) not in c.z:  # a shared network appears under both names; the fixture stores it once
            continue
        assert p.grad is not None, k
        g, ref = p.grad.cpu().numpy(), c.z["grad_" + k]
        if g.ndim == 2 and g.shape[0] > 3:
            g = g[::8]
        assert g.shape == ref.shape, k
        if kinked:
            assert_parity(g, ref, tol, kinked=True, what=k)
        else:
            assert nerr(g, ref) < tol, (k, nerr(g, ref))
        checked += 1
    assert checked == len([k for k in c.z if k.startswith("grad_")])


def field_backward_matches_reference_gradients(name):
    """Field level: the recorded upstream gradients of both passes into NeRF.forward_rays under autograd."""
    import neddf_b200
    c = TrainCase(name)
    render, _ = build(c)
    d, o = orc.make_rays(c.t("uv"), c.cam)
    radius = neddf_b200.ray.CONE_RAY_RADIUS if c.rc.sampling_type == "cone" else 0.0
    loss = 0
    for tag, net, dists in (("coarse", render.network_coarse, orc.coarse_dists(c.rc, c.t("u_coarse"))),
                            ("fine", render.network_fine, c.t("dists_fine"))):
        out = net.forward_rays(d.to(DEV), o.to(DEV), dists.to(DEV), c.rc.sampling_type, radius)
        assert out["density"].requires_grad
        for k in ("density", "color"):
            assert nerr(out[k].detach().cpu().numpy(), c.z[f"field_{tag}_{k}"]) < 1e-4, (tag, k)
        loss = loss + (out["density"] * c.t(f"up_{tag}_density").to(DEV)).sum() + (out["color"] * c.t(f"up_{tag}_color").to(DEV)).sum()
    render.zero_grad()
    loss.backward()
    check_grads(c, render, 1e-4)


def render_rays_training_matches_reference(name):
    """End to end: render_rays under autograd (field forward, compositing, resampling, compositing backward, field
    backward, weight gradients) - loss and parameter gradients of the reference's own training graph."""
    c = TrainCase(name)
    render, cam = build(c)
    out = render.render_rays(c.t("uv").to(DEV), cam, uniforms=(c.t("u_coarse").to(DEV), c.t("u_fine").to(DEV)))
    loss = (out["color"].sum() + 0.1 * out["depth"].sum() + 0.05 * out["transmittance"].sum()
            + 0.1 * out["color_coarse"].sum() + 0.02 * out["depth_coarse"].sum())
    assert abs(float(loss.detach()) - float(c.z["loss"])) < 1e-4 * abs(float(c.z["loss"]))
    render.zero_grad()
    loss.backward()
    check_grads(c, render, 2e-4)  # through the resampling, like test_render_rays_training_matches_reference_gradients


if __name__ == "__main__":
    check, case = sys.argv[1], sys.argv[2]
    {"field": field_backward_matches_reference_gradients, "render": render_rays_training_matches_reference}[check](case)
    torch.cuda.synchronize()
    print(f"nerf_train_gpu_child: {check} {case} ok")
