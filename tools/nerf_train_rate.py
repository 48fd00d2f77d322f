"""NeRF variant, training step probe (the training kernel of csrc/nerf.cu + neddf_wgrad; opt-in path, DESIGN 4.7): forward + backward of
NeRF.forward_rays on a slice of the bench frame, and the worst parameter-gradient distance from torch autograd through the
oracle on a small batch.  First thing to run when a GPU is available again (the kernel has only run in host emulation)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import neddf_b200
from oracle import neddf_oracle as orc  # tools may use the oracle (reference values)

dev = torch.device("cuda:0")
net = neddf_b200.NeRF().to(dev)
net.set_iter(-1)
net.training_kernels = True
g = torch.Generator().manual_seed(0)


def batch(n_rays, n_edges=65):
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g), dim=-1)
    o = torch.randn(n_rays, 3, generator=g) * 0.1
    dists = 2.0 + 4.0 * torch.rand(n_rays, n_edges, generator=g).sort(dim=1).values
    return d, o, dists


# parity on a small batch against autograd through the oracle
d, o, dists = batch(37, 9)
gd, gc = torch.randn(37, 9, generator=g), torch.randn(37, 9, 3, generator=g)
out = net.forward_rays(d.to(dev), o.to(dev), dists.to(dev), "cone", neddf_b200.CONE_RAY_RADIUS)
((out["density"] * gd.to(dev)).sum() + (out["color"] * gc.to(dev)).sum()).backward()
nc = orc.NerfConfig()
P = {k: (v.detach().cpu().t().contiguous() if k.endswith(".weight") else v.detach().cpu()).requires_grad_(True) for k, v in net.state_dict().items()}
pos, dd, var = orc.make_samples(orc.RenderConfig(sampling_type="cone"), d, o, dists)
ref = orc.nerf_forward(P, nc, nc.lowpass_alpha_at(-1), pos, dd, var)
((ref["density"] * gd).sum() + (ref["color"] * gc).sum()).backward()
worst = 0.0
for k, p in net.named_parameters():
    r = P[k].grad.t() if k.endswith(".weight") else P[k].grad
    worst = max(worst, float((p.grad.cpu() - r).abs().max() / r.abs().max()))
print(f"worst parameter-gradient distance from oracle autograd: {worst:.2e}")

# throughput
n_rays = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
d, o, dists = (t.to(dev) for t in batch(n_rays))
for it in range(4):
    if it == 1:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    net.zero_grad()
    out = net.forward_rays(d, o, dists, "cone", neddf_b200.CONE_RAY_RADIUS)
    (out["density"].sum() + out["color"].sum()).backward()
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 3
print(f"NeRF forward + backward: {n_rays * 65 / ms * 1e3:.3e} evaluations/s ({ms:.1f} ms for {n_rays * 65} evaluations)")
