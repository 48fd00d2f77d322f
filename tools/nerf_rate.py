"""Throughput of the NeRF variant's kernel (csrc/nerf.cu): fused-ray forward on a slice of the bench frame.
FLOP per evaluation = 2 x sum of in x out over its linear layers (padding not counted)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import neddf_b200
from oracle import neddf_oracle as orc  # shapes only (tools may use the oracle's config helpers)

n_rays = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
dev = torch.device("cuda:0")
net = neddf_b200.NeRF().to(dev)
net.set_iter(-1)
flop = 2 * sum(i * o for _, i, o in orc.nerf_layer_shapes(orc.NerfConfig()))
g = torch.Generator().manual_seed(0)
d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g), dim=-1).to(dev)
o = (torch.randn(n_rays, 3, generator=g) * 0.1).to(dev)
dists = (2.0 + 4.0 * torch.rand(n_rays, 65, generator=g).sort(dim=1).values).to(dev)
with torch.no_grad():
    net.forward_rays(d, o, dists, "cone", neddf_b200.CONE_RAY_RADIUS)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        net.forward_rays(d, o, dists, "cone", neddf_b200.CONE_RAY_RADIUS)
    e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 3
ev = n_rays * 65
print(f"NeRF kernel: {ev / ms * 1e3:.3e} evaluations/s, {ev * flop / ms * 1e-9:.1f} TFLOP/s fp32 FMA "
      f"({flop} FLOP/evaluation, {ms:.2f} ms for {ev} evaluations)")
