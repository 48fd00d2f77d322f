"""Drop-in for neddf.network.NeRF (neddf/network/nerf.py:13-178) on the B200 path: same constructor, same
module / state_dict layout (``layers.N``, ``outL_density``, ``outL_color.0`` / ``.2``), ``forward(Sampling)`` and
``set_iter``; the network itself runs in one CUDA kernel (``csrc/nerf.cu`` behind ``neddf_nerf_*``).

Scope (SURVEY 8(f) item 3): inference - ``forward`` / ``forward_rays`` under ``torch.no_grad()``, i.e. everything
``NeRFRender.render_image`` and ``render_rays`` in eval need.  By default a call with autograd enabled on trainable
parameters raises (train it with the reference, load the checkpoint here).  No CPU / PyTorch fallback.

Training (opt-in: ``net.training_kernels = True`` or NEDDF_NERF_TRAIN=1): the backward of the autograd graph of
nerf.py:107-165 with respect to the parameters runs in the training kernel of ``csrc/nerf.cu`` (the forward's tile
program, recomputed per tile, then the data gradients in fp32 FMA) + ``neddf_wgrad`` / ``neddf_colsum_value_rows``
(weight / bias gradients).  That kernel has so far been validated through the host emulation of its tile program only
(tests/test_nerf_train_emul.py: the real reference's autograd gradients, sanitizers), hence the opt-in."""
import ctypes as C
import math
import os
from typing import Dict, List, Optional

import torch
from torch import Tensor, nn

from . import _lib as L
from .network import BaseNeuralField
from .ray import Sampling


def lowpass_scale(embed_dim: int, alpha: float) -> List[float]:
    """PositionalEncoding.get_lowpass_scale per frequency (nn_module/positional_encoding.py:67-89)."""
    if alpha >= embed_dim:
        return [1.0] * embed_dim
    s = [1.0] * embed_dim
    k = int(alpha)
    s[k] = 0.5 * (1.0 - math.cos(math.pi * (alpha - k))) + 1e-7
    for i in range(k + 1, embed_dim):
        s[i] = 1e-7
    return s


class _NerfTrainFn(torch.autograd.Function):
    """NeRF.forward under autograd.  forward: the inference kernel (neddf_nerf_forward[_rays]); backward:
    neddf_nerf_train_backward[_rays] (recomputes the forward per tile, leaves layer inputs X and pre-activation gradients
    G in global memory), then gW = X^T G as tensor-core split-K GEMMs (neddf_wgrad) and bias gradients as column sums.
    Gradients flow to the module's parameters only (nerf_trainer.py:38-42 optimises nothing else)."""

    @staticmethod
    def forward(ctx, net, a, b, c, sampling_type, ray_radius, *params):
        """(a, b, c) = (ray_dir[B,3], ray_orig[B,3], dists[B,S]) with a sampling type, or the Sampling tensors
        (pos, dir, var)[B,S,3] when sampling_type is None."""
        from_rays = sampling_type is not None
        with torch.no_grad():
            out = net._launch_forward(a, b, c, sampling_type, ray_radius)
        ctx.net, ctx.meta = net, (sampling_type, float(ray_radius), net._lowpass_list())
        ctx.save_for_backward(a, b, c)
        return out["density"], out["color"]

    @staticmethod
    def backward(ctx, g_density, g_color):
        net = ctx.net
        a, b, c = ctx.saved_tensors
        sampling_type, ray_radius, lowpass = ctx.meta
        from_rays = sampling_type is not None
        B, S = (c.shape if from_rays else a.shape[:2])
        n = B * S
        device = a.device
        Lh, W = net.layer_count, 256
        n_e, n_d = 6 * net.embed_pos_rank, 6 * net.embed_dir_rank

        def prep(g, shape):
            if g is None:
                return torch.zeros(shape, device=device, dtype=torch.float32)
            return g.contiguous().to(torch.float32)

        g_density, g_color = prep(g_density, (B, S)), prep(g_color, (B, S, 3))
        X = torch.empty(Lh, n, W, device=device, dtype=torch.float32)
        G = torch.empty(Lh, n, W, device=device, dtype=torch.float32)
        E = torch.empty(n, n_e, device=device, dtype=torch.float32)
        D = torch.empty(n, n_d, device=device, dtype=torch.float32)
        C1 = torch.empty(n, W, device=device, dtype=torch.float32)
        GC1 = torch.empty(n, W, device=device, dtype=torch.float32)
        GZD = torch.empty(n, device=device, dtype=torch.float32)
        lib = L.lib()
        h = net._kernel_handle(device, "_train")
        stream = L.stream_ptr(device)
        with torch.cuda.device(device):
            if from_rays:
                L.check(lib.neddf_nerf_train_backward_rays(
                    h, L.fbuf(lowpass), L.ptr(a), L.ptr(b), L.ptr(c), B, S, L.SAMPLING_IDS[sampling_type], ray_radius,
                    L.ptr(g_density), L.ptr(g_color), L.ptr(X), L.ptr(G), L.ptr(E), L.ptr(D), L.ptr(C1), L.ptr(GC1), L.ptr(GZD), stream),
                    "nerf_train_backward_rays")
            else:
                L.check(lib.neddf_nerf_train_backward(
                    h, L.fbuf(lowpass), L.ptr(a), L.ptr(b), L.ptr(c), n, L.ptr(g_density), L.ptr(g_color), L.ptr(X), L.ptr(G),
                    L.ptr(E), L.ptr(D), L.ptr(C1), L.ptr(GC1), L.ptr(GZD), stream), "nerf_train_backward")
            ws = getattr(net, "_wgrad_ws", None)
            if ws is None or ws.device != device:
                ws = torch.empty(int(lib.neddf_wgrad_workspace_bytes()) // 4, device=device, dtype=torch.float32)
                net._wgrad_ws = ws

            def wgrad_into(out, row0, A, lda, ka, Bm, n_cols):
                """out[row0 : row0 + ka, :n_cols] = A[:, :ka]^T Bm[:, :n_cols] (Bm has 256 columns), 128 columns of A at a time."""
                for c0 in range(0, ka, 128):
                    kk = min(128, ka - c0)
                    L.check(lib.neddf_wgrad(L.ptr(A), lda, c0, kk, L.ptr(Bm), W, n,
                                            C.c_void_p(out.data_ptr() + 4 * (row0 + c0) * out.shape[1]), out.shape[1], n_cols,
                                            L.ptr(ws), stream), "wgrad")

            def colsum(Gm):
                out = torch.empty(W, device=device, dtype=torch.float32)
                L.check(lib.neddf_colsum_value_rows(L.ptr(Gm), n, W, L.ptr(out), L.ptr(ws), stream), "colsum")
                return out

            grads = []
            for l in range(Lh):  # layers.l: d W^T [in, 256] = in_l^T G_l with in_0 = E, in_l = [h_{l-1} | E if l-1 in skips]
                parts = [(E, n_e)] if l == 0 else ([(X[l - 1], W)] + ([(E, n_e)] if (l - 1) in net.skips else []))
                gWt = torch.empty(sum(k for _, k in parts), W, device=device, dtype=torch.float32)
                row0 = 0
                for Xp, k_in in parts:
                    wgrad_into(gWt, row0, Xp, k_in, k_in, G[l], W)
                    row0 += k_in
                grads += [gWt.t().contiguous(), colsum(G[l])]
            gwd = torch.empty(1, W, device=device, dtype=torch.float32)  # outL_density: GZD^T h_{L-1}
            wgrad_into(gwd, 0, GZD, 1, 1, X[Lh - 1], W)
            grads += [gwd, GZD.sum().reshape(1)]
            # (all GEMMs with n_cols = ld_out = 256, the parameters test_wgrad_gemm holds on hardware; the colour branch is
            #  128 wide, the upper half of GC1 / C1 is zero and sliced away)
            gc1t = torch.empty(W + n_d, W, device=device, dtype=torch.float32)  # outL_color.0: [h_{L-1} | D]^T GC1
            wgrad_into(gc1t, 0, X[Lh - 1], W, W, GC1, W)
            wgrad_into(gc1t, W, D, n_d, n_d, GC1, W)
            grads += [gc1t[:, :W // 2].t().contiguous(), colsum(GC1)[:W // 2].contiguous()]
            gc2 = torch.empty(3, W, device=device, dtype=torch.float32)  # outL_color.2: g_color^T C1
            g_col2 = g_color.reshape(n, 3)
            wgrad_into(gc2, 0, g_col2, 3, 3, C1, W)
            grads += [gc2[:, :W // 2].contiguous(), g_col2.sum(0)]
        return (None, None, None, None, None, None) + tuple(grads)


class NeRF(BaseNeuralField):
    def __init__(
        self,
        embed_pos_rank: int = 10,
        embed_dir_rank: int = 4,
        layer_count: int = 8,
        layer_width: int = 256,
        activation_type: str = "ReLU",
        density_activation_type: str = "ReLU",
        skips: Optional[List[int]] = None,
        lowpass_alpha_offset: float = 10.0,
    ) -> None:
        super().__init__()
        input_pos_dim, input_dir_dim = embed_pos_rank * 6, embed_dir_rank * 6
        if skips is None:
            skips = [4]
        self.skips = [int(s) for s in skips]
        if activation_type not in L.ACT_IDS or density_activation_type not in L.ACT_IDS:
            raise KeyError(f"unknown activation {activation_type!r}/{density_activation_type!r}")  # nerf.py:72-81
        self.activation_type, self.density_activation_type = activation_type, density_activation_type
        self.embed_pos_rank, self.embed_dir_rank = int(embed_pos_rank), int(embed_dir_rank)
        self.layer_count, self.layer_width = int(layer_count), int(layer_width)
        # identical construction order and shapes to nerf.py:86-103 (same parameters for the same torch seed)
        layers: List[nn.Module] = [nn.Linear(input_pos_dim, layer_width)]
        for layer_id in range(layer_count - 1):
            layers.append(nn.Linear(layer_width + (input_pos_dim if layer_id in self.skips else 0), layer_width))
        self.layers = nn.ModuleList(layers)
        self.outL_density = nn.Linear(layer_width, 1)
        self.outL_color = nn.Sequential(nn.Linear(layer_width + input_dir_dim, layer_width // 2), nn.ReLU(),
                                        nn.Linear(layer_width // 2, 3))
        self.lowpass_alpha_offset = float(lowpass_alpha_offset)
        self.lowpass_alpha = float(lowpass_alpha_offset)
        # kernel-side state
        self.engine = "fp32"  # the only engine of this variant; NeRFRender.set_engine may overwrite the attribute
        self._handle = None
        self._handle_device = None
        self._packed_key = None
        self._profile_events = None
        # training backward (neddf_nerf_train_*): opt-in until it has been run on hardware (module docstring)
        self.training_kernels = os.environ.get("NEDDF_NERF_TRAIN", "0") not in ("", "0")
        self._train_handle = None
        self._train_handle_device = None
        self._train_packed_key = None

    # ------------------------------------------------------------------ kernel plumbing --
    def _ordered_layers(self) -> List[nn.Linear]:
        return list(self.layers) + [self.outL_density, self.outL_color[0], self.outL_color[2]]

    def _lowpass_list(self) -> List[float]:
        return lowpass_scale(self.embed_pos_rank, self.lowpass_alpha)

    def _kernel_handle(self, device: torch.device, kind: str):
        """Handle of neddf_nerf_* (kind "") or of the training backward's neddf_nerf_train_* (kind "_train", which also
        holds the transposed weight packs) on ``device``: created on first use or a device change, re-packed when a
        parameter changed."""
        lib = L.lib()
        api = "neddf_nerf" + kind
        if getattr(self, kind + "_handle") is None or getattr(self, kind + "_handle_device") != device:
            self._release_handle(kind)
            h = C.c_void_p()
            with torch.cuda.device(device):
                cfg = self._config_struct()
                L.check(getattr(lib, api + "_create")(C.byref(cfg), C.byref(h)), api[6:] + "_create")
            setattr(self, kind + "_handle", h)
            setattr(self, kind + "_handle_device", device)
        layers = self._ordered_layers()
        key = tuple((p.data_ptr(), p._version) for l in layers for p in (l.weight, l.bias))
        if key != getattr(self, kind + "_packed_key"):
            for l in layers:
                if l.weight.dtype != torch.float32 or not l.weight.is_contiguous() or l.weight.device != device:
                    raise RuntimeError("neddf_b200: parameters must be contiguous fp32 tensors on the module's device")
            n = len(layers)
            ws = (C.c_void_p * n)(*[l.weight.data_ptr() for l in layers])
            bs = (C.c_void_p * n)(*[l.bias.data_ptr() for l in layers])
            with torch.cuda.device(device):
                L.check(getattr(lib, api + "_set_weights")(getattr(self, kind + "_handle"), ws, bs, n, L.stream_ptr(device)),
                        api[6:] + "_set_weights")
            setattr(self, kind + "_packed_key", key)
        return getattr(self, kind + "_handle")

    def _release_handle(self, kind: str) -> None:
        h = getattr(self, kind + "_handle", None)
        if h is not None:
            getattr(L.lib(), "neddf_nerf" + kind + "_destroy")(h)
        setattr(self, kind + "_handle", None)
        setattr(self, kind + "_handle_device", None)
        setattr(self, kind + "_packed_key", None)

    def _config_struct(self) -> L.NerfConfig:
        c = L.NerfConfig()
        c.embed_pos_rank, c.embed_dir_rank = self.embed_pos_rank, self.embed_dir_rank
        c.layer_count, c.layer_width = self.layer_count, self.layer_width
        c.activation_type = L.ACT_IDS[self.activation_type]
        c.density_activation_type = L.ACT_IDS[self.density_activation_type]
        if len(self.skips) > L.MAX_SKIPS:
            raise NotImplementedError("neddf_b200: more than 8 skip connections")
        c.n_skips = len(self.skips)
        for i, s in enumerate(self.skips):
            c.skips[i] = s
        return c

    def _release(self) -> None:
        self._release_handle("")
        self._release_handle("_train")

    def __del__(self):
        try:
            self._release()
        except Exception:  # interpreter shutdown
            pass

    def _field(self, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("neddf_b200.NeRF runs on CUDA devices only: move the module with .to('cuda') "
                               "(the hot path has no CPU implementation)")
        return self._kernel_handle(device, "")

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._packed_key = None  # .to()/.cuda() replaced the parameter storage
        self._train_packed_key = None
        return r

    def invalidate(self) -> None:
        self._packed_key = None
        self._train_packed_key = None

    def __getstate__(self):
        d = self.__dict__.copy()
        d["_handle"], d["_handle_device"], d["_packed_key"], d["_profile_events"] = None, None, None, None
        d["_train_handle"], d["_train_handle_device"], d["_train_packed_key"] = None, None, None
        d.pop("_wgrad_ws", None)
        return d

    def check_engine_status(self) -> None:
        """(fp32 kernel: no range checks to report)"""

    def _wants_grad(self) -> bool:
        """Autograd is recording and some parameter is trainable.  Without the opt-in that is refused."""
        if not (torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())):
            return False
        if not self.training_kernels:
            raise NotImplementedError(
                "neddf_b200.NeRF is forward-only on the B200 path by default: wrap the call in torch.no_grad() / use "
                "render_image, or train with the reference and load the checkpoint.  The training backward kernel "
                "(neddf_nerf_train_*) is opt-in - net.training_kernels = True or NEDDF_NERF_TRAIN=1 - until it has been "
                "run on hardware (so far: host emulation against the reference's autograd gradients)")
        return True

    def _launch_forward(self, a: Tensor, b: Tensor, c: Tensor, sampling_type, ray_radius: float) -> Dict[str, Tensor]:
        """The inference kernels on rays (sampling_type given) or explicit samples; called under no_grad."""
        if sampling_type is not None:
            return self.forward_rays(a, b, c, sampling_type, ray_radius)
        return self.forward(Sampling(a, b, c))

    def _forward_autograd(self, a: Tensor, b: Tensor, c: Tensor, sampling_type, ray_radius: float) -> Dict[str, Tensor]:
        flat = [t for l in self._ordered_layers() for t in (l.weight, l.bias)]
        density, color = _NerfTrainFn.apply(self, a, b, c, sampling_type, float(ray_radius), *flat)
        return {"density": density, "color": color}

    def _lowpass(self):
        return L.fbuf(lowpass_scale(self.embed_pos_rank, self.lowpass_alpha))

    # ----------------------------------------------------------------------- forward --
    def forward(self, sampling: Sampling) -> Dict[str, Tensor]:
        """nerf.py:107-165: {'density': [B,S], 'color': [B,S,3]}."""
        pos = L.require_cuda_f32(sampling.sample_pos, "sample_pos")
        sdir = L.require_cuda_f32(sampling.sample_dir, "sample_dir")
        var = L.require_cuda_f32(sampling.diag_variance, "diag_variance")
        B, S = pos.shape[0], pos.shape[1]
        if self._wants_grad():
            return self._forward_autograd(pos.reshape(B, S, 3), sdir.reshape(B, S, 3), var.reshape(B, S, 3), None, 0.0)
        device = pos.device
        out = {"density": torch.empty(B, S, device=device, dtype=torch.float32),
               "color": torch.empty(B, S, 3, device=device, dtype=torch.float32)}
        h = self._field(device)
        with torch.cuda.device(device):
            L.check(L.lib().neddf_nerf_forward(h, self._lowpass(), L.ptr(pos), L.ptr(sdir), L.ptr(var), B * S,
                                               L.ptr(out["density"]), L.ptr(out["color"]), L.stream_ptr(device)),
                    "nerf_forward")
        return out

    def forward_rays(self, ray_dir: Tensor, ray_orig: Tensor, dists: Tensor, sampling_type: str, ray_radius: float,
                     need_penalty: bool = True, need_aux: bool = True) -> Dict[str, Tensor]:
        """Same network with the sample geometry fused into the kernel (what NeRFRender calls; the NeRF variant has
        neither penalties nor auxiliary fields, the flags are accepted for interface parity)."""
        ray_dir = L.require_cuda_f32(ray_dir, "ray_dir")
        ray_orig = L.require_cuda_f32(ray_orig, "ray_orig")
        dists = L.require_cuda_f32(dists, "dists")
        if self._wants_grad():
            return self._forward_autograd(ray_dir, ray_orig, dists, sampling_type, ray_radius)
        B, S = dists.shape
        device = dists.device
        out = {"density": torch.empty(B, S, device=device, dtype=torch.float32),
               "color": torch.empty(B, S, 3, device=device, dtype=torch.float32)}
        h = self._field(device)
        prof = self._profile_events
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(torch.cuda.current_stream(device))
        with torch.cuda.device(device):
            L.check(L.lib().neddf_nerf_forward_rays(h, self._lowpass(), L.ptr(ray_dir), L.ptr(ray_orig), L.ptr(dists), B, S,
                                                    L.SAMPLING_IDS[sampling_type], float(ray_radius), L.ptr(out["density"]),
                                                    L.ptr(out["color"]), L.stream_ptr(device)), "nerf_forward_rays")
        if prof is not None:
            e1.record(torch.cuda.current_stream(device))
            prof.append((e0, e1, B * S))
        return out

    def set_iter(self, iter: int) -> None:
        """nerf.py:167-178."""
        if iter == -1:
            self.lowpass_alpha = float(self.embed_pos_rank)
        else:
            self.lowpass_alpha = self.lowpass_alpha_offset + 0.001 * iter
