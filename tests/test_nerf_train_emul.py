"""The NeRF variant's kernels (csrc/nerf.cu), forward and training backward, executed on the CPU.

Their tile program (neddf_b200/csrc/nerf_train_kernel.cuh) is compiled by g++ into tests/emul/libnerf_train_emul.so
(a CTA = 256 OS threads, pthread barrier for __syncthreads).  The forward is checked against the field goldens of the real reference and
the oracle.  The backward is run on the samples and the upstream gradients (d loss / d density,
d loss / d colour per sample, captured with tensor hooks) of fixtures recorded from the REAL reference's autograd
(tests/golden/make_nerf_train_golden.py).  The parameter gradients are then assembled exactly as the GPU path does -
gW = X^T G over all samples, bias = column sums - with numpy standing in for neddf_wgrad, and compared with the
reference's.  STATUS of the backward kernel itself: not yet passed on hardware; tests/test_zzz_nerf_train_gpu.py holds
its GPU tests."""
import ctypes as C
import json
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import neddf_oracle as orc
from tests.helpers import GOLDEN, PARITY_TOL, assert_parity, nerr
from tests.test_nerf_oracle import NerfCase

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "nerf_train_emul.cpp")
LIB = os.path.join(HERE, "emul", "libnerf_train_emul.so")
CUDA_INC = "/usr/local/cuda/include"
FP = C.POINTER(C.c_float)


class TrainCase:
    def __init__(self, name: str):
        z = np.load(os.path.join(GOLDEN, f"case_nerf_train_{name}.npz"), allow_pickle=False)
        self.z = {k: z[k] for k in z.files}
        meta = json.loads(str(self.z["cfg"]))
        self.net_cfg, self.render_cfg, self.iter = meta["net"], meta["render"], int(meta["iter"])
        self.nc = orc.NerfConfig.from_dict(self.net_cfg)
        self.rc = orc.RenderConfig.from_dict(self.render_cfg)
        self.alpha = self.nc.lowpass_alpha_at(self.iter)
        cal = [float(v) for v in self.z["cam_calib"]]
        self.cam = orc.CameraPose(torch.from_numpy(self.z["cam_R"]), torch.from_numpy(self.z["cam_T"]), *cal)
        self.separate = "w_coarse.layers.0.weight" in self.z

    def weights(self, tag):
        """torch layout ([out,in] weights, [out] biases) in the order of neddf_nerf_layer_shapes."""
        pre = f"w_{tag}." if (tag == "fine" or self.separate) else "w_fine."
        names = [n for n, _, _ in orc.nerf_layer_shapes(self.nc)]
        return names, [np.ascontiguousarray(self.z[pre + n + ".weight"], np.float32) for n in names], \
            [np.ascontiguousarray(self.z[pre + n + ".bias"], np.float32) for n in names]

    def t(self, k):
        return torch.from_numpy(self.z[k])


@pytest.fixture(scope="module")
def emul():
    if shutil.which("g++") is None or not os.path.isdir(CUDA_INC):
        pytest.skip("g++ / CUDA headers not available")
    deps = [SRC, os.path.join(HERE, "emul", "emul_common.h"), os.path.join(HERE, "..", "neddf_b200", "csrc", "nerf_train_kernel.cuh"),
            os.path.join(HERE, "..", "neddf_b200", "csrc", "simt_mlp.cuh"), os.path.join(HERE, "..", "neddf_b200", "csrc", "common.cuh"),
            os.path.join(HERE, "..", "include", "neddf_b200.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-I" + CUDA_INC, SRC, "-o", LIB],
                       check=True)
    lib = C.CDLL(LIB)
    lib.nerf_train_emul.restype = C.c_int
    lib.nerf_forward_emul.restype = C.c_int
    return lib


def cfg_struct(nc: orc.NerfConfig):
    from neddf_b200 import _lib as L
    c = L.NerfConfig()
    c.embed_pos_rank, c.embed_dir_rank, c.layer_count, c.layer_width = nc.embed_pos_rank, nc.embed_dir_rank, nc.layer_count, nc.layer_width
    c.activation_type, c.density_activation_type = L.ACT_IDS[nc.activation_type], L.ACT_IDS[nc.density_activation_type]
    c.n_skips = len(nc.skips)
    for i, s in enumerate(nc.skips):
        c.skips[i] = s
    return c


def run_backward(lib, nc, alpha, ws, bs, ray_dir, ray_orig, dists, sampling_type, g_density, g_color, nblocks=2):
    """The emulated kernel on rays (fused geometry); returns the buffers of neddf_nerf_train_backward_rays."""
    L = nc.layer_count
    rd, ro, di = (np.ascontiguousarray(t.numpy(), np.float32) for t in (ray_dir, ray_orig, dists))
    B, S = di.shape
    n = B * S
    gd = np.ascontiguousarray(g_density, np.float32).reshape(n)
    gc = np.ascontiguousarray(g_color, np.float32).reshape(n, 3)
    n_e, n_d = 6 * nc.embed_pos_rank, 6 * nc.embed_dir_rank
    buf = {"X": np.full((L, n, 256), np.nan, np.float32), "G": np.full((L, n, 256), np.nan, np.float32),
           "E": np.full((n, n_e), np.nan, np.float32), "D": np.full((n, n_d), np.nan, np.float32),
           "C1": np.full((n, 256), np.nan, np.float32), "GC1": np.full((n, 256), np.nan, np.float32), "GZD": np.full((n,), np.nan, np.float32)}
    lowpass = orc.lowpass_scale(nc.embed_pos_rank, alpha).numpy().astype(np.float32)

    def p(a):
        return a.ctypes.data_as(FP)

    wp = (FP * len(ws))(*[p(a) for a in ws])
    bp = (FP * len(bs))(*[p(a) for a in bs])
    cfg = cfg_struct(nc)
    radius = orc.CONE_RAY_RADIUS if sampling_type == "cone" else 0.0
    rc = lib.nerf_train_emul(C.byref(cfg), wp, bp, len(ws), p(lowpass), None, None, None, p(rd), p(ro), p(di), C.c_longlong(B), C.c_int(S),
                             C.c_int({"point": 0, "cone": 1}[sampling_type]), C.c_float(radius), p(gd), p(gc), p(buf["X"]), p(buf["G"]),
                             p(buf["E"]), p(buf["D"]), p(buf["C1"]), p(buf["GC1"]), p(buf["GZD"]), C.c_int(nblocks))
    assert rc == 0
    assert all(np.isfinite(v).all() for v in buf.values())
    return buf, gd, gc


def run_forward(lib, nc, alpha, ws, bs, sampling_type, pos=None, dirs=None, var=None, rays=None, nblocks=2):
    """The emulated forward kernel on explicit samples (pos, dirs, var [..., 3]) or rays ((ray_dir, ray_orig, dists),
    fused geometry): {'density': [...], 'color': [..., 3]}."""
    def p(a):
        return None if a is None else a.ctypes.data_as(FP)

    if rays is not None:
        rd, ro, di = (np.ascontiguousarray(t.numpy(), np.float32) for t in rays)
        n, n_edges = di.shape
        shape = di.shape
        pa = da = va = None
    else:
        pa, da, va = (np.ascontiguousarray(t.reshape(-1, 3).numpy(), np.float32) for t in (pos, dirs, var))
        rd = ro = di = None
        n, n_edges, shape = pa.shape[0], 0, tuple(pos.shape[:-1])
    total = int(np.prod(shape))
    density, color = np.full((total,), np.nan, np.float32), np.full((total, 3), np.nan, np.float32)
    lowpass = orc.lowpass_scale(nc.embed_pos_rank, alpha).numpy().astype(np.float32)
    wp = (FP * len(ws))(*[p(a) for a in ws])
    bp = (FP * len(bs))(*[p(a) for a in bs])
    cfg = cfg_struct(nc)
    radius = orc.CONE_RAY_RADIUS if sampling_type == "cone" else 0.0
    rc = lib.nerf_forward_emul(C.byref(cfg), wp, bp, len(ws), p(lowpass), p(pa), p(da), p(va), p(rd), p(ro), p(di), C.c_longlong(n),
                               C.c_int(n_edges), C.c_int({"point": 0, "cone": 1}[sampling_type]), C.c_float(radius), p(density),
                               p(color), C.c_int(nblocks))
    assert rc == 0
    return {"density": density.reshape(shape), "color": color.reshape(shape + (3,))}


def _case_weights(c: NerfCase, tag: str):
    """torch layout ([out,in] weights, [out] biases) of a NerfCase in the order of neddf_nerf_layer_shapes."""
    pre = f"w_{tag}." if f"w_{tag}.layers.0.weight" in c.z else "w_fine."
    names = [n for n, _, _ in orc.nerf_layer_shapes(c.nc)]
    return ([np.ascontiguousarray(c.z[pre + n + ".weight"], np.float32) for n in names],
            [np.ascontiguousarray(c.z[pre + n + ".bias"], np.float32) for n in names])


@pytest.mark.parametrize("name", ["relu", "tanhexp"])
def test_emulated_forward_matches_reference_goldens(emul, name):
    """The forward kernel's coarse and fine fields, explicit samples and fused geometry, against the real reference's
    (a slice of the rays: full + ragged tiles over two CTAs at a few seconds of emulation)."""
    c = NerfCase(name)
    d, o = orc.make_rays(c.t("uv"), c.cam)
    for tag, dists, n_rays in (("coarse", orc.coarse_dists(c.rc, c.t("u_coarse")), 3), ("fine", c.t("dists_fine"), 2)):
        sl = slice(0, n_rays)
        ws, bs = _case_weights(c, tag)
        pos, dd, var = orc.make_samples(c.rc, d[sl], o[sl], dists[sl])
        fused = run_forward(emul, c.nc, c.alpha, ws, bs, c.rc.sampling_type, rays=(d[sl], o[sl], dists[sl]))
        explicit = run_forward(emul, c.nc, c.alpha, ws, bs, c.rc.sampling_type, pos=pos, dirs=dd.contiguous(), var=var, nblocks=1)
        for k in ("density", "color"):
            ref = c.z[f"field_{tag}_{k}"][sl]
            for what, got in (("explicit samples", explicit[k]), ("fused geometry", fused[k])):
                assert got.shape == ref.shape, (tag, k, what)
                assert np.isfinite(got).all(), (tag, k, what)
                assert nerr(got, ref) < PARITY_TOL, (tag, k, what, nerr(got, ref))


def test_emulated_forward_ragged_tiles(emul):
    """Sample counts that are not multiples of the 64-sample tile, against the oracle field on the same samples."""
    c = NerfCase("relu")
    ws, bs = _case_weights(c, "fine")
    g = torch.Generator().manual_seed(5)
    for n in (1, 63, 65, 1000):
        pos = (torch.rand(1, n, 3, generator=g) * 2 - 1)
        dd = torch.nn.functional.normalize(torch.randn(1, n, 3, generator=g), dim=-1)
        var = torch.rand(1, n, 3, generator=g) * 1e-3
        out = run_forward(emul, c.nc, c.alpha, ws, bs, "cone", pos=pos, dirs=dd, var=var)
        with torch.no_grad():
            ref = orc.nerf_forward(c.params("fine"), c.nc, c.alpha, pos, dd, var)
        for k in ("density", "color"):
            a, r = out[k], ref[k].numpy()
            assert np.abs(a - r).max() <= PARITY_TOL * max(np.abs(r).max(), 1.0), (n, k)


def oracle_grads(c: TrainCase, dtype):
    """Parameter gradients of the fixture's two passes by torch autograd through oracle.nerf_forward, torch layout."""
    d, o = orc.make_rays(c.t("uv"), c.cam)
    grads = {}
    for tag, dists in (("coarse", orc.coarse_dists(c.rc, c.t("u_coarse"))), ("fine", c.t("dists_fine"))):
        names, ws, bs = c.weights(tag)
        P = {}
        for n, w, b in zip(names, ws, bs):
            P[n + ".weight"] = torch.from_numpy(w).t().contiguous().to(dtype).requires_grad_(True)
            P[n + ".bias"] = torch.from_numpy(b).to(dtype).requires_grad_(True)
        pos, dd, var = orc.make_samples(c.rc, d.to(dtype), o.to(dtype), dists.to(dtype))
        out = orc.nerf_forward(P, c.nc, c.alpha, pos, dd, var)
        ((out["density"] * c.t(f"up_{tag}_density").to(dtype)).sum() + (out["color"] * c.t(f"up_{tag}_color").to(dtype)).sum()).backward()
        net = "network_" + (tag if c.separate else "fine")
        for k, v in P.items():
            g = v.grad.numpy()
            grads[net + "." + k] = grads.get(net + "." + k, 0) + (g.T if k.endswith(".weight") else g)
    return grads


def assemble_grads(nc, names, buf, gd, gc):
    """What neddf_b200/nerf.py does with neddf_wgrad / neddf_colsum_value_rows, in float64 numpy: {state_dict key: gradient
    in torch's layout}."""
    L = nc.layer_count
    X, G = buf["X"].astype(np.float64), buf["G"].astype(np.float64)
    E, D = buf["E"].astype(np.float64), buf["D"].astype(np.float64)
    C1, GC1, GZD = buf["C1"].astype(np.float64), buf["GC1"].astype(np.float64), buf["GZD"].astype(np.float64)
    out = {}
    for l in range(L):
        inp = E if l == 0 else (np.concatenate([X[l - 1], E], 1) if (l - 1) in nc.skips else X[l - 1])
        out[f"layers.{l}.weight"] = (inp.T @ G[l]).T
        out[f"layers.{l}.bias"] = G[l].sum(0)
    out["outL_density.weight"] = (GZD[:, None].T @ X[L - 1])
    out["outL_density.bias"] = GZD.sum(keepdims=True)
    out["outL_color.0.weight"] = (np.concatenate([X[L - 1], D], 1).T @ GC1[:, :128]).T
    out["outL_color.0.bias"] = GC1[:, :128].sum(0)
    out["outL_color.2.weight"] = gc.astype(np.float64).T @ C1[:, :128]
    out["outL_color.2.bias"] = gc.astype(np.float64).sum(0)
    assert set(out) == {f"{n}.{p}" for n in names for p in ("weight", "bias")}
    return out


@pytest.mark.parametrize("name", ["relu", "tanhexp"])
def test_emulated_backward_matches_the_reference_gradients(emul, name):
    c = TrainCase(name)
    d, o = orc.make_rays(c.t("uv"), c.cam)
    passes = (("coarse", orc.coarse_dists(c.rc, c.t("u_coarse"))), ("fine", c.t("dists_fine")))
    grads = {}
    for tag, dists in passes:
        names, ws, bs = c.weights(tag)
        buf, gd, gc = run_backward(emul, c.nc, c.alpha, ws, bs, d, o, dists, c.rc.sampling_type, c.z[f"up_{tag}_density"], c.z[f"up_{tag}_color"])
        # the forward the kernel recomputed: activations of the last hidden layer reproduce the reference's field outputs
        n = gd.shape[0]
        wd, bd = ws[c.nc.layer_count], bs[c.nc.layer_count]
        zd = buf["X"][c.nc.layer_count - 1].astype(np.float64) @ wd[0].astype(np.float64) + bd[0]
        dens = orc.density_act(c.nc.density_activation_type, torch.from_numpy(zd)).numpy().reshape(dists.shape)
        assert nerr(dens, c.z[f"field_{tag}_density"]) < 5e-5, (tag, "density from the recomputed forward")
        col = buf["C1"][:, :128].astype(np.float64) @ ws[-1].astype(np.float64).T + bs[-1]
        assert nerr(col.reshape(dists.shape + (3,)), c.z[f"field_{tag}_color"]) < 5e-5, (tag, "colour from the recomputed forward")
        net = "network_" + (tag if c.separate else "fine")
        for k, v in assemble_grads(c.nc, names, buf, gd, gc).items():
            grads[net + "." + k] = grads.get(net + "." + k, 0) + v  # a shared network accumulates both passes
    exact = oracle_grads(c, torch.float64)  # the arbiter: autograd through the restatement in fp64
    checked = 0
    for k, g in grads.items():
        ref, ex = c.z["grad_" + k], exact[k]
        if g.ndim == 2 and g.shape[0] > 3:
            g, ex = g[::8], ex[::8]
        assert g.shape == ref.shape, (k, g.shape, ref.shape)
        # tanhExp: 1e-4 of the reference's fp32 gradients (measured 2e-6).  ReLU: the reference's own fp32 run sits
        # 1.5e-4 from the exact gradient on layers.1.weight (a hidden unit on the other side of its kink); the kernel
        # is held to the exact gradient and may be as far from the reference as the exact gradient is
        # is held to the exact gradient too - with the same allowance, because any fp32 evaluation of a ReLU network
        # (this one included: measured 8e-5 on layers.0.weight) has a few of its 3,108 x 2,048 hidden units on the other
        # side of a kink than the fp64 run (tests/test_arbiter.py, tests/test_neus_oracle.py show the mechanism)
        kinked = c.nc.activation_type != "tanhExp"
        if kinked:
            # ReLU, 1,036 samples: every fp32 evaluation (the reference's, the oracle's, this kernel's) has a few hidden
            # units on the other side of a kink than the fp64 run and then differs from it by up to 5e-4 on 1-5 % of a
            # tensor's elements (measured: reference vs fp64 91 of 1,920 elements of layers.0.weight) - but two fp32
            # evaluations mostly agree on the side.  So: the reference's fp32 gradients with the kinked-configuration
            # rule of helpers.assert_parity (all but max(2, 1 %) of the elements within 1e-4, outliers below 5e-2), and
            # the fp64 run only as a sanity bound
            assert_parity(g, ref, 1e-4, kinked=True, what=k + " vs the reference")
            assert nerr(g, ex) < 2e-2, (k, "vs fp64 autograd", nerr(g, ex))
        else:
            assert nerr(g, ex) < 5e-5, (k, "vs fp64 autograd", nerr(g, ex))
            assert nerr(g, ref) < 1e-4, (k, "vs the reference", nerr(g, ref), nerr(ex, ref))
        checked += 1
    assert checked == len([k for k in c.z if k.startswith("grad_")])


def test_emulated_backward_leaky_density_and_ragged_tiles(emul):
    """LeakyReLU hidden + density (the reference's own backward raises once coarse weights go negative, so its autograd
    is taken through the oracle restatement here), 3 skips, 70 and 2 samples (ragged tiles), against torch autograd."""
    nc = orc.NerfConfig(embed_pos_rank=4, embed_dir_rank=2, layer_count=5, activation_type="LeakyReLU",
                        density_activation_type="LeakyReLU", skips=[0, 1, 3], lowpass_alpha_offset=2.0)
    alpha = nc.lowpass_alpha_at(700)
    P = orc.nerf_init_params(nc, 11)
    names = [n for n, _, _ in orc.nerf_layer_shapes(nc)]
    ws = [np.ascontiguousarray(P[n + ".weight"].t().numpy()) for n in names]
    bs = [np.ascontiguousarray(P[n + ".bias"].numpy()) for n in names]
    g = torch.Generator().manual_seed(3)
    for B, S in ((10, 7), (1, 2)):
        d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1)
        o = torch.randn(B, 3, generator=g) * 0.2
        dists = 2.0 + torch.rand(B, S, generator=g).sort(dim=1).values * 3
        gd, gc = torch.randn(B, S, generator=g), torch.randn(B, S, 3, generator=g)
        rc = orc.RenderConfig(sampling_type="cone")
        pos, dd, var = orc.make_samples(rc, d, o, dists)
        Pg = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        out = orc.nerf_forward(Pg, nc, alpha, pos, dd, var)
        ((out["density"] * gd).sum() + (out["color"] * gc).sum()).backward()
        buf, gdn, gcn = run_backward(emul, nc, alpha, ws, bs, d, o, dists, "cone", gd.numpy(), gc.numpy())
        got = assemble_grads(nc, names, buf, gdn, gcn)
        for k, v in got.items():
            ref = Pg[k].grad.numpy()
            ref = ref.T if k.endswith(".weight") else ref  # the oracle keeps [in,out]
            assert nerr(v, ref) < 2e-5, (B, S, k, nerr(v, ref))


class _FakeLib:
    """Stands in for libneddf_b200.so under neddf_b200.NeRF's autograd function on a box without a GPU: the training
    kernel is the host emulation, neddf_wgrad / neddf_colsum_value_rows are numpy on the very pointers, strides and tile
    arguments the glue passes (their CUDA versions are held to fp64 by tests/test_gpu_parity.py::test_wgrad_gemm)."""

    def __init__(self, emul_lib):
        self.emul, self.handles, self.calls = emul_lib, {}, []

    @staticmethod
    def _arr(p, n):
        addr = p.value if hasattr(p, "value") else p
        return np.ctypeslib.as_array(C.cast(addr, FP), shape=(int(n),))

    def neddf_last_error(self):
        return b"fake"

    def neddf_nerf_train_create(self, cfg_ref, h_ref):
        cfg = type(cfg_ref._obj)()
        C.memmove(C.byref(cfg), C.byref(cfg_ref._obj), C.sizeof(cfg))
        h_ref._obj.value = 4096 + len(self.handles)
        self.handles[h_ref._obj.value] = {"cfg": cfg}
        return 0

    def neddf_nerf_train_destroy(self, h):
        self.handles.pop(h.value, None)

    def neddf_nerf_train_set_weights(self, h, ws, bs, n, stream):
        self.handles[h.value].update(w=[C.cast(ws[i], FP) for i in range(n)], b=[C.cast(bs[i], FP) for i in range(n)], n=n)
        return 0

    def _backward(self, h, lowpass, pos, dirs, var, rd, ro, dists, n, n_edges, stype, radius, bufs):
        st = self.handles[h.value]
        wp, bp = (FP * st["n"])(*st["w"]), (FP * st["n"])(*st["b"])
        cast = [None if b is None else C.cast(b.value, FP) for b in (pos, dirs, var, rd, ro, dists)] + [C.cast(b.value, FP) for b in bufs]
        self.calls.append("train_backward")
        return self.emul.nerf_train_emul(C.byref(st["cfg"]), wp, bp, st["n"], C.cast(lowpass, FP), *cast[:6], C.c_longlong(n), C.c_int(n_edges),
                                         C.c_int(stype), C.c_float(radius), *cast[6:], C.c_int(2))

    def neddf_nerf_train_backward_rays(self, h, lowpass, rd, ro, dists, n_rays, n_edges, stype, radius, *rest):
        return self._backward(h, lowpass, None, None, None, rd, ro, dists, n_rays, n_edges, stype, radius, rest[:9])

    def neddf_nerf_train_backward(self, h, lowpass, pos, dirs, var, n, *rest):
        return self._backward(h, lowpass, pos, dirs, var, None, None, None, n, 0, 0, 0.0, rest[:9])

    def neddf_wgrad_workspace_bytes(self):
        return 4096

    def neddf_wgrad(self, a, lda, a_col0, ka, b, ldb, rows, out, ld_out, n_cols, ws, stream):
        assert 0 < ka <= 128 and n_cols == 256 and ld_out == 256 and ldb == 256  # the parameters test_wgrad_gemm holds on hardware
        A = self._arr(a, rows * lda).reshape(rows, lda).astype(np.float64)
        B = self._arr(b, rows * ldb).reshape(rows, ldb).astype(np.float64)
        O = self._arr(out, (ka - 1) * ld_out + n_cols)
        res = A[:, a_col0:a_col0 + ka].T @ B[:, :n_cols]
        for m in range(ka):
            O[m * ld_out:m * ld_out + n_cols] = res[m]
        self.calls.append("wgrad")
        return 0

    def neddf_colsum_value_rows(self, g, n_samples, stride, out, ws, stream):
        Gm = self._arr(g, (n_samples - 1) * stride + 256)
        self._arr(out, 256)[:] = np.stack([Gm[s * stride:s * stride + 256] for s in range(n_samples)]).astype(np.float64).sum(0)
        self.calls.append("colsum")
        return 0


@pytest.mark.parametrize("name", ["tanhexp"])  # separate coarse / fine networks, two skips; "relu" also passes (shared network)
def test_autograd_glue_with_emulated_kernels(emul, name, monkeypatch):
    """neddf_b200.NeRF with training_kernels=True, end to end through torch autograd on CPU tensors: the module's own
    _NerfTrainFn (buffer allocation, pointer arithmetic of the 128-column wgrad tiles, transposes, gradient order) over a
    fake library, against the real reference's parameter gradients.  Default (opt-out) behaviour: the call is refused."""
    import contextlib

    import neddf_b200
    from neddf_b200 import _lib as L
    c = TrainCase(name)
    fake = _FakeLib(emul)
    monkeypatch.setattr(L, "lib", lambda: fake)
    monkeypatch.setattr(L, "stream_ptr", lambda device=None: None)
    monkeypatch.setattr(L, "require_cuda_f32", lambda t, name: t.to(torch.float32).contiguous())
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    d, o = orc.make_rays(c.t("uv"), c.cam)
    radius = orc.CONE_RAY_RADIUS if c.rc.sampling_type == "cone" else 0.0
    nets = {}
    for tag in (("coarse", "fine") if c.separate else ("fine",)):
        net = neddf_b200.NeRF(**{k: v for k, v in c.net_cfg.items() if k != "_target_"})
        pre = f"w_{tag}."
        net.load_state_dict({k[len(pre):]: torch.from_numpy(v) for k, v in c.z.items() if k.startswith(pre)})
        net.set_iter(c.iter)
        monkeypatch.setattr(net, "_release", lambda: None)
        # the inference kernel is not under test here: the forward values come from the oracle
        params = c.weights(tag)

        def launch(a, b, cc, stype, rr, _p=params):
            names, ws, bs = _p
            P = {}
            for n, w, bb in zip(names, ws, bs):
                P[n + ".weight"], P[n + ".bias"] = torch.from_numpy(w).t().contiguous(), torch.from_numpy(bb)
            pos, dd, var = orc.make_samples(c.rc, a, b, cc)
            return orc.nerf_forward(P, c.nc, c.alpha, pos, dd, var)

        monkeypatch.setattr(net, "_launch_forward", launch)
        nets[tag] = net
    with pytest.raises(NotImplementedError, match="opt-in"):
        nets["fine"].forward_rays(d, o, c.t("dists_fine"), c.rc.sampling_type, radius)  # the default
    for net in nets.values():
        net.training_kernels = True
    loss = 0
    for tag, dists in (("coarse", orc.coarse_dists(c.rc, c.t("u_coarse"))), ("fine", c.t("dists_fine"))):
        net = nets[tag if c.separate else "fine"]
        out = net.forward_rays(d, o, dists, c.rc.sampling_type, radius)
        assert out["density"].requires_grad and out["color"].requires_grad
        loss = loss + (out["density"] * c.t(f"up_{tag}_density")).sum() + (out["color"] * c.t(f"up_{tag}_color")).sum()
    loss.backward()
    assert fake.calls.count("train_backward") == 2
    kinked = c.nc.activation_type != "tanhExp"
    checked = 0
    for tag, net in nets.items():
        for k, p in net.named_parameters():
            g, ref = p.grad.numpy(), c.z[f"grad_network_{tag}.{k}"]
            if g.ndim == 2 and g.shape[0] > 3:
                g = g[::8]
            assert g.shape == ref.shape
            if kinked:
                assert_parity(g, ref, 1e-4, kinked=True, what=f"{tag} {k}")
            else:
                assert nerr(g, ref) < 1e-4, (tag, k, nerr(g, ref))
            checked += 1
    assert checked == len([k for k in c.z if k.startswith("grad_")])
    for net in nets.values():  # fake handles must never reach the real library's destroy (module __del__ after the patches are gone)
        net._train_handle, net._handle = None, None


def _san_build(tmp_path, name, flags):
    exe = str(tmp_path / name)
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-pthread", "-I" + CUDA_INC] + flags +
                       [os.path.join(HERE, "emul", "nerf_train_emul_main.cpp"), "-o", exe], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + r.stderr[-300:])
    return exe


def test_emulated_backward_under_sanitizers(emul, tmp_path):
    """AddressSanitizer + UBSan (memcheck: exact-size buffers, float4 alignment) and ThreadSanitizer (racecheck, best
    effort) on the emulated forward and training-backward kernels (the negative controls that show the detectors see this kind of code
    live in tests/test_neus_emul.py: same harness, same GEMM loop)."""
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    r = subprocess.run([_san_build(tmp_path, "asan", ["-fsanitize=address,undefined", "-fno-sanitize-recover=all"])], capture_output=True,
                       text=True, env=env, timeout=600)
    assert r.returncode == 0 and "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-1500:]
    assert r.stdout.count("rc 0 checksum") == 4  # two configurations, forward and backward
    r = subprocess.run([_san_build(tmp_path, "tsan", ["-fsanitize=thread"])], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "ThreadSanitizer" not in r.stderr, r.stderr[-1500:]
