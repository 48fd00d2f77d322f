"""The NeuS CUDA kernel's tile program, executed on the CPU.

neddf_b200/csrc/neus_kernel.cuh (index arithmetic, layer table, packing, barrier placement of csrc/neus_simt.cu) is
compiled by g++ into tests/emul/libneus_emul.so - a CTA is 256 OS threads with a pthread barrier for __syncthreads -
and run against the goldens recorded from the REAL reference (tests/golden/make_neus_golden.py).  The build
container has no GPU; this is how the kernel's logic is checked before it ever reaches one (the GPU tests in
tests/test_neus_gpu.py check the compiled kernel itself)."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import neddf_oracle as orc
from tests.helpers import PARITY_TOL, nerr
from tests.test_neus_oracle import NeusCase

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emul", "neus_emul.cpp")
LIB = os.path.join(HERE, "emul", "libneus_emul.so")
CUDA_INC = "/usr/local/cuda/include"


@pytest.fixture(scope="module")
def emul():
    if shutil.which("g++") is None or not os.path.isdir(CUDA_INC):
        pytest.skip("g++ / CUDA headers not available")
    deps = [SRC, os.path.join(HERE, "emul", "emul_common.h"), os.path.join(HERE, "..", "neddf_b200", "csrc", "neus_kernel.cuh"),
            os.path.join(HERE, "..", "neddf_b200", "csrc", "simt_mlp.cuh"), os.path.join(HERE, "..", "neddf_b200", "csrc", "common.cuh"),
            os.path.join(HERE, "..", "include", "neddf_b200.h")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-I" + CUDA_INC,
                        SRC, "-o", LIB], check=True)
    lib = C.CDLL(LIB)
    lib.neus_emul_forward.restype = C.c_int
    return lib


def _cfg_struct(nc: orc.NeusConfig):
    from neddf_b200 import _lib as L
    c = L.NeusConfig()
    c.embed_pos_rank, c.embed_dir_rank = nc.embed_pos_rank, nc.embed_dir_rank
    c.sdf_layer_count, c.sdf_layer_width = nc.sdf_layer_count, nc.sdf_layer_width
    c.col_layer_count, c.col_layer_width = nc.col_layer_count, nc.col_layer_width
    c.activation_type = L.ACT_IDS[nc.activation_type]
    c.n_skips = len(nc.skips)
    for i, s in enumerate(nc.skips):
        c.skips[i] = s
    return c


def run_emul(lib, c, tag: str, pos=None, dirs=None, rays=None, nblocks=2):
    """The emulated kernel on explicit samples (pos, dirs [n,3]) or rays ((ray_dir, ray_orig, dists), fused geometry);
    weights in torch's own [out,in] layout, straight from the reference's state_dict (``c`` = a NeusCase, or any
    object with ``nc``, ``rc`` and a dict ``z`` of ``w_fine.<state_dict key>`` arrays)."""
    pre = f"w_{tag}." if f"w_{tag}.layers_sdf.0.weight" in c.z else "w_fine."
    names = [n for n, _, _ in orc.neus_layer_shapes(c.nc)]
    ws = [np.ascontiguousarray(c.z[pre + n + ".weight"], dtype=np.float32) for n in names]
    bs = [np.ascontiguousarray(c.z[pre + n + ".bias"], dtype=np.float32) for n in names]
    var = np.ascontiguousarray(c.z[pre + "variance"], dtype=np.float32).reshape(1)
    fp = C.POINTER(C.c_float)

    def p(a):
        return None if a is None else a.ctypes.data_as(fp)

    wp = (fp * len(ws))(*[p(a) for a in ws])
    bp = (fp * len(bs))(*[p(a) for a in bs])
    if rays is not None:
        rd, ro, dists = (np.ascontiguousarray(t.numpy(), dtype=np.float32) for t in rays)
        n, n_edges = dists.shape
        total = n * n_edges
        shape = (n, n_edges)
        a_pos = a_dir = None
    else:
        a_pos = np.ascontiguousarray(pos.reshape(-1, 3).numpy(), dtype=np.float32)
        a_dir = np.ascontiguousarray(dirs.reshape(-1, 3).numpy(), dtype=np.float32)
        rd = ro = dists = None
        n, n_edges, total = a_pos.shape[0], 0, a_pos.shape[0]
        shape = tuple(pos.shape[:-1])
    out = {k: np.full((total,) + s, np.nan, np.float32) for k, s in (("sdf", ()), ("density", ()), ("color", (3,)), ("normal", (3,)))}
    radius = orc.CONE_RAY_RADIUS if c.rc.sampling_type == "cone" else 0.0
    cfg = _cfg_struct(c.nc)
    rc = lib.neus_emul_forward(C.byref(cfg), wp, bp, len(ws), p(var), p(a_pos), p(a_dir), p(rd), p(ro), p(dists), C.c_longlong(n),
                               C.c_int(n_edges), C.c_int({"point": 0, "cone": 1}[c.rc.sampling_type]), C.c_float(radius),
                               p(out["sdf"]), p(out["density"]), p(out["color"]), p(out["normal"]), C.c_int(nblocks))
    assert rc == 0
    return {k: v.reshape(shape + v.shape[1:]) for k, v in out.items()}


@pytest.mark.parametrize("name", ["relu", "tanhexp"])
def test_emulated_kernel_matches_reference_goldens(emul, name):
    c = NeusCase(name)
    d, o = orc.make_rays(c.t("uv"), c.cam)
    # coarse: 3 x 65 / 3 x 25 samples (full + ragged tiles over two CTAs), fine: 1 x 194 / 2 x 66 (a barrier of 256 OS
    # threads costs ~0.2 ms, a tile ~1400 of them: the sample counts are what keeps this test at half a minute)
    for tag, dists, n_rays in (("coarse", orc.coarse_dists(c.rc, c.t("u_coarse")), 3),
                               ("fine", c.t("dists_fine"), 1 if name == "relu" else 2)):
        sl = slice(0, n_rays)
        fused = run_emul(emul, c, tag, rays=(d[sl], o[sl], dists[sl]))
        pos, dd, _ = orc.make_samples(c.rc, d[sl], o[sl], dists[sl])
        explicit = run_emul(emul, c, tag, pos=pos, dirs=dd.contiguous(), nblocks=1) if tag == "coarse" else fused
        twin = orc.neus_forward_jac(c.params(tag), c.nc, pos, dd)
        for k in ("sdf", "density", "color"):
            ref = c.z[f"field_{tag}_{k}"][sl]
            scale = np.abs(c.z[f"field_{tag}_{k}"]).max()
            for what, got in (("fused geometry", fused[k]), ("explicit samples", explicit[k])):
                assert got.shape == ref.shape
                assert np.isfinite(got).all(), (tag, k, what)
                assert np.abs(got - ref).max() / scale < PARITY_TOL, (tag, k, what)
        assert nerr(fused["normal"], twin["gradients"].numpy()) < PARITY_TOL
        assert nerr(explicit["normal"], twin["gradients"].numpy()) < PARITY_TOL


def test_emulated_kernel_refuses_what_the_abi_refuses(emul):
    c = NeusCase("relu")
    bad = orc.NeusConfig(**{**c.nc.__dict__, "skips": [c.nc.sdf_layer_count - 1]})
    cfg = _cfg_struct(bad)
    assert emul.neus_emul_forward(C.byref(cfg), None, None, 0, None, None, None, None, None, None, C.c_longlong(0), 0, 0,
                                  C.c_float(0.0), None, None, None, None, 1) == -1


class _Synthetic:
    """Seeded weights for configurations the goldens do not cover (stored like a golden: torch's [out,in])."""

    def __init__(self, nc: orc.NeusConfig, seed: int):
        self.nc, self.rc = nc, orc.RenderConfig(sampling_type="point")
        self.P = orc.neus_init_params(nc, seed)
        self.z = {"w_fine." + k: (v.t().contiguous().numpy() if k.endswith(".weight") else v.numpy()) for k, v in self.P.items()}


@pytest.mark.parametrize("kw", [
    # largest embeddings the kernel accepts (60 + 30 rows), shallowest trunks, a skip right after the first layer
    dict(embed_pos_rank=10, embed_dir_rank=4, sdf_layer_count=2, col_layer_count=1, activation_type="tanhExp", skips=[0]),
    # one SDF layer (sdf = channel 0 of the first layer), no skip at all, smallest embeddings
    dict(embed_pos_rank=1, embed_dir_rank=1, sdf_layer_count=1, col_layer_count=2, activation_type="ReLU", skips=[]),
], ids=["max-embeddings-skip0", "one-sdf-layer"])
def test_emulated_kernel_layer_table_extremes(emul, kw):
    """Configurations at the edges of what neddf_neus_create accepts, against the oracle (70 samples: one full tile
    and a ragged one whose last SDF sub-tile is partly empty)."""
    c = _Synthetic(orc.NeusConfig(**kw), seed=5)
    g = torch.Generator().manual_seed(9)
    pos = torch.rand(1, 70, 3, generator=g) * 2 - 1
    dd = torch.nn.functional.normalize(torch.randn(1, 70, 3, generator=g), dim=-1)
    got = run_emul(emul, c, "fine", pos=pos, dirs=dd, nblocks=2)
    ref = orc.neus_forward(c.P, c.nc, pos, dd)
    for k, rk in (("sdf", "sdf"), ("density", "density"), ("color", "color"), ("normal", "gradients")):
        r = ref[rk].numpy()
        assert np.isfinite(got[k]).all(), k
        assert np.abs(got[k] - r).max() <= 2e-5 * max(np.abs(r).max(), 1.0), (k, float(np.abs(got[k] - r).max()))


def _san_build(tmp_path, name, flags):
    exe = str(tmp_path / name)
    r = subprocess.run(["g++", "-std=c++17", "-O1", "-g", "-ffp-contract=off", "-pthread", "-I" + CUDA_INC] + flags +
                       [os.path.join(HERE, "emul", "neus_emul_main.cpp"), "-o", exe], capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer runtime not available: " + r.stderr[-300:])
    return exe


def test_emulated_kernel_under_sanitizers(emul, tmp_path):
    """memcheck / racecheck without a GPU: the same tile program under AddressSanitizer + UBSan (out-of-bounds or
    misaligned accesses to the emulated shared memory, the packed weights, the exact-size outputs) and under
    ThreadSanitizer (conflicting accesses of a CTA's threads not ordered by the barrier that stands in for
    __syncthreads).  Full + ragged tiles, explicit and fused geometry, two configurations, two CTAs.  Two negative
    controls show the detectors see this code: a shared-memory base off by one float must trip the alignment check of
    the float4 accesses, and dropping every thread's first __syncthreads must be reported as a data race.
    (Best effort for races: ThreadSanitizer keeps four accesses per 8-byte cell, so it proves presence, not absence.)"""
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=0 exitcode=66", ASAN_OPTIONS="detect_leaks=0")
    clean = _san_build(tmp_path, "asan", ["-fsanitize=address,undefined", "-fno-sanitize-recover=all"])
    r = subprocess.run([clean], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-1500:]
    assert r.stdout.count("rc 0 checksum") == 2
    tsan = _san_build(tmp_path, "tsan", ["-fsanitize=thread"])
    r = subprocess.run([tsan], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "ThreadSanitizer" not in r.stderr, r.stderr[-1500:]
    bad_align = _san_build(tmp_path, "misalign", ["-fsanitize=address,undefined", "-fno-sanitize-recover=all", "-DNEUS_EMUL_MISALIGN"])
    r = subprocess.run([bad_align], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode != 0 and "misaligned address" in r.stderr, "negative control: the alignment check did not fire"
    no_barrier = _san_build(tmp_path, "nobar", ["-fsanitize=thread", "-DNEUS_EMUL_DROP_BARRIER=1"])
    r = subprocess.run([no_barrier], capture_output=True, text=True, env=env, timeout=600)
    assert "ThreadSanitizer: data race" in r.stderr, "negative control: the dropped barrier was not reported"
