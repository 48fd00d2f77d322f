"""CPU: host-side mirror of the reference interface (no kernels run)."""
import os

import numpy as np
import pytest
import torch

import neddf_b200
from oracle import neddf_oracle as orc
from tests.helpers import GOLDEN, Case


def test_state_dict_surface_matches_reference_checkpoint():
    c = Case("bunny")
    r = neddf_b200.NeRFRender(network_config=c.net_cfg, **{k: v for k, v in c.render_cfg.items() if k != "_target_"})
    sd = r.state_dict()
    assert len(sd) == 52  # SURVEY 3.3: network_fine.* and network_coarse.* alias the same tensors
    assert r.network_coarse is r.network_fine
    res = r.load_state_dict(c.state_dict())
    assert not res.missing_keys and not res.unexpected_keys
    assert len(r.get_parameters_list()) == 26
    r2 = neddf_b200.NeRFRender(network_config=c.net_cfg, use_coarse_network=True)
    assert r2.network_coarse is not r2.network_fine and len(r2.get_parameters_list()) == 52


def test_set_iter_schedule_matches_reference():
    net = neddf_b200.NeDDF(lowpass_alpha_offset=4.0)
    cfg = orc.FieldConfig(lowpass_alpha_offset=4.0)
    for it in (-1, 0, 50, 2500, 20000):
        net.set_iter(it)
        st = orc.FieldState.at_iter(cfg, it)
        assert (net.aux_grad_scale, net.distance_range_max, net.lowpass_alpha) == \
            (st.aux_grad_scale, st.distance_range_max, st.lowpass_alpha)
    r = neddf_b200.NeRFRender(network_config={"_target_": "neddf.network.NeDDF"})
    r.set_iter(7)
    r.next_iter()
    assert r.iteration == 8 and r.network_fine.aux_grad_scale == pytest.approx(0.01)


def test_cpu_tensors_are_rejected_loudly():
    net = neddf_b200.NeDDF()
    s = neddf_b200.Sampling(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        net(s)


def test_unknown_network_target_is_rejected():
    with pytest.raises(NotImplementedError):
        neddf_b200.NeRFRender(network_config={"_target_": "neddf.network.SomethingElse"})
    with pytest.raises(KeyError):
        neddf_b200.NeDDF(activation_type="gelu")
    with pytest.raises(KeyError):  # neus.py:70-75 knows ReLU and tanhExp only
        neddf_b200.NeuS(activation_type="LeakyReLU")


def test_neus_module_surface_matches_the_reference():
    """Same constructor, parameter names / shapes and initial values as neddf.network.NeuS for the same torch seed;
    NeRFRender resolves the reference's _target_ to it; the C ABI reports the same layer shapes and refusals."""
    import ctypes as C
    import json

    from neddf_b200 import _lib as L
    from oracle import neddf_oracle as orc
    from tests.golden.make_host_golden import NEUS_KW as kw
    from tests.golden.make_host_golden import tensor_digest, tensor_sample
    torch.manual_seed(7)
    net = neddf_b200.NeuS(**kw)
    sd = net.state_dict()
    shapes = orc.neus_layer_shapes(orc.NeusConfig(**kw))
    assert set(sd) == {f"{n}.{p}" for n, _, _ in shapes for p in ("weight", "bias")} | {"variance"}
    for n, cin, cout in shapes:  # torch nn.Linear keeps [out, in]
        assert tuple(sd[n + ".weight"].shape) == (cout, cin) and tuple(sd[n + ".bias"].shape) == (cout,)
    assert abs(float(sd["variance"]) - 0.45) < 1e-7
    # the reference's NeuS(**kw) after the same seed (tests/golden/make_host_golden.py): key order, values bit for bit
    z = np.load(os.path.join(GOLDEN, "case_host.npz"))
    assert json.loads(str(z["neus_keys"])) == list(sd)
    for i, (k, v) in enumerate(sd.items()):
        assert np.array_equal(tensor_sample(v), z[f"neus_sample_{i}"]), k
    assert [tensor_digest(v) for v in sd.values()] == json.loads(str(z["neus_sha256"]))
    r = neddf_b200.NeRFRender(network_config={"_target_": "neddf.network.NeuS", **kw}, use_coarse_network=False)
    assert isinstance(r.network_fine, neddf_b200.NeuS) and r.network_coarse is r.network_fine
    assert len(r.get_parameters_list()) == 2 * len(shapes) + 1
    lib = L.lib()
    cfg = net._config_struct()
    buf = (C.c_int32 * 64)()
    n = lib.neddf_neus_layer_shapes(C.byref(cfg), buf, 32)
    assert [(buf[2 * i], buf[2 * i + 1]) for i in range(n)] == [(a, b) for _, a, b in shapes]
    bad = neddf_b200.NeuS(sdf_layer_count=4, skips=[3])._config_struct()
    assert lib.neddf_neus_layer_shapes(C.byref(bad), None, 0) == -3 and b"skip" in lib.neddf_last_error()
    s = neddf_b200.Sampling(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        net(s)  # CPU tensors are refused, nothing is computed on the host
    with pytest.raises(NotImplementedError, match="forward-only"):
        net(s)  # autograd enabled on trainable parameters


def test_camera_standin_matches_reference_pose():
    c = Case("bunny")
    cam = neddf_b200.Camera.from_matrix(neddf_b200.PinholeCalib(c.z["cam_calib"]), c.z["cam_R"], c.z["cam_T"])
    assert np.allclose(cam.R.numpy(), c.z["cam_R"]) and np.allclose(cam.T.numpy(), c.z["cam_T"])
    # rotvec path: Rodrigues of a known rotation
    from scipy.spatial.transform import Rotation
    rv = np.array([0.3, -1.1, 0.7])
    cam2 = neddf_b200.Camera(neddf_b200.PinholeCalib([100, 100, 50, 50]), np.concatenate([rv, [1, 2, 3]]))
    assert np.allclose(cam2.R.numpy(), Rotation.from_rotvec(rv).as_matrix(), atol=1e-6)
    assert np.allclose(cam2.T.numpy(), [1, 2, 3])


def test_install_rebinds_reference_targets(repo_root):
    """neddf_b200.install makes the saved `_target_` strings resolve to the B200 classes and the
    pretrained checkpoint loads unchanged (subprocess: do not pollute this interpreter's modules).
    The reference's packages are empty stand-in modules here: install only rebinds their attributes.
    The checkpoint is the bunny_smoke run's (its key order from case_host.npz, its tensors in bunny_smoke_weights.npz)."""
    import os
    import subprocess
    import sys
    code = (
        "import sys, types, json, yaml, numpy as np, torch, hydra\n"
        "from tests.helpers import GOLDEN\n"
        "for name in ('neddf', 'neddf.render', 'neddf.network'):\n"
        "    sys.modules[name] = types.ModuleType(name)\n"
        "import neddf_b200.install as I; I.install()\n"
        "cfg = yaml.safe_load(open(GOLDEN + '/bunny_smoke_config.yaml'))\n"
        "r = hydra.utils.instantiate(dict(cfg['render']), network_config=cfg['network'])\n"
        "assert type(r).__module__ == 'neddf_b200.render' and type(r.network_fine).__module__ == 'neddf_b200.network'\n"
        "w = np.load(GOLDEN + '/bunny_smoke_weights.npz')\n"
        "keys = json.loads(str(np.load(GOLDEN + '/case_host.npz')['ckpt_keys']))\n"
        "res = r.load_state_dict({k: torch.from_numpy(w[k.split('.', 1)[1]]) for k in keys})\n"
        "assert not res.missing_keys and not res.unexpected_keys\n"
        "print('ok')\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(repo_root, "tests/golden/_refstub"), repo_root]))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def _loop_targets(item, us_int, vs_int, loss_types):
    """Restatement of the per-pixel loop of base_trainer.py:222-243 (test oracle)."""
    out = {}
    if "ColorLoss" in loss_types:
        rgb = item["rgb_images"]
        out["color"] = torch.from_numpy(((1.0 / 256) * np.stack([rgb[v, u, :] for u, v in zip(us_int, vs_int)])).astype(np.float32))
    if "MaskBCELoss" in loss_types or "MaskMSELoss" in loss_types:
        mask = item["mask_images"]
        out["mask"] = torch.from_numpy(((1.0 / 256) * np.stack([mask[v, u] for u, v in zip(us_int, vs_int)])).astype(np.float32))
    if "FieldsConstraintLoss" in loss_types:
        out["fields_penalty"] = torch.zeros(us_int.shape, dtype=torch.float32)
    return out


def test_vectorised_ground_truth_gather_is_bit_exact():
    from neddf_b200.trainer_glue import gather_targets
    rng = np.random.default_rng(0)
    item = {"rgb_images": rng.integers(0, 256, (37, 53, 3), dtype=np.uint8),
            "mask_images": rng.integers(0, 256, (37, 53), dtype=np.uint8)}
    g = torch.Generator().manual_seed(1)
    us = (torch.rand(300, generator=g) * 52).to(torch.int16)  # nerf_trainer.py:92-97
    vs = (torch.rand(300, generator=g) * 36).to(torch.int16)
    kinds = ["ColorLoss", "MaskBCELoss", "FieldsConstraintLoss"]
    got, ref = gather_targets(item, us, vs, kinds, "cpu"), _loop_targets(item, us, vs, kinds)
    assert set(got) == set(ref) == {"color", "mask", "fields_penalty"}
    for k in ref:
        assert got[k].dtype == torch.float32 and got[k].shape == ref[k].shape and torch.equal(got[k], ref[k]), k
    assert set(gather_targets(item, us, vs, ["MaskMSELoss"], "cpu")) == {"mask"}
    assert gather_targets(item, us[:0], vs[:0], ["ColorLoss"], "cpu")["color"].shape == (0, 3)


def test_trainer_patch_matches_reference_method(repo_root):
    """install(patch_trainer=True) swaps BaseTrainer.construct_ground_truth for the vectorised gather;
    it gives the tensors the reference's own method gave on the same seeded inputs (case_host.npz, recorded by
    tests/golden/make_host_golden.py).  Subprocess; the reference's packages are empty stand-in modules."""
    import os
    import subprocess
    import sys
    code = (
        "import sys, types, numpy as np, torch\n"
        "from tests.golden.make_host_golden import GATHER_KINDS, gather_inputs\n"
        "from tests.helpers import GOLDEN\n"
        "for name in ('neddf', 'neddf.render', 'neddf.network', 'neddf.loss', 'neddf.trainer', 'neddf.trainer.base_trainer'):\n"
        "    sys.modules[name] = types.ModuleType(name)\n"
        "class BaseTrainer:\n"
        "    def construct_ground_truth(self, camera_id, us_int, vs_int, loss_types):\n"
        "        raise NotImplementedError\n"
        "sys.modules['neddf.trainer.base_trainer'].BaseTrainer = BaseTrainer\n"
        "ref_fn = BaseTrainer.construct_ground_truth\n"
        "import neddf_b200.install as I; I.install(patch_trainer=True)\n"
        "assert BaseTrainer.construct_ground_truth is not ref_fn\n"
        "rgb, mask, us, vs = gather_inputs()\n"
        "t = types.SimpleNamespace(device=torch.device('cpu'), dataset=[dict(rgb_images=rgb, mask_images=mask)])\n"
        "z = np.load(GOLDEN + '/case_host.npz')\n"
        "a = {k[len('gather_'):]: torch.from_numpy(z[k]) for k in z.files if k.startswith('gather_')}\n"
        "b = BaseTrainer.construct_ground_truth(t, 0, us, vs, GATHER_KINDS)\n"
        "assert set(a) == set(b) and all(torch.equal(a[k], b[k]) and a[k].dtype == b[k].dtype for k in a)\n"
        "print('ok')\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(repo_root, "tests/golden/_refstub"), repo_root]))
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_module_copies_and_pickles_without_the_kernel_handle():
    """The reference module is deep-copyable / picklable (EMA copies, whole-module checkpoints); the
    process-local kernel handle must not travel with it."""
    import copy
    import ctypes
    import pickle
    net = neddf_b200.NeDDF(col_layer_count=4)
    net._handle = ctypes.c_void_p(1234)  # as after a first forward
    net._handle_device = torch.device("cpu")
    net._packed_key = ("stale",)
    twin = copy.deepcopy(net)
    assert twin._handle is None and twin._packed_key is None
    assert all(torch.equal(a, b) and a.data_ptr() != b.data_ptr()
               for a, b in zip(net.state_dict().values(), twin.state_dict().values()))
    blob = pickle.dumps(net)
    back = pickle.loads(blob)
    assert back._handle is None and back.penalty_weight == net.penalty_weight
    net._handle = None  # nothing real to destroy


def test_state_struct_reads_penalty_weights_on_every_call():
    """neddf.py:296-299 reads the dict on every forward: mutating it must reach the next launch."""
    from neddf_b200 import _lib as L
    net = neddf_b200.NeDDF(penalty_weight={"constraints_dDdt": 0.5})
    st = net._state_struct()
    w = dict(zip(L.PENALTY_KEYS, list(st.penalty_weight)))
    assert w["constraints_dDdt"] == 0.5 and w["range_color"] == 1.0  # absent key -> unweighted
    net.penalty_weight["range_color"] = 0.25
    assert dict(zip(L.PENALTY_KEYS, list(net._state_struct().penalty_weight)))["range_color"] == 0.25
    net._packed_key = ("x",)
    net.invalidate()
    assert net._packed_key is None


def test_eval_io_writer_matches_the_reference_tail(tmp_path):
    """eval_io.FrameWriter / render_all keep render_test's arithmetic, file names and frame order
    (base_trainer.py:146-187); here with CPU tensors and a stub renderer."""
    import cv2
    from neddf_b200 import eval_io
    g = torch.Generator().manual_seed(0)
    h, w = 20, 24

    class StubRender:
        def __init__(self):
            self.iter = None

        def set_iter(self, it):
            self.iter = it

        def render_image(self, width, height, camera, target_types, downsampling, chunk):
            assert (width, height, list(target_types), downsampling, chunk) == (w, h, ["color", "depth"], 1, 7)
            return {"color": torch.rand(h, w, 3, generator=g) * 1.2 - 0.1, "depth": torch.rand(h, w, 1, generator=g) * 5 + 1.5}

    class Cam:
        def __init__(self):
            self.updated = 0

        def update_transform(self):
            self.updated += 1

    class StubTrainer:
        pass

    tr = StubTrainer()
    tr.neural_render, tr.chunk = StubRender(), 7
    tr.dataset = [{"rgb_images": (torch.rand(h, w, 3, generator=g) * 255).numpy()} for _ in range(3)]
    tr.cameras = [Cam() for _ in range(3)]
    eval_io.render_all(tr, tmp_path)
    assert tr.neural_render.iter == -1 and all(c.updated == 1 for c in tr.cameras)
    # replay the same random stream through the reference's expressions
    g = torch.Generator().manual_seed(0)
    gts = [(torch.rand(h, w, 3, generator=g) * 255).numpy().astype(np.uint8) for _ in range(3)]  # the dataset came first
    frames = []
    for _ in range(3):
        frames.append((torch.rand(h, w, 3, generator=g) * 1.2 - 0.1, torch.rand(h, w, 1, generator=g) * 5 + 1.5))
    for i, (col, dep) in enumerate(frames):
        rgb_ref = torch.clamp(col * 255, 0, 255).numpy().astype(np.uint8)
        dep_ref = torch.clamp((dep - 2.0) / 4.0 * 50000 / 256, 0, 255).numpy().astype(np.uint8)
        assert np.array_equal(cv2.imread(str(tmp_path / f"{i:03}_rgb.png")), rgb_ref)
        assert np.array_equal(cv2.imread(str(tmp_path / f"{i:03}_depth.png"), cv2.IMREAD_UNCHANGED), dep_ref[:, :, 0])
        assert np.array_equal(cv2.imread(str(tmp_path / f"{i:03}_rgb_gt.png")), gts[i])
        mse = np.mean((rgb_ref.astype(np.float64) - gts[i].astype(np.float64)) ** 2)
        assert abs(eval_io.psnr_uint8(rgb_ref, gts[i]) - 10 * np.log10(255.0 ** 2 / mse)) < 1e-12


def test_engine_range_fallback_host_logic(monkeypatch):
    """Engine "auto" leaving fp16 range (status bit 4 of neddf_field_status): the network marks itself and raises
    EngineRangeError once, the renderer reads BOTH networks' flags, clears its own NaN flags of the invalid run and
    re-raises; explicit engines raise plain FloatingPointError; set_engine starts afresh.  (The device side and the
    re-run are covered by tests/test_gpu_parity.py::test_auto_engine_leaves_fp16_range_gracefully.)"""
    import ctypes as C

    from neddf_b200 import _lib as L
    from neddf_b200.network import EngineRangeError

    class FakeLib:
        def __init__(self):
            self.status = {}

        def neddf_field_status(self, handle, out, stream):
            out._obj.value = self.status.pop(handle.value, 0)  # read-and-clear, like the kernel-side word
            return 0

    fake = FakeLib()
    monkeypatch.setattr(L, "lib", lambda: fake)
    monkeypatch.setattr(L, "stream_ptr", lambda device=None: None)
    monkeypatch.setattr(torch.cuda, "device", lambda d: __import__("contextlib").nullcontext())
    r = neddf_b200.NeRFRender(network_config={"_target_": "neddf.network.NeDDF"}, use_coarse_network=True)
    for i, net in enumerate((r.network_coarse, r.network_fine)):
        net._handle, net._handle_device = C.c_void_p(100 + i), torch.device("cpu")
        monkeypatch.setattr(net, "_release", lambda: None)
    r._status_buf = torch.tensor([1, 0], dtype=torch.int32)  # a NaN flag left by the invalid run
    fake.status = {100: 4, 101: 4}
    with pytest.raises(EngineRangeError):
        r.check_status()
    assert fake.status == {}  # both words were read although the first network already raised
    assert r.network_coarse._range_fallback and r.network_fine._range_fallback
    assert int(r._status_buf[0]) == 0  # flags of the invalid run are gone: the re-run starts clean
    assert r.network_fine._engine_id() == L.ENGINE_IDS["fp32"]
    r.check_status()  # nothing pending any more
    fake.status = {101: 4}  # still out of range although already on fp32?  that is an error, not another detour
    with pytest.raises(FloatingPointError) as ei:
        r.check_status()
    assert not isinstance(ei.value, EngineRangeError)
    r.set_engine("tc")
    assert not r.network_fine._range_fallback and r.network_fine._engine_id() == L.ENGINE_IDS["tc"]
    fake.status = {100: 4}
    with pytest.raises(FloatingPointError) as ei:
        r.check_status()
    assert not isinstance(ei.value, EngineRangeError)
    r.set_engine("auto")
    assert r.network_fine._engine_id() == L.ENGINE_IDS["auto"]
    for net in (r.network_coarse, r.network_fine):
        net._handle = None
