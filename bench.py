#!/usr/bin/env python
"""Benchmark of the NeDDF render hot path (BASELINE.json metric: ray-samples/s, 800x800x192).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on host cores

A "step" is one 800x800 frame (640,000 rays, 64 coarse + 128 fine samples/ray = 192 nominal
ray-samples = 259 MLP evaluations per ray), synthetic camera on the radius-4.03 sphere, seeded
random-init NeDDF weights of the reference architecture (8x256 distance trunk with skip, 4x256
colour trunk, tanhExp, cone sampling).  With N GPUs a step is N frames, every frame ray-sharded
over the N ranks with ONE all-gather of image tiles per frame (weak scaling: 640k rays per rank
per step).

Prints ONE JSON line (rank 0).  `value` = nominal ray-samples/s with the frame's uniforms
resident in HBM; `e2e` = the same through NeRFRender.render_image with HOST buffers (uniforms
copied from pinned memory, image copied back) inside the timed region.

`--dump-outputs DIR` writes what the last timed step returned (render: colour and depth of every frame of the step;
train: the loss, the render outputs and the updated weights) as DIR/<name>.npy.  Weights, cameras, uniforms and
batches are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W = H = 800
S_COARSE, S_FINE = 64, 128
NOMINAL_PER_RAY = S_COARSE + S_FINE            # 192
EVALS_PER_RAY = (S_COARSE + 1) + (S_COARSE + 1 + S_FINE + 1)  # 65 + 194 = 259
# algorithmic FLOP per MLP evaluation (SURVEY 8(d)): 4 rows through the distance trunk + heads,
# 1 row through the colour trunk (eval outputs) / 4 rows everywhere (fields_penalty produced)
F_EVAL, F_FULL = 3_834_880, 5_152_768

NET_CFG = dict(_target_="neddf.network.NeDDF", embed_pos_rank=10, embed_dir_rank=4, ddf_layer_count=8,
               ddf_layer_width=256, col_layer_count=4, col_layer_width=256, d_near=0.001,
               activation_type="tanhExp", density_activation_type="ReLU", lowpass_alpha_offset=10,
               penalty_weight=dict(constraints_aux_grad=0.05, constraints_dDdt=1.0, constraints_color=0.0001,
                                   range_distance=1.0, range_aux_grad=1.0, range_color=0.1), skips=[4])
RENDER_CFG = dict(sample_coarse=S_COARSE, sample_fine=S_FINE, dist_near=2.0, dist_far=6.0, max_dist=6.0,
                  use_coarse_network=False, sampling_type="cone")
WEIGHT_SEED = 3408
DUMP_LIMIT = 64 << 20  # bytes of --dump-outputs in all


def write_outputs(path: str, arrays) -> None:
    """--dump-outputs: every array as <path>/<name>.npy, float64 kept, everything else as float32."""
    import numpy as np
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT})")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def frame_outputs(outs, n_pix: int):
    """Colour [frames, pixels, 3] and depth [frames, pixels, 1] of one step's frames on the host (each frame either
    render_pixels' dict or the all-gathered [pixels, 4] colour + depth tiles).  When the frames do not fit half of
    DUMP_LIMIT, every frame keeps the same fixed, seeded sample of pixels, listed in ``pixel_index``."""
    import numpy as np
    img = torch.stack([o if torch.is_tensor(o) else torch.cat([o["color"], o["depth"]], 1) for o in outs]).cpu().numpy()
    res = {}
    keep = (DUMP_LIMIT // 2) // (img.shape[0] * img.shape[2] * img.itemsize)
    if keep < n_pix:
        idx = np.sort(np.random.default_rng(0).choice(n_pix, keep, replace=False))
        img = img[:, idx]
        res["pixel_index"] = idx.astype(np.float64)
    res["color"], res["depth"] = img[..., :3], img[..., 3:]
    return res


def synthetic_pose(seed: int):
    """Camera on the radius-4.0311 sphere looking at the origin (SURVEY 8(d))."""
    import numpy as np
    g = np.random.default_rng(seed)
    v = g.normal(size=3)
    v /= np.linalg.norm(v)
    back = v
    right = np.cross([0.0, 0.0, 1.0], back)
    right /= np.linalg.norm(right)
    up = np.cross(back, right)
    R = np.stack([right, up, back], 1).astype(np.float32)
    T = (4.0311 * v).astype(np.float32)
    focal = 0.5 * W / np.tan(0.5 * 0.6911112070083618)
    return R, T, np.array([focal, focal, 0.5 * W, 0.5 * H], dtype=np.float32)


def seeded_params(seed: int = WEIGHT_SEED, bias_std: float = 0.05):
    """Xavier-normal weights [in,out] like LinearGradLayer's init (nn_module/with_grad/linear.py:113-116)
    from a fixed seed, biases perturbed so the bias path is exercised.  Built from the product's own
    module (its parameter order is the reference's); tests/test_bench_contract.py pins that this is the
    stream the oracle's init_params draws, so the CPU legs see identical weights."""
    import math

    import neddf_b200
    net = neddf_b200.NeDDF(**{k: v for k, v in NET_CFG.items() if k != "_target_"})
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, v in net.state_dict().items():
        if name.endswith(".weight"):
            cin, cout = v.shape
            out[name] = torch.randn(cin, cout, generator=g) * math.sqrt(2.0 / (cin + cout))
        else:
            out[name] = torch.randn(v.shape[0], generator=g) * bias_std
    return out


def seeded_state_dict():
    """(state_dict of NeRFRender, per-network parameter dict) - no test infrastructure involved."""
    p = seeded_params()
    sd = {"network_fine." + k: v for k, v in p.items()}
    sd.update({"network_coarse." + k: v for k, v in p.items()})
    return sd, p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax = float(r[2])
            except Exception:
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for n, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_rate(n_rays: int, threads: int, keep=None):
    """The reference algorithm (oracle port, torch CPU fp32, same op structure as the reference)
    on a bounded sample of the workload: `n_rays` rays of the same frame.  ``keep`` (a dict) receives
    the sample's inputs and the port's outputs for the in-run parity check."""
    from oracle import neddf_oracle as orc
    torch.set_num_threads(threads)
    _, p = seeded_state_dict()
    fc = orc.FieldConfig.from_dict(NET_CFG)
    rc = orc.RenderConfig(**RENDER_CFG)
    st = orc.FieldState.at_iter(fc, -1)
    R, T, calib = synthetic_pose(0)
    cam = orc.CameraPose(torch.from_numpy(R), torch.from_numpy(T), *[float(c) for c in calib])
    uv = orc.image_uv(W, H)
    g = torch.Generator().manual_seed(1)
    sel = torch.randint(0, uv.shape[0], (n_rays,), generator=g)
    u_c = torch.rand(n_rays, S_COARSE + 1, generator=g)
    u_f = torch.rand(n_rays, S_FINE + 1, generator=g)
    with torch.no_grad():
        orc.render_rays(p, p, fc, st, rc, uv[sel[:32]], cam, u_c[:32], u_f[:32])  # warm-up
        t0 = time.perf_counter()
        taps = {} if keep is not None else None
        out = orc.render_rays(p, p, fc, st, rc, uv[sel], cam, u_c, u_f, taps=taps)
        dt = time.perf_counter() - t0
        if keep is not None:
            cdf = orc.pdf_cdf(out["weight_coarse"])
            _, ids = orc.invert_cdf(taps["dists_coarse"], cdf, u_f)
            keep.update(uv=uv[sel], u_c=u_c, u_f=u_f, out=out, ids=ids)
    return n_rays * NOMINAL_PER_RAY / dt, dt


def parity_block(render, cam, dev, keep):
    """BASELINE.md section 4 step 5: the CUDA path on the SAME rays and uniforms the CPU leg just
    rendered.  max|new - ref| / max|ref| per output, and the end-to-end mismatch rate of the
    searchsorted indices (bit-exact given the same cdf - tests/test_gpu_parity.py; here each side
    inverts its own coarse weights)."""
    uv, u_c, u_f, ref = keep["uv"].to(dev), keep["u_c"].to(dev), keep["u_f"].to(dev), keep["out"]
    with torch.no_grad():
        got = render.render_rays(uv, cam, uniforms=(u_c, u_f))
        dists_c = torch.empty_like(u_c)
        from neddf_b200 import _lib as L
        L.check(L.lib().neddf_coarse_dists(L.ptr(u_c), u_c.shape[0], u_c.shape[1], render.dist_near, render.dist_far,
                                           L.ptr(dists_c), L.stream_ptr(dev)), "coarse_dists")
        _, ids = render.sample_pdf(dists_c, got["weight_coarse"].clone(), u_f.shape[1], uniform_rands=u_f, return_ids=True)
    res = {}
    for k in ("color", "depth", "transmittance", "fields_penalty", "color_coarse", "depth_coarse"):
        a, b = got[k].detach().cpu().double(), ref[k].double()
        res[k] = float((a.reshape(b.shape) - b).abs().max() / b.abs().max())
    res["ids_mismatch_rate"] = float((ids.cpu() != keep["ids"]).double().mean())
    mse = float(((got["color"].detach().cpu().double() - ref["color"].double()) ** 2).mean())
    res["psnr_new_vs_ref_db"] = float("inf") if mse == 0 else 10.0 * math.log10(1.0 / mse)
    res["rays"] = int(uv.shape[0])
    res["reference"] = "oracle port (torch CPU fp32), same rays / uniforms / weights"
    return res


def best_cpu_threads():
    """Thread count for the CPU arm: the batched small GEMMs of the reference path do not scale to
    every core of a big host (128 threads measured 10x slower than 8 on the same work), so a tiny
    probe picks the fastest of a few counts - the baseline gets its best configuration.
    Returns (threads, ray-samples/s of the probe)."""
    n = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, n) if c <= n})
    best, best_rate = cands[0], 0.0
    for c in cands:
        r, _ = cpu_port_rate(48, c)
        if r > best_rate:
            best, best_rate = c, r
    return best, best_rate


def bounded_cpu_rays(max_rays: int, rate: float, seconds: float) -> int:
    """Rays in one CPU sample: at most `max_rays`, sized from the probe rate to about `seconds`."""
    if rate <= 0:
        return max_rays
    return int(max(48, min(max_rays, rate * seconds / NOMINAL_PER_RAY)))


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; /root/reference does not exist on
    the GPU box) timed on host cores, same workload/metric, bounded sample per step (about 10 s of
    CPU work each, so that W + K steps end within a few minutes on any host)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads, probe_rate = best_cpu_threads()
    n_rays = bounded_cpu_rays(args.cpu_rays, probe_rate, 10.0)
    rates = []
    for i in range(args.warmup + args.steps):
        r, dt = cpu_port_rate(n_rays, threads)
        if i >= args.warmup:
            rates.append((r, dt))
    value = sum(r for r, _ in rates) / len(rates)
    ms = 1e3 * sum(dt for _, dt in rates) / len(rates)
    line = {
        "impl": "reference", "metric": "ray-samples/s (800x800x192)", "value": value, "unit": "ray-samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus, "cpu"),
        "cpu_baseline": {"value": value, "unit": "ray-samples/s", "cores": threads, "kind": "port",
                         "sample": f"{n_rays} random rays of the 800x800 frame per step ({n_rays * EVALS_PER_RAY} MLP evaluations)"},
        "e2e": {"value": value, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus, engine):
    return {"workload": "lego-shaped synthetic 800x800 frame, 64 coarse + 128 fine samples/ray, cone sampling, "
                        "NeDDF 8x256 + 4x256 tanhExp, seeded random-init weights",
            "rays_per_frame": W * H, "frames_per_step": n_gpus, "nominal_samples_per_ray": NOMINAL_PER_RAY,
            "mlp_evaluations_per_ray": EVALS_PER_RAY, "engine": engine,
            "parallelism": f"ray-sharded x{n_gpus}, one all-gather of image tiles per frame" if n_gpus > 1 else "single GPU",
            "l2": "per-frame uniforms are 497 MB (> 126 MB L2) and every step reads fresh ones; no explicit flush"}


# --------------------------------------------------------------------------------------------------
# workload "train": BASELINE.json configs[3] - the training inner loop (nerf_trainer.py:100-134) on 1 GPU
# --------------------------------------------------------------------------------------------------
TRAIN_RAYS = 1024           # config/trainer/nerf_trainer.yaml:3
TRAIN_LR = 5e-4             # optimizer_lr
# config/loss/neddf_loss.yaml: (weight, weight_coarse) of ColorLoss, MaskBCELoss, FieldsConstraintLoss
LOSS_W = {"color": (1.0, 0.1), "mask": (0.05, 0.005), "fields_penalty": (0.01, 0.01)}


def train_loss(out, target_color, target_mask):
    """The reference's objective (loss/color_loss.py:41-55, mask_bce_loss.py:41-59,
    fields_constraint_loss.py:40-54, summed as nerf_trainer.py:118-121) in plain torch ops."""
    total = 0.0
    for suffix, wi in (("", 0), ("_coarse", 1)):
        total = total + LOSS_W["color"][wi] * torch.mean(torch.square(out["color" + suffix] - target_color))
        m = torch.clamp(1.0 - out["transmittance" + suffix], 1e-6, 1.0 - 1e-6)
        total = total + LOSS_W["mask"][wi] * -torch.mean(target_mask * torch.log(m) + (1.0 - target_mask) * torch.log(1.0 - m))
        total = total + LOSS_W["fields_penalty"][wi] * torch.mean(out["fields_penalty" + suffix])
    return total


def train_batch(step: int, n_rays: int):
    """Host-side batch like the trainer draws it: int16 pixel ids (nerf_trainer.py:100-106), synthetic
    colour / mask targets (there is no dataset here)."""
    g = torch.Generator().manual_seed(77 + step)
    us = (torch.rand(n_rays, generator=g) * (W - 1)).to(torch.int16)
    vs = (torch.rand(n_rays, generator=g) * (H - 1)).to(torch.int16)
    uv = torch.stack([us, vs], 1)
    color = torch.rand(n_rays, 3, generator=g)
    mask = (torch.rand(n_rays, generator=g) > 0.5).float()
    return uv, color, mask


def cpu_port_train_rate(n_rays: int, threads: int):
    """Forward + backward (autograd through the oracle port) + Adam on `n_rays` rays, host cores."""
    from oracle import neddf_oracle as orc
    torch.set_num_threads(threads)
    _, p = seeded_state_dict()
    p = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    fc = orc.FieldConfig.from_dict(NET_CFG)
    rc = orc.RenderConfig(**RENDER_CFG)
    R, T, calib = synthetic_pose(0)
    cam = orc.CameraPose(torch.from_numpy(R), torch.from_numpy(T), *[float(c) for c in calib])
    opt = torch.optim.Adam(list(p.values()), lr=TRAIN_LR)
    dts = []
    for it in range(2):
        uv, color, mask = train_batch(it, n_rays)
        g = torch.Generator().manual_seed(it)
        u_c, u_f = torch.rand(n_rays, S_COARSE + 1, generator=g), torch.rand(n_rays, S_FINE + 1, generator=g)
        st = orc.FieldState.at_iter(fc, it)
        t0 = time.perf_counter()
        out = orc.render_rays(p, p, fc, st, rc, uv.long(), cam, u_c, u_f)
        loss = train_loss(out, color, mask)
        opt.zero_grad()
        loss.backward()
        opt.step()
        dts.append(time.perf_counter() - t0)
    dt = dts[-1]
    return n_rays * NOMINAL_PER_RAY / dt, dt


def train_config(engine):
    return {"workload": "drums-shaped synthetic training step: 1024 random pixels of an 800x800 view, 64 coarse + 128 "
                        "fine samples/ray, forward + backward + Adam (nerf_trainer.py:100-134, neddf_loss.yaml), "
                        "NeDDF 8x256 + 4x256 tanhExp, seeded random-init weights, set_iter(k)",
            "rays_per_step": TRAIN_RAYS, "nominal_samples_per_ray": NOMINAL_PER_RAY,
            "mlp_evaluations_per_ray": EVALS_PER_RAY, "engine": engine, "parallelism": "single GPU",
            "l2": "1.3e9 B of per-step activations (> 126 MB L2) are written and re-read every step; no explicit flush"}


def run_train(args):
    metric = "ray-samples/s (training step, 1024 rays x 192)"
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if rank != 0:
            return
        n = max(8, min(32, args.cpu_rays))
        threads = min(32, os.cpu_count() or 1)
        rates = []
        for i in range(args.warmup + args.steps):
            r, dt = cpu_port_train_rate(n, threads)
            if i >= args.warmup:
                rates.append((r, dt))
        value = sum(r for r, _ in rates) / len(rates)
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": value, "unit": "ray-samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(d for _, d in rates) / len(rates),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": train_config("cpu"),
            "cpu_baseline": {"value": value, "unit": "ray-samples/s", "cores": threads, "kind": "port",
                             "sample": f"{n} rays per step: forward + autograd backward + Adam"},
            "e2e": {"value": value, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}), flush=True)
        return
    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("bench.py --workload train is a single-GPU workload (BASELINE.json configs[3])")
    import neddf_b200
    from neddf_b200 import _lib as L
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the training path has no CPU implementation")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    torch.manual_seed(0)  # render_rays draws the training uniforms from torch's generator: same run, same numbers
    sd, _ = seeded_state_dict()
    render = neddf_b200.NeRFRender(network_config=NET_CFG, **RENDER_CFG)
    render.load_state_dict(sd)
    render.to(dev)
    render.set_engine(args.engine)
    render.check_nan = False
    R, T, calib = synthetic_pose(0)
    cam = neddf_b200.Camera.from_matrix(neddf_b200.PinholeCalib(calib), R, T).to(dev)
    cam.update_transform()
    from neddf_b200 import losses, optim
    opt = optim.FusedAdam.for_render(render, lr=TRAIN_LR)          # one launch per network + re-pack
    loss_fn = losses.RenderLoss(**{k: v for k, v in LOSS_W.items()})  # the six loss terms in one launch
    n_batches = 8
    host = [tuple(x.pin_memory() for x in train_batch(i, TRAIN_RAYS)) for i in range(n_batches)]
    resident = [tuple(x.to(dev) for x in b) for b in host]
    it = [0]

    def one_step(uv, color, mask):
        render.set_iter(it[0])
        it[0] += 1
        out = render.render_rays(uv, cam)
        loss = torch.sum(torch.stack(list(loss_fn(out, {"color": color, "mask": mask}).values())))  # nerf_trainer.py:121
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss, out

    def step_device(i):
        return one_step(*resident[i % n_batches])

    def step_e2e(i):
        uv, color, mask = (x.to(dev, non_blocking=True) for x in host[i % n_batches])
        return float(one_step(uv, color, mask)[0].item())  # the loss the trainer logs (nerf_trainer.py:124)

    def timed(fn, steps):
        """(ms per step, what the last step returned)"""
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            last = fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps, last

    for i in range(args.warmup):
        step_device(i)
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = L.lib().neddf_launch_count()
    ms_step, (loss, out) = timed(step_device, args.steps)
    launches = L.lib().neddf_launch_count() - launches0
    clocks = sampler.stop()
    render.check_status()
    if args.dump_outputs:  # the loss, the render outputs and the weights after the optimiser step
        dump = {"loss": loss.detach().cpu().numpy()}
        dump.update({k: v.detach().cpu().numpy() for k, v in out.items()})
        dump.update({"param." + k: v.detach().cpu().numpy() for k, v in render.network_fine.state_dict().items()})
    for i in range(2):
        step_e2e(i)
    ms_e2e, _ = timed(step_e2e, args.steps)
    value = TRAIN_RAYS * NOMINAL_PER_RAY / (ms_step * 1e-3)
    evals = TRAIN_RAYS * EVALS_PER_RAY
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    achieved = evals * 3 * F_FULL / (ms_step * 1e-3) / 1e12
    cpu = None
    if not args.no_cpu_baseline:
        threads = min(32, os.cpu_count() or 1)
        v, dt = cpu_port_train_rate(16, threads)
        cpu = {"value": v, "unit": "ray-samples/s", "cores": threads, "kind": "port",
               "sample": f"16 rays: forward + autograd backward + Adam ({dt:.1f} s)"}
    engine = render.network_fine.resolved_engine(dev)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, dump)
    print(json.dumps({
        "metric": metric, "value": value, "unit": "ray-samples/s", "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if engine == "fp32" else "f16x3-split operands, f32 accumulate (forward and data-gradient GEMMs); f32 elsewhere",
        "data": "synthetic", "config": train_config(engine),
        "mlp_evaluations_per_s": evals / (ms_step * 1e-3),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                     "frac": achieved / peak if peak else None, "traffic": None,
                     "kernel": "whole training step (field forward x2, field backward x2, weight gradients, Adam)",
                     "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback",
                     "flop_per_evaluation": 3 * F_FULL},
        "cpu_baseline": cpu,
        "e2e": {"value": TRAIN_RAYS * NOMINAL_PER_RAY / (ms_e2e * 1e-3), "unit": "ray-samples/s",
                "h2d_bytes_per_step": TRAIN_RAYS * (2 * 2 + 3 * 4 + 4), "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e},
        "gpu_launches": int(launches), "clocks": clocks,
        "peak_memory_gib": torch.cuda.max_memory_allocated() / 2 ** 30}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--engine", default="auto", choices=["auto", "fp32", "tc", "tc2"])
    ap.add_argument("--workload", default="render", choices=["render", "train"],
                    help="render = BASELINE.json configs[1] (800x800 frame, the headline); train = configs[3] "
                         "(1024-ray training step: forward + backward + Adam)")
    ap.add_argument("--cpu-rays", type=int, default=384, help="rays in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eps", type=float, default=0.0,
                    help="early ray termination threshold on the transmittance (BASELINE.json configs[4]; 0 = off = "
                         "the reference's behaviour, the default workload)")
    ap.add_argument("--segments", type=int, default=4, help="depth segments of the fine pass when --eps > 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB; seeded inputs, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path; --impl reference has none")
    if args.warmup < 3:
        args.warmup = 3  # timing rules: W >= 3
    if args.workload == "train":
        return run_train(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    import neddf_b200
    from neddf_b200 import _lib as L
    from neddf_b200.dist import render_image_sharded, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the render hot path has no CPU implementation "
                         "(use --impl reference for the host-core baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    sd, _ = seeded_state_dict()
    render = neddf_b200.NeRFRender(network_config=NET_CFG, **RENDER_CFG)
    render.load_state_dict(sd)
    render.to(dev)
    render.set_iter(-1)
    render.set_engine(args.engine)
    render.check_nan = False  # no host sync inside the timed region; checked once after it
    render.transmittance_eps, render.termination_segments = float(args.eps), int(args.segments)
    n_pix = W * H
    first, count = shard_range(n_pix, world, rank)
    n_frames = n_gpus  # frames per step
    cams = []
    for f in range(n_frames):
        R, T, calib = synthetic_pose(f)
        cam = neddf_b200.Camera.from_matrix(neddf_b200.PinholeCalib(calib), R, T).to(dev)
        cam.update_transform()
        cams.append(cam)

    # host-side inputs of one step (pinned): the uniforms of this rank's slice of every frame
    g = torch.Generator().manual_seed(1234 + rank)
    host_u = [(torch.rand(count, S_COARSE + 1, generator=g).pin_memory(),
               torch.rand(count, S_FINE + 1, generator=g).pin_memory()) for _ in range(n_frames)]
    dev_u = [(a.to(dev), b.to(dev)) for a, b in host_u]
    targets = ["color", "depth"]

    def step_device():
        outs = []
        for f in range(n_frames):
            flat = render.render_pixels(W, H, cams[f], targets, 1, first, count, dev_u[f])
            if world > 1:
                from neddf_b200.dist import gather_tiles
                packed = torch.cat([flat["color"], flat["depth"]], 1)
                outs.append(gather_tiles(packed, n_pix))
            else:
                outs.append(flat)
        return outs

    def step_e2e():
        """Public API with host buffers: H2D of the uniforms, render_image (sharded when N>1),
        D2H of colour + depth."""
        res = []
        for f in range(n_frames):
            u = (host_u[f][0].to(dev, non_blocking=True), host_u[f][1].to(dev, non_blocking=True))
            if world > 1:
                flat = render.render_pixels(W, H, cams[f], targets, 1, first, count, u)
                from neddf_b200.dist import gather_tiles
                img = gather_tiles(torch.cat([flat["color"], flat["depth"]], 1), n_pix)
                if rank == 0:
                    res.append(img.to("cpu", non_blocking=False))
            else:
                img = render.render_image(W, H, cams[f], targets, 1, 1024, uniforms=u)
                res.append((img["color"].cpu(), img["depth"].cpu()))
        return res

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if profile:
            render.network_fine._profile_events = []
        ev0.record()
        for _ in range(steps):
            last = fn()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        evs = None
        if profile:
            evs = render.network_fine._profile_events
            render.network_fine._profile_events = None
        return float(t.item()), evs, last

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    render.termination_stats()  # reset the executed / nominal counters after the warm-up
    launches0 = L.lib().neddf_launch_count()
    ms_total, evs, last = timed(step_device, args.steps, profile=True)
    launches = L.lib().neddf_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    # copied now: the renders below may reuse the buffers behind the last step's outputs
    dump = frame_outputs(last, n_pix) if args.dump_outputs and rank == 0 else None
    del last
    render.check_status()
    term = render.termination_stats()  # fine-pass evaluations of this rank inside the timed region
    if world > 1:
        tt = torch.tensor([term["executed"], term["nominal"]], device=dev, dtype=torch.int64)
        dist.all_reduce(tt)
        term = {"executed": int(tt[0]), "nominal": int(tt[1])}
    ms_step = ms_total / args.steps
    rays_per_step = n_pix * n_frames
    value = rays_per_step * NOMINAL_PER_RAY / (ms_step * 1e-3)

    # dominant kernel: the field megakernel.  Launch durations from CUDA events recorded around
    # every launch on the launching stream, inside the timed region above.
    evals, kms = 0, 0.0
    for (e0, e1, n_eval) in evs:
        kms += e0.elapsed_time(e1)
        evals += n_eval or 0
    if args.eps > 0:  # segment launches carry no static count: coarse passes + what the fine passes really ran
        evals = args.steps * n_frames * count * (S_COARSE + 1) + term["executed"] // world
    flop = F_EVAL
    achieved_tflops = evals * flop / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"
    # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture; only valid for the
    # kernel source it was taken from (hash of field_tc.cu + tc_ptx.cuh) and the engine it profiled
    traffic, traffic_note = None, None
    try:
        import hashlib
        tj = json.load(open(os.path.join(ROOT, "profiles", "field_kernel_traffic.json")))
        h = hashlib.sha256(b"".join(open(os.path.join(ROOT, f), "rb").read() for f in tj["source_files"])).hexdigest()
        if h != tj["source_sha256"]:
            traffic_note = "profiles/field_kernel_traffic.json was captured from a different kernel source - re-run the ncu capture"
        elif render.network_fine.resolved_engine(dev) != "tc":
            traffic_note = "the committed capture is of the tc engine"
        else:
            traffic = tj["dram_bytes_per_launch"]
            traffic_note = tj["launch"]
    except Exception as e:  # noqa: BLE001
        traffic_note = f"no capture available ({e})"

    # end to end through the public API with host buffers
    for _ in range(2):
        step_e2e()
    ms_e2e, _, _ = timed(step_e2e, max(1, args.steps))
    ms_e2e /= max(1, args.steps)
    e2e_value = rays_per_step * NOMINAL_PER_RAY / (ms_e2e * 1e-3)
    h2d = n_frames * count * (S_COARSE + 1 + S_FINE + 1) * 4 + n_frames * 16 * 4
    d2h = n_frames * n_pix * 4 * 4 if rank == 0 else 0

    # strong scaling: ONE frame ray-sharded over the N ranks (latency of a frame), device-resident uniforms
    strong = None
    if world > 1:
        from neddf_b200.dist import gather_tiles

        def one_frame():
            flat = render.render_pixels(W, H, cams[0], targets, 1, first, count, dev_u[0])
            return gather_tiles(torch.cat([flat["color"], flat["depth"]], 1), n_pix)

        one_frame()
        ms_frame, _, _ = timed(one_frame, max(3, args.steps))
        ms_frame /= max(3, args.steps)
        strong = {"frame_ms": ms_frame, "ray_samples_per_s": n_pix * NOMINAL_PER_RAY / (ms_frame * 1e-3),
                  "note": "one 800x800 frame sharded over the ranks + the all-gather of the image tiles"}

    cpu, parity = None, None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:  # reported at N=1 only
        threads, probe_rate = best_cpu_threads()
        cpu_rays = bounded_cpu_rays(args.cpu_rays, probe_rate, 20.0)
        keep = {}
        v, dt = cpu_port_rate(cpu_rays, threads, keep)
        cpu = {"value": v, "unit": "ray-samples/s", "cores": threads, "kind": "port",
               "sample": f"{cpu_rays} random rays of the same 800x800 frame ({cpu_rays * EVALS_PER_RAY} MLP evaluations, {dt:.1f} s)"}
        parity = parity_block(render, cams[0], dev, keep)

    if rank == 0:
        engine = render.network_fine.resolved_engine(dev)
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        line = {
            "metric": "ray-samples/s (800x800x192)", "value": value, "unit": "ray-samples/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if engine == "fp32" else "f16x3-split operands, f32 accumulate",
            "data": "synthetic", "config": workload_config(n_gpus, engine),
            "mlp_evaluations_per_s": rays_per_step * EVALS_PER_RAY / (ms_step * 1e-3),
            "roofline": {"bound": "tensor", "achieved": achieved_tflops, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved_tflops / peak if peak else None, "traffic": traffic, "traffic_note": traffic_note,
                         "kernel": "field megakernel (NeDDF.forward fused)", "peak_source": peak_src,
                         "flop_per_evaluation": flop, "launches_timed": len(evs),
                         "kernel_share_of_step": kms / ms_total if ms_total else None},
            "cpu_baseline": cpu,
            "parity": parity,
            "strong_scaling": strong,
            "early_termination": None if args.eps <= 0 else {
                "transmittance_eps": args.eps, "segments": args.segments,
                "fine_evaluations_executed": term["executed"], "fine_evaluations_nominal": term["nominal"],
                "note": "value / e2e count NOMINAL ray-samples; executed < nominal is work skipped under the error bound "
                        "|d color| <= eps max|c| (not in the reference: opt-in)"},
            "e2e": {"value": e2e_value, "unit": "ray-samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
