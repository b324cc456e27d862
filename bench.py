#!/usr/bin/env python
"""bench.py -- benchmarks of the NeRSemble render hot path on B200 (one JSON line on rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2|2occ|3|4|5] [--scaling strong|weak] [--impl reference]
                    [--dump-outputs DIR]

Default (what the driver runs): BASELINE.json config 2 -- 4096 rays x 256 samples = 2^20 samples, 32-member hash
ensemble with full-size tables (16 levels x 2^19), T = 24, fused forward + alpha composite.

  value     device-resident inputs, ONE kernel launch per step: fixed-stride march -> fused field -> composite
            (nsb_render_forward through the op layer).
            N > 1: STRONG scaling of the 4096-ray batch (SURVEY 8e: "partition the ray batch 1/N per GPU"), the
            per-ray RGB all-gathered to every rank INSIDE the timed region (NCCL); the weak-scaling number (every
            rank renders its own 4096 rays, no collective) is measured in the same run and reported under "weak".
  e2e       the same metric through the reference-facing plugin call `NeRSembleNGPModel.get_outputs_for_camera_ray_bundle`
            (evaluate_nersemble.py:143) with HOST buffers: pinned H2D of the rays and D2H of the RGB inside the timed
            region, occupancy-grid sampler, 256 samples per ray via the bundle's nears / fars.
  parity    RGB of the first 64 rays of the SAME batch and parameters against the CPU oracle (north-star tolerance:
            per-pixel L2 < 1e-3); the run fails when it is exceeded.
  roofline  HBM: 16 384 algorithmic bytes per sample / time of the fused render kernel (CUDA events around its launch).
  cpu_baseline  the oracle port timed on the host cores on those 64 rays (1 warm-up + median of 5).

Other configs (BASELINE.json configs[2..4]; `--config`): 2occ = config 2 with a seeded blob occupancy grid through the
plugin sampler; 3 = full training step of the seq-30 recipe (jittered occupancy march + visibility pre-pass, six losses,
backward, FusedFieldsAdam) on one GPU; 4 = 1088x1920 frames, rays sharded over the ranks, RGB all-gathered; 5 = dense
march (--disable_occupancy_grid) full gradient step on N GPUs with the gradient all-reduce inside the timed region.

`--impl reference` times the CPU oracle port of the reference's path (its GPU dependencies tiny-cuda-nn / nerfacc /
nerfstudio are not installable here) on the host cores, on a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned to its caller as DIR/<name>.npy
(float32, or float64 for integers): config 2 the render op's per-ray outputs (rgb, accumulation, depth, deformation,
num_samples_per_ray, packed_info) and the plugin call's as e2e_<name>; configs 3 / 5 the training step's per-ray outputs
and loss; config 4 the gathered frame (rgb) and rank 0's rows of the other outputs.  Inputs are seeded, so two builds
run with the same arguments can be compared file for file; above 64 MB in all a fixed, seeded sample is written.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

RAYS = 4096
SAMPLES_PER_RAY = 256
STEP = 0.011
NEAR = 0.2
N_TIMESTEPS = 24
LOG2T = 19
SEED = 19980801                   # the reference's seed (train_nersemble.py:116)
ALG_BYTES_PER_SAMPLE = 16384      # 16 levels x 8 corners x 32 members x 2 feats x 2 B (SURVEY 8d)
AABB = ((-2.5, -1.8, -2.5), (2.2, 1.8, 2.0))   # sequence-30 box (train_nersemble.py:42)
PARITY_RAYS = 64
WORKLOAD2 = "config2: 4096 rays x 256 samples = 2^20 samples, 32x(16 lvl, 2^19) fp16 hash ensemble, T=24, fwd+composite"


# ------------------------------------------------------------------------------------------------ synthetic data
def synthetic_rays(R, seed, device="cpu"):
    """16 pinhole cameras on a ring of radius 9 aimed at the head volume (SURVEY 8d config 2)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    cam = torch.randint(0, 16, (R,), generator=g)
    ang = cam.float() / 16 * 2 * torch.pi
    o = torch.stack([9.0 * torch.sin(ang), 0.3 * torch.cos(3 * ang), 9.0 * torch.cos(ang)], -1)
    target = (torch.rand((R, 3), generator=g) * 2 - 1) * 1.2
    d = target - o
    d = d / d.norm(dim=-1, keepdim=True)
    times = torch.rand((R, 1), generator=g)
    return o.float().to(device), d.float().to(device), times.float().to(device)


def synthetic_params(seed=SEED, n_timesteps=N_TIMESTEPS, log2T=LOG2T):
    """Random-init parameters of the named architecture on the CPU (trained-like scale so that densities and colours
    are non-trivial): ONE parameter set feeds the CUDA path, the plugin model and the CPU oracle leg."""
    import torch
    from nersemble_b200 import packing
    g = torch.Generator().manual_seed(seed)
    lv = packing.level_table(log2_hashmap_size=log2T)

    def U(shape, b):
        return (torch.rand(shape, generator=g) * 2 - 1) * b

    xav = lambda o, i: U((o, i), math.sqrt(6.0 / (i + o)))
    dims = [(128, 173), (128, 128), (128, 128), (128, 128), (128, 301), (128, 128)]
    return dict(
        levels=lv, aabb=torch.tensor(AABB),
        tables=U((lv["total_entries"], 32, 2), 0.5),
        base_w=[xav(64, 32), xav(16, 64)], head_w=[xav(64, 32), xav(64, 64), xav(16, 64)],
        stem_w=[U((o, i), 1 / math.sqrt(i)) for o, i in dims], stem_b=[U((o,), 1 / math.sqrt(i)) for o, i in dims],
        r_w=U((3, 128), 1e-3), r_b=torch.zeros(3), v_w=U((3, 128), 1e-3), v_b=torch.zeros(3),
        time_emb=torch.randn((n_timesteps, 32), generator=g) * 0.18,
        time_emb_deform=torch.randn((n_timesteps, 128), generator=g) * 0.09)


def native_params(S, device):
    from nersemble_b200 import ops
    deform = dict(stem_w=S["stem_w"], stem_b=S["stem_b"], r_w=S["r_w"], r_b=S["r_b"], v_w=S["v_w"], v_b=S["v_b"])
    return ops.NativeParams.build(tables=S["tables"], base_w=S["base_w"], head_w=S["head_w"], time_emb=S["time_emb"],
                                  aabb=S["aabb"], levels=S["levels"], deform=deform, time_emb_deform=S["time_emb_deform"],
                                  device=device)


def recipe_config(n_timesteps=N_TIMESTEPS, log2T=LOG2T, **over):
    """The hyper-parameters of scripts/train/train_nersemble.py:184-240 (seq-30 defaults) on the plugin config."""
    from nersemble_b200.plugin.components import HashEnsembleConfig, SE3DeformationFieldConfig, TCNNHashEncodingConfig
    from nersemble_b200.plugin.model import NeRSembleNGPModelConfig
    kw = dict(render_step_size=STEP, near_plane=NEAR, far_plane=1e3, cone_angle=0.0, alpha_thre=1e-2, occ_thre=1e-2,
              early_stop_eps=0, background_color="white", grid_levels=1, disable_scene_contraction=True,
              n_timesteps=n_timesteps, latent_dim_time=32, use_masked_rgb_loss=True, alpha_mask_threshold=0,
              lambda_alpha_loss=1e-2, lambda_near_loss=1e-4, lambda_empty_loss=1e-2, lambda_depth_loss=1e-4,
              lambda_dist_loss=1e-4, use_hash_ensemble=True,
              hash_ensemble_config=HashEnsembleConfig(32, TCNNHashEncodingConfig(log2_hashmap_size=log2T), True, True),
              use_deformation_field=True, use_separate_deformation_time_embedding=True,
              deformation_field_config=SE3DeformationFieldConfig(warp_code_dim=128, mlp_num_layers=6, mlp_layer_width=128),
              window_hash_encodings_begin=40000, window_hash_encodings_end=80000, window_deform_begin=0,
              window_deform_end=20000, use_view_frustum_culling=False, eval_num_rays_per_chunk=RAYS)
    kw.update(over)
    return NeRSembleNGPModelConfig(**kw)


def build_model(S, device, **over):
    """The reference-facing plugin model (NeRSembleNGPModel) holding the synthetic parameters, windows at their final
    values (w_hash = 32, w_deform = 7)."""
    import torch
    from nersemble_b200.nerfstudio_shim import SceneBox
    cfg = recipe_config(n_timesteps=S["time_emb"].shape[0], log2T=int(math.log2(max(S["levels"]["entries"]))), **over)
    m = cfg.setup(scene_box=SceneBox(S["aabb"].clone()), num_train_data=16, metadata={"camera_frustums": None})
    with torch.no_grad():
        m.field.hash_ensemble.tables.copy_(S["tables"])
        m.field.mlp_base.params.copy_(torch.cat([w.reshape(-1) for w in S["base_w"]]))
        m.field.mlp_head.params.copy_(torch.cat([w.reshape(-1) for w in S["head_w"]]))
        se3 = m.deformation_field.se3_field
        for i, layer in enumerate(se3.mlp_stem.layers):
            layer.weight.copy_(S["stem_w"][i]); layer.bias.copy_(S["stem_b"][i])
        se3.mlp_r.layers[0].weight.copy_(S["r_w"]); se3.mlp_r.layers[0].bias.copy_(S["r_b"])
        se3.mlp_v.layers[0].weight.copy_(S["v_w"]); se3.mlp_v.layers[0].bias.copy_(S["v_b"])
        m.time_embedding.weight.copy_(S["time_emb"])
        m.time_embedding_deformation.weight.copy_(S["time_emb_deform"])
    m = m.to(device)
    m.sched_window_hash_encodings.value = 32.0
    m.sched_window_deform.value = 7.0
    return m


def blob_occupancy(res=128, seed=5, n_blobs=6):
    """Seeded union of spheres in grid coordinates (the `occ` variant of config 2 and configs 3/4)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    ax = (torch.arange(res).float() + 0.5) / res
    X, Y, Z = torch.meshgrid(ax, ax, ax, indexing="ij")
    occ = torch.zeros((res, res, res), dtype=torch.bool)
    for _ in range(n_blobs):
        c = 0.25 + 0.5 * torch.rand(3, generator=g)
        r = 0.12 + 0.14 * float(torch.rand(1, generator=g))
        occ |= ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) < r * r
    return occ


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Polls SM clock and throttle reasons through NVML every few ms while `active` is set (the timed regions)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.active = False
        self.stop_flag = False

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            while not self.stop_flag:
                if self.active:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for n, bit in names.items():
                        if r & bit:
                            self.reasons.add(n)
                time.sleep(0.002)
        except Exception as e:  # noqa: BLE001
            self.error = repr(e)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "n_samples": 0,
                    "error": getattr(self, "error", None)}
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "n_samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU oracle leg
def oracle_field_params(S):
    """The SAME synthetic parameters as an oracle FieldParams (test infrastructure: checker / CPU baseline only)."""
    from oracle import pipeline as pl
    from oracle.tp.tcnn_cpu import hashgrid_levels
    lv = hashgrid_levels(16, int(math.log2(max(S["levels"]["entries"]))), 16, 1.4472692012786865)
    return pl.FieldParams(S["aabb"].float(), S["tables"], S["base_w"], S["head_w"], S["stem_w"], S["stem_b"],
                          S["r_w"], S["r_b"], S["v_w"], S["v_b"], S["time_emb"], S["time_emb_deform"], lv)


def cpu_oracle(S, o, d, times, repeats=5, mode="none"):
    """Renders rays (o, d, times) x 256 samples with the CPU oracle port (oracle/pipeline.py, fp32 torch ops on the
    fp16-stored tables): returns (rgb, median seconds of `repeats` runs after one warm-up, threads, n_samples)."""
    import torch
    from oracle import pipeline as pl
    from oracle.tp.tcnn_cpu import Precision
    avail = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    P = oracle_field_params(S)
    Precision.mode = mode
    ts, te, ri = pl.fixed_samples(o, d, P.aabb, SAMPLES_PER_RAY, STEP, near=NEAR)
    # thread count: the oracle is gather-bound torch code that does NOT scale to every hardware thread (r1: the same
    # code gave 0.0007 .. 0.0089 M samples/s between boxes with torch.set_num_threads(os.cpu_count())); calibrate on
    # 8 rays and keep the fastest setting -- `cores` reports what was used
    global _ORACLE_THREADS
    if "_ORACLE_THREADS" not in globals():
        best = None
        n8 = 8 * SAMPLES_PER_RAY
        for c in sorted({min(avail, c) for c in (8, 16, 32, 64, avail)}):
            torch.set_num_threads(c)
            with torch.no_grad():
                for it in range(2):
                    t0 = time.perf_counter()
                    pl.render(P, o[:8], d[:8], times[:8], ts[:n8], te[:n8], ri[:n8], window_hash=32.0, window_deform=7.0, training=False)
                    dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, c)
        _ORACLE_THREADS = best[1]
    torch.set_num_threads(_ORACLE_THREADS)
    secs, out = [], None
    with torch.no_grad():
        for it in range(repeats + 1):
            t0 = time.perf_counter()
            out = pl.render(P, o, d, times, ts, te, ri, window_hash=32.0, window_deform=7.0, training=False)
            if it > 0:
                secs.append(time.perf_counter() - t0)
    Precision.mode = "reference"
    return out["rgb"], statistics.median(secs), torch.get_num_threads(), int(ts.numel())


def run_reference(args):
    """The reference arm: the CPU oracle port on a bounded sample (64 rays x 256 samples per step) of config 2."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    S = synthetic_params()
    o, d, t = synthetic_rays(RAYS, 1000)
    reps = args.steps
    rgb, sec, threads, n = cpu_oracle(S, o[:PARITY_RAYS], d[:PARITY_RAYS], t[:PARITY_RAYS], repeats=reps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, host_arrays({"rgb": rgb}))
    v = n / sec / 1e6
    sample = f"{PARITY_RAYS} rays x {SAMPLES_PER_RAY} samples ({n} samples) per step, full-size tables, oracle/pipeline.py torch CPU fp32; 1 warm-up + median of {reps}"
    print(json.dumps({
        "impl": "reference", "metric": "M ray-samples/sec", "value": v, "unit": "M ray-samples/s", "n_gpus": args.gpus,
        "steps": reps, "warmup": 1, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 and args.scaling != "weak" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOAD2, "sample": sample},
        "cpu_baseline": {"value": v, "unit": "M ray-samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "M ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ------------------------------------------------------------------------------------------------ helpers
class Dist:
    def __init__(self, gpus):
        import torch
        import torch.distributed as dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        assert self.world == gpus or self.world == 1, (self.world, gpus)
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.dist = dist

    def barrier(self):
        import torch
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, *vals):
        import torch
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.cpu()]

    def sum(self, *vals):
        import torch
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.cpu()]

    def close(self):
        """End of the run.  N > 1: communicators that were captured into CUDA graphs made destroy_process_group() hang
        (r2i: rank 0 had printed its line, then torchrun sat until the outer timeout), so the graphs are reset first and
        the process leaves through os._exit after a last barrier."""
        import torch
        for g in _GRAPHS:
            try:
                g.reset()
            except Exception:  # noqa: BLE001
                pass
        _GRAPHS.clear()
        torch.cuda.synchronize()
        if self.world > 1:
            try:
                self.dist.barrier()
                torch.cuda.synchronize()
            except Exception:  # noqa: BLE001
                pass
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(0)


_GRAPHS: list = []


def timed(D, fn, K, sampler=None):
    """K calls of fn bracketed by barrier + synchronize on both sides; returns (CUDA-event milliseconds of this rank,
    what the last call returned)."""
    import torch
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    D.barrier()
    if sampler is not None:
        sampler.active = True
    e0.record()
    for _ in range(K):
        last = fn()
    e1.record()
    D.barrier()
    if sampler is not None:
        sampler.active = False
    return e0.elapsed_time(e1), last


DUMP_BYTES = 60 << 20             # 62.9 MB of array data: the files stay under 64 MB with their .npy headers


def host_arrays(outputs, prefix=""):
    """The tensors among a call's outputs (name -> tensor; other values and names starting with '_' are skipped), copied
    to the host: float64 as it is, other floating point as float32, integers and booleans as float64 (exact)."""
    import torch
    arrs = {}
    for k, v in outputs.items():
        if torch.is_tensor(v) and not k.startswith("_"):
            v = v.detach().cpu()
            arrs[prefix + k] = (v.float() if v.is_floating_point() and v.dtype != torch.float64 else v.double()).numpy()
    return arrs


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes every array as out_dir/<name>.npy, so that two builds run with the same arguments (same
    seeded inputs) can be compared output for output.  Above DUMP_BYTES in all, every array is cut to the same fraction
    of its elements, flattened, at positions drawn with a fixed seed (the same for every run of the same shapes)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, a.size * DUMP_BYTES // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(SEED).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def graphed(fn, dev):
    """Capture fn (kernels + NCCL collectives on the current stream) into a CUDA graph; returns (replay, captured?)."""
    import torch
    try:
        s = torch.cuda.Stream(dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(s):
            for _ in range(3):
                fn()
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        torch.cuda.synchronize()
        _GRAPHS.append(g)
        return g.replay, True
    except Exception as e:  # noqa: BLE001  (capture of a collective can be refused: fall back to eager launches)
        sys.stderr.write(f"[bench] CUDA-graph capture failed, running eagerly: {e!r}\n")
        torch.cuda.synchronize()
        return fn, False


# ------------------------------------------------------------------------------------------------ config 2
def run_config2(args, occ=False):
    import torch
    from nersemble_b200 import ops
    from nersemble_b200.distributed import shard_bounds
    from nersemble_b200.nerfstudio_shim import RayBundle
    D = Dist(args.gpus)
    dev, rank, world = D.dev, D.rank, D.world
    W, K = max(args.warmup, 3), args.steps
    strong = world > 1 and args.scaling != "weak"
    S = synthetic_params()
    P = native_params(S, dev)
    model = build_model(S, dev).eval()
    if occ:
        model.occupancy_grid.binaries[0] = blob_occupancy().to(dev)
    else:
        model.occupancy_grid.binaries[:] = True
    aabb = P.aabb
    n_samples = RAYS * SAMPLES_PER_RAY

    # one global 4096-ray batch (seed 1000) for the strong-scaling / parity / e2e legs; rank-private batches for weak scaling
    o_g, d_g, t_g = synthetic_rays(RAYS, 1000)
    lo, hi = shard_bounds(RAYS, rank, world) if strong else (0, RAYS)
    o_s, d_s, t_s = o_g[lo:hi].to(dev), d_g[lo:hi].to(dev), t_g[lo:hi].to(dev)
    o_w, d_w, t_w = [x.to(dev) for x in synthetic_rays(RAYS, 1000 + rank)]
    ev_field = []

    def render(o, d, t, time_field=False):
        """ONE launch: fixed-stride march -> fused field -> composite + depth clip (nsb_render_forward)."""
        if time_field:
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
        out = ops.render_rays(P, o, d, t, window_hash=32.0, window_deform=7.0, sampler="fixed", n_per_ray=SAMPLES_PER_RAY,
                              near_plane=NEAR, step=STEP)
        if time_field:
            e1.record(); ev_field.append((e0, e1))
        return out

    # ---- parity: the first 64 rays of the global batch, CUDA vs CPU oracle on the same parameters (rank 0) ----
    parity = cpu = None
    if rank == 0:
        got = render(o_g[:PARITY_RAYS].to(dev), d_g[:PARITY_RAYS].to(dev), t_g[:PARITY_RAYS].to(dev))["rgb"].cpu()
        if not args.no_cpu_baseline:
            want, sec, threads, n = cpu_oracle(S, o_g[:PARITY_RAYS], d_g[:PARITY_RAYS], t_g[:PARITY_RAYS],
                                               repeats=5 if world == 1 else 1)
            l2 = (got - want).norm(dim=-1)
            mse = float(((got - want) ** 2).mean())
            parity = {"rgb_l2_max": float(l2.max()), "rgb_l2_mean": float(l2.mean()),
                      "psnr_db": (-10.0 * math.log10(mse)) if mse > 0 else float("inf"), "n_rays": PARITY_RAYS,
                      "tolerance": 1e-3, "against": "oracle/pipeline.py (fp32 on the fp16-stored tables), same parameters and rays"}
            if world == 1:
                cpu = {"value": n / sec / 1e6, "unit": "M ray-samples/s", "cores": threads, "kind": "port",
                       "sample": f"{PARITY_RAYS} rays x {SAMPLES_PER_RAY} samples ({n} samples) of the same batch, full-size tables, "
                                 "oracle/pipeline.py torch CPU fp32; 1 warm-up + median of 5"}
    ev_field.clear()

    sampler = ClockSampler(D.local_rank)
    if rank == 0:
        sampler.start(); time.sleep(0.05)

    # ---- timed region 1 (value): device-resident inputs ----
    rgb_all = torch.empty((RAYS, 3), device=dev)
    if strong:
        def step_value():
            out = render(o_s, d_s, t_s)
            D.dist.all_gather_into_tensor(rgb_all, out["rgb"])      # balanced shards: 4096 % world == 0
        assert RAYS % world == 0
        step_fn, was_graphed = graphed(step_value, dev)
    else:
        step_fn, was_graphed = (lambda: render(o_w, d_w, t_w)), False
    for _ in range(W):
        step_fn()
    ms_value, last = timed(D, step_fn, K, sampler)
    dump = {}
    if args.dump_outputs and rank == 0:     # strong scaling replays a graph: its result is the all-gathered RGB
        dump = host_arrays({"rgb": rgb_all} if strong else last)
    # fused field kernel alone (CUDA events around the launch, separate pass so that the events do not sit in the graph)
    for _ in range(2):
        render(o_s, d_s, t_s, time_field=False)
    D.barrier()
    for _ in range(min(K, 10)):
        render(o_s, d_s, t_s, time_field=True)
    D.barrier()
    field_ms = sum(a.elapsed_time(b) for a, b in ev_field) / len(ev_field)
    # weak-scaling companion number (N > 1 only): every rank its own 4096 rays, no collective
    ms_weak = None
    if strong:
        weak_fn, _ = graphed(lambda: render(o_w, d_w, t_w), dev)
        for _ in range(W):
            weak_fn()
        ms_weak, _ = timed(D, weak_fn, K)

    # ---- timed region 2 (e2e): the plugin call with HOST buffers ----
    n_loc = hi - lo
    rows = 1 << (int(math.log2(n_loc)) // 2)           # the shard as an [rows, cols] "image" for the camera-ray-bundle call
    cols = n_loc // rows
    assert rows * cols == n_loc, "ray shards are rendered as rectangular camera bundles"
    o_pin, d_pin, t_pin = o_g[lo:hi].contiguous().pin_memory(), d_g[lo:hi].contiguous().pin_memory(), t_g[lo:hi].contiguous().pin_memory()
    rgb_pin = torch.empty((n_loc, 3), dtype=torch.float32).pin_memory()
    with torch.no_grad():     # per-ray far plane = entry + 256 steps: the sampler marches exactly the config's samples
        ts0 = ops.march_fixed(o_s, d_s, aabb, 1, STEP, NEAR)[0]
    torch.cuda.synchronize()
    nears_h = ts0.cpu().reshape(n_loc, 1).pin_memory()
    fars_h = (nears_h + SAMPLES_PER_RAY * STEP).pin_memory()
    model.config.eval_num_rays_per_chunk = n_loc
    e2e_samples = torch.zeros((), dtype=torch.long, device=dev)

    def step_e2e(count=False):
        cu = lambda x: x.to(dev, non_blocking=True).view(rows, cols, -1)
        rb = RayBundle(origins=cu(o_pin), directions=cu(d_pin), pixel_area=torch.ones((rows, cols, 1), device=dev),
                       camera_indices=torch.zeros((rows, cols, 1), dtype=torch.long, device=dev),
                       nears=cu(nears_h), fars=cu(fars_h), times=cu(t_pin))
        out = model.get_outputs_for_camera_ray_bundle(rb)
        rgb = out["rgb"].view(n_loc, 3)
        if strong:
            D.dist.all_gather_into_tensor(rgb_all, rgb)
        rgb_pin.copy_(rgb, non_blocking=True)
        if count:
            e2e_samples.add_(out["num_samples_per_ray"].sum())
        return out

    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    e2e_samples.zero_()
    step_e2e(count=True)
    samples_e2e_step = int(e2e_samples.item())                  # marched by the occupancy sampler (~256 per ray)
    ms_e2e, last_e2e = timed(D, step_e2e, K, sampler)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump.update(host_arrays(last_e2e, prefix="e2e_"))
    e2e_l2 = None
    if rank == 0 and not occ:
        # the plugin path (occupancy march) and the op path (fixed march) integrate the same medium over the same span
        ref_rgb = render(o_s, d_s, t_s)["rgb"]
        e2e_l2 = float((rgb_pin.to(dev) - ref_rgb).norm(dim=-1).max())

    ms_value, ms_e2e, field_ms = D.max_ms(ms_value, ms_e2e, field_ms)
    if ms_weak is not None:
        (ms_weak,) = D.max_ms(ms_weak)
    (samples_e2e_total,) = D.sum(float(samples_e2e_step))
    if rank == 0:
        hbm_peak, peak_src = peaks()
        total = n_samples * (1 if strong or world == 1 else world)
        value = total * K / (ms_value / 1e3) / 1e6
        e2e_val = samples_e2e_total * K / (ms_e2e / 1e3) / 1e6
        field_samples = (hi - lo) * SAMPLES_PER_RAY
        achieved = ALG_BYTES_PER_SAMPLE * field_samples / (field_ms / 1e3) / 1e9
        traffic = None
        from nersemble_b200 import ops as _ops
        kname = "render_kernel_tc" if _ops.USE_TCGEN05 else "render_kernel_ws"      # NSB_TCGEN05=0 selects the mma.sync role
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and world == 1:
            traffic = json.load(open(tp)).get(f"{kname}_dram_bytes_per_launch")
        line = {
            "metric": "M ray-samples/sec", "value": value, "unit": "M ray-samples/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": ms_value / K, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f16 tables/MLP operands, f32 accumulate", "data": "synthetic",
            "config": {"workload": WORKLOAD2 + ("; seeded blob occupancy grid" if occ else ""),
                       "rays_total": RAYS if (strong or world == 1) else RAYS * world, "rays_per_gpu": hi - lo,
                       "samples_per_ray": SAMPLES_PER_RAY,
                       "parallelism": (f"rays sharded 1/{world} per GPU, per-ray RGB all-gathered (NCCL) inside the timed region"
                                       if strong else f"ray-sharded x{world} (no collective)"),
                       "cuda_graph": was_graphed,
                       "l2": "806 MB of hash tables are gathered every step (>> 126 MB L2); no explicit flush"},
            "e2e": {"value": e2e_val, "unit": "M ray-samples/s", "h2d_bytes_per_step": RAYS * 9 * 4 * (1 if strong or world == 1 else world),
                    "d2h_bytes_per_step": RAYS * 3 * 4 * (1 if strong or world == 1 else world),
                    "call": "NeRSembleNGPModel.get_outputs_for_camera_ray_bundle (occupancy sampler, nears/fars = 256 steps): "
                            "cooperative march launch + one fused field/composite launch, no host sync",
                    "samples_per_step": samples_e2e_total, "ms_per_step": ms_e2e / K, "rgb_l2_max_vs_op_path": e2e_l2},
            "gpu_launches": 1 * K,
            "roofline": {"bound": "hbm", "kernel": f"nsb::{kname}<fixed march> (march + field + composite, one launch; deformation MLP on "
                                                      + ("tcgen05/TMEM)" if _ops.USE_TCGEN05 else "mma.sync)"), "achieved": achieved,
                         "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": traffic, "kernel_ms": field_ms, "samples_per_launch": field_samples},
            "clocks": sampler.summary(),
        }
        if ms_weak is not None:
            line["weak"] = {"value": n_samples * world * K / (ms_weak / 1e3) / 1e6, "unit": "M ray-samples/s",
                            "ms_per_step": ms_weak / K, "rays_per_gpu": RAYS, "parallelism": "every rank renders its own 4096 rays, no collective"}
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
        if parity is not None and not (parity["rgb_l2_max"] < 1e-3):
            sys.stderr.write(f"parity FAILED: max per-ray RGB L2 vs the oracle = {parity['rgb_l2_max']:.3e} >= 1e-3\n")
            sys.stdout.flush(); sys.stderr.flush()
            os._exit(1)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 20; config 4: 24, every timestep's frame once)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="2", choices=["2", "2occ", "3", "4", "5"])
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ab", action="store_true", help="config 5, N > 1: also time all-reduce + full step vs the sharded optimiser in the same process")
    ap.add_argument("--no-shard", action="store_true", help="config 5: all-reduce the table gradient and step the full table on every rank")
    ap.add_argument("--overlap", action="store_true", help="config 5: issue the table-gradient all-reduce on a side stream as soon as the "
                    "gradient is parked (measured SLOWER on 2 x B200: 30.8 vs 22.9 ms per step, see DESIGN.md section 6)")
    ap.add_argument("--height", type=int, default=1088)
    ap.add_argument("--width", type=int, default=1920)
    args = ap.parse_args()
    if args.steps is None:
        args.steps = N_TIMESTEPS if args.config == "4" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    import torch
    torch.manual_seed(SEED)           # the training configs' sampler jitter: the same inputs on every run
    if args.impl == "reference":
        return run_reference(args)
    if args.config in ("2", "2occ"):
        return run_config2(args, occ=args.config == "2occ")
    from tools import bench_configs
    return {"3": bench_configs.run_config3, "4": bench_configs.run_config4, "5": bench_configs.run_config5}[args.config](args)


if __name__ == "__main__":
    main()
