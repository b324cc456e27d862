"""bench.py --config 3 | 4 | 5: the BASELINE.json configurations beyond the headline forward (configs[2..4]).

  3  train_nersemble.py seq-30 default hparams, 1 x B200: one optimiser step = jittered occupancy march + visibility
     pre-pass (alpha_thre 1e-2) -> differentiable fused render -> six losses -> backward -> FusedFieldsAdam (fields) +
     Adam (embeddings, deformation field).  Synthetic multi-view batch (image, alpha map, depth map per ray).
  4  novel-view frames (default 1088 x 1920, T = 24), rays of every frame sharded 1/N per GPU, per-ray RGB all-gathered
     (NCCL) inside the timed region; through NeRSembleNGPModel.get_outputs_for_camera_ray_bundle.
  5  seq-97 recipe: --disable_occupancy_grid (dense march through the box) --lambda_dist_loss 0, 4096 rays per GPU, full
     gradient step on N GPUs with the gradient all-reduce INSIDE the timed region (data parallel: weak scaling).

Every function prints ONE JSON line on rank 0 with the bench.py contract's keys."""
from __future__ import annotations

import json
import math
import os
import sys
import time

import bench as B

SEQ97_AABB = ((-2.2, -2.8, -2.5), (2.2, 2.2, 2.0))     # train_nersemble.py:45


def _optimizers(model, fused=True):
    """One optimiser per parameter group like nerfstudio's Optimizers (train_nersemble.py:243-256: Adam eps 1e-15,
    fields 5e-3, embeddings 5e-3, deformation field 1e-3)."""
    import torch
    from nersemble_b200.optim import FusedFieldsAdam
    groups = model.get_param_groups()
    F = FusedFieldsAdam if fused else torch.optim.Adam
    opts = [F(groups["fields"], lr=5e-3, eps=1e-15), torch.optim.Adam(groups["embeddings"], lr=5e-3, eps=1e-15),
            torch.optim.Adam([p for p in groups["deformation_field"] if p.requires_grad], lr=1e-3, eps=1e-15)]
    return opts, [p for g in groups.values() for p in g]


def _train_batch(dev, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    return {"image": torch.rand((B.RAYS, 3), generator=g).to(dev),
            "alpha_map": torch.randint(0, 256, (B.RAYS, 1), generator=g).float().to(dev),
            "depth_maps": ((torch.rand(B.RAYS, generator=g) * 4 + 7) * (torch.rand(B.RAYS, generator=g) > 0.2)).to(dev)}


def _train_loop(args, D, model, opts, params, batch, rb, with_allreduce, reduce_pending=True):
    """W warm-up + K timed optimiser steps; per-phase CUDA-event times of the timed steps (ms, this rank)."""
    import torch
    from nersemble_b200.distributed import allreduce_gradients
    HE = [model.field.hash_ensemble]
    W, K = max(args.warmup, 3), args.steps
    phases = {k: 0.0 for k in ("forward", "losses", "backward", "allreduce", "optimizer")}
    host = {k: 0.0 for k in phases}          # host time to ENQUEUE each phase (no synchronisation inside the loop except the sampler's)
    marks, hmarks = [], []

    def ev():
        e = torch.cuda.Event(enable_timing=True); e.record(); return e

    def step(record):
        e = [ev()]; h = [time.perf_counter()]
        for o in opts:
            o.zero_grad(set_to_none=True)
        out = model.get_outputs(rb); e.append(ev()); h.append(time.perf_counter())
        loss = sum(model.get_loss_dict(out, batch).values()); e.append(ev()); h.append(time.perf_counter())
        loss.backward(); e.append(ev()); h.append(time.perf_counter())
        if with_allreduce:
            allreduce_gradients(params, hash_ensembles=HE, reduce_pending=reduce_pending)
        e.append(ev()); h.append(time.perf_counter())
        for o in opts:
            o.step()
        e.append(ev()); h.append(time.perf_counter())
        if record:
            marks.append(e); hmarks.append(h)
        return out, loss

    for _ in range(W):
        out, loss = step(False)
    sampler = B.ClockSampler(D.local_rank)
    if D.rank == 0:
        sampler.start(); time.sleep(0.05)
    n_samples = torch.zeros((), dtype=torch.long, device=D.dev)

    def timed_step():
        out, loss = step(True)
        n_samples.add_(out["num_samples_per_ray"].sum())
        return out, loss
    ms, (last_out, last_loss) = B.timed(D, timed_step, K, sampler)
    sampler.stop_flag = True
    if args.dump_outputs and D.rank == 0:
        B.dump_outputs(args.dump_outputs, B.host_arrays({**last_out, "loss": last_loss}))
    for e, h in zip(marks, hmarks):
        for i, k in enumerate(phases):
            phases[k] += e[i].elapsed_time(e[i + 1]) / len(marks)
            host[k] += (h[i + 1] - h[i]) * 1e3 / len(marks)
    phases["host_enqueue"] = host
    return ms, int(n_samples.item()), phases, float(loss.detach()), sampler


def run_config3(args, config5=False):
    import torch
    from nersemble_b200.nerfstudio_shim import RayBundle
    D = B.Dist(args.gpus)
    dev, rank, world = D.dev, D.rank, D.world
    if not config5 and world != 1:
        raise SystemExit("config 3 is the single-GPU training step; use --config 5 for the multi-GPU gradient step")
    K = args.steps
    S = B.synthetic_params()
    if config5:
        S["aabb"] = torch.tensor(SEQ97_AABB)
        model = B.build_model(S, dev, disable_occupancy_grid=True, lambda_dist_loss=0.0).train()
        model.occupancy_grid.binaries[:] = True               # what the first occupancy update yields for density == 1
        model.occupancy_grid.occs.fill_(1.0 * B.STEP)
    else:
        model = B.build_model(S, dev).train()
        occ = B.blob_occupancy(seed=5)
        model.occupancy_grid.binaries[0] = occ.to(dev)
        model.occupancy_grid.occs.copy_((occ.flatten().float() * 0.05).to(dev))
    opts, params = _optimizers(model)
    shard = world > 1 and not args.no_shard and not args.overlap
    opts[0].shard_tables = shard              # reduce-scatter -> Adam on 1/N of the entries -> all-gather of the fp16 table
    if world > 1 and args.overlap:
        from nersemble_b200.distributed import overlap_table_allreduce
        overlap_table_allreduce(model.field.hash_ensemble)        # table-gradient all-reduce overlaps the deformation backward
    o, d, t = B.synthetic_rays(B.RAYS, 1000 + rank, dev)
    rb = RayBundle(origins=o, directions=d, pixel_area=torch.ones(B.RAYS, 1, device=dev),
                   camera_indices=torch.zeros(B.RAYS, 1, dtype=torch.long, device=dev), times=t)
    batch = _train_batch(dev, 7 + rank)
    variants = {}
    if world > 1 and args.ab:
        # in-process A/B (box-to-box variance of the host side is larger than the effect): blocking all-reduce + full
        # table step on every rank, then the sharded optimiser; both on the same model state, same batches
        for tag, sh in (("allreduce_full_step", False), ("sharded_optimiser", True)):
            opts[0].shard_tables = sh
            if not sh:
                opts[0].consolidate()
            v_ms, v_n, v_ph, _, _ = _train_loop(args, D, model, opts, params, batch, rb, with_allreduce=True, reduce_pending=not sh)
            v_ph.pop("host_enqueue")
            (v_ms,) = D.max_ms(v_ms)
            variants[tag] = {"ms_per_step": v_ms / K, "phases_ms": dict(zip(v_ph.keys(), D.max_ms(*v_ph.values())))}
        opts[0].shard_tables = shard
    ms, n_samples, phases, loss, sampler = _train_loop(args, D, model, opts, params, batch, rb, with_allreduce=world > 1,
                                                       reduce_pending=not shard)
    (ms,) = D.max_ms(ms)
    (tot_samples,) = D.sum(float(n_samples))
    host = phases.pop("host_enqueue")
    ph = D.max_ms(*phases.values())
    if rank == 0:
        name = ("config5: seq-97 recipe, --disable_occupancy_grid dense march, lambda_dist 0, 4096 rays per GPU, full gradient step"
                if config5 else "config3: seq-30 default hparams training step (jittered occupancy march + visibility pre-pass, "
                "six losses, backward, FusedFieldsAdam), 4096 rays")
        line = {"metric": "M ray-samples/sec", "value": tot_samples / (ms / 1e3) / 1e6, "unit": "M ray-samples/s",
                "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms / K,
                "it_per_s": K / (ms / 1e3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16 tables/MLP operands, f32 accumulate / master / Adam", "data": "synthetic",
                "config": {"workload": name, "rays_per_gpu": B.RAYS, "samples_per_step_per_gpu": n_samples / K,
                           "parallelism": (f"data parallel x{world}: NCCL "
                                           + ("reduce-scatter of the table gradient -> Adam on 1/N of the entries -> all-gather of the fp16 table; all-reduce of the MLP / embedding gradients"
                                              if shard else "all-reduce of all gradients") + ", every step inside the timed region"
                                           + ("; the 1.2 GB table-gradient reduction is issued on a side stream during the backward" if args.overlap else "")
                                           if world > 1 else "single GPU"),
                           "tables": "32 x (16 levels, 2^19) fp32 master + fp16 shadow", "n_timesteps": B.N_TIMESTEPS},
                "phases_ms": dict(zip(phases.keys(), ph)), "host_enqueue_ms": host, "loss": loss, "clocks": sampler.summary(),
                "gpu_launches": None}
        if variants:
            line["ab_same_process"] = variants
        print(json.dumps(line), flush=True)
    D.close()


def run_config5(args):
    return run_config3(args, config5=True)


def run_config4(args):
    import torch
    from nersemble_b200.distributed import shard_bounds
    from nersemble_b200.nerfstudio_shim import RayBundle
    D = B.Dist(args.gpus)
    dev, rank, world = D.dev, D.rank, D.world
    H, Wd, T = args.height, args.width, B.N_TIMESTEPS
    n_frames = T
    S = B.synthetic_params()
    model = B.build_model(S, dev, eval_num_rays_per_chunk=1 << 19).eval()
    ax = (torch.arange(128, device=dev).float() + 0.5) / 128
    X, Y, Z = torch.meshgrid(ax, ax, ax, indexing="ij")
    model.occupancy_grid.binaries[0] = ((X - 0.5) ** 2 + (Y - 0.5) ** 2 + (Z - 0.5) ** 2) < 0.33 ** 2   # a head-sized blob
    assert H % world == 0, "frames are sharded by rows"
    rows = H // world
    # rows are dealt out round-robin (row r -> rank r % N), not in contiguous blocks: the head sits in the middle of the
    # frame, and with contiguous blocks the central ranks marched 4x the samples of the outer ones (r2m: 8 GPUs only 2.85x)
    from nersemble_b200.distributed import gather_rows_round_robin, shard_rows_round_robin
    my_rows = shard_rows_round_robin(H, rank, world, device=dev)

    def camera_rays(frame, row_idx=None):
        row_idx = my_rows if row_idx is None else row_idx
        n_rows = int(row_idx.shape[0])
        ang = torch.tensor(2 * torch.pi * frame / n_frames)
        o = torch.tensor([9.0 * torch.sin(ang), 0.0, 9.0 * torch.cos(ang)], device=dev)
        fwd = -o / o.norm()
        right = torch.linalg.cross(fwd, torch.tensor([0.0, 1.0, 0.0], device=dev)); right = right / right.norm()
        up = torch.linalg.cross(right, fwd)
        ys, xs = torch.meshgrid(torch.linspace(0.25, -0.25, H, device=dev)[row_idx],
                                torch.linspace(-0.25 * Wd / H, 0.25 * Wd / H, Wd, device=dev), indexing="ij")
        d = fwd[None, None] + xs[..., None] * right + ys[..., None] * up
        d = d / d.norm(dim=-1, keepdim=True)
        return RayBundle(origins=o.expand(n_rows, Wd, 3).contiguous(), directions=d.contiguous(),
                         pixel_area=torch.ones((n_rows, Wd, 1), device=dev),
                         camera_indices=torch.zeros((n_rows, Wd, 1), dtype=torch.long, device=dev),
                         times=torch.full((n_rows, Wd, 1), frame / max(T - 1, 1), device=dev))

    gather_buf = torch.empty((world, rows, Wd, 3), device=dev)
    frame_buf = torch.empty((H, Wd, 3), device=dev)
    n_samples = torch.zeros((), dtype=torch.long, device=dev)
    state = {"f": 0}

    def render_frame():
        rb = camera_rays(state["f"] % n_frames)
        out = model.get_outputs_for_camera_ray_bundle(rb)
        gather_rows_round_robin(out["rgb"], out=frame_buf, scratch=gather_buf)      # NCCL all-gather + one strided copy
        n_samples.add_(out["num_samples_per_ray"].sum())
        state["f"] += 1
        return out

    with torch.no_grad():
        render_frame(); render_frame()
        n_samples.zero_(); state["f"] = 0
        sampler = B.ClockSampler(D.local_rank)
        if rank == 0:
            sampler.start(); time.sleep(0.05)
        K = args.steps
        ms, last = B.timed(D, render_frame, K, sampler)
        sampler.stop_flag = True
        if args.dump_outputs and rank == 0:     # the gathered frame, and this rank's rows of the other outputs
            B.dump_outputs(args.dump_outputs, B.host_arrays({**last, "rgb": frame_buf}))
        # sharded vs unsharded: the last frame again on rank 0 alone (chunk boundaries differ, pixels must not)
        max_diff = None
        if rank == 0 and world > 1:
            rb = camera_rays((state["f"] - 1) % n_frames, row_idx=torch.arange(H, device=dev))
            full = model.get_outputs_for_camera_ray_bundle(rb)["rgb"]
            max_diff = float((full - frame_buf).abs().max())
    (ms,) = D.max_ms(ms)
    (tot,) = D.sum(float(n_samples.item()))
    if rank == 0:
        line = {"metric": "M ray-samples/sec", "value": tot / (ms / 1e3) / 1e6, "unit": "M ray-samples/s", "n_gpus": world,
                "steps": K, "warmup": 2, "ms_per_step": ms / K, "frames_per_s": K / (ms / 1e3), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16 tables/MLP operands, f32 accumulate", "data": "synthetic",
                "config": {"workload": f"config4: {H}x{Wd} novel-view frames, T={T} timesteps (one frame per step), eval mode, "
                                       "head-sized occupancy blob", "rays_per_frame": H * Wd, "samples_per_frame": tot / K,
                           "parallelism": f"rows dealt round-robin to {world} GPU(s), RGB all-gathered (NCCL) per frame inside the timed region",
                           "eval_num_rays_per_chunk": model.config.eval_num_rays_per_chunk},
                "max_abs_rgb_diff_vs_unsharded": max_diff, "clocks": sampler.summary(), "gpu_launches": None}
        print(json.dumps(line), flush=True)
    D.close()
