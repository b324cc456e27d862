"""GPU tests on a long sequence: T = 257 timesteps (the reference recipe trains on every frame of a sequence,
n_timesteps = -1, and a NeRSemble sequence has far more than 32 frames).

Beyond 32 timesteps the rank-1 table-gradient scatter indexes a non-identity timestep -> slot map (ops._rank1_slots),
and a batch with more than 32 distinct timesteps falls back to the direct scatter with a dense table gradient.  Both
are compared with autograd through the CPU oracle here, with the timestep changing from ray to ray as in training.

With T - 1 = 256, (k + 1/2) / 256 and t * 256 are exact in fp32, so round(t (T - 1)) meets exact ties: every place
that computes the timestep must round them half to even, as torch.round does in the reference."""
import pytest
import torch

from conftest import native_from_oracle, oracle_params
from oracle import pipeline as pl
from oracle.tp import nerfacc_cpu
from oracle.tp.tcnn_cpu import Precision

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
T = 257
LONG = dict(seed=19980801, n_timesteps=T, log2_hashmap_size=14, table_scale=0.5, time_std_scale=100.0,
            deform_last_scale=1e-3)
TIE_KS = (0, 1, 2, 3, 64, 65, 200, 255)          # ties at (k + 1/2) / 256 for even and odd k


@pytest.fixture(autouse=True)
def _mode():
    Precision.mode = "kernel"; Precision.autocast = False
    yield
    Precision.mode = "reference"


@pytest.fixture(scope="module")
def long_params():
    P = oracle_params(LONG)
    return P, {"tcgen05": native_from_oracle(P, DEV, tcgen05=True), "mma.sync": native_from_oracle(P, DEV, tcgen05=False)}


def _relerr(got, want):
    return ((got - want).abs().max() / want.abs().max().clamp_min(1e-30)).item()


def _even_odd(k):
    """(even, odd) neighbour of the tie (k + 1/2) / 256: round half to even picks the even one."""
    return (k, k + 1) if k % 2 == 0 else (k + 1, k)


def _tie_rays():
    """For each tie k: three rays with the same origin and direction, at t = (k + 1/2) / 256, at the even neighbour
    k' / 256 and at the odd neighbour.  Then one ray at t = 0 and one at t = 1.  Rays aim at the box centre so that
    every ray has density along it."""
    from oracle.gen_golden import ring_rays
    n = len(TIE_KS)
    o, d, _, _ = ring_rays(n + 2, 29, spread=0.6)
    times, tie_idx, even_idx, odd_idx = [], [], [], []
    oo, dd = [], []
    for i, k in enumerate(TIE_KS):
        ev, od = _even_odd(k)
        for t in ((k + 0.5) / 256, ev / 256, od / 256):
            oo.append(o[i]); dd.append(d[i]); times.append(t)
        tie_idx.append(3 * i); even_idx.append(3 * i + 1); odd_idx.append(3 * i + 2)
    for j, t in enumerate((0.0, 1.0)):
        oo.append(o[n + j]); dd.append(d[n + j]); times.append(t)
    times = torch.tensor(times, dtype=torch.float32)[:, None]
    return torch.stack(oo), torch.stack(dd), times, torch.tensor(tie_idx), torch.tensor(even_idx), torch.tensor(odd_idx)


# ------------------------------------------------------------------------------------------------------------------
# forward
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tensor_role", ["tcgen05", "mma.sync"])
@pytest.mark.parametrize("w_hash,w_deform", [(32.0, 7.0), (1.5, 3.3)])
def test_forward_vs_oracle_random_times(long_params, tensor_role, w_hash, w_deform):
    """render_packed with an unsorted random time per ray (most rays on a different timestep of the 257) against the
    oracle, at the tolerances of the T = 4 test (test_gpu_parity.py::test_field_and_composite_vs_oracle)."""
    from nersemble_b200 import ops
    from oracle.gen_golden import ring_rays
    P, NPs = long_params
    NP = NPs[tensor_role]
    R = 40
    o, d, times, _ = ring_rays(R, 31)
    assert pl.timesteps_from_times(times, T).unique().numel() > 32
    ts, te, ri = pl.fixed_samples(o, d, P.aabb, 50, 0.011, near=0.2)
    with torch.no_grad():
        want = pl.render(P, o, d, times, ts, te, ri, window_hash=w_hash, window_deform=w_deform, training=False)
    info = nerfacc_cpu.pack_info(ri, R)
    got = ops.render_packed(NP, o.to(DEV), d.to(DEV), times.to(DEV), ts.to(DEV), te.to(DEV), ri.to(DEV), info.to(DEV),
                            window_hash=w_hash, window_deform=w_deform, training=False)
    got = {k: v.cpu() for k, v in got.items()}
    torch.testing.assert_close(got["offsets"], want["offsets"], rtol=2e-3, atol=3e-6)
    torch.testing.assert_close(got["density"], want["density"], rtol=5e-3, atol=1e-5)
    torch.testing.assert_close(got["rgb_samples"], want["rgb_samples"], rtol=0, atol=2e-3)
    torch.testing.assert_close(got["weights"], want["weights"], rtol=5e-3, atol=2e-5)
    assert (got["rgb"] - want["rgb"]).norm(dim=-1).max() < 1e-3
    torch.testing.assert_close(got["accumulation"], want["accumulation"], rtol=0, atol=1e-3)
    torch.testing.assert_close(got["depth"], want["depth"], rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(got["deformation"], want["deformation"], rtol=5e-3, atol=1e-5)


def test_rounding_ties_pick_the_even_timestep(long_params):
    """t = (k + 1/2) / 256: the oracle (torch.round), the training forward (field_forward with the training outputs)
    and the fused render (fixed march; tcgen05 and mma.sync roles) all use timestep k' = the even neighbour.  A tie ray
    must reproduce the ray at k' / 256 bit for bit, and differ from the ray at the odd neighbour by more than the
    tolerance (so the comparison can fail)."""
    from nersemble_b200 import ops
    P, NPs = long_params
    o, d, times, tie, even, odd = _tie_rays()
    R, S = o.shape[0], 50
    want_ts = torch.tensor([_even_odd(k)[0] for k in TIE_KS])
    assert torch.equal(pl.timesteps_from_times(times[tie], T), want_ts)
    assert torch.equal(pl.timesteps_from_times(times[-2:], T), torch.tensor([0, T - 1]))
    ts, te, ri = pl.fixed_samples(o, d, P.aabb, S, 0.011, near=0.2)
    with torch.no_grad():
        want = pl.render(P, o, d, times, ts, te, ri, window_hash=32.0, window_deform=7.0, training=False)
    assert torch.equal(want["rgb"][tie], want["rgb"][even])

    # training forward: per-sample outputs of a tie ray == those of its even neighbour, bit for bit
    kw = dict(origins=o.to(DEV), directions=d.to(DEV), ray_times=times.to(DEV), t_starts=ts.to(DEV), t_ends=te.to(DEV),
              ray_indices=ri.to(DEV))
    f = ops.field_forward(NPs["mma.sync"], window_hash=32.0, window_deform=7.0, use_deformation=True,
                          want=("sigma", "rgb", "offsets", "feat", "xs", "deform_acts", "corner_vals"), **kw)
    for k in ("sigma", "rgb", "offsets", "feat", "xs", "corner_vals"):
        v = f[k].cpu().reshape(R, S, -1)
        assert torch.equal(v[tie], v[even]), k
    sg = f["sigma"].cpu().reshape(R, S)
    torch.testing.assert_close(sg, want["density"][:, 0].reshape(R, S), rtol=5e-3, atol=1e-5)
    # the odd neighbour is clearly another timestep: its densities fail the oracle tolerance on every tie ray
    off = ((sg[tie] - sg[odd]).abs() - (1e-5 + 5e-3 * sg[odd].abs())).amax(dim=1)
    print("ties: max excess of |sigma(tie) - sigma(odd)| over the tolerance per ray", off.tolist())
    assert (off > 0).all()

    # fused render, both inference roles
    for role, NP in NPs.items():
        got = ops.render_rays(NP, o.to(DEV), d.to(DEV), times.to(DEV), window_hash=32.0, window_deform=7.0,
                              sampler="fixed", n_per_ray=S, near_plane=0.2, step=0.011)
        got = {k: got[k].cpu() for k in ("rgb", "accumulation", "depth", "deformation")}
        for k, v in got.items():
            assert torch.equal(v[tie], v[even]), (role, k)
        l2 = (got["rgb"] - want["rgb"]).norm(dim=-1)
        assert l2.max() < 1e-3, (role, l2.max())
        torch.testing.assert_close(got["accumulation"], want["accumulation"], rtol=0, atol=1e-3)
        torch.testing.assert_close(got["depth"], want["depth"], rtol=1e-3, atol=1e-3)
        l2_odd = (got["rgb"][tie] - got["rgb"][odd]).norm(dim=-1)
        print(f"ties ({role}): max RGB L2 vs oracle {l2.max().item():.3e}; tie vs odd neighbour L2 {l2_odd.tolist()}")
        assert (l2_odd > 1e-3).all(), (role, l2_odd)


@pytest.mark.parametrize("k", [64, 65])
def test_frame_table_at_a_tie(long_params, k):
    """uniform_time = (k + 1/2) / 256 (one camera frame at a tie): the frame table (NativeParams.frame_table) is the
    blend with the EVEN timestep's member weights, and the image agrees with the per-sample path and the oracle."""
    from nersemble_b200 import ops, packing
    P, NPs = long_params
    NP = NPs["tcgen05"]
    ev, od = _even_odd(k)
    t0 = (k + 0.5) / 256
    w_hash = 32.0
    ft = NP.frame_table(t0, w_hash, True, True).cpu()
    sc, bi = packing.blend_fold(w_hash, 32, True, True)
    tabs = NP.tables.float().cpu()

    def blended(tsi):
        return torch.einsum("emf,m->ef", tabs, P.time_emb[tsi].float() * torch.tensor(sc) + torch.tensor(bi))

    torch.testing.assert_close(ft, blended(ev), rtol=1e-5, atol=1e-6)
    assert not torch.allclose(ft, blended(od), rtol=1e-5, atol=1e-6)
    from oracle.gen_golden import ring_rays
    R = 40
    o, d, times, _ = ring_rays(R, 3)
    times = torch.full_like(times, t0)
    ts, te, ri = pl.fixed_samples(o, d, P.aabb, 50, 0.011, near=0.2)
    with torch.no_grad():
        want = pl.render(P, o, d, times, ts, te, ri, window_hash=w_hash, window_deform=7.0, training=False)
    kw = dict(origins=o.to(DEV), directions=d.to(DEV), ray_times=times.to(DEV), t_starts=ts.to(DEV), t_ends=te.to(DEV),
              ray_indices=ri.to(DEV), window_hash=w_hash, window_deform=7.0)
    per_sample = ops.field_forward(NP, **kw)
    frame = ops.field_forward(NP, uniform_time=t0, **kw)
    assert torch.equal(frame["offsets"], per_sample["offsets"])
    torch.testing.assert_close(frame["sigma"], per_sample["sigma"], rtol=5e-3, atol=1e-5)
    torch.testing.assert_close(frame["rgb"], per_sample["rgb"], rtol=0, atol=2e-3)
    torch.testing.assert_close(frame["sigma"].cpu(), want["density"][:, 0], rtol=5e-3, atol=1e-5)
    torch.testing.assert_close(frame["rgb"].cpu(), want["rgb_samples"], rtol=0, atol=2e-3)
    got = ops.render_rays(NP, o.to(DEV), d.to(DEV), times.to(DEV), window_hash=w_hash, window_deform=7.0, sampler="fixed",
                          n_per_ray=50, near_plane=0.2, step=0.011, uniform_time=t0)
    assert (got["rgb"].cpu() - want["rgb"]).norm(dim=-1).max() < 1e-3
    torch.testing.assert_close(got["accumulation"].cpu(), want["accumulation"], rtol=0, atol=1e-3)
    torch.testing.assert_close(got["depth"].cpu(), want["depth"], rtol=1e-3, atol=1e-3)


# ------------------------------------------------------------------------------------------------------------------
# backward
# ------------------------------------------------------------------------------------------------------------------
def _batch_times(regime, R, gen):
    """Per-ray times in a shuffled order.  few: 20 distinct timesteps, 6 of them reached through a tie;
    many: 48 distinct timesteps (more than the 32 slots of the rank-1 scatter)."""
    if regime == "few":
        ties = torch.tensor([(k + 0.5) / 256 for k in (10, 11, 100, 101, 254, 255)])
        rest = torch.randperm(T, generator=gen)
        rest = rest[(rest != 10) & (rest != 12) & (rest != 100) & (rest != 102) & (rest != 254) & (rest != 256)][:14]
        pool = torch.cat([ties, rest.float() / 256])
        times = pool[torch.cat([torch.arange(pool.numel()), torch.randint(0, pool.numel(), (R - pool.numel(),), generator=gen)])]
    else:
        times = torch.randperm(T, generator=gen)[:48].float() / 256
        times = times[torch.cat([torch.arange(48), torch.randint(0, 48, (R - 48,), generator=gen)])]
    return times[torch.randperm(R, generator=gen)][:, None].contiguous()


_ORACLE_BWD = {}


def _oracle_field_grads(regime):
    """Inputs and oracle autograd gradients of one batch (shared by the four scatter variants): 2048 rays x 10
    samples.  At this size the hash backward kernels give each warp a run of 3 consecutive samples, so runs cross ray
    boundaries -- and with them timesteps -- as they do in training."""
    if regime not in _ORACLE_BWD:
        from oracle.gen_golden import ring_rays
        P = pl.random_params(**LONG)
        NP = native_from_oracle(P, DEV)
        gen = torch.Generator().manual_seed(5)
        R, S = 2048, 10
        o, d, _, _ = ring_rays(R, 13)
        times = _batch_times(regime, R, gen)
        ts, te, ri = pl.fixed_samples(o, d, P.aabb, S, 0.04, near=0.2)
        tsteps = pl.timesteps_from_times(times[ri], T)
        w_hash = 20.25
        P.requires_grad_(True)
        pos = (o[ri] + d[ri] * ((ts + te)[:, None] / 2)).requires_grad_(True)
        sigma, geo = pl.field_density(P, pos, P.time_emb[tsteps], w_hash)
        rgb = pl.field_rgb(P, d[ri], geo)
        g_sigma = torch.randn((ri.numel(),), generator=gen) * 0.1
        g_rgb = torch.randn((ri.numel(), 3), generator=gen)
        ((sigma[:, 0] * g_sigma).sum() + (rgb * g_rgb).sum()).backward()
        _ORACLE_BWD[regime] = dict(P=P, NP=NP, o=o, d=d, times=times, ts=ts, te=te, ri=ri, present=torch.unique(tsteps),
                                   w_hash=w_hash, pos=pos, sigma=sigma.detach(), g_sigma=g_sigma, g_rgb=g_rgb)
    return _ORACLE_BWD[regime]


@pytest.mark.parametrize("regime", ["few", "many"])
@pytest.mark.parametrize("rank1", [True, False, "saved_corners", "deferred"])
def test_field_backward_vs_autograd_long_sequence(regime, rank1):
    """field_backward on the ray/sample inputs training uses (consecutive samples of a ray share its time, the time
    changes from ray to ray) against autograd through the oracle.  few: the rank-1 scatter through a non-identity slot
    map; many: the direct scatter with a dense table gradient, even when a deferred gradient was asked for.

    The max-norm bounds of the T = 4 test (test_gpu_backward.py::test_field_backward_vs_autograd, 700 samples) are
    loosened for d_xs, d_tables, d_base_w and d_blend_codes: a max-norm error is set by the worst of 20 480 samples,
    where a rounding of an fp16 operand lands differently.  Measured on a B200 (kernel vs oracle, few / many, identical
    for all four variants): d_xs 0.32 / 0.26, d_tables 0.12 / 0.10, d_base_w 0.026 / 0.017, d_blend_codes
    0.025 / 0.028, d_head_w 0.009 / 0.006.  The oracle's own fp16-rounding mode differs from its fp32 mode by the same
    order on these inputs (d_xs 0.13, d_tables 0.065, relative L2 error 1.5 %).  The slot-map, zero-row, touched-set
    and cosine checks are unchanged, and a timestep mix-up moves whole rows of the gradient, far outside these bounds."""
    cv = rank1 in ("saved_corners", "deferred")
    deferred = rank1 == "deferred"
    rank1 = bool(rank1)
    from nersemble_b200 import ops
    c = _oracle_field_grads(regime)
    P, NP, o, d, times, ts, te, ri = (c[k] for k in ("P", "NP", "o", "d", "times", "ts", "te", "ri"))
    present, w_hash, pos, sigma, g_sigma, g_rgb = (c[k] for k in ("present", "w_hash", "pos", "sigma", "g_sigma", "g_rgb"))
    assert (present.numel() <= 32) == (regime == "few")
    kw = dict(origins=o.to(DEV), directions=d.to(DEV), ray_times=times.to(DEV), t_starts=ts.to(DEV), t_ends=te.to(DEV),
              ray_indices=ri.to(DEV))
    # the path: a slot per timestep present (in increasing order), or no rank-1 scatter at all
    slot, n_slots = ops._rank1_slots(NP, DEV, kw)
    if regime == "few":
        want_slot = torch.full((T,), -1, dtype=torch.int32)
        want_slot[present] = torch.arange(present.numel(), dtype=torch.int32)
        assert n_slots == present.numel() and torch.equal(slot.cpu(), want_slot)
        assert not torch.equal(present, torch.arange(present.numel()))             # not the identity
    else:
        assert slot is None and n_slots == 0
    saved = ops.field_forward(NP, window_hash=w_hash, use_deformation=False,
                              want=("sigma", "rgb", "feat", "xs") + (("corner_vals",) if cv else ()), **kw)
    torch.testing.assert_close(saved["sigma"].cpu(), sigma[:, 0], rtol=5e-3, atol=1e-5)
    grads = ops.field_backward(NP, saved, g_sigma.to(DEV), g_rgb.to(DEV), window_hash=w_hash, loss_scale=128.0, want_dx=True,
                               rank1=rank1, defer_tables=deferred, **kw)
    if deferred and regime == "few":
        assert "d_tables" not in grads
        pend = grads["pending"]
        assert pend["n_slots"] == present.numel() and pend["slots_are_timesteps"] is False
        grads["d_tables"] = ops.rank1_expand(pend, P.tables.shape[0])
    else:
        assert "pending" not in grads and grads["d_tables"].shape == P.tables.shape
    lo, hi = P.aabb[0], P.aabb[1]
    dpos = grads["d_xs"].cpu() / (hi - lo)
    errs = {"d_xs": _relerr(dpos, pos.grad)}
    assert (dpos[saved["xs"].cpu()[:, 3] == 0] == 0).all()
    gb = torch.cat([w.grad.reshape(-1) for w in P.base_w]); gh = torch.cat([w.grad.reshape(-1) for w in P.head_w])
    errs["d_head_w"] = _relerr(grads["d_head_w"].cpu(), gh)
    errs["d_base_w"] = _relerr(grads["d_base_w"].cpu(), gb)
    dc = grads["d_blend_codes"].cpu()
    errs["d_blend_codes"] = _relerr(dc, P.time_emb.grad)
    dt = grads["d_tables"].cpu()
    errs["d_tables"] = _relerr(dt, P.tables.grad)
    touched = ((dt != 0) == (P.tables.grad != 0)).float().mean().item()
    cos = torch.nn.functional.cosine_similarity(dt.double().reshape(1, -1), P.tables.grad.double().reshape(1, -1)).item()
    print(f"field_backward T=257 rank1={rank1} cv={cv} deferred={deferred} {regime}: {errs} touched {touched} cos {cos}")
    assert errs["d_xs"] < 0.45
    assert errs["d_head_w"] < 2e-2 and errs["d_base_w"] < 4e-2
    assert errs["d_blend_codes"] < 4e-2
    absent = torch.ones(T, dtype=torch.bool); absent[present] = False
    assert (dc[absent] == 0).all()                                   # codes of timesteps absent from the batch: exactly 0
    assert (dc[present].abs().amax(dim=1) > 0).all()
    assert errs["d_tables"] < 0.16
    assert touched > 0.999
    assert cos > 0.9995, cos


def test_deform_backward_vs_autograd_long_sequence():
    """The SE(3) deformation backward with a random timestep per sample (unsorted, half of them at ties), so the
    timestep changes inside nearly every warp: the warp-code gradient takes its per-row branch.  Bounds of the T = 4
    test (test_gpu_backward.py::test_deform_backward_vs_autograd)."""
    from nersemble_b200 import ops
    P = pl.random_params(**dict(LONG, deform_last_scale=0.05))
    NP = native_from_oracle(P, DEV)
    g = torch.Generator().manual_seed(9)
    n = 999
    lo, hi = P.aabb[0], P.aabb[1]
    pos = lo + (torch.rand((n, 3), generator=g) * 0.9 + 0.05) * (hi - lo)
    k = torch.randint(0, T - 1, (n,), generator=g)
    times = torch.where(torch.rand((n,), generator=g) < 0.5, (k.float() + 0.5) / 256, k.float() / 256)[:, None]
    tsteps = pl.timesteps_from_times(times, T)
    present = torch.unique(tsteps)
    w_deform = 5.5
    P.requires_grad_(True)
    off = pl.compute_offsets(P, pos, P.time_emb_deform[tsteps], w_deform)
    g_off = torch.randn((n, 3), generator=g)
    (off * g_off).sum().backward()

    kw = dict(positions=pos.to(DEV), sample_times=times.to(DEV))
    saved = ops.field_forward(NP, window_hash=None, window_deform=w_deform, use_deformation=True,
                              want=("offsets", "deform_acts"), **kw)
    torch.testing.assert_close(saved["offsets"].cpu(), off.detach(), rtol=5e-3, atol=5e-5)
    d_xs = (g_off * (hi - lo)).to(DEV)
    gr = ops.deform_backward(NP, saved, d_xs, window_deform=w_deform, loss_scale=64.0, **kw)
    errs = {}
    for l in range(6):
        errs[f"d_stem_w{l}"] = _relerr(gr["d_stem_w"][l].cpu(), P.deform_w[l].grad)
        errs[f"d_stem_b{l}"] = _relerr(gr["d_stem_b"][l].cpu(), P.deform_b[l].grad)
    for name, ref in (("d_r_w", P.r_w), ("d_v_w", P.v_w), ("d_r_b", P.r_b), ("d_v_b", P.v_b)):
        errs[name] = _relerr(gr[name].cpu(), ref.grad)
    dw = gr["d_warp_codes"].cpu()
    errs["d_warp_codes"] = _relerr(dw, P.time_emb_deform.grad)
    print("deform_backward T=257:", errs)
    for l in range(6):
        assert errs[f"d_stem_w{l}"] < 4e-2 and errs[f"d_stem_b{l}"] < 4e-2, l
    assert max(errs[k] for k in ("d_r_w", "d_v_w", "d_r_b", "d_v_b")) < 3e-2
    assert errs["d_warp_codes"] < 4e-2
    absent = torch.ones(T, dtype=torch.bool); absent[present] = False
    assert absent.any() and (dw[absent] == 0).all()
    assert (dw[present].abs().amax(dim=1) > 0).all()


# ------------------------------------------------------------------------------------------------------------------
# model + optimiser
# ------------------------------------------------------------------------------------------------------------------
def _model_times(regime, it):
    gen = torch.Generator().manual_seed(100 + it)
    return _batch_times(regime, 64, gen)


def _make_long_model():
    from test_plugin_cpu import make_model
    from oracle.gen_golden import blob_grid
    torch.manual_seed(0)
    m = make_model(T=T, log2T=14, lambda_near_loss=0, lambda_empty_loss=0, lambda_depth_loss=0).to(DEV).train()
    with torch.no_grad():
        m.field.hash_ensemble.tables.uniform_(-0.5, 0.5)
        m.time_embedding.weight.normal_(0, 0.18)
    occ = blob_grid(3)
    m.occupancy_grid.binaries[0] = occ.to(DEV)
    m.occupancy_grid.occs.copy_((occ.flatten().float() * 0.05).to(DEV))
    m.sampler.eval()
    return m


def _bundle(regime, it):
    from oracle.gen_golden import ring_rays
    from nersemble_b200.nerfstudio_shim import RayBundle
    o, d, _, cams = ring_rays(64, 21 + it)
    gen = torch.Generator().manual_seed(it)
    batch = {"image": torch.rand((64, 3), generator=gen), "alpha_map": torch.randint(0, 256, (64, 1), generator=gen).float()}
    rb = RayBundle(origins=o.to(DEV), directions=d.to(DEV), pixel_area=torch.ones(64, 1, device=DEV),
                   camera_indices=cams.to(DEV), times=_model_times(regime, it).to(DEV))
    return rb, batch


@pytest.mark.parametrize("regime", ["few", "many"])
def test_fused_fields_adam_tracks_torch_adam_long_sequence(regime):
    """test_gpu_optim.py::test_fused_fields_adam_tracks_torch_adam_on_the_model with 257 timesteps.  few: the backward
    parks a rank-1 gradient whose slots are NOT timesteps; many: it cannot, and leaves a dense tables.grad, which
    FusedFieldsAdam steps with its dense branch."""
    from nersemble_b200.optim import FusedFieldsAdam

    def run(fused):
        m = _make_long_model()
        he = m.field.hash_ensemble
        t0 = he.tables.detach().clone()
        groups = m.get_param_groups()
        fields = (FusedFieldsAdam if fused else torch.optim.Adam)(groups["fields"], lr=5e-3, eps=1e-8)
        rest = torch.optim.Adam(groups["embeddings"], lr=5e-3, eps=1e-8)
        losses = []
        for it in range(3):
            rb, batch = _bundle(regime, it)
            fields.zero_grad(); rest.zero_grad()
            loss = sum(m.get_loss_dict(m.get_outputs(rb), batch).values())
            loss.backward()
            if fused and regime == "few":
                assert he.tables.grad is None and he.pending_table_grad is not None
                assert he.pending_table_grad["slots_are_timesteps"] is False
            elif fused:
                assert he.pending_table_grad is None
                assert he.tables.grad is not None and he.tables.grad.shape == he.tables.shape
                assert he.tables.grad.abs().max().item() > 0
            fields.step(); rest.step()
            losses.append(loss.item())
        assert torch.equal(he.native_tables(), he.tables.detach().half())
        return losses, he.tables.detach() - t0, m.field.mlp_base.params.detach().clone()

    l_f, t_f, b_f = run(True)
    l_t, t_t, b_t = run(False)
    for a, b in zip(l_f, l_t):
        assert abs(a - b) < 1e-4 * abs(b) + 1e-6, (l_f, l_t)
    cos = torch.nn.functional.cosine_similarity(t_f.reshape(1, -1), t_t.reshape(1, -1)).item()
    print(f"model T=257 {regime}: losses {l_f} vs {l_t}; table update cos {cos}; "
          f"mlp_base max diff {(b_f - b_t).abs().max().item():.3e}")
    assert cos > 0.995, cos
    assert (t_f != 0).float().mean().item() > 0.01
    assert (b_f - b_t).abs().max().item() < 5e-3 * 0.05


def test_grad_scaler_skips_a_non_finite_dense_table_gradient():
    """More than 32 timesteps in the batch: the table gradient is a dense tables.grad (no parked gradient, no NaN flag
    folded into mlp_base's gradient), so GradScaler's own inf check must see it.  A non-finite entry skips the whole
    step -- table, fp16 copy, every other parameter untouched -- and halves the scale."""
    from nersemble_b200.optim import FusedFieldsAdam
    m = _make_long_model()
    he = m.field.hash_ensemble
    groups = m.get_param_groups()
    fields = FusedFieldsAdam(groups["fields"], lr=5e-3, eps=1e-15)
    scaler = torch.amp.GradScaler("cuda", init_scale=1024.0)
    rb, batch = _bundle("many", 0)
    loss = sum(m.get_loss_dict(m.get_outputs(rb), batch).values())
    scaler.scale(loss).backward()
    assert he.pending_table_grad is None and he.tables.grad is not None
    assert all(torch.isfinite(p.grad).all() for p in groups["fields"] if p.grad is not None)
    he.tables.grad[he.tables.shape[0] // 2, 7, 1] = float("inf")
    before = [p.detach().clone() for p in groups["fields"]]
    half0 = he.native_tables().clone()
    scaler.step(fields); scaler.update()
    assert fields.last_step_skipped
    assert all(torch.equal(p.detach(), b) for p, b in zip(groups["fields"], before))
    assert torch.equal(he.native_tables(), half0)
    assert len(fields.state[he.tables]) == 0 and scaler.get_scale() == 512.0
