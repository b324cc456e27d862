"""The backward and the table optimiser AT THE BENCHMARKED TABLE SIZE (log2_hashmap_size = 19, T = 24: the `FULL`
knobs of test_gpu_fullsize.py, which the training benchmarks run).  At this size levels 0-4 are dense, the level
offsets reach 6.3 M lines, the resolution-4096 level wraps the 32-bit hash, and the 6 299 960-line table ends 24 lines
into a 32-line block of the expansion and optimiser kernels.  The backward kernels compute the corner indices in
copies of their own, so they are checked here against autograd through the CPU oracle."""
import pytest
import torch

from conftest import native_from_oracle, oracle_params
from oracle import pipeline as pl
from oracle.tp.tcnn_cpu import Precision

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FULL = dict(seed=19980801, n_timesteps=24, log2_hashmap_size=19, table_scale=0.5, time_std_scale=100.0,
            deform_last_scale=1e-3)


@pytest.fixture(autouse=True)
def _mode():
    Precision.mode = "kernel"; Precision.autocast = False
    yield
    Precision.mode = "reference"


def _relerr(got, want):
    return ((got - want).abs().max() / want.abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def full_case():
    """2048 samples over the box: uniform ones, points within 1e-4 of each of the six faces, points just below x = 1
    (where the resolution-4096 level's hash wraps) and a few outside the box; random unsorted timesteps.  The oracle's
    gradients are computed once for the four scatter variants."""
    P0 = oracle_params(FULL)
    NP = native_from_oracle(P0, DEV)
    # fresh leaves that share the cached parameters' storage: gradients land on these only
    P = pl.FieldParams(P0.aabb, P0.tables.detach(), [w.detach() for w in P0.base_w], [w.detach() for w in P0.head_w],
                       P0.deform_w, P0.deform_b, P0.r_w, P0.r_b, P0.v_w, P0.v_b, P0.time_emb.detach(),
                       P0.time_emb_deform, P0.levels)
    g = torch.Generator().manual_seed(23)
    n = 2048
    u = torch.rand((n, 3), generator=g) * 0.998 + 0.001
    eps = torch.rand((96, 6), generator=g) * 1e-4
    for f in range(6):                                              # 96 points within 1e-4 of each face
        rows = slice(96 * f, 96 * (f + 1))
        u[rows, f % 3] = eps[:, f] if f < 3 else 1.0 - eps[:, f]
    u[576:704, 0] = 1.0 - torch.rand((128,), generator=g) * 2e-3    # x just below 1: the top level's last cells
    u[704:720] = u[704:720] * 1.2 - 0.1                             # some outside the box
    lo, hi = P.aabb[0], P.aabb[1]
    pos = lo + u * (hi - lo)
    dirs = torch.randn((n, 3), generator=g); dirs = dirs / dirs.norm(dim=-1, keepdim=True)
    tsteps = torch.randint(0, 24, (n,), generator=g)
    times = tsteps.float()[:, None] / 23
    assert torch.equal(pl.timesteps_from_times(times, 24), tsteps)
    w_hash = 20.25
    for t in [P.tables, P.time_emb] + P.base_w + P.head_w:
        t.requires_grad_(True)
    pos = pos.requires_grad_(True)
    sigma, geo = pl.field_density(P, pos, P.time_emb[tsteps], w_hash)
    rgb = pl.field_rgb(P, dirs, geo)
    g_sigma = torch.randn((n,), generator=g) * 0.1
    g_rgb = torch.randn((n, 3), generator=g)
    ((sigma[:, 0] * g_sigma).sum() + (rgb * g_rgb).sum()).backward()
    yield dict(P=P, NP=NP, pos=pos, dirs=dirs, times=times, w_hash=w_hash, sigma=sigma.detach(), g_sigma=g_sigma, g_rgb=g_rgb)
    torch.cuda.empty_cache()


def _kernel_grads(c, rank1, deferred=False, cv=False):
    from nersemble_b200 import ops
    kw = dict(positions=c["pos"].detach().to(DEV), sample_times=c["times"].to(DEV), sample_directions=c["dirs"].to(DEV))
    saved = ops.field_forward(c["NP"], window_hash=c["w_hash"], use_deformation=False,
                              want=("sigma", "rgb", "feat", "xs") + (("corner_vals",) if cv else ()), **kw)
    grads = ops.field_backward(c["NP"], saved, c["g_sigma"].to(DEV), c["g_rgb"].to(DEV), window_hash=c["w_hash"],
                               loss_scale=128.0, want_dx=True, rank1=rank1, defer_tables=deferred, **kw)
    return saved, grads


@pytest.mark.parametrize("rank1", [True, False, "saved_corners", "deferred"])
def test_full_size_field_backward_vs_autograd(full_case, rank1):
    """Table, time-code and position gradients at 2^19 against the oracle.  The table gradient is compared over table
    LINES (32 members x 2 features): relative error over the lines the oracle touched, agreement of the touched sets
    over every line either side touched, and the cosine over the whole table.

    Bounds: those of the 2^14 test (test_gpu_backward.py::test_field_backward_vs_autograd) except the max-norm errors
    of d_xs, d_base_w, d_blend_codes and d_tables.  Measured on a B200 (all four variants alike): d_xs 0.088,
    d_base_w 0.052, d_blend_codes 0.026, d_tables 0.096, d_head_w 0.008; every line and every entry touched on one
    side is touched on the other.  The oracle's own fp16-rounding mode differs from its fp32 mode by the same order
    on these inputs (d_xs 0.067, d_base_w 0.024, d_blend_codes 0.030, d_tables 0.119): a max-norm error is set by
    the one sample where an fp16 rounding lands differently."""
    from nersemble_b200 import ops
    c = full_case
    P = c["P"]
    cv = rank1 in ("saved_corners", "deferred")
    deferred = rank1 == "deferred"
    saved, grads = _kernel_grads(c, bool(rank1), deferred, cv)
    torch.testing.assert_close(saved["sigma"].cpu(), c["sigma"][:, 0], rtol=5e-3, atol=1e-5)
    outside = saved["xs"].cpu()[:, 3] == 0
    if deferred:
        assert "d_tables" not in grads and grads["pending"]["slots_are_timesteps"] is True
        grads["d_tables"] = ops.rank1_expand(grads["pending"], P.tables.shape[0])
    del saved
    lo, hi = P.aabb[0], P.aabb[1]
    dpos = grads["d_xs"].cpu() / (hi - lo)
    errs = {"d_xs": _relerr(dpos, c["pos"].grad), "d_blend_codes": _relerr(grads["d_blend_codes"].cpu(), P.time_emb.grad)}
    gb = torch.cat([w.grad.reshape(-1) for w in P.base_w]); gh = torch.cat([w.grad.reshape(-1) for w in P.head_w])
    errs["d_head_w"] = _relerr(grads["d_head_w"].cpu(), gh)
    errs["d_base_w"] = _relerr(grads["d_base_w"].cpu(), gb)
    dt = grads.pop("d_tables").cpu()
    ref = P.tables.grad
    line_t, line_r = (dt != 0).any(-1).any(-1), (ref != 0).any(-1).any(-1)
    errs["d_tables"] = _relerr(dt[line_r], ref[line_r])
    either = line_t | line_r
    touched = (line_t[either] == line_r[either]).float().mean().item()
    elem = ((dt[either] != 0) == (ref[either] != 0)).float().mean().item()
    cos = torch.nn.functional.cosine_similarity(dt.double().reshape(1, -1), ref.double().reshape(1, -1)).item()
    print(f"full-size field_backward rank1={rank1}: {errs}; lines touched {int(line_r.sum())}, line agreement {touched}, "
          f"element agreement on those lines {elem}, cos {cos}")
    assert errs["d_xs"] < 0.13
    assert outside.sum() > 0 and (dpos[outside] == 0).all()
    assert errs["d_head_w"] < 2e-2 and errs["d_base_w"] < 0.08
    assert errs["d_blend_codes"] < 4e-2
    assert errs["d_tables"] < 0.14
    assert touched > 0.999 and elem > 0.999
    assert cos > 0.9995, cos


def test_full_size_rank1_expand_matches_direct_scatter(full_case):
    """The deferred rank-1 gradient, expanded by nsb_rank1_expand, equals the direct scatter's dense gradient from the
    same inputs up to the order of the float sums."""
    from nersemble_b200 import ops
    c = full_case
    _, direct = _kernel_grads(c, rank1=False)
    _, deferred = _kernel_grads(c, rank1=True, deferred=True, cv=True)
    E = c["P"].tables.shape[0]
    dense = ops.rank1_expand(deferred["pending"], E)
    scale = direct["d_tables"].abs().max().item()
    err = (dense - direct["d_tables"]).abs().max().item()
    print(f"full-size rank1_expand vs direct scatter: max abs diff {err:.3e} (max |g| {scale:.3e})")
    assert err <= 1e-5 * scale, (err, scale)
    assert ((dense != 0) == (direct["d_tables"] != 0)).float().mean().item() > 0.9999
    torch.testing.assert_close(deferred["d_blend_codes"], direct["d_blend_codes"], rtol=1e-4, atol=1e-6 * deferred["d_blend_codes"].abs().max().item())
    del dense, direct, deferred
    torch.cuda.empty_cache()


def test_full_size_table_adam_step_matches_torch_adam():
    """One nsb_table_adam_step over the whole 6 299 960-line table (dense gradient, rank-1 gradient, both) against
    torch.optim.Adam, as test_gpu_optim.py::test_table_adam_step_matches_torch_adam does at 2053 lines.  The table
    ends 24 lines into a 32-line block: those lines carry gradients in every slot.

    The gradients are multiples of 2^-24 below 2^-5 and the member weights multiples of 1/16, so every product and
    sum is exact in fp32 and both sides see the same gradient.  With random fp32 values, 400 M elements include sums
    that cancel to ~1e-10, whose sign then depends on the summation order, and at eps = 1e-15 Adam turns that sign
    into a full +-lr step (measured with random fp32 gradients, dense + rank-1: max |p - p_torch| = 2 lr).
    About 13 GB of device memory, released at the end."""
    from nersemble_b200 import ops
    E, n_slots = 6299960, 24
    assert E % 32 == 24
    gen = torch.Generator(device=DEV).manual_seed(7)

    def grid(shape):                                  # integers in [-1023, 1023] x 2^-20
        return torch.randint(-1023, 1024, shape, generator=gen, device=DEV).float() * 2.0 ** -20

    p0 = (torch.rand((E, 32, 2), generator=gen, device=DEV) * 2 - 1) * 1e-2
    for mode in ("dense", "rank1", "both"):
        ref = torch.nn.Parameter(p0.clone())
        opt = torch.optim.Adam([ref], lr=5e-3, eps=1e-15, foreach=False)
        p = p0.clone()
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        shadow = torch.empty(p.shape, dtype=torch.float16, device=DEV)
        g1 = grid((n_slots, E, 2))
        g1 *= torch.rand((n_slots, E, 1), generator=gen, device=DEV) < 0.3
        g1[:, -24:] = grid((n_slots, 24, 2))
        cw = torch.randint(0, 17, (n_slots, 32), generator=gen, device=DEV).float() / 16
        pend = {"g_rank1": g1, "cw_slots": cw, "n_slots": n_slots}
        dense = grid((E, 32, 2))
        dense[torch.rand((E,), generator=gen, device=DEV) < 0.5] = 0
        dense[-24:] = grid((24, 32, 2))
        total = torch.zeros_like(p)
        if mode != "rank1":
            total += dense
        if mode != "dense":
            for s in range(n_slots):                  # einsum("sm,sef->emf") slot by slot: no 24x-sized temporary
                total.addcmul_(cw[s][None, :, None], g1[s][:, None, :])
        ref.grad = total.mul_(0.25)
        opt.step()
        ops.table_adam_step(p, m, v, shadow, step=1, lr=5e-3, eps=1e-15, grad=dense if mode != "rank1" else None,
                            pending=pend if mode != "dense" else None, grad_scale=0.25)
        st = opt.state[ref]
        m_err = ((m - st["exp_avg"]).abs() / st["exp_avg"].abs().clamp_min(1e-10)).max().item()
        p_err = (p - ref.detach()).abs().max().item()
        print(f"full-size table_adam_step {mode}: max rel exp_avg diff {m_err:.3e}, max |p - p_torch| {p_err:.3e}")
        torch.testing.assert_close(m, st["exp_avg"], rtol=2e-5, atol=1e-10)
        torch.testing.assert_close(v, st["exp_avg_sq"], rtol=2e-5, atol=1e-20)
        assert p_err < 5e-3 * 1e-4
        assert torch.equal(shadow, p.half())
        last = ref.grad[-24:] != 0
        assert last.float().mean() > 0.9 and (p[-24:] != p0[-24:])[last].all()     # the partial last block moved
        del ref, opt, st, p, m, v, shadow, g1, cw, pend, dense, total, last
        torch.cuda.empty_cache()
    del p0
    torch.cuda.empty_cache()
