"""Scenes with up to NRB_MAX_ACTORS (256) dynamic actors on the actor kernels.

* The assignment's per-ray pre-cull keeps one bit set of ceil(A / 32) words per ray: inert actors (never valid, or
  placed where no ray line passes their sphere) around 16 real ones at high indices change nothing, bit for bit.
* The assignment agrees with a float64 box test of every (sample, actor) pair.
* The kernel route agrees with the torch bookkeeping when actors above index 32 are hit, and the whole hot path with
  64 trained actor trajectories runs without host synchronisation and replays as a CUDA graph.
* Routing and the C ABI: up to 256 actor grids take the kernels, 257 the torch route; every entry point that takes
  actor grids accepts 256 and refuses 257 before any launch.
"""
import ctypes

import pytest
import torch

from tests.parity_utils import rel_err
from tests.test_gpu_actor_pose_grad import aimed_samples, make_field, mlp_of, partly_valid_actors, set_flip, world2boxes_of
from tests.test_gpu_field_gather import leaves

DEV = "cuda"


@pytest.fixture(scope="module")
def nb():
    import neuradar_b200

    assert torch.cuda.is_available()
    return neuradar_b200


def make_proposal(nb, actors, log2_actor=9):
    pcfg = nb.NeuRADProposalFieldConfig()
    pcfg.grid.static.log2_hashmap_size = 13
    pcfg.grid.actor.log2_hashmap_size = log2_actor
    pcfg.grid.actor.flip_prob = 0.25
    prop = nb.NeuRADProposalField(pcfg, actors=actors, static_scale=100.0)
    with torch.no_grad():
        prop.hashgrid.static_grid.hash_table.mul_(2000.0)
        for g in prop.hashgrid.actor_grids:
            g.hash_table.mul_(2000.0)
    return prop


def grad_or_zero(t):
    return torch.zeros_like(t) if t.grad is None else t.grad


# ------------------------------------------------------------------------------------------------ 1. the cull is exact
def pad_scene(w2b16, valid16, bounds16, a2i16, A, off):
    """The 16 actors at indices off..off+15 of an A-actor scene; the others are inert: even ones never valid, odd ones
    axis-aligned boxes 10 km up, where no ray line of the batch passes their sphere."""
    N = w2b16.shape[0]
    w2b = torch.zeros((N, A, 3, 4), device=DEV)
    w2b[..., :3] = torch.eye(3, device=DEV)
    w2b[..., 2, 3] = -(1.0e4 + 10.0 * torch.arange(A, device=DEV, dtype=torch.float32))
    w2b[:, off:off + 16] = w2b16
    valid = (torch.arange(A, device=DEV) % 2 == 1)[None, :].repeat(N, 1)
    valid[:, off:off + 16] = valid16
    bounds = bounds16[:1].repeat(A, 1)
    bounds[off:off + 16] = bounds16
    a2i = torch.arange(A, device=DEV)
    a2i[off:off + 16] = a2i16 + off
    return w2b.contiguous(), valid, bounds, a2i


def shifted(ids, off):
    return torch.where(ids >= 0, ids + off, ids)


@pytest.mark.gpu
@pytest.mark.parametrize("S", [8, 33, 48, 128])
@pytest.mark.parametrize("A,off", [(40, 24), (256, 200)])
def test_cull_is_exact(nb, A, off, S):
    from neuradar_b200 import functional as Fn
    from neuradar_b200.fields import get_normalized_directions
    from neuradar_b200.synthetic import SyntheticActors

    n = 384
    actors = SyntheticActors(16, device=DEV)
    fld = make_field(nb, actors, require_actor_grad=False, seed=S)
    prop = make_proposal(nb, actors).to(DEV)
    rs = aimed_samples(nb, actors, n, S, seed=S + 3)
    rays, iv = rs.per_ray()
    times = rs.times.reshape(n, -1)[:, 0]
    b2w, valid16 = actors.get_boxes2world(times, flatten=False)
    w2b16 = world2boxes_of(b2w).contiguous()
    valid16 = valid16.clone()
    valid16[: n // 2, 3] = False  # a per-ray valid mask on a real actor
    g = torch.Generator(device=DEV).manual_seed(S)
    flip = (torch.rand(n, device=DEV, generator=g) < 0.5).float() * -2 + 1
    scale = fld.hashgrid.actor_scale
    w2bA, validA, boundsA, a2iA = pad_scene(w2b16, valid16, actors.bounds, actors.actor_to_id, A, off)

    def assign(w2b, valid, bounds, a2i):
        index = torch.empty((n * S,), device=DEV, dtype=torch.int32)
        return (*Fn.actor_assign(rays, iv, w2b, valid, bounds, a2i, flip, scale, index), index)

    gid16, pos16, std16, dirs16, idx16 = assign(w2b16, valid16, actors.bounds, actors.actor_to_id)
    gidA, posA, stdA, dirsA, idxA = assign(w2bA, validA, boundsA, a2iA)
    assert int((gid16 >= 0).sum()) > n // 32, int((gid16 >= 0).sum())
    assert torch.equal(gidA, shifted(gid16, off)) and torch.equal(idxA, shifted(idx16, off))
    assert torch.equal(posA, pos16) and torch.equal(stdA, std16) and torch.equal(dirsA, dirs16)

    # fused field forward + backward, with the pose gradient
    x3, std = Fn.frustum_gaussians(rays, iv, fld.hashgrid.static_scale)
    sh = fld.direction_encoding(get_normalized_directions(rays.directions))
    grid = fld.hashgrid.static_grid
    spec = fld.hashgrid.actor_grids[0].spec
    real = [t.hash_table.detach() for t in fld.hashgrid.actor_grids]
    inert = [torch.randn_like(real[0]) for _ in range(A - 16)]
    M = n * S
    ups = [torch.randn((M, 32), device=DEV, generator=g), torch.randn((M,), device=DEV, generator=g),
           torch.randn((M,), device=DEV, generator=g)]

    def field(tables, gid, pos, sd, dirs, idx, w2b):
        tk = grid.hash_table.detach().clone().requires_grad_(True)
        w, b = mlp_of(fld)
        wk, bk = leaves(w, torch.float32), leaves(b, torch.float32)
        (betak,) = leaves([fld.sdf_to_density.beta], torch.float32)
        ak = leaves(tables, torch.float32)
        wl = w2b.detach().clone().requires_grad_(True)
        pose = Fn.ActorPose(wl, idx, flip, scale, rays, iv)
        batch = Fn.ActorBatch(gid, pos, sd, dirs, ak, spec, pose)
        outs = Fn.field_fused(tk, None, x3, std, sh, S, grid.spec, wk, bk, betak, fld.sdf_to_density.beta_min_value, batch)
        sum((o * u).sum() for o, u in zip(outs, ups)).backward()
        grads = [tk.grad, betak.grad] + [t.grad for t in wk + bk]
        return [o.detach() for o in outs], grads, [grad_or_zero(t) for t in ak], wl.grad

    o16, g16, a16, p16 = field(real, gid16, pos16, std16, dirs16, idx16, w2b16)
    oA, gA, aA, pA = field(inert[:off] + real + inert[off:], gidA, posA, stdA, dirsA, idxA, w2bA)
    assert all(torch.equal(a, b) for a, b in zip(oA, o16))
    # sums over samples in any order (atomics): 1e-5 of the largest magnitude, as test_gpu_actor_pose_grad
    for k, (a, b) in enumerate(zip(gA, g16)):
        assert rel_err(a, b) <= 1e-5, (k, rel_err(a, b))
    for k in range(16):
        assert rel_err(aA[off + k], a16[k]) <= 1e-5 if float(a16[k].abs().max()) > 0 else float(aA[off + k].abs().max()) == 0
    assert sum(float(t.abs().max()) > 0 for t in a16) >= 4
    inert_ids = [a for a in range(A) if not off <= a < off + 16]
    assert all(float(aA[a].abs().max()) == 0.0 for a in inert_ids)
    assert rel_err(pA[:, off:off + 16], p16) <= 1e-5 and float(p16.abs().max()) > 0
    assert float(pA[:, inert_ids].abs().max()) == 0.0

    # proposal round forward + backward
    pspec = prop.hashgrid.actor_grids[0].spec
    preal = [t.hash_table.detach() for t in prop.hashgrid.actor_grids]
    pinert = [torch.randn_like(preal[0]) for _ in range(A - 16)]
    pgrid = prop.hashgrid.static_grid
    gw = torch.randn((n, S), device=DEV, generator=g)

    def proposal(tables, gid, pos, sd, dirs):
        tk = pgrid.hash_table.detach().clone().requires_grad_(True)
        dk = prop.density_decoder.weight.detach().clone().requires_grad_(True)
        ak = leaves(tables, torch.float32)
        batch = Fn.ActorBatch(gid, pos, sd, dirs, ak, pspec)
        dens, w = Fn.proposal_round(tk, dk, rays, iv, pgrid.spec, prop.hashgrid.static_scale, actors=batch)
        (w * gw).sum().backward()
        return dens.detach(), w.detach(), [tk.grad, dk.grad], [grad_or_zero(t) for t in ak]

    d16, w16, pg16, pa16 = proposal(preal, gid16, pos16, std16, dirs16)
    dA, wA, pgA, paA = proposal(pinert[:off] + preal + pinert[off:], gidA, posA, stdA, dirsA)
    assert torch.equal(dA, d16) and torch.equal(wA, w16)
    for a, b in zip(pgA, pg16):
        assert rel_err(a, b) <= 1e-5, rel_err(a, b)
    for k in range(16):
        assert rel_err(paA[off + k], pa16[k]) <= 1e-5 if float(pa16[k].abs().max()) > 0 else float(paA[off + k].abs().max()) == 0
    assert all(float(paA[a].abs().max()) == 0.0 for a in inert_ids)


# ------------------------------------------------------------------------------------------------ 2. float64 box tests
@pytest.mark.gpu
@pytest.mark.parametrize("A", [64, 256])
def test_assignment_vs_float64_box_tests(nb, A):
    """Every (sample, actor) box test in float64.  The lattice is pulled in to 3.6 m so that boxes overlap (the highest
    index wins) and every world point stays within |x| < 40 m, where the kernel's fp32 box-frame point is off by a few
    1e-6: samples within 1e-5 of a face plane of any valid actor are left out."""
    from neuradar_b200 import functional as Fn
    from neuradar_b200.synthetic import SyntheticActors, synthetic_rays

    n, S = 512, 48
    actors = SyntheticActors(A, device=DEV, seed=A)
    with torch.no_grad():
        actors.centres.mul_(0.3)
        actors.actor_to_id[1::5] = actors.actor_to_id[0::5][: actors.actor_to_id[1::5].numel()]
    r = synthetic_rays(n, seed=A)
    k = 2 * n // 3
    targets = actors.centres.detach().cpu()[torch.randint(0, A, (k,), generator=torch.Generator().manual_seed(A))]
    d = targets - r["origins"][:k]
    r["directions"][:k] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = torch.linspace(0.5, 15.0, S + 1)[None, :].repeat(n, 1).to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    rays, iv = rs.per_ray()
    b2w, valid = actors.get_boxes2world(rs.times.reshape(n, -1)[:, 0], flatten=False)
    valid = valid.clone()
    valid[:, 3::7] = (rs.times.reshape(n, -1)[:, :1] < 10)  # per-ray valid masks
    w2b = world2boxes_of(b2w).contiguous()
    flip = (torch.rand(n, device=DEV) < 0.5).float() * -2 + 1
    index = torch.empty((n * S,), device=DEV, dtype=torch.int32)
    gid, *_ = Fn.actor_assign(rays, iv, w2b, valid, actors.bounds, actors.actor_to_id, flip, 10.0, index)

    st, en = iv.starts.double(), iv.ends.double()
    t = st + (en - st) / 2
    x = rays.origins.double()[:, None, :] + rays.directions.double()[:, None, :] * t[..., None]     # [N,S,3]
    W = w2b.double()
    p = torch.einsum("nsk,naik->nsai", x, W[..., :3]) + W[..., 3][:, None]                          # [N,S,A,3]
    b = actors.bounds.double()
    inside = (p.abs() < b).all(-1) & valid[:, None, :]
    want = torch.where(inside, torch.arange(A, device=DEV), -1).amax(-1).reshape(-1)
    near = (((p.abs() - b).abs().amin(-1) < 1e-5) & valid[:, None, :]).any(-1).reshape(-1)
    assert float(x.abs().max()) < 40.0
    assert int(near.sum()) < n * S // 100, int(near.sum())
    keep = ~near
    assert torch.equal(index.long()[keep], want[keep])
    assert torch.equal(gid.long()[keep], torch.where(want >= 0, actors.actor_to_id[want.clamp_min(0)], -1)[keep])
    hits = want[keep]
    assert int((hits > 32).sum()) > 200 and int((inside.sum(-1) > 1).sum()) > 0, (int((hits > 32).sum()),)


# ------------------------------------------------------------------------------------------------ 3. kernel vs torch route
def rays_near(actors, first, n, seed):
    """Synthetic rays on the device; a third of them start 15 m from an actor of index >= `first` and aim at it."""
    from neuradar_b200.synthetic import synthetic_rays

    r = synthetic_rays(n, seed=seed)
    k = n // 3
    g = torch.Generator().manual_seed(seed)
    targets = actors.centres.detach().cpu()[first + torch.arange(k) % (actors.n_actors - first)]
    away = torch.randn((k, 3), generator=g)
    away[:, 2] = away[:, 2].abs() * 0.3
    r["origins"][:k] = targets + 15.0 * away / away.norm(dim=-1, keepdim=True)
    d = targets - r["origins"][:k]
    r["directions"][:k] = d / d.norm(dim=-1, keepdim=True)
    return {key: v.to(DEV) for key, v in r.items()}


def samples_of(nb, r, S):
    rb = nb.RayBundle(origins=r["origins"], directions=r["directions"], pixel_area=r["pixel_area"], times=r["times"],
                      metadata={})
    bins = torch.linspace(0.5, 60.0, S + 1)[None, :].repeat(r["origins"].shape[0], 1).to(DEV)
    return rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])


def high_index_scene(A, n, seed):
    """Trained actors, actor 3 valid only at times < 10, actors 5 -> grid 4 and 41 -> grid 40 sharing; a third of the rays
    aim at actors above index 32."""
    actors = partly_valid_actors(A)
    actors.actor_to_id[41] = 40
    return actors, rays_near(actors, 33, n, seed)


def record_boxes2world(actors):
    """Keep the [N,A,4,4] boxes2world of each get_boxes2world call, with its gradient."""
    seen = []
    base = actors.get_boxes2world

    def wrapped(times, flatten=False):
        b2w, valid = base(times, flatten=flatten)
        if b2w.requires_grad:
            b2w.retain_grad()
        seen.append(b2w)
        return b2w, valid

    actors.get_boxes2world = wrapped
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("A", [64, 256])
def test_kernel_route_matches_torch_route_high_indices(nb, A):
    n, S = 512, 64
    actors, r = high_index_scene(A, n, seed=A)
    fld = make_field(nb, actors, seed=A)
    rs = samples_of(nb, r, S)
    set_flip(fld.hashgrid, n, seed=A)
    seen = record_boxes2world(actors)
    g = torch.Generator(device=DEV).manual_seed(0)
    gf, ga = torch.randn((n, S, 32), device=DEV, generator=g), torch.randn((n, S, 1), device=DEV, generator=g)

    def run():
        fld.zero_grad(set_to_none=True)
        seen.clear()
        out = fld(rs)
        feat, alpha = out[nb.FieldHeadNames.FEATURE], out[nb.FieldHeadNames.ALPHA]
        ((feat * gf).sum() + (alpha * ga).sum()).backward()
        db2w = sum(grad_or_zero(t) for t in seen if t.requires_grad)
        return feat.detach(), alpha.detach(), {k: p.grad.clone() for k, p in fld.named_parameters() if p.grad is not None}, db2w

    assert fld.hashgrid.can_assign_in_kernel()
    rays, iv = rs.per_ray()
    batch = fld.hashgrid.assign_actors(rays, iv, rs.times.reshape(n, -1)[:, 0])
    hit = batch.pose.actor_index.long()
    assert int((hit > 32).sum()) > 200 and bool((hit == 41).any()) and bool((hit == 40).any()), int((hit > 32).sum())
    fk, ak, gk, bk = run()
    fld.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    ft, at, gt, bt = run()
    assert rel_err(fk, ft) <= 1e-3 and rel_err(ak, at) <= 1e-3
    for k in set(gk) - set(gt):  # grids the torch route never reads: zero on the kernel route
        assert float(gk[k].abs().max()) == 0.0, k
    tables = 0
    for k in gt:  # static and per-actor tables one by one, the MLPs, beta, the trajectory parameters
        if float(gt[k].abs().max()) == 0.0:
            assert float(gk[k].abs().max()) == 0.0, k
            continue
        e = rel_err(gk[k], gt[k])
        assert e <= 1e-3, (k, e)
        tables += k.startswith("hashgrid.actor_grids.") and int(k.split(".")[2]) > 32
    assert tables >= 8, tables
    # per (ray, actor) d loss / d boxes2world, each block against its own largest magnitude (floor 1 % of the largest)
    top = bt.abs().amax(dim=(-2, -1))
    err = (bk - bt).abs().amax(dim=(-2, -1))
    worst = float((err / top.clamp_min(1e-2 * float(top.max()))).max())
    print(f"[measured] A={A} kernel vs torch route d boxes2world: worst per-block {worst:.3e}")
    assert worst <= 2e-3 and int((top[:, 33:] > 0).sum()) > 50

    # the proposal rounds (no pose gradient, as the reference's default)
    prop = make_proposal(nb, actors).to(DEV)
    prop.train()
    set_flip(prop.hashgrid, n, seed=A + 1)
    gw = torch.randn((n, S, 1), device=DEV, generator=g)

    def run_prop():
        prop.zero_grad(set_to_none=True)
        dens, w = prop.density_and_weights(rs)
        (w * gw).sum().backward()
        return dens.detach(), w.detach(), {k: p.grad.clone() for k, p in prop.named_parameters() if p.grad is not None}

    assert prop.hashgrid.can_assign_in_kernel(proposal=True)
    dk, wk, pk = run_prop()
    prop.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    dt, wt, pt = run_prop()
    assert rel_err(dk, dt) <= 3e-5 and rel_err(wk, wt) <= 3e-5
    for k in pt:
        if float(pt[k].abs().max()) == 0.0:
            assert float(pk[k].abs().max()) == 0.0, k
            continue
        assert rel_err(pk[k], pt[k]) <= 1e-3, (k, rel_err(pk[k], pt[k]))


# ------------------------------------------------------------------------------------------------ 4. the whole hot path
@pytest.mark.gpu
def test_hot_path_64_trained_actors(nb):
    from neuradar_b200.synthetic import build_hot_path

    n, A = 1024, 64
    actors, r = high_index_scene(A, n, seed=7)
    model = build_hot_path(log2_main=14, log2_prop=14, num_proposal_samples=(64, 48), num_nerf_samples=48, main_levels=8,
                           main_features=4, main_res=(32, 8192), seed=1, actors=actors)
    model.train()
    model.sampler.eval()  # no jitter: the eager and graph steps see the same samples
    with torch.no_grad():
        for g in model.field.hashgrid.actor_grids:
            g.hash_table.mul_(300.0)
    for h in [model.field.hashgrid] + [p.hashgrid for p in model.proposal_fields]:
        set_flip(h, n, seed=8)
        assert h.can_assign_in_kernel(proposal=h is not model.field.hashgrid)

    def step():
        out = model(nb.RayBundle(origins=r["origins"].clone(), directions=r["directions"].clone(),
                                 pixel_area=r["pixel_area"].clone(), nears=r["nears"].clone(), fars=r["fars"].clone(),
                                 times=r["times"], metadata={"is_lidar": r["is_lidar"], "is_radar": r["is_radar"]}))
        nb.bench_loss(out).backward()

    def grads():
        return {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        model.zero_grad(set_to_none=True)
        step()  # warm-up (allocations, caches, side streams)
        torch.cuda.synchronize()
        model.zero_grad(set_to_none=True)
        torch.cuda.set_sync_debug_mode("error")
        try:
            step()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        torch.cuda.synchronize()
        eager = grads()
        eager_poses = [p.grad.detach().clone() for p in actors.parameters()]
        model.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            step()
        graph.replay()
        torch.cuda.synchronize()
    replay = grads()
    assert set(eager) == set(replay)
    assert all(float(g.abs().max()) > 0 for g in eager_poses[:3])  # (yaw_rate's gradient is scaled by the times)
    for e, p in zip(eager_poses, actors.parameters()):
        assert rel_err(p.grad, e) <= 1e-5
    touched = [k for k in eager if k.startswith("field.hashgrid.actor_grids.") and int(k.split(".")[3]) > 32
               and float(eager[k].abs().max()) > 0]
    assert len(touched) >= 1, touched
    for k in eager:
        assert rel_err(replay[k], eager[k]) <= 1e-5, (k, rel_err(replay[k], eager[k]))


# ------------------------------------------------------------------------------------------------ 5. routing
def _modules(nb, A, device="cpu"):
    from neuradar_b200.synthetic import SyntheticActors

    actors = SyntheticActors(A, device=device)
    cfg = nb.NeuRADFieldConfig(grid=nb.NeuRADHashEncodingConfig(
        static=nb.StaticSettings(hashgrid_dim=4, num_levels=8, base_res=32, max_res=8192, log2_hashmap_size=12),
        actor=nb.ActorSettings(log2_hashmap_size=6)))
    fld = nb.NeuRADField(cfg, actors=actors, static_scale=100.0).to(device)
    prop = make_proposal(nb, actors, log2_actor=6).to(device)
    return actors, fld, prop


@pytest.mark.parametrize("A", [33, 256, 257])
def test_routing_by_actor_count(A):
    """No device needed: up to _lib.MAX_ACTORS actor grids take the kernels in the field and the proposal networks."""
    import neuradar_b200 as nb
    from neuradar_b200 import _lib

    assert _lib.MAX_ACTORS == 256
    _, fld, prop = _modules(nb, A)
    on_kernels = A <= 256
    assert fld.hashgrid.can_assign_in_kernel() == on_kernels
    assert prop.hashgrid.can_assign_in_kernel(proposal=True) == on_kernels


@pytest.mark.gpu
@pytest.mark.parametrize("A", [33, 256, 257])
def test_routes_run(nb, A):
    """33 and 256 actor grids never enter the torch bookkeeping; 257 take it and still run."""
    n, S = 256, 48
    actors, fld, prop = _modules(nb, A, device=DEV)
    rs = samples_of(nb, rays_near(actors, A - 16, n, seed=1), S)
    fld.train(), prop.train()
    calls = []
    for h in (fld.hashgrid, prop.hashgrid):
        base = h._apply_actors

        def apply(*a, base=base, **kw):
            calls.append(1)
            return base(*a, **kw)

        h._apply_actors = apply
    out = fld(rs)
    dens, w = prop.density_and_weights(rs)
    (out[nb.FieldHeadNames.FEATURE].sum() + out[nb.FieldHeadNames.ALPHA].sum() + w.sum()).backward()
    assert len(calls) == 0 if A <= 256 else len(calls) >= 2, len(calls)
    touched = sum(float(g.hash_table.grad.abs().max()) > 0 for g in list(fld.hashgrid.actor_grids)[A - 16:]
                  if g.hash_table.grad is not None)
    assert touched >= 4, touched
    assert bool(torch.isfinite(dens).all()) and bool(torch.isfinite(out[nb.FieldHeadNames.FEATURE]).all())


# ------------------------------------------------------------------------------------------------ 6. C ABI
def test_actor_cap_abi():
    """No device needed: the library's cap is the binding's, and each entry point that takes actor grids accepts 256 and
    refuses 257 with NRB_ERR_UNSUPPORTED before any launch (empty batches: nothing is launched either way)."""
    from neuradar_b200 import _lib

    lib = _lib.load()
    assert lib.nrb_max_actors() == _lib.MAX_ACTORS == 256
    raw = (ctypes.c_float * 4096)()
    p = (ctypes.addressof(raw) + 15) // 16 * 16
    rays, iv = _lib.Rays(), _lib.Intervals()
    rays.origins = rays.directions = rays.pixel_area = rays.nears = rays.fars = p
    rays.num_rays = 0
    iv.starts = iv.ends = p
    iv.row_stride, iv.num_samples = 8, 8
    grid = _lib.Grid()
    grid.table, grid.num_levels, grid.features_per_level, grid.log2_hashmap_size = p, 8, 4, 4
    grids, samples = _lib.ActorGrids(), _lib.ActorSamples()
    for i in range(_lib.MAX_ACTORS):
        grids.tables[i] = p
    grids.num_levels, grids.features_per_level, grids.log2_hashmap_size = 4, 4, 4
    samples.grid_id = samples.pos = samples.std = samples.dirs = p
    mlp = _lib.FieldMlp()
    for i in range(5):
        mlp.weights[i] = p
    mlp.beta = p
    dtables = (ctypes.c_void_p * _lib.MAX_ACTORS)(*([p] * _lib.MAX_ACTORS))
    r, i_, g_, a_, s_ = (ctypes.byref(x) for x in (rays, iv, grid, grids, samples))
    calls = {
        "nrb_field_fused_fwd": lambda: lib.nrb_field_fused_fwd(ctypes.byref(mlp), g_, p, p, None, p, 8, 0, p, p, p, None, a_, s_,
                                                               None),
        "nrb_proposal_fwd": lambda: lib.nrb_proposal_fwd(r, g_, p, 1.0, i_, p, p, None, None, a_, s_, None),
        "nrb_proposal_bwd": lambda: lib.nrb_proposal_bwd(r, g_, p, 1.0, i_, p, p, p, None, p, p, None, 0, a_, s_, dtables, None),
        "nrb_actor_scatter": lambda: lib.nrb_actor_scatter(a_, dtables, s_, p, None, 0, None),
        "nrb_actor_pose_grad": lambda: lib.nrb_actor_pose_grad(r, i_, p, 2, p, None, 10.0, a_, s_, p, p, None),
    }
    launches = lib.nrb_launch_count()
    for name, call in calls.items():
        grids.num_grids = 256
        assert call() == 0, (name, lib.nrb_last_error_string())
        grids.num_grids = 257
        assert call() == -3, name  # NRB_ERR_UNSUPPORTED
    assert lib.nrb_launch_count() == launches
