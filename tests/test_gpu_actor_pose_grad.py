"""Trained actor trajectories on the kernel path: nrb_actor_pose_grad (csrc/actors.cu), the pose context of
functional.ActorBatch and the routing of NeuRADHashEncoding.

The main reference is float64, built like the references of test_gpu_field_gather.py:
* cells are located from the kernel's own fp32 `ActorBatch.pos`, and the actor assignment is the kernel's own
  `actor_index`, so a cell or box-face decision is never compared across two roundings;
* everything that depends on the poses W = world2boxes is float64 - the box-frame point p = R x + t, the flip, the
  contraction, pos and std - with in-cell offsets o_fp32 + (pos64 - pos64.detach()) * scal;
* the MLPs, the SH concatenation and the compositing are float64 too.
Pose gradients are compared per (ray, actor) block against that block's largest magnitude: a bar over the whole tensor
would hide a wrong small actor.  The bar 1e-4 follows the bf16 hi / mid error model of the fused backward.
"""
import copy
import ctypes
import math
from dataclasses import replace

import pytest
import torch
import torch.nn.functional as TF

from oracle import neuradar_oracle as O
from tests.parity_utils import rel_err
from tests.test_gpu_field_gather import leaves, near_kink, ref_encode, ref_field, ref_sh, tiles_for

DEV = "cuda"
POSE_TOL = 1e-4


@pytest.fixture(scope="module")
def nb():
    import neuradar_b200

    assert torch.cuda.is_available()
    return neuradar_b200


def partly_valid_actors(n_actors, trainable=True, **kw):
    """SyntheticActors whose actor 3 is valid only at times < 10 (a per-ray valid mask, as DynamicActors gives), with
    actors 4 and 5 sharing grid 4 (actor_to_id is not the identity; grid 5 is never read)."""
    from neuradar_b200.synthetic import SyntheticActors

    class PartlyValid(SyntheticActors):
        def get_boxes2world(self, times, flatten=False):
            assert not flatten
            b2w, valid = super().get_boxes2world(times, flatten=False)
            valid = valid.clone()
            if self.n_actors > 3:
                valid[:, 3] = times.reshape(-1) < 10
            return b2w, valid

    actors = PartlyValid(n_actors, device=DEV, trainable=trainable, **kw)
    if n_actors > 5:
        actors.actor_to_id[5] = 4
    return actors


def make_field(nb, actors, require_actor_grad=True, seed=0):
    cfg = nb.NeuRADFieldConfig(grid=nb.NeuRADHashEncodingConfig(
        static=nb.StaticSettings(hashgrid_dim=4, num_levels=8, base_res=32, max_res=8192, log2_hashmap_size=14),
        actor=nb.ActorSettings(flip_prob=0.5, log2_hashmap_size=10), require_actor_grad=require_actor_grad))
    torch.manual_seed(seed)
    fld = nb.NeuRADField(cfg, actors=actors, static_scale=100.0).to(DEV)
    fld.train()
    with torch.no_grad():
        fld.hashgrid.static_grid.hash_table.mul_(300.0)
        for g in fld.hashgrid.actor_grids:
            g.hash_table.mul_(300.0)
    return fld


def aimed_samples(nb, actors, n, S, seed, near=0.5, far=60.0, targets=None):
    """n synthetic rays, a third of them aimed at actor boxes (or at `targets` [k,3]), with S samples on [near, far]."""
    from neuradar_b200.synthetic import synthetic_rays

    r = synthetic_rays(n, seed=seed)
    if targets is None:
        targets = actors.centres.detach()[torch.arange(n // 3) % actors.n_actors].cpu()
    k = targets.shape[0]
    d = targets - r["origins"][:k]
    r["directions"][:k] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = torch.linspace(near, far, S + 1)[None, :].repeat(n, 1).to(DEV)
    return rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])


def set_flip(hashgrid, n, seed):
    g = torch.Generator().manual_seed(seed)
    hashgrid.ray_flip_override = ((torch.rand(n, generator=g) < 0.5).float() * -2 + 1).to(DEV)


def kernel_inputs(fld, rs):
    from neuradar_b200 import functional as Fn
    from neuradar_b200.fields import get_normalized_directions

    rays, iv = rs.per_ray()
    x3, std = Fn.frustum_gaussians(rays, iv, fld.hashgrid.static_scale)
    sh = fld.direction_encoding(get_normalized_directions(rays.directions))
    batch = fld.hashgrid.assign_actors(rays, iv, rs.times.reshape(rays.num_rays, -1)[:, 0])
    return rays, iv, x3, std, sh, batch


def world2boxes_of(boxes2world):
    """NeuRADHashEncoding.assign_actors' element-wise inverse."""
    Ri = boxes2world[..., :3, :3].transpose(-2, -1)
    return torch.cat([Ri, -(Ri * boxes2world[..., None, :3, 3]).sum(-1, keepdim=True)], dim=-1)


def mlp_of(fld):
    geo, feat = fld.mlp_geo.layers, fld.mlp_feature.layers
    return ([geo[0].weight, geo[1].weight, feat[0].weight, feat[1].weight, feat[2].weight],
            [geo[0].bias, geo[1].bias, feat[0].bias, feat[1].bias, feat[2].bias])


# ------------------------------------------------------------------------------------------------ float64 reference
class Ref:
    """The field on the kernel's assignment, float64 in everything that depends on the poses."""

    def __init__(self, fld, actors, times, rays, iv, x3, std, sh, batch, with_std=True):
        from neuradar_b200.field_components import NeuRADHashEncoding

        N, S = rays.num_rays, iv.num_samples
        M = N * S
        self.N, self.S, self.A = N, S, actors.n_actors
        self.actors64 = copy.deepcopy(actors).double()
        self.params64 = list(self.actors64.parameters())
        self.times = times
        W = world2boxes_of(self.actors64.get_boxes2world(times, flatten=False)[0])
        W.retain_grad()
        self.W = W
        idx = batch.pose.actor_index.long()
        m = (idx >= 0).nonzero()[:, 0]
        rn, ra = m // S, idx[m]
        self.claimed = torch.zeros((N, self.A), dtype=torch.bool, device=DEV)
        self.claimed[rn, ra] = True
        # world-space gaussians (cameras/rays.py:109-124), independent of W
        st, en = iv.starts.double(), iv.ends.double()
        dist = (en - st) / 2
        t = st + dist
        xw = (rays.origins.double()[:, None, :] + rays.directions.double()[:, None, :] * t[..., None]).reshape(M, 3)
        sw = (rays.pixel_area.double()[:, None] * t * t * dist).pow(1 / 3).reshape(M)
        Wm = W[rn, ra]
        p = (Wm[:, :, :3] @ xw[m][..., None])[..., 0] + Wm[:, :, 3]
        flip = batch.pose.flip
        f = torch.ones_like(p[:, 0]) if flip is None else flip.double()[rn]
        q = torch.cat([p[:, :1] * f[:, None], p[:, 1:]], dim=-1)
        pos64, std64 = NeuRADHashEncoding._contract(q, sw[m][:, None], batch.pose.actor_scale)
        std64 = std64[:, 0] if with_std else std64[:, 0].detach()
        self.m, self.pos64, self.std64 = m, pos64, std64
        # features: static grid for every sample, the sample's actor grid for claimed ones
        grid = fld.hashgrid.static_grid
        self.t64 = grid.hash_table.detach().double().requires_grad_(True)
        self.a64 = leaves([g.hash_table for g in fld.hashgrid.actor_grids], torch.float64)
        static = ref_encode(x3, std, self.t64, grid.scalings, grid.log2_hashmap_size)
        ascal, Ta = fld.hashgrid.actor_grids[0].scalings, fld.hashgrid.actor_grids[0].log2_hashmap_size
        gid = batch.grid_id[m]
        afeat = torch.zeros((m.numel(), 32), dtype=torch.float64, device=DEV)
        for g in torch.unique(gid).tolist():
            sel = (gid == g).nonzero()[:, 0]
            f16 = ref_encode(batch.pos[m[sel]], std64[sel], self.a64[g], ascal, Ta, x_leaf=pos64[sel])
            afeat = afeat.index_put((sel,), TF.pad(f16, (0, 16)))
        self.feats = static.index_put((m,), afeat)
        sh_rows = sh.double()[torch.arange(M, device=DEV) // S]
        self.sh_rows = sh_rows.index_put((m,), ref_sh(batch.dirs[m]))
        w, b = mlp_of(fld)
        self.w64, self.b64 = leaves(w, torch.float64), leaves(b, torch.float64)
        (self.beta64,) = leaves([fld.sdf_to_density.beta], torch.float64)
        self.kink = near_kink(self.feats.detach(), self.sh_rows, self.w64, self.b64)

    def field(self):
        return ref_field(self.feats, self.sh_rows, self.w64, self.b64, self.beta64)

    def param_grads(self, dW):
        """d loss / d trajectory parameters for a given d loss / d world2boxes, through the float64 trajectory."""
        W = world2boxes_of(self.actors64.get_boxes2world(self.times, flatten=False)[0])
        return torch.autograd.grad(W, self.params64, dW)


def make_ref(fld, actors, rs, inputs, with_std=True):
    return Ref(fld, actors, rs.times.reshape(inputs[0].num_rays, -1)[:, 0], *inputs, with_std=with_std)


def composite64(ra, rf, iv, N, S):
    """The oracle's compositing with the sky fix-up, float64 on the CPU (test_gpu_field_gather.test_gather_backward_render)."""
    starts, ends = iv.starts.double().cpu(), iv.ends.double().cpu()
    alpha, feats = ra.view(N, S).cpu(), rf.view(N, S, 32).cpu()
    comp = O.composite(alpha, feats, starts, ends, 0.0)
    raw, _ = O.alpha_weights(alpha, 0.0)
    w = torch.cat([comp["weights"][..., 0], raw[:, -1:] + 1 - comp["accumulation"]], dim=-1)
    return w, comp["features"], comp["depth"][:, 0], comp["accumulation"][:, 0]


def upstream(kind, N, S, seed, kink=None):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if kind == "fused":
        M = N * S
        gf, gs, ga = (torch.randn((M, 32), device=DEV, generator=g), torch.randn((M,), device=DEV, generator=g),
                      torch.randn((M,), device=DEV, generator=g))
        gf[kink], gs[kink], ga[kink] = 0, 0, 0
        return gf, gs, ga
    return (torch.randn((N, S), device=DEV, generator=g), torch.randn((N, 32), device=DEV, generator=g),
            torch.randn((N,), device=DEV, generator=g) * 1e-3, torch.randn((N,), device=DEV, generator=g))


def loss_of(outs, ups):
    return sum((o * u.to(o.dtype)).sum() for o, u in zip(outs, ups))


def run_kernel(kind, fld, inputs, batch, ups):
    """One forward + backward of Fn.field_fused / Fn.field_render on fresh leaves; returns (outputs, grads by name)."""
    from neuradar_b200 import functional as Fn

    rays, iv, x3, std, sh, _ = inputs
    grid = fld.hashgrid.static_grid
    w, b = mlp_of(fld)
    tk = grid.hash_table.detach().clone().requires_grad_(True)
    wk, bk = leaves(w, torch.float32), leaves(b, torch.float32)
    (betak,) = leaves([fld.sdf_to_density.beta], torch.float32)
    ak = leaves([g.hash_table for g in fld.hashgrid.actor_grids], torch.float32)
    batch = batch.with_tables(ak)
    beta_min = fld.sdf_to_density.beta_min_value
    if kind == "fused":
        outs = Fn.field_fused(tk, None, x3, std, sh, iv.num_samples, grid.spec, wk, bk, betak, beta_min, batch)
    else:
        outs = Fn.field_render(tk, x3, std, sh, iv, grid.spec, wk, bk, betak, beta_min, 0.0, batch)
    loss_of(outs, ups).backward()
    grads = {"table": tk.grad, "beta": betak.grad}
    grads.update({f"w{k}": t.grad for k, t in enumerate(wk)})
    grads.update({f"b{k}": t.grad for k, t in enumerate(bk)})
    grads.update({f"actor{k}": t.grad for k, t in enumerate(ak)})
    return [o.detach() for o in outs], grads


def check_blocks(tag, got, want, claimed, skip=None, tol=POSE_TOL):
    """Per (ray, actor) block of d loss / d world2boxes [N,A,3,4]: max error over the block's own largest magnitude."""
    got, want = got.detach().double(), want.detach().double()
    err, top = (got - want).abs().amax(dim=(-2, -1)), want.abs().amax(dim=(-2, -1))
    # blocks below 1e-6 of the largest are held to that floor: behind an opaque surface a sample's compositing weight
    # underflows in fp32 (float64 keeps gradients of 1e-60 and less)
    floor = 1e-6 * float(top.max())
    use = claimed & (top > 0) & (torch.ones_like(claimed) if skip is None else ~skip)
    assert int((use & (top > floor)).sum()) >= 8, int(use.sum())
    worst = float((err[use] / top[use].clamp_min(floor)).max())
    print(f"[measured] {tag}: worst per-block max-rel {worst:.3e} over {int(use.sum())} blocks")
    assert worst <= tol, (tag, worst)
    zero = claimed & (top == 0)
    assert float(err[zero].max()) == 0.0 if bool(zero.any()) else True
    assert float(got[~claimed].abs().max()) == 0.0, "an unclaimed or invalid actor received a pose gradient"
    return worst


def actor_param_grads(actors):
    return [p.grad for p in actors.parameters()]


def zero_actor_grads(actors):
    for p in actors.parameters():
        p.grad = None


# ------------------------------------------------------------------------------------------------ 1. field, float64
@pytest.mark.gpu
@pytest.mark.parametrize("S,kind", [(33, "few"), (128, "few"), (48, "multi")])
@pytest.mark.parametrize("fn", ["fused", "render"])
def test_pose_grad_vs_float64(nb, fn, S, kind):
    n = -(-tiles_for(3, S)[0] // S) if kind == "multi" else 384
    actors = partly_valid_actors(16)
    fld = make_field(nb, actors, seed=S)
    rs = aimed_samples(nb, actors, n, S, seed=S + 1)
    set_flip(fld.hashgrid, n, seed=S)
    inputs = kernel_inputs(fld, rs)
    batch = inputs[-1]
    assert fld.hashgrid.can_assign_in_kernel() and batch.pose is not None and batch.pose.flip is not None
    assert bool((batch.pose.flip < 0).any()) and bool((batch.pose.flip > 0).any())
    ref = make_ref(fld, actors, rs, inputs)
    assert ref.m.numel() > 100, ref.m.numel()
    # actor 3 is invalid on some rays aimed at it, and grids 4 (actors 4 and 5) serve two actors
    assert bool(ref.claimed[:, 4].any()) and bool(ref.claimed[:, 5].any())
    N = n
    ups = upstream(fn, N, S, seed=S, kink=ref.kink)
    rf, rsdf, ra = ref.field()
    if fn == "fused":
        loss_of((rf, rsdf, ra), ups).backward()
        skip = torch.zeros_like(ref.claimed)
    else:
        loss_of(composite64(ra, rf, inputs[1], N, S), [u.double().cpu() for u in ups]).backward()
        # a hidden unit at a ReLU kink may switch sides between fp32 and float64, and compositing couples a ray's samples
        skip = ref.kink.view(N, S).any(dim=1)[:, None].expand_as(ref.claimed)
    zero_actor_grads(actors)
    w2b = batch.pose.world2boxes
    w2b.retain_grad()
    outs, grads = run_kernel(fn, fld, inputs, batch, ups)
    tag = f"{fn} S{S} {kind}"
    # (render: a block sums the few samples of one ray in one box, each a product of fp32 compositing factors; the
    # measured worst block is 1.1e-4 on a B200)
    check_blocks(f"{tag} dworld2boxes", w2b.grad, ref.W.grad, ref.claimed, skip, POSE_TOL if fn == "fused" else 2 * POSE_TOL)
    # trajectory parameters: the float64 chain of the reference's dW (the kernel's on skipped blocks)
    dW = torch.where(skip[..., None, None], w2b.grad.double(), ref.W.grad)
    for (name, p), want in zip(actors.named_parameters(), ref.param_grads(dW)):
        e = rel_err(p.grad, want)
        print(f"[measured] {tag} d{name}: max-rel {e:.3e}")
        assert e <= POSE_TOL, (name, e)
    # the same inputs with frozen poses: identical forward, the same table / MLP / beta gradients up to atomics order
    outs0, grads0 = run_kernel(fn, fld, inputs, replace(batch, pose=None), ups)
    assert all(torch.equal(a, b) for a, b in zip(outs, outs0))
    for k in grads:
        if grads0[k] is None or float(grads0[k].abs().max()) == 0.0:
            assert grads[k] is None or float(grads[k].abs().max()) == 0.0, k
            continue
        # (sums over many samples in any order: measured up to 1.7e-6 of the largest magnitude on a B200)
        assert rel_err(grads[k], grads0[k]) <= 1e-5, (k, rel_err(grads[k], grads0[k]))


# ------------------------------------------------------------------------------------------------ 2. outside the linear region
@pytest.mark.gpu
def test_pose_grad_outside_linear_region(nb):
    """A truck-sized box (half-extent 12 m > actor_scale = 10 m) seen by radar-footprint rays from ~50 m: samples beyond
    |u| = 1 are contracted, their std depends on the pose, and 2 scal std > 1 on the coarse actor levels."""
    S, n = 32, 256
    actors = partly_valid_actors(1)
    with torch.no_grad():
        actors.bounds.copy_(torch.tensor([[12.0, 3.0, 2.0]], device=DEV))
        actors.yaw_rate.zero_()
        actors.velocity.zero_()
    fld = make_field(nb, actors, seed=7)
    g = torch.Generator().manual_seed(3)
    # targets in the box's end regions |x| in [9, 12) (box frame), rotated into the world at yaw0
    k = n // 2
    bx = (torch.rand(k, generator=g) * 3 + 9) * torch.where(torch.rand(k, generator=g) < 0.5, -1.0, 1.0)
    local = torch.stack([bx, (torch.rand(k, generator=g) - 0.5) * 4, (torch.rand(k, generator=g) - 0.5) * 2], -1)
    yaw = float(actors.yaw0[0])
    c, s = math.cos(yaw), math.sin(yaw)
    rot = torch.tensor([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    targets = local @ rot.T + actors.centres.detach().cpu()[0]
    from neuradar_b200.synthetic import synthetic_rays

    r = synthetic_rays(n, seed=11, mix="radar")  # radar pixel areas
    away = torch.randn((k, 3), generator=g)
    away[:, 2] = away[:, 2].abs() * 0.2
    away = away / away.norm(dim=-1, keepdim=True)
    r["origins"][:k] = targets + away * 50.0
    d = targets - r["origins"][:k]
    r["directions"][:k] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = torch.linspace(40.0, 60.0, S + 1)[None, :].repeat(n, 1).to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    set_flip(fld.hashgrid, n, seed=5)
    inputs = kernel_inputs(fld, rs)
    batch = inputs[-1]
    ref = make_ref(fld, actors, rs, inputs)
    scal = fld.hashgrid.actor_grids[0].scalings.to(DEV, torch.float64)
    outside = (ref.pos64.detach() * 4 - 2).abs().amax(dim=-1) >= 1  # max |u| >= 1: the contracted region
    assert int(outside.sum()) > 50, int(outside.sum())
    assert bool((2 * scal[:2] * ref.std64.detach()[outside][:, None] > 1).all())
    ups = upstream("fused", n, S, seed=2, kink=ref.kink)
    rf, rsdf, ra = ref.field()
    loss_of((rf, rsdf, ra), ups).backward()
    ref_nostd = make_ref(fld, actors, rs, inputs, with_std=False)
    loss_of(ref_nostd.field(), ups).backward()
    zero_actor_grads(actors)
    w2b = batch.pose.world2boxes
    w2b.retain_grad()
    run_kernel("fused", fld, inputs, batch, ups)
    check_blocks("outside linear region dworld2boxes", w2b.grad, ref.W.grad, ref.claimed)
    for (name, p), want in zip(actors.named_parameters(), ref.param_grads(ref.W.grad)):
        assert rel_err(p.grad, want) <= POSE_TOL, (name, rel_err(p.grad, want))
    # the std term is what this case tests: without it the reference moves well beyond the bar
    top = ref.W.grad.abs().amax(dim=(-2, -1))
    moved = ((ref_nostd.W.grad - ref.W.grad).abs().amax(dim=(-2, -1))[ref.claimed] / top[ref.claimed]).max()
    print(f"[measured] dropping the std term moves a block by {float(moved):.3e}")
    assert float(moved) > 10 * POSE_TOL


# ------------------------------------------------------------------------------------------------ 3. kernel vs torch route
@pytest.mark.gpu
def test_kernel_route_matches_torch_route(nb):
    """NeuRADField.forward on the kernel route against the reference's torch bookkeeping of the same module (the std
    term is zero here: every box lies inside the contraction's linear region)."""
    n, S = 512, 64
    actors = partly_valid_actors(16)
    fld = make_field(nb, actors, seed=4)
    rs = aimed_samples(nb, actors, n, S, seed=9)
    set_flip(fld.hashgrid, n, seed=9)
    g = torch.Generator(device=DEV).manual_seed(0)
    gf, ga = torch.randn((n, S, 32), device=DEV, generator=g), torch.randn((n, S, 1), device=DEV, generator=g)

    def run():
        fld.zero_grad(set_to_none=True)
        out = fld(rs)
        feat, alpha = out[nb.FieldHeadNames.FEATURE], out[nb.FieldHeadNames.ALPHA]
        ((feat * gf).sum() + (alpha * ga).sum()).backward()
        return feat.detach(), alpha.detach(), {k: p.grad.clone() for k, p in fld.named_parameters() if p.grad is not None}

    assert fld.hashgrid.can_assign_in_kernel()
    fk, ak, gk = run()
    fld.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    ft, at, gt = run()
    assert rel_err(fk, ft) <= 1e-3 and rel_err(ak, at) <= 1e-3
    for k in set(gk) - set(gt):  # actor grid 5 is never read: the kernel route returns it a zero gradient
        assert float(gk[k].abs().max()) == 0.0, k
    assert set(gt) <= set(gk)
    poses = 0
    for k in gt:
        if float(gt[k].abs().max()) == 0.0:
            assert float(gk[k].abs().max()) == 0.0, k
            continue
        e = rel_err(gk[k], gt[k])
        print(f"[measured] kernel vs torch route {k}: max-rel {e:.3e}")
        assert e <= 1e-3, (k, e)
        poses += k.startswith("hashgrid.actors.")
    assert poses == 4  # centres, velocity, yaw0, yaw_rate


# ------------------------------------------------------------------------------------------------ 4. proposal rounds
@pytest.mark.gpu
def test_proposal_rounds_with_trained_poses(nb):
    """Proposal networks (require_actor_grad=False, as the reference) stay on the fused round with trained poses: the
    same density and weights as with frozen poses, and no pose gradient from a proposal loss."""
    n, S = 384, 96
    actors = partly_valid_actors(16)
    pcfg = nb.NeuRADProposalFieldConfig()
    pcfg.grid.static.log2_hashmap_size = 13
    pcfg.grid.actor.log2_hashmap_size = 9
    pcfg.grid.actor.flip_prob = 0.25
    prop = nb.NeuRADProposalField(pcfg, actors=actors, static_scale=100.0).to(DEV)
    prop.train()
    with torch.no_grad():
        prop.hashgrid.static_grid.hash_table.mul_(2000.0)
        for g in prop.hashgrid.actor_grids:
            g.hash_table.mul_(2000.0)
    rs = aimed_samples(nb, actors, n, S, seed=4)
    set_flip(prop.hashgrid, n, seed=4)
    assert prop.hashgrid.can_assign_in_kernel(proposal=True)
    gw = torch.randn((n, S, 1), device=DEV)

    def run():
        dens, w = prop.density_and_weights(rs)
        (w * gw).sum().backward()
        return dens.detach(), w.detach()

    dens_t, w_t = run()
    assert all(p.grad is None for p in actors.parameters())
    for p in actors.parameters():
        p.requires_grad_(False)
    dens_f, w_f = run()
    assert torch.equal(dens_t, dens_f) and torch.equal(w_t, w_f)
    # a proposal network that asks for pose gradients keeps the torch route
    for p in actors.parameters():
        p.requires_grad_(True)
    prop.hashgrid.config.require_actor_grad = True
    assert not prop.hashgrid.can_assign_in_kernel(proposal=True)


# ------------------------------------------------------------------------------------------------ 5. field without pose grad
@pytest.mark.gpu
def test_field_without_actor_grad_keeps_poses_constant(nb):
    n, S = 256, 48
    actors = partly_valid_actors(16)
    fld = make_field(nb, actors, require_actor_grad=False, seed=2)
    rs = aimed_samples(nb, actors, n, S, seed=3)
    assert fld.hashgrid.can_assign_in_kernel()
    inputs = kernel_inputs(fld, rs)
    assert inputs[-1].pose is None and int((inputs[-1].grid_id >= 0).sum()) > 50
    out = fld(rs)
    (out[nb.FieldHeadNames.FEATURE].sum() + out[nb.FieldHeadNames.ALPHA].sum()).backward()
    assert all(p.grad is None for p in actors.parameters())
    assert sum(float(g.hash_table.grad.abs().max()) > 0 for g in fld.hashgrid.actor_grids) >= 4


# ------------------------------------------------------------------------------------------------ 6. the whole hot path
def _hot_path(nb, n):
    from neuradar_b200.synthetic import build_hot_path, synthetic_rays

    actors = partly_valid_actors(16)
    model = build_hot_path(log2_main=14, log2_prop=14, num_proposal_samples=(64, 48), num_nerf_samples=48, main_levels=8,
                           main_features=4, main_res=(32, 8192), seed=1, actors=actors)
    model.train()
    model.sampler.eval()  # no jitter: the eager, graph and torch-route steps see the same samples
    with torch.no_grad():
        for g in model.field.hashgrid.actor_grids:
            g.hash_table.mul_(300.0)
    r = synthetic_rays(n, seed=6)
    k = n // 3
    d = actors.centres.detach()[torch.arange(k) % 16].cpu() - r["origins"][:k]
    r["directions"][:k] = d / d.norm(dim=-1, keepdim=True)
    r = {key: v.to(DEV) for key, v in r.items()}
    for h in [model.field.hashgrid] + [p.hashgrid for p in model.proposal_fields]:
        set_flip(h, n, seed=8)

    def bundle():
        return nb.RayBundle(origins=r["origins"].clone(), directions=r["directions"].clone(), pixel_area=r["pixel_area"].clone(),
                            nears=r["nears"].clone(), fars=r["fars"].clone(), times=r["times"],
                            metadata={"is_lidar": r["is_lidar"], "is_radar": r["is_radar"]})

    return model, actors, bundle


@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True])
def test_hot_path_with_trained_poses(nb, autocast):
    n = 1024
    model, actors, bundle = _hot_path(nb, n)
    assert model.field.hashgrid.can_assign_in_kernel()

    def step():
        with torch.autocast("cuda", torch.float16, enabled=autocast):
            out = model(bundle())
            loss = nb.bench_loss(out)
        loss.backward()

    def grads():
        return [p.grad.detach().clone() for p in actors.parameters()]

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
        assert all(float(g.abs().max()) > 0 for g in eager[:3])  # (yaw_rate's gradient is scaled by the times)
        model.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            step()
        graph.replay()
        torch.cuda.synchronize()
    for (name, _), e, g in zip(actors.named_parameters(), eager, grads()):
        assert rel_err(g, e) <= 1e-5, (name, rel_err(g, e))
    if autocast:
        return
    # the torch bookkeeping of the field (the proposals take no pose gradient on either route)
    model.field.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    model.zero_grad(set_to_none=True)
    step()
    for (name, _), e, t in zip(actors.named_parameters(), eager, grads()):
        print(f"[measured] hot path d{name} kernel vs torch route: max-rel {rel_err(e, t):.3e}")
        assert rel_err(e, t) <= 1e-3, (name, rel_err(e, t))


# ------------------------------------------------------------------------------------------------ 7. C ABI
def test_pose_grad_abi_rejects_bad_arguments():
    """No GPU needed: the symbol is exported, and null pointers or bad sizes return a negative code before any launch."""
    from neuradar_b200 import _lib

    lib = _lib.load()
    assert hasattr(lib, "nrb_actor_pose_grad")
    buf = (ctypes.c_float * 4096)()
    p = ctypes.addressof(buf)
    rays, iv = _lib.Rays(), _lib.Intervals()
    rays.origins = rays.directions = rays.pixel_area = p
    rays.num_rays = 4
    iv.starts = iv.ends = p
    iv.row_stride, iv.num_samples = 8, 8
    grids, samples = _lib.ActorGrids(), _lib.ActorSamples()
    grids.tables[0] = p
    grids.num_levels, grids.features_per_level, grids.log2_hashmap_size, grids.num_grids = 4, 4, 4, 1
    samples.grid_id = samples.pos = samples.std = samples.dirs = p
    launches = lib.nrb_launch_count()

    def call(rays_=rays, iv_=iv, w2b=p, A=2, index=p, scale=10.0, grids_=grids, samples_=samples, img=p, out=p):
        return lib.nrb_actor_pose_grad(None if rays_ is None else ctypes.byref(rays_), None if iv_ is None else ctypes.byref(iv_),
                                       w2b, A, index, None, scale, None if grids_ is None else ctypes.byref(grids_),
                                       None if samples_ is None else ctypes.byref(samples_), img, out, None)

    assert call(rays_=None) < 0
    assert call(iv_=None) < 0
    assert call(w2b=None) < 0
    assert call(index=None) < 0
    assert call(out=None) < 0
    assert call(img=None) < 0
    assert call(samples_=None) < 0
    assert call(grids_=None) < 0
    assert call(A=0) < 0
    assert call(scale=0.0) < 0
    assert call(img=p + 4) < 0
    grids.num_levels = 3
    assert call() < 0
    grids.num_levels = 4
    iv.num_samples = 0
    assert call() < 0
    iv.num_samples = 8
    rays.num_rays = 0
    assert call() == 0  # no rays: a valid no-op
    assert lib.nrb_launch_count() == launches
