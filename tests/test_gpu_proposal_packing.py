"""Single-feature (F = 1) grids and the proposal backward's packed scatter.

* F = 1 x-corner pairs are scattered with one 16-byte reduction whenever the floor and ceil rows share an aligned
  group of four rows (floor(x) mod 4 != 3, whatever the y / z part of the hash).  The tests place points on
  every residue of floor(x) mod 4 under hash offsets of both parities, on integral x (ceil == floor), and on tables so
  small that rows collide (2 and 4 rows per level; 2 rows is too small for a 16-byte group).
* The proposal backward scatters the samples of several rays per block in full chunks of 32 lanes, and a chunk may
  cross a ray boundary.  The tests cover sample counts that fill whole chunks and ones that do not, ray counts that are
  not a multiple of the rays per block, and the actor branch.
"""
import pytest
import torch

from oracle import neuradar_oracle as O
from tests.parity_utils import build_hot_path, oracle_params, rel_err, scaled_pixel_area, synthetic_rays

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def nb():
    import neuradar_b200

    assert torch.cuda.is_available()
    return neuradar_b200


def _x_pair_points(M: int, seed: int) -> torch.Tensor:
    """Points whose level-0 x coordinate (scaling 16) runs through every residue of floor(x) mod 4, with random y / z
    (so the hash offset takes both parities), runs of identical points and integral x."""
    g = torch.Generator().manual_seed(seed)
    k = torch.randint(0, 4, (M,), generator=g)
    r = torch.arange(M) % 4
    u = torch.rand((M,), generator=g) * 0.98 + 0.01
    x = torch.stack([(4 * k + r + u) / 16.0, torch.rand((M,), generator=g), torch.rand((M,), generator=g)], dim=-1)
    x[5:9] = x[4]  # identical points: one run of the merge
    x[16:80:2, 0] = torch.arange(32, dtype=torch.float32) % 17 / 16.0  # integral x on the level-0 grid
    return x.clamp(0, 1)


@pytest.mark.parametrize("log2T,M", [(1, 4000), (2, 4000), (12, 4000), (19, 65600)])
def test_hash_f1_x_pairs(nb, log2T, M):
    """nrb_hash_fwd / nrb_hash_bwd at F = 1 against the oracle; T = 2^19 with M >= 2^16 also scatters into the
    dense-lattice replicas of the coarse levels."""
    from neuradar_b200 import functional as Fn
    from neuradar_b200.functional import GridSpec

    L = 4
    scal = O.level_scalings(L, 16, 512)
    assert float(scal[0]) == 16.0
    spec = GridSpec(L, 1, log2T, tuple(float(s) for s in scal))
    x = _x_pair_points(M, seed=log2T)
    idx, _ = O.hash_corner_indices(x, scal, log2T)
    row_f, row_c = idx[:, 0, 3], idx[:, 0, 0]  # level 0, x pair (floor, ceil) = corners (3, 0)
    xf = torch.floor(x[:, 0] * 16.0).to(torch.int64)
    assert bool((row_f == row_c).any())  # integral x
    if log2T >= 2:
        h_parity = (row_f ^ xf) & 1
        seen = {(int(a), int(b)) for a, b in zip((xf % 4).tolist(), h_parity.tolist())}
        assert seen == {(a, b) for a in range(4) for b in range(2)}, seen
        d = row_f ^ row_c  # 1: floor(x) even; 3: floor(x) mod 4 == 1; >= 4: floor(x) mod 4 == 3 (two operations)
        assert bool((d == 1).any()) and bool((d == 3).any()) and (log2T == 2 or bool((d >= 4).any()))
    g = torch.Generator().manual_seed(M)
    table = torch.rand(((1 << log2T) * L, 1), generator=g) * 2 - 1
    dy = torch.randn((M, L), generator=g)
    t_ref = table.clone().requires_grad_(True)
    y_ref = O.hash_encode(x, t_ref, scal, log2T)
    (y_ref * dy).sum().backward()
    t_dev = table.to(DEV).requires_grad_(True)
    y = Fn.hash_encode(x.to(DEV), t_dev, spec)
    assert rel_err(y, y_ref) <= 1e-6
    (y * dy.to(DEV)).sum().backward()
    assert rel_err(t_dev.grad, t_ref.grad) <= 1e-5  # fp32 sums in a different order


@pytest.mark.parametrize("S", [33, 40, 48, 64, 96, 128])
def test_proposal_round_packed_scatter_vs_oracle(nb, S):
    """A proposal round (F = 1 grid) forward and backward against the oracle; 203 rays is not a multiple of 4, 8 or 16
    rays per block."""
    from neuradar_b200 import functional as Fn

    N = 203
    model = build_hot_path(log2_main=12, log2_prop=14, table_gain=(300.0, 2000.0), seed=4, device=DEV)
    pf = model.proposal_fields[1]
    assert pf.hashgrid.static_grid.spec.features_per_level == 1
    rays = synthetic_rays(N, seed=S)
    pa = scaled_pixel_area(rays)
    g = torch.Generator().manual_seed(S)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), S, torch.rand((N, S + 1), generator=g))
    eb = eb.contiguous()
    _, props = oracle_params(model)
    p = props[1]
    dens_ref = O.proposal_density(p, rays["origins"], rays["directions"], pa, eb[:, :-1], eb[:, 1:])
    w_ref = O.density_weights(dens_ref, (eb[:, 1:] - eb[:, :-1])[..., None])
    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), pa.to(DEV))
    dens, w = Fn.proposal_round(pf.hashgrid.static_grid.hash_table, pf.density_decoder.weight, rd,
                                Fn.SampleIntervals.from_bins(eb.to(DEV)), pf.hashgrid.static_grid.spec, 100.0)
    assert rel_err(dens, dens_ref[..., 0]) <= 1e-4
    assert rel_err(w, w_ref[..., 0]) <= 1e-4
    gw = torch.randn((N, S), generator=g)
    gd = torch.randn((N, S), generator=g) * 1e-3
    ((w * gw.to(DEV)).sum() + (dens * gd.to(DEV)).sum()).backward()
    ((w_ref[..., 0] * gw).sum() + (dens_ref[..., 0] * gd).sum()).backward()
    assert rel_err(pf.hashgrid.static_grid.hash_table.grad, p.grid.table.grad) <= 1e-3
    assert rel_err(pf.density_decoder.weight.grad, p.decoder_w.grad) <= 1e-3


@pytest.mark.parametrize("S", [33, 40, 48, 64, 96, 128])
def test_proposal_round_packed_scatter_with_actors(nb, S):
    """The same with dynamic actors: the fused round with the in-kernel actor branch against the torch bookkeeping of
    the same module, forward and every gradient (static table, decoder and actor tables)."""
    import neuradar_b200 as pkg
    from neuradar_b200.synthetic import SyntheticActors, synthetic_rays as actor_rays

    n = 203
    actors = SyntheticActors(16, device=DEV)
    pcfg = pkg.NeuRADProposalFieldConfig()
    pcfg.grid.static.log2_hashmap_size = 13
    pcfg.grid.actor.log2_hashmap_size = 9
    prop = pkg.NeuRADProposalField(pcfg, actors=actors, static_scale=100.0).to(DEV)
    prop.train()
    with torch.no_grad():
        prop.hashgrid.static_grid.hash_table.mul_(2000.0)
        for grid in prop.hashgrid.actor_grids:
            grid.hash_table.mul_(2000.0)
    r = actor_rays(n, seed=S)
    centres = actors.centres[torch.arange(n // 2) % 16].cpu()
    d = centres - r["origins"][: n // 2]
    r["directions"][: n // 2] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = (torch.linspace(0.5, 60.0, S + 1)[None, :].repeat(n, 1)).to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    g = torch.Generator(device=DEV).manual_seed(S)
    # the same actor flips in both runs (training draws them at random per call)
    prop.hashgrid.ray_flip_override = (torch.rand(n, device=DEV, generator=g) < 0.25).float() * -2 + 1
    assert prop.hashgrid.can_assign_in_kernel(proposal=True)
    gw = torch.randn((n, S, 1), device=DEV, generator=g)
    gd = torch.randn((n, S, 1), device=DEV, generator=g) * 1e-3

    def run():
        for p in prop.parameters():
            p.grad = None
        dens, w = prop.density_and_weights(rs)
        ((w * gw).sum() + (dens * gd).sum()).backward()
        return dens.detach(), w.detach(), {k: p.grad.clone() for k, p in prop.named_parameters() if p.grad is not None}

    dens_k, w_k, grads_k = run()
    rays, iv = rs.per_ray()
    assert int((prop.hashgrid.assign_actors(rays, iv, rs.times.reshape(n, -1)[:, 0]).grid_id >= 0).sum()) > 50
    prop.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    dens_t, w_t, grads_t = run()
    assert rel_err(dens_k, dens_t) <= 3e-5 and rel_err(w_k, w_t) <= 3e-5
    assert set(grads_k) == set(grads_t)
    nonzero_actor_tables = 0
    for k in grads_t:
        if float(grads_t[k].abs().max()) == 0.0:
            assert float(grads_k[k].abs().max()) == 0.0, k
            continue
        assert rel_err(grads_k[k], grads_t[k]) <= 1e-4, (k, rel_err(grads_k[k], grads_t[k]))
        nonzero_actor_tables += "actor_grids" in k
    assert nonzero_actor_tables >= 2
