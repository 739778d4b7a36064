"""GPU parity tests: every kernel behind the C ABI against the CPU oracle and the committed golden vectors.

Bars (BASELINE.md section 5): hash-table rows and searchsorted indices bit-exact at stage level (identical inputs
-> identical integers); floating-point outputs and gradients within 1e-3 relative of the fp32 reference path (most
kernels are held to 1e-5 here, the tolerance is written at each assert).
"""
import pytest
import torch

from oracle import neuradar_oracle as O
from tests.parity_utils import (
    FixedJitter,
    build_hot_path,
    make_ray_bundle,
    oracle_params,
    rel_err,
    run_path_parity,
    scaled_pixel_area,
    synthetic_rays,
)

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(scope="module")
def nb():
    import neuradar_b200

    assert torch.cuda.is_available()
    return neuradar_b200


def spec_for(nb, L, F, log2T, lo, hi):
    from neuradar_b200.functional import GridSpec

    return GridSpec(L, F, log2T, tuple(float(s) for s in O.level_scalings(L, lo, hi)))


# ------------------------------------------------------------------------------------------------ hash grid
def test_hash_indices_bit_exact(nb, golden):
    from neuradar_b200 import functional as Fn

    g = torch.Generator().manual_seed(0)
    x = torch.rand((20000, 3), generator=g)
    x[:4] = torch.tensor([[0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [0.5, 0.25, 0.125], [1.0, 0.0, 0.5]])
    for (L, lo, hi, log2T) in [(16, 16, 1024, 19), (8, 32, 8192, 22), (6, 128, 4096, 20), (4, 64, 1024, 17)]:
        spec = spec_for(nb, L, 2, log2T, lo, hi)
        got = Fn.hash_indices(x.to(DEV), spec).cpu()
        want, _ = O.hash_corner_indices(x, O.level_scalings(L, lo, hi), log2T)
        assert got.dtype == torch.int64
        assert torch.equal(got, want), f"hash rows differ for L={L} T=2^{log2T}"
    # points outside [0,1] (negative grid coordinates) hash like the reference's int64 arithmetic
    xo = (torch.rand((4096, 3), generator=g) - 0.5) * 6
    spec = spec_for(nb, 16, 2, 19, 16, 1024)
    want, _ = O.hash_corner_indices(xo, O.level_scalings(16, 16, 1024), 19)
    assert torch.equal(Fn.hash_indices(xo.to(DEV), spec).cpu(), want)


@pytest.mark.parametrize("L,F,M", [(16, 2, 1000), (16, 2, 33), (16, 2, 31), (8, 4, 4097), (4, 4, 640), (6, 1, 500)])
def test_hash_clustered_samples_run_merging(nb, L, F, M):
    """The sample-major forward and the run-merging backward on what they are built for: ray-ordered samples that
    pile into the same cells (identical points, integral coordinates, runs crossing warp boundaries), ragged M, and
    the shapes that take the level-major fallback (M < 32, L*F not a power of two).  The table gradient must equal
    the oracle's index_add whatever the grouping."""
    from neuradar_b200 import functional as Fn

    g = torch.Generator().manual_seed(M + L)
    log2T = 12
    anchors = torch.rand((max(M // 40, 1), 3), generator=g)
    x = anchors.repeat_interleave(40, dim=0)[:M].clone()
    if x.shape[0] < M:
        x = torch.cat([x, torch.rand((M - x.shape[0], 3), generator=g)])
    x = x + torch.rand((M, 3), generator=g) * torch.rand((M, 1), generator=g).pow(4) * 0.02  # mostly tiny offsets
    x[5:9] = x[4]                          # exactly identical points
    x[10:14] = torch.tensor([0.5, 0.25, 0.75])  # integral grid coordinates on the power-of-two levels
    x = x.clamp(0, 1)
    scal = O.level_scalings(L, 16, 512)
    spec = spec_for(nb, L, F, log2T, 16, 512)
    table = (torch.rand(((1 << log2T) * L, F), generator=g) * 2 - 1)
    dy = torch.randn((M, L * F), generator=g)
    t_ref = table.clone().requires_grad_(True)
    y_ref = O.hash_encode(x, t_ref, scal, log2T)
    (y_ref * dy).sum().backward()
    t_dev = table.to(DEV).requires_grad_(True)
    y = Fn.hash_encode(x.to(DEV), t_dev, spec)
    assert rel_err(y, y_ref) <= 1e-6
    (y * dy.to(DEV)).sum().backward()
    assert rel_err(t_dev.grad, t_ref.grad) <= 1e-5  # fp32 sums in a different order


@pytest.mark.parametrize("F", [1, 2, 4])
def test_hash_forward_backward_golden(nb, golden, F):
    from neuradar_b200 import functional as Fn

    g = golden("hash")
    spec = spec_for(nb, 16, F, 10, 16, 1024)
    table = g[f"F{F}_table"].to(DEV).requires_grad_(True)
    x = g["x"].to(DEV).requires_grad_(True)
    y = Fn.hash_encode(x, table, spec)
    assert rel_err(y, g[f"F{F}_y"]) <= 1e-6
    (y * g[f"F{F}_dy"].to(DEV)).sum().backward()
    assert rel_err(table.grad, g[f"F{F}_dtable"]) <= 1e-5
    assert rel_err(x.grad, g[f"F{F}_dx"]) <= 1e-5


def test_hash_module_matches_reference_api(nb, golden):
    g = golden("hash")
    enc = nb.HashEncoding(num_levels=16, min_res=16, max_res=1024, log2_hashmap_size=10, features_per_level=2).to(DEV)
    assert torch.equal(enc.scalings.cpu(), g["scalings_A"])
    assert list(enc.state_dict().keys()) == ["hash_table", "scalings"]
    with torch.no_grad():
        enc.hash_table.copy_(g["F2_table"])
    y = enc(g["x"].to(DEV).view(11, 23, 3))
    assert y.shape == (11, 23, 32)
    assert rel_err(y.reshape(-1, 32), g["F2_y"]) <= 1e-6
    big = nb.HashEncoding(num_levels=8, min_res=32, max_res=8192, log2_hashmap_size=4, features_per_level=4)
    assert big.scalings[-1].item() == 8191.0
    # shape-only tests of the reference (tests/field_components/test_encodings.py:142-168)
    enc2 = nb.HashEncoding(num_levels=4, features_per_level=4, log2_hashmap_size=5).to(DEV)
    assert enc2(torch.rand((10, 3), device=DEV)).shape == (10, 16)
    assert enc2.get_out_dim() == 16


def test_hash_linearity_full_size(nb):
    """Size-independent property at BASELINE config-2 size: the encoding is linear in the table."""
    from neuradar_b200 import functional as Fn

    spec = spec_for(nb, 16, 2, 19, 16, 1024)
    M = 65536 * 48
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.rand((M, 3), device=DEV, generator=g)
    t1 = torch.randn((spec.rows, 2), device=DEV, generator=g)
    t2 = torch.randn((spec.rows, 2), device=DEV, generator=g)
    y1, y2 = Fn.hash_encode(x, t1, spec), Fn.hash_encode(x, t2, spec)
    y12 = Fn.hash_encode(x, 0.5 * t1 - 2.0 * t2, spec)
    assert float((y12 - (0.5 * y1 - 2.0 * y2)).abs().max()) <= 1e-4
    # a constant table interpolates to the constant (partition of unity of the trilinear weights)
    yc = Fn.hash_encode(x, torch.full((spec.rows, 2), 3.0, device=DEV), spec)
    assert float((yc - 3.0).abs().max()) <= 1e-5
    # backward is the adjoint of forward: <enc(T), dY> == <T, enc^T(dY)>
    dy = torch.randn((M, 32), device=DEV, generator=g)
    t1.requires_grad_(True)
    (Fn.hash_encode(x, t1, spec) * dy).sum().backward()
    lhs = (y1.double() * dy.double()).sum()
    rhs = (t1.detach().double() * t1.grad.double()).sum()
    assert abs(lhs.item() - rhs.item()) <= 1e-4 * abs(lhs.item())


def test_frustum_gaussians(nb):
    from neuradar_b200 import functional as Fn

    rays = synthetic_rays(512, seed=5)
    pa = scaled_pixel_area(rays)
    sb, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), 64, None)
    eb = eb.contiguous()
    mean, std = O.fast_isotropic_gaussian(rays["origins"], rays["directions"], eb[:, :-1], eb[:, 1:], pa)
    cmean, cstd = O.contract(mean, std, 100.0)
    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), pa.to(DEV))
    x, s = Fn.frustum_gaussians(rd, Fn.SampleIntervals.from_bins(eb.to(DEV)), 100.0)
    assert torch.equal(x.cpu(), cmean.reshape(-1, 3)), "contracted sample means must be bit-exact (they feed the hash)"
    assert rel_err(s, cstd.reshape(-1)) <= 1e-5
    # generic Frustums API
    fr = nb.Frustums(origins=rays["origins"].to(DEV)[:, None, :], directions=rays["directions"].to(DEV)[:, None, :],
                     starts=eb[:, :-1, None].to(DEV), ends=eb[:, 1:, None].to(DEV), pixel_area=pa.to(DEV)[:, None, :])
    gs = fr.get_fast_isotropic_gaussian(1, contraction_scale=100.0)
    assert gs.mean.shape == (512, 64, 1, 3) and torch.equal(gs.mean.reshape(-1, 3), x)
    world = fr.get_fast_isotropic_gaussian(1)
    assert rel_err(world.mean, mean[:, :, None, :]) <= 1e-6


# ------------------------------------------------------------------------------------------------ MLP / SH
@pytest.mark.parametrize("tag,cfg", [("geo", (32, 2, 32, 33)), ("feat", (48, 3, 32, 32)), ("lidar", (48, 3, 32, 2)),
                                     ("radar", (48, 3, 16, 3))])
def test_mlp_golden(nb, golden, tag, cfg):
    g = golden("kats")
    i, n, w, o = cfg
    m = nb.MLP(in_dim=i, num_layers=n, layer_width=w, out_dim=o).to(DEV)
    assert [k for k in m.state_dict()] == [f"layers.{k}.{p}" for k in range(n) for p in ("weight", "bias")]
    with torch.no_grad():
        for k, layer in enumerate(m.layers):
            layer.weight.copy_(g[f"mlp_{tag}_w{k}"])
            layer.bias.copy_(g[f"mlp_{tag}_b{k}"])
    x = g[f"mlp_{tag}_x"].to(DEV).requires_grad_(True)
    y = m(x)
    assert rel_err(y, g[f"mlp_{tag}_y"]) <= 1e-5
    (y * g[f"mlp_{tag}_dy"].to(DEV)).sum().backward()
    assert rel_err(x.grad, g[f"mlp_{tag}_dx"]) <= 1e-5
    for k, layer in enumerate(m.layers):
        assert rel_err(layer.weight.grad, g[f"mlp_{tag}_dw{k}"]) <= 1e-5
        assert rel_err(layer.bias.grad, g[f"mlp_{tag}_db{k}"]) <= 1e-5


def test_mlp_many_tiles_and_ragged(nb):
    torch.manual_seed(0)
    m = nb.MLP(in_dim=32, num_layers=2, layer_width=32, out_dim=33).to(DEV)
    for M in (1, 127, 128, 129, 100003):
        x = torch.randn((M, 32), device=DEV, requires_grad=True)
        y = m(x)
        xr = x.detach().cpu().requires_grad_(True)
        ws = [l.weight.detach().cpu().requires_grad_(True) for l in m.layers]
        bs = [l.bias.detach().cpu().requires_grad_(True) for l in m.layers]
        yr = O.mlp(xr, ws, bs)
        assert rel_err(y, yr) <= 1e-5
        dy = torch.randn_like(yr)
        m.zero_grad()
        (y * dy.to(DEV)).sum().backward()
        (yr * dy).sum().backward()
        assert rel_err(x.grad, xr.grad) <= 1e-5
        assert rel_err(m.layers[0].weight.grad, ws[0].grad) <= 2e-5
        assert rel_err(m.layers[1].bias.grad, bs[1].grad) <= 2e-5
    assert m(torch.empty((0, 32), device=DEV)).shape == (0, 33)


def test_sh16(nb, golden):
    from neuradar_b200 import functional as Fn

    g = golden("kats")
    assert rel_err(Fn.sh16(g["sh_dirs"].to(DEV), normalize_to_unit_cube=True), g["sh_out"]) <= 1e-6
    enc = nb.SHEncoding(levels=4)
    assert rel_err(enc(g["sh_dirs"].to(DEV)), g["sh_enc"]) <= 1e-6


# ------------------------------------------------------------------------------------------------ samplers
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_samplers_golden(nb, golden, mode):
    from neuradar_b200 import functional as Fn

    g = golden("samplers")
    N = 96
    rd = Fn.RayData(torch.zeros((N, 3), device=DEV), torch.ones((N, 3), device=DEV), torch.ones((N,), device=DEV),
                    g["nears"].to(DEV), g["fars"].to(DEV))
    j0 = g[f"{mode}_j0"].to(DEV) if mode == "train" else None
    j1 = g[f"{mode}_j1"].to(DEV) if mode == "train" else None
    sb0, eb0 = Fn.spaced_bins(rd, 64, j0, -1.0, 0.1)
    assert torch.equal(sb0.cpu(), g[f"{mode}_sbins0"]), "initial spacing bins must be bit-exact"
    assert torch.equal(eb0.cpu(), g[f"{mode}_ebins0"]), "initial euclidean bins must be bit-exact"
    w = g[f"{mode}_w"][..., 0].to(DEV)
    sb1, eb1, inds, cdf = Fn.pdf_sample(rd, w, sb0, 48, j1, -1.0, 0.1, return_debug=True)
    # stage-level exactness: the kernel's indices are torch.searchsorted of the kernel's own cdf and the exact u
    u = O.pdf_u(N, 48, None if j1 is None else j1.cpu())
    assert torch.equal(inds.cpu(), torch.searchsorted(cdf.cpu().contiguous(), u, side="right"))
    # and the cdf / indices / bins agree with the reference's
    ref_cdf = O.pdf_cdf(g[f"{mode}_w"][..., 0])
    assert float((cdf.cpu() - ref_cdf).abs().max()) <= 2e-7
    ref_bins, ref_inds = O.pdf_invert(ref_cdf, u, g[f"{mode}_sbins0"])
    assert float((inds.cpu() != ref_inds).float().mean()) <= 1e-3
    # bins in low-density intervals amplify the 1-ulp cdf difference by 1/pdf (<= 1/histogram_padding)
    assert float((sb1.cpu() - g[f"{mode}_sbins1"]).abs().max()) <= 5e-6
    # stage level: the kernel's euclidean bins are the reference's spacing_to_euclidean_fn of the kernel's own bins
    sp = O.Spacing(O.power_fn(g["nears"] * 0.1, -1.0), O.power_fn(g["fars"] * 0.1, -1.0), -1.0, 0.1)
    assert torch.equal(eb1.cpu(), sp.to_euclidean(sb1.cpu()))
    # end to end the inverse power transform amplifies bin differences by up to ~1e7 m per unit of s at the far end
    assert rel_err(eb1, g[f"{mode}_ebins1"]) <= 1e-3
    assert bool((sb1[:, 1:] >= sb1[:, :-1]).all()), "sampled bins must be sorted"


def test_pdf_indices_mismatch_rate_at_scale(nb):
    """393 K inverse-cdf look-ups against the oracle on the same weights, bins and u: the kernel's cdf differs from the
    reference's by at most one ulp (a different but fixed summation order), so an index can only differ where u falls
    within that ulp of a cdf value; the rate of such samples must stay at the 1e-5 level, and every one of them must be
    an adjacent bin."""
    from neuradar_b200 import functional as Fn

    N, S_in, S_out = 8192, 64, 48
    g = torch.Generator().manual_seed(21)
    w = torch.rand((N, S_in), generator=g).pow(4) * (torch.rand((N, 1), generator=g) * 3)
    nears, fars = torch.zeros((N,)), torch.full((N,), 2.0e4)
    rd = Fn.RayData(torch.zeros((N, 3), device=DEV), torch.ones((N, 3), device=DEV), torch.ones((N,), device=DEV),
                    nears.to(DEV), fars.to(DEV))
    j0, j1 = torch.rand((N, S_in + 1), generator=g), torch.rand((N, 1), generator=g)
    sb0, _ = Fn.spaced_bins(rd, S_in, j0.to(DEV), -1.0, 0.1)
    sb1, eb1, inds, cdf = Fn.pdf_sample(rd, w.to(DEV), sb0, S_out, j1.to(DEV), -1.0, 0.1, return_debug=True)
    u = O.pdf_u(N, S_out, j1)
    ref_cdf = O.pdf_cdf(w)
    assert float((cdf.cpu() - ref_cdf).abs().max()) <= 2.4e-7
    _, ref_inds = O.pdf_invert(ref_cdf, u, sb0.cpu())
    diff = inds.cpu() != ref_inds
    rate = float(diff.float().mean())
    assert rate <= 2e-5, rate
    assert int((inds.cpu() - ref_inds).abs().max()) <= 1
    # stage-level exactness (the bit-exact bar for index work): the kernel's indices ARE searchsorted of its own cdf
    assert torch.equal(inds.cpu(), torch.searchsorted(cdf.cpu().contiguous(), u, side="right"))


def test_pdf_sampler_known_answer(nb, golden):
    from neuradar_b200 import functional as Fn

    g = golden("samplers")
    rd = Fn.RayData(torch.zeros((2, 3), device=DEV), torch.ones((2, 3), device=DEV), torch.ones((2,), device=DEV),
                    torch.full((2,), 2.0, device=DEV), torch.full((2,), 6.0, device=DEV))
    sb, eb = Fn.pdf_sample(rd, g["kat_w"][..., 0].to(DEV), g["kat_in_sbins"].to(DEV), 4, None, -1.0, 0.1)
    assert float((sb.cpu() - g["kat_sbins"]).abs().max()) <= 2.5e-7
    torch.testing.assert_close(sb.cpu()[1], torch.tensor([0.1, 0.3, 0.5, 0.7, 0.9]), rtol=1e-6, atol=1e-7)


def test_sampler_modules(nb):
    rays = synthetic_rays(300, seed=8)
    rb = make_ray_bundle(rays, DEV)
    rb.fars.clamp_max_(20000.0)
    ps = nb.PowerSampler(lambda_=-1.0, scaling=0.1)
    ps.eval()
    rs = ps(rb, num_samples=64)
    assert rs.shape == (300, 64)
    assert rs.frustums.origins.shape == (300, 64, 3) and rs.frustums.origins.stride(1) == 0
    assert rs.frustums.starts.shape == (300, 64, 1) and rs.deltas.shape == (300, 64, 1)
    eb = torch.cat([rs.frustums.starts[..., 0], rs.frustums.ends[..., -1:, 0]], -1)
    assert rel_err(rs.spacing_to_euclidean_fn(rs.spacing_bins), eb) <= 1e-5
    pdf = nb.PDFSampler(include_original=False, single_jitter=True)
    pdf.eval()
    rs2 = pdf(rb, rs, torch.rand((300, 64, 1), device=DEV), num_samples=48)
    assert rs2.shape == (300, 48)
    assert bool((rs2.frustums.ends >= rs2.frustums.starts).all())
    # reference test: "just check that it doesn't crash" + sample count (tests/model_components/test_ray_sampler.py)
    assert rs2.frustums.get_positions().shape == (300, 48, 3)


# ------------------------------------------------------------------------------------------------ compositing
def test_density_weights_golden(nb, golden):
    from neuradar_b200 import functional as Fn

    g = golden("kats")
    bins = g["gw_bins"].to(DEV)
    dens = g["gw_dens"][..., 0].to(DEV).requires_grad_(True)
    w = Fn.density_weights(dens, Fn.SampleIntervals.from_bins(bins))
    ref = g["gw_w"][..., 0]
    finite = torch.isfinite(ref)
    assert rel_err(w.cpu()[finite], ref[finite]) <= 1e-5
    (w * g["gw_dw"][..., 0].to(DEV)).sum().backward()
    gref = g["gw_ddens"][..., 0]
    ok = torch.isfinite(gref) & (g["gw_dens"][..., 0] < 1e20)
    assert rel_err(dens.grad.cpu()[ok], gref[ok]) <= 1e-4
    kat = Fn.density_weights(torch.tensor([[1.0, 2.0, 0.5, 3.0]], device=DEV),
                             Fn.SampleIntervals.from_bins(torch.tensor([[0.0, 0.5, 1.0, 2.0, 3.0]], device=DEV)))
    torch.testing.assert_close(kat.cpu()[0], torch.tensor([0.39346933, 0.3834005, 0.08779488, 0.12859733]), rtol=1e-6, atol=0)


def test_ray_samples_weight_api(nb, golden):
    g = golden("kats")
    w, T = nb.RaySamples.get_weights_and_transmittance_from_alphas(g["alpha2_in"].to(DEV))
    assert w.shape == (37, 48, 1) and T.shape == (37, 49, 1)
    assert rel_err(w, g["alpha2_w"]) <= 1e-5
    assert rel_err(T, g["alpha2_T"]) <= 1e-5
    w1 = nb.RaySamples.get_weights_and_transmittance_from_alphas(g["alpha_in"].to(DEV), weights_only=True)
    torch.testing.assert_close(w1.cpu().flatten(), torch.tensor([0.1, 0.45000005, 0.40500015, 0.0090000136]), rtol=1e-6, atol=0)
    from neuradar_b200 import nerfacc_compat

    wn, tn = nerfacc_compat.render_weight_from_alpha(g["alpha2_in"][..., 0].to(DEV))
    w0, t0 = O.alpha_weights(g["alpha2_in"][..., 0], eps=0.0)
    assert rel_err(wn, w0) <= 1e-5 and rel_err(tn, t0[:, :-1]) <= 1e-5


def test_renderers_golden(nb, golden):
    g = golden("kats")
    bins = g["gw_bins"].to(DEV)
    rb = nb.RayBundle(origins=torch.zeros((37, 3), device=DEV), directions=torch.ones((37, 3), device=DEV),
                      pixel_area=torch.ones((37, 1), device=DEV))
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    feats, w = g["rend_feats"].to(DEV), g["rend_w"].to(DEV)
    assert rel_err(nb.FeatureRenderer()(features=feats, weights=w), g["rend_feature"]) <= 1e-5
    assert rel_err(nb.AccumulationRenderer()(weights=w), g["rend_acc"]) <= 1e-5
    assert rel_err(nb.DepthRenderer(method="expected")(weights=w, ray_samples=rs), g["rend_depth_expected"]) <= 1e-5
    assert rel_err(nb.DepthRenderer(method="median")(weights=w * 3, ray_samples=rs), g["rend_depth_median"]) <= 1e-6
    # the reference's renderer tests use loose inequalities (tests/model_components/test_renderers.py)
    acc = nb.AccumulationRenderer()(weights=torch.ones((3, 5, 1), device=DEV))
    assert bool((acc > 0.9).all())


@pytest.mark.parametrize("eps", [0.0, 1e-7])
@pytest.mark.parametrize("S", [48, 128, 33])
def test_alpha_composite_forward_backward(nb, eps, S):
    from neuradar_b200 import functional as Fn

    g = torch.Generator().manual_seed(S)
    N, C = 257, 32
    alphas = torch.rand((N, S), generator=g) ** 3
    alphas[0] = 0.0
    alphas[1, 5] = 1.0  # opaque sample: later transmittance is exactly 0 when eps == 0
    alphas[2] = 1.0
    feats = torch.randn((N, S, C), generator=g)
    bins = torch.cumsum(torch.rand((N, S + 1), generator=g), dim=-1)
    a_ref = alphas.clone().requires_grad_(True)
    f_ref = feats.clone().requires_grad_(True)
    ref = O.composite(a_ref, f_ref, bins[:, :-1], bins[:, 1:], eps)
    a = alphas.to(DEV).requires_grad_(True)
    f = feats.to(DEV).requires_grad_(True)
    w, feat, depth, acc = Fn.alpha_composite(a, f, Fn.SampleIntervals.from_bins(bins.to(DEV)), eps, True)
    assert rel_err(feat, ref["features"]) <= 1e-5
    assert rel_err(depth, ref["depth"][:, 0]) <= 1e-5
    assert rel_err(acc, ref["accumulation"][:, 0]) <= 1e-5
    assert rel_err(w[:, :-1], ref["weights"][..., 0]) <= 1e-5
    gw = torch.randn((N, S - 1), generator=g)
    gf = torch.randn((N, C), generator=g)
    gd = torch.randn((N,), generator=g)
    ga = torch.randn((N,), generator=g)
    loss = (w[:, :-1] * gw.to(DEV)).sum() + (feat * gf.to(DEV)).sum() + (depth * gd.to(DEV)).sum() + (acc * ga.to(DEV)).sum()
    loss.backward()
    lref = (ref["weights"][..., 0] * gw).sum() + (ref["features"] * gf).sum() + (ref["depth"][:, 0] * gd).sum() \
        + (ref["accumulation"][:, 0] * ga).sum()
    lref.backward()
    assert rel_err(f.grad, f_ref.grad) <= 1e-5
    assert rel_err(a.grad, a_ref.grad) <= 1e-4


# ------------------------------------------------------------------------------------------------ fields / whole path
def test_proposal_round_vs_oracle(nb):
    model = build_hot_path(log2_main=12, log2_prop=14, table_gain=(300.0, 2000.0), seed=4, device=DEV)
    rays = synthetic_rays(384, seed=6)
    pa = scaled_pixel_area(rays)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), 64, torch.rand((384, 65)))
    eb = eb.contiguous()
    fld, props = oracle_params(model)
    p = props[1]
    dens_ref = O.proposal_density(p, rays["origins"], rays["directions"], pa, eb[:, :-1], eb[:, 1:])
    w_ref = O.density_weights(dens_ref, (eb[:, 1:] - eb[:, :-1])[..., None])
    from neuradar_b200 import functional as Fn

    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), pa.to(DEV))
    pf = model.proposal_fields[1]
    dens, w = Fn.proposal_round(pf.hashgrid.static_grid.hash_table, pf.density_decoder.weight, rd,
                                Fn.SampleIntervals.from_bins(eb.to(DEV)), pf.hashgrid.static_grid.spec, 100.0)
    assert rel_err(dens, dens_ref[..., 0]) <= 1e-4
    assert rel_err(w, w_ref[..., 0]) <= 1e-4
    gw = torch.randn((384, 64))
    (w * gw.to(DEV)).sum().backward()
    (w_ref[..., 0] * gw).sum().backward()
    assert rel_err(pf.hashgrid.static_grid.hash_table.grad, p.grid.table.grad) <= 1e-3
    assert rel_err(pf.density_decoder.weight.grad, p.decoder_w.grad) <= 1e-3
    # the unfused API (get_density + RaySamples.get_weights) gives the same numbers
    rb = make_ray_bundle(rays, DEV)
    rb.pixel_area = pa.to(DEV)
    rs = rb.get_ray_samples(bin_starts=eb[:, :-1, None].to(DEV), bin_ends=eb[:, 1:, None].to(DEV))
    d2, _ = pf.get_density(rs)
    assert d2.shape == (384, 64, 1) and rel_err(d2, dens_ref) <= 1e-4
    assert rel_err(rs.get_weights(d2), w_ref) <= 1e-4


def test_maximum_samples_per_ray(nb):
    """NRB_MAX_SAMPLES = 256 samples per ray is the most the warp-per-ray kernels hold (8 chunks of 32 lanes): 256 must agree
    with the oracle (proposal round, PDF sampling, compositing), 257 must be refused with an error, not truncated."""
    import neuradar_b200 as pkg
    from neuradar_b200 import functional as Fn

    N, S = 96, 256
    model = build_hot_path(log2_main=12, log2_prop=13, table_gain=(300.0, 2000.0), seed=4, device=DEV)
    rays = synthetic_rays(N, seed=16)
    pa = scaled_pixel_area(rays)
    g = torch.Generator().manual_seed(2)
    sb, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), S, torch.rand((N, S + 1), generator=g))
    eb = eb.contiguous()
    _, props = oracle_params(model)
    dens_ref = O.proposal_density(props[1], rays["origins"], rays["directions"], pa, eb[:, :-1], eb[:, 1:])
    w_ref = O.density_weights(dens_ref, (eb[:, 1:] - eb[:, :-1])[..., None])
    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), pa.to(DEV), rays["nears"].to(DEV),
                    rays["fars"].clamp_max(20000.0).to(DEV))
    pf = model.proposal_fields[1]
    dens, w = Fn.proposal_round(pf.hashgrid.static_grid.hash_table, pf.density_decoder.weight, rd,
                                Fn.SampleIntervals.from_bins(eb.to(DEV)), pf.hashgrid.static_grid.spec, 100.0)
    assert rel_err(dens, dens_ref[..., 0]) <= 1e-4 and rel_err(w, w_ref[..., 0]) <= 1e-4
    (w * w).sum().backward()
    (w_ref * w_ref).sum().backward()
    assert rel_err(pf.hashgrid.static_grid.hash_table.grad, props[1].grid.table.grad) <= 1e-3
    # PDF sampling from 256 input bins into 256 output bins
    j1 = torch.rand((N, 1), generator=g)
    sb1, eb1, inds, cdf = Fn.pdf_sample(rd, w.detach(), sb.to(DEV), S, j1.to(DEV), -1.0, 0.1, return_debug=True)
    u = O.pdf_u(N, S, j1)
    assert torch.equal(inds.cpu(), torch.searchsorted(cdf.cpu().contiguous(), u, side="right"))
    assert float((cdf.cpu() - O.pdf_cdf(w.detach().cpu())).abs().max()) <= 5e-7
    assert bool((sb1[:, 1:] >= sb1[:, :-1]).all())
    # compositing of 256 samples
    alpha = torch.rand((N, S), generator=g) * 0.05
    feats = torch.randn((N, S, 32), generator=g)
    wts, feat, depth, acc = Fn.alpha_composite(alpha.to(DEV), feats.to(DEV), Fn.SampleIntervals.from_bins(eb.to(DEV)),
                                               trans_eps=0.0, sky_sample=True)
    ref_w, _ = O.alpha_weights(alpha, eps=0.0)
    assert rel_err(wts[:, :-1], ref_w[:, :-1]) <= 1e-5
    # one sample more than the kernels hold: refused
    eb257 = torch.cat([eb, eb[:, -1:] + 1.0], dim=-1).to(DEV)
    with pytest.raises(pkg._lib.NeuradarB200Error):
        Fn.proposal_round(pf.hashgrid.static_grid.hash_table, pf.density_decoder.weight, rd,
                          Fn.SampleIntervals.from_bins(eb257), pf.hashgrid.static_grid.spec, 100.0)
    with pytest.raises(pkg._lib.NeuradarB200Error):
        Fn.alpha_composite(torch.rand((N, S + 1), device=DEV), torch.randn((N, S + 1, 32), device=DEV),
                           Fn.SampleIntervals.from_bins(eb257), trans_eps=0.0, sky_sample=True)


def test_field_forward_vs_oracle(nb):
    model = build_hot_path(log2_main=14, log2_prop=12, table_gain=(300.0, 2000.0), seed=9, device=DEV)
    rays = synthetic_rays(320, seed=10)
    pa = scaled_pixel_area(rays)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), 48, torch.rand((320, 49)))
    eb = eb.contiguous()
    fld, _ = oracle_params(model)
    ref = O.field_forward(fld, rays["origins"], rays["directions"], pa, eb[:, :-1], eb[:, 1:])
    rb = make_ray_bundle(rays, DEV)
    rb.pixel_area = pa.to(DEV)
    rs = rb.get_ray_samples(bin_starts=eb[:, :-1, None].to(DEV), bin_ends=eb[:, 1:, None].to(DEV))
    out = model.field(rs)
    assert out[nb.FieldHeadNames.FEATURE].shape == (320, 48, 32)
    assert rel_err(out[nb.FieldHeadNames.FEATURE], ref["feature"]) <= 1e-4
    assert rel_err(out[nb.FieldHeadNames.SDF], ref["sdf"]) <= 1e-4
    assert float((out[nb.FieldHeadNames.ALPHA].cpu() - ref["alpha"]).abs().max()) <= 1e-4


@pytest.mark.parametrize("train", [True, False])
def test_whole_path_vs_oracle(nb, train):
    report = run_path_parity(num_rays=512, device=DEV, seed=11, train=train)
    assert report["ok"], report


@pytest.mark.parametrize("num_rays", [1, 3, 131])
def test_whole_path_ragged_ray_counts_vs_oracle(nb, num_rays):
    """Ray counts that leave every kernel with a partial last tile / warp / block (a single ray: 48 samples in a 128-sample
    tile; 131 rays: 6288 samples = 49 tiles + 16 rows)."""
    report = run_path_parity(num_rays=num_rays, device=DEV, seed=5 + num_rays, train=True)
    assert report["ok"], report


def test_whole_path_zero_rays(nb):
    """An empty batch (a rank whose shard is empty, the tail chunk of an inference sweep) passes through every kernel
    entry point without a launch and yields empty outputs of the right shapes, forward and backward."""
    model = build_hot_path(log2_main=10, log2_prop=10, device=DEV)
    model.train()
    rays = synthetic_rays(4, seed=1)
    rb = make_ray_bundle({k: v[:0] for k, v in rays.items()}, DEV)
    out = model(rb)
    assert out["features"].shape == (0, 32) and out["depth"].shape == (0, 1) and out["accumulation"].shape == (0, 1)
    assert [w.shape for w in out["weights_list"]] == [(0, 64, 1), (0, 48, 1), (0, 47, 1)]  # (the sky sample is dropped)
    loss = out["features"].sum() + out["depth"].sum() + sum(w.sum() for w in out["weights_list"])
    loss.backward()
    for name, p in model.named_parameters():
        assert p.grad is None or float(p.grad.abs().sum()) == 0.0, name


def test_whole_path_with_regularisers_vs_oracle(nb):
    """The step as the model trains it: path + interlevel + distortion losses, gradients of every parameter."""
    report = run_path_parity(num_rays=384, device=DEV, seed=17, train=True, with_losses=True)
    assert report["ok"], report


def test_whole_path_under_autocast_vs_oracle(nb):
    """The step under torch.autocast(float16), as the reference's trainer runs it (engine/trainer.py:564): outputs and
    every gradient still within the 1e-3 bar of the fp32 oracle."""
    with torch.autocast("cuda", dtype=torch.float16):
        report = run_path_parity(num_rays=384, device=DEV, seed=19, train=True)
    assert report["ok"], report


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_whole_path_golden(nb, golden, mode):
    """The path on the reference's own outputs (tests/golden/path.npz, made by running the reference)."""
    g = golden("path")
    model = build_hot_path(log2_main=10, log2_prop=10, late_binding=False, device=DEV)
    sd = {"field.hashgrid.static_grid.hash_table": g["main_table"], "field.sdf_to_density.beta": g["beta"]}
    for k in range(2):
        sd[f"field.mlp_geo.layers.{k}.weight"], sd[f"field.mlp_geo.layers.{k}.bias"] = g[f"geo_w{k}"], g[f"geo_b{k}"]
    for k in range(3):
        sd[f"field.mlp_feature.layers.{k}.weight"], sd[f"field.mlp_feature.layers.{k}.bias"] = g[f"feat_w{k}"], g[f"feat_b{k}"]
    for i in range(2):
        sd[f"proposal_fields.{i}.hashgrid.static_grid.hash_table"] = g[f"prop{i}_table"]
        sd[f"proposal_fields.{i}.density_decoder.weight"] = g[f"prop{i}_w"]
    missing = model.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all(k.endswith(("scalings", "beta_min")) for k in missing.missing_keys)
    model.train(mode == "train")
    N = 64
    rb = nb.RayBundle(origins=g["origins"].to(DEV), directions=g["directions"].to(DEV), pixel_area=g["pixel_area"].to(DEV),
                      nears=g["nears"].to(DEV), fars=g["fars"].to(DEV), times=g["times"].to(DEV), metadata={})
    pre = mode + "_"
    # golden rays were generated without the x9 camera scaling: bypass _scale_pixel_area
    model._scale_pixel_area = lambda bundle: None
    if mode == "train":
        with FixedJitter([g[f"{pre}jitter{i}"] for i in range(3)]):
            out = model(rb)
    else:
        with torch.no_grad():
            out = model(rb)
    # the golden composite uses the in-tree 1e-7 formula; the model uses nerfacc's (eps=0): <=6e-6 apart (SURVEY 8a C3)
    assert rel_err(out["features"], g[f"{pre}features"]) <= 1e-3
    assert rel_err(out["depth"], g[f"{pre}depth"]) <= 1e-3
    assert rel_err(out["accumulation"], g[f"{pre}accumulation"]) <= 1e-3
    if mode == "train":
        for i in range(2):
            assert rel_err(out["weights_list"][i], g[f"{pre}prop_w{i}"]) <= 1e-3
            rs = out["ray_samples_list"][i]
            assert float((rs.spacing_bins.cpu() - g[f"{pre}sbins{i}"]).abs().max()) <= 2e-6
        assert rel_err(out["weights_list"][2], g[f"{pre}weights"]) <= 1e-3
        nb.bench_loss(out).backward()
        assert rel_err(model.field.hashgrid.static_grid.hash_table.grad, g[f"{pre}d_main_table"]) <= 1e-3
        for k in range(2):
            assert rel_err(model.field.mlp_geo.layers[k].weight.grad, g[f"{pre}d_geo_w{k}"]) <= 1e-3
        for k in range(3):
            assert rel_err(model.field.mlp_feature.layers[k].weight.grad, g[f"{pre}d_feat_w{k}"]) <= 1e-3
            assert rel_err(model.field.mlp_feature.layers[k].bias.grad, g[f"{pre}d_feat_b{k}"]) <= 1e-3
        assert rel_err(model.field.sdf_to_density.beta.grad, g[f"{pre}d_beta"]) <= 1e-3
        for i in range(2):
            assert rel_err(model.proposal_fields[i].hashgrid.static_grid.hash_table.grad, g[f"{pre}d_prop{i}_table"]) <= 1e-3
            assert rel_err(model.proposal_fields[i].density_decoder.weight.grad, g[f"{pre}d_prop{i}_w"]) <= 1e-3


def test_full_size_properties(nb):
    """BASELINE config 2 (65536 mixed rays, 2^19 main table, 48 samples): size-independent invariants."""
    model = build_hot_path(device=DEV)  # cfg-A main grid, cfg-P proposals, (64,48)/48 samples
    model.train()
    rays = synthetic_rays(65536, seed=42)
    out = model(make_ray_bundle(rays, DEV))
    acc = out["accumulation"]
    assert out["features"].shape == (65536, 32) and out["depth"].shape == (65536, 1)
    assert bool(torch.isfinite(out["features"]).all()) and bool(torch.isfinite(out["depth"]).all())
    assert float(acc.min()) >= 0.0 and float(acc.max()) <= 1.0 + 1e-5
    for w in out["weights_list"]:
        assert float(w.min()) >= 0.0 and float(w.sum(dim=1).max()) <= 1.0 + 1e-4
    for rs in out["ray_samples_list"][:2]:
        eb = rs.euclidean_bins
        assert bool((eb[:, 1:] >= eb[:, :-1]).all()) and float(eb.min()) >= 0.0 and float(eb.max()) <= 20000.0 * (1 + 1e-3)  # the inverse power transform amplifies 1 ulp of s by ~1e3 at the far end
    nb.bench_loss(out).backward()
    for name, p in model.named_parameters():
        if name.startswith("proposal_fields.0"):
            assert p.grad is None  # never evaluated (late-binding density_fns, SURVEY.md section 0 item 4)
        else:
            assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name
    assert float(model.field.hashgrid.static_grid.hash_table.grad.abs().sum()) > 0


# ------------------------------------------------------------------------------------------------ other BASELINE configs
def test_config4_large_scene_shapes_vs_oracle(nb):
    """BASELINE config 4 without actors at reduced table size: main grid L8/F4 (res 32..8191), 128 samples per ray,
    proposals (128, 64).  Exercises F=4 gathers/reductions, 4-chunk warp scans and the 8191 top level."""
    S0, S1, S2 = 128, 64, 128
    model = build_hot_path(log2_main=15, log2_prop=14, num_proposal_samples=(S0, S1), num_nerf_samples=S2, main_levels=8,
                           main_features=4, main_res=(32, 8192), table_gain=(300.0, 2000.0), seed=5, device=DEV)
    assert model.field.hashgrid.static_grid.scalings[-1].item() == 8191.0
    model.train()
    N = 300
    rays = synthetic_rays(N, seed=13)
    g = torch.Generator().manual_seed(14)
    jit = [torch.rand((N, S0 + 1), generator=g), torch.rand((N, 1), generator=g), torch.rand((N, 1), generator=g)]
    fld, props = oracle_params(model)
    with FixedJitter(jit):
        out = model(make_ray_bundle(rays, DEV))
    cfg = O.PathConfig(num_proposal_samples=(S0, S1), num_nerf_samples=S2)
    ref = O.nff_forward(fld, [props[-1], props[-1]], rays["origins"], rays["directions"], scaled_pixel_area(rays),
                        rays["nears"], rays["fars"], cfg, jit, composite_eps=0.0)
    assert rel_err(out["features"], ref.features) <= 1e-3
    assert rel_err(out["depth"], ref.depth) <= 1e-3
    assert rel_err(out["accumulation"], ref.accumulation) <= 1e-3
    for i in range(3):
        assert rel_err(out["weights_list"][i], ref.weights_list[i]) <= 1e-3
    nb.bench_loss(out).backward()
    O.bench_loss(ref).backward()
    assert rel_err(model.field.hashgrid.static_grid.hash_table.grad, fld.grid.table.grad) <= 1e-3
    assert rel_err(model.field.mlp_geo.layers[0].weight.grad, fld.geo_w[0].grad) <= 1e-3
    assert rel_err(model.proposal_fields[1].hashgrid.static_grid.hash_table.grad, props[1].grid.table.grad) <= 1e-3


def test_config5_inference_sweep(nb):
    """BASELINE config 5: radar point-cloud render sweep, eval mode (deterministic u), forward only, chunks of 32768
    rays (eval_num_rays_per_chunk, configs/method_configs.py:380).  One chunk is compared with the oracle on a slice;
    the sweep itself checks size-independent invariants and chunking invariance."""
    model = build_hot_path(log2_main=16, log2_prop=16, table_gain=(300.0, 2000.0), seed=6, device=DEV)
    model.eval()
    rays = synthetic_rays(4 * 32768, seed=21, mix="radar")
    depth, acc = [], []
    with torch.no_grad():
        for lo in range(0, 4 * 32768, 32768):
            chunk = {k: v[lo : lo + 32768] for k, v in rays.items()}
            out = model(make_ray_bundle(chunk, DEV))
            depth.append(out["depth"])
            acc.append(out["accumulation"])
        whole = model(make_ray_bundle({k: v[:65536] for k, v in rays.items()}, DEV))
    depth, acc = torch.cat(depth), torch.cat(acc)
    assert bool(torch.isfinite(depth).all()) and float(acc.min()) >= 0 and float(acc.max()) <= 1 + 1e-5
    assert torch.equal(whole["depth"], depth[:65536]), "eval mode is deterministic: chunking must not change a bit"
    # radar point head (models/neuradar.py:1025-1029) on the rendered depth vs the oracle, on a 512-ray slice
    sl = {k: v[:512] for k, v in rays.items()}
    fld, props = oracle_params(model)
    ref = O.nff_forward(fld, [props[-1], props[-1]], sl["origins"], sl["directions"], scaled_pixel_area(sl), sl["nears"],
                        sl["fars"], O.PathConfig(num_proposal_samples=(64, 48), num_nerf_samples=48), None)
    assert rel_err(depth[:512], ref.depth) <= 1e-3
    d = sl["directions"]
    theta, phi = torch.asin(d[:, 2:3]), torch.atan2(d[:, 1:2], d[:, 0:1])
    pts = O.radar_points(depth[:512].cpu(), theta, phi)
    assert rel_err(pts, O.radar_points(ref.depth, theta, phi)) <= 1e-3
    assert rel_err(pts, d * depth[:512].cpu()) <= 1e-5  # unit directions: the point head is direction * depth


# ------------------------------------------------------------------------------------------------ dynamic actors (H8)
class GoldenActors(torch.nn.Module):
    """Stand-in for the reference's DynamicActors (trajectory interpolation is outside the path): replays the
    boxes2world / valid tensors the reference produced for the golden rays."""

    def __init__(self, g, mode, device):
        super().__init__()
        self.n_actors = 3
        self.b2w = g[f"{mode}_boxes2world"].to(device)
        self.valid = g[f"{mode}_valid"].to(device)
        self.bounds = g["actor_bounds"].to(device)
        self.actor_to_id = g["actor_to_id"].to(device)

    def get_boxes2world(self, query_times, flatten=True):
        assert not flatten and query_times.shape[0] == self.b2w.shape[0]
        return self.b2w, self.valid

    def actor_bounds(self):
        return self.bounds


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_dynamic_actor_branch_golden(nb, golden, mode):
    """NeuRADField in a scene with dynamic actors against the reference's own outputs (tests/golden/actors.npz)."""
    import neuradar_b200 as pkg

    g = golden("actors")
    actors = GoldenActors(g, mode, DEV)
    cfg = pkg.NeuRADFieldConfig(grid=pkg.NeuRADHashEncodingConfig(
        static=pkg.StaticSettings(hashgrid_dim=2, num_levels=16, base_res=16, max_res=1024, log2_hashmap_size=10),
        actor=pkg.ActorSettings(flip_prob=0.25, log2_hashmap_size=9)))
    fld = pkg.NeuRADField(cfg, actors=actors, static_scale=100.0).to(DEV)
    sd = {k[2:].replace("__", "."): v for k, v in g.items() if k.startswith("p_")}
    res = fld.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and not res.missing_keys
    fld.train(mode == "train")
    bins = g["bins"].to(DEV)
    rb = nb.RayBundle(origins=g["origins"].to(DEV), directions=g["directions"].to(DEV), pixel_area=g["pixel_area"].to(DEV),
                      times=g["times"].to(DEV), metadata={})
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    if mode == "train":  # replay the reference's per-ray flip draw
        flip = g["train_ray_flip"].to(DEV)
        fld.hashgrid.ray_flip_override = flip
    assert fld.hashgrid.can_assign_in_kernel()  # the actor kernels (csrc/actors.cu), not the torch bookkeeping
    out = fld(rs)
    ref_inside = (g[f"{mode}_grid_features"][:, 16:] == 0).all(dim=-1)
    assert int(ref_inside.sum()) > 100
    assert rel_err(out[nb.FieldHeadNames.FEATURE], g[f"{mode}_feature"]) <= 1e-3
    assert float((out[nb.FieldHeadNames.ALPHA].detach().cpu() - g[f"{mode}_alpha"]).abs().max()) <= 1e-3
    # the grid stage alone, through the reference-shaped API (GaussiansStd in, features + directions out)
    gs = rs.frustums.get_fast_isotropic_gaussian(1)
    feats, dirs = fld.hashgrid(gs, rs.times, rs.frustums.directions)
    assert torch.equal((feats[:, 16:] == 0).all(dim=-1).cpu(), ref_inside), "the same samples must be claimed by actors"
    assert rel_err(feats, g[f"{mode}_grid_features"]) <= 1e-4
    assert rel_err(dirs, g[f"{mode}_grid_directions"]) <= 1e-5
    if mode == "train":
        ((out[nb.FieldHeadNames.FEATURE] * g["train_gf"].to(DEV)).sum()
         + (out[nb.FieldHeadNames.ALPHA] * g["train_ga"].to(DEV)).sum()).backward()
        assert rel_err(fld.hashgrid.static_grid.hash_table.grad, g["train_d_static_table"]) <= 1e-3
        for i in range(3):
            got = fld.hashgrid.actor_grids[i].hash_table.grad
            ref = g[f"train_d_actor_table{i}"]
            if float(ref.abs().max()) > 0:
                assert rel_err(got, ref) <= 1e-3, i
        assert rel_err(fld.mlp_geo.layers[0].weight.grad, g["train_d_geo_w0"]) <= 1e-3


def test_actor_path_has_no_host_sync(nb):
    """The field forward + backward in a scene with dynamic actors (config-4 shape, 16 actors) must not synchronise the
    host: the reference's three nonzero() round trips and its python loop over actors are one kernel here."""
    import neuradar_b200 as pkg
    from neuradar_b200.synthetic import SyntheticActors, synthetic_rays

    n, S = 512, 64
    actors = SyntheticActors(16, device=DEV)
    cfg = pkg.NeuRADFieldConfig(grid=pkg.NeuRADHashEncodingConfig(
        static=pkg.StaticSettings(hashgrid_dim=4, num_levels=8, base_res=32, max_res=8192, log2_hashmap_size=14),
        actor=pkg.ActorSettings(flip_prob=0.25, log2_hashmap_size=10)))
    fld = pkg.NeuRADField(cfg, actors=actors, static_scale=100.0).to(DEV)
    fld.train()
    with torch.no_grad():
        fld.hashgrid.static_grid.hash_table.mul_(300.0)
        for g in fld.hashgrid.actor_grids:
            g.hash_table.mul_(300.0)
    r = synthetic_rays(n, seed=2)
    # aim a third of the rays at actor boxes so that they are certainly hit
    centres = actors.centres[torch.arange(n // 3) % 16].cpu()
    d = centres - r["origins"][: n // 3]
    r["directions"][: n // 3] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = (torch.linspace(0.5, 60.0, S + 1)[None, :].repeat(n, 1)).to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    out = fld(rs)  # warm-up (allocations, caches)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = fld(rs)
        (out[nb.FieldHeadNames.FEATURE].sum() + out[nb.FieldHeadNames.ALPHA].sum()).backward()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    rays, iv = rs.per_ray()
    batch = fld.hashgrid.assign_actors(rays, iv, rs.times.reshape(n, -1)[:, 0])
    inside = int((batch.grid_id >= 0).sum())
    assert inside > 50, inside
    assert sum(float(g.hash_table.grad.abs().sum()) > 0 for g in fld.hashgrid.actor_grids) >= 4
    # against the torch bookkeeping of the same module (the reference's algorithm, round 1) on the same samples
    fld.eval()
    feats_kernel = fld(rs)[nb.FieldHeadNames.FEATURE]
    fld.hashgrid.can_assign_in_kernel = lambda proposal=False: False
    feats_torch = fld(rs)[nb.FieldHeadNames.FEATURE]
    # (box-frame positions differ by an ulp between the torch path's matmul and the kernel's fused multiply-adds; the
    #  finest actor level multiplies that by its resolution)
    assert rel_err(feats_kernel, feats_torch) <= 3e-5


def test_proposal_round_with_actors_matches_torch_bookkeeping(nb):
    """NeuRADProposalField in a scene with dynamic actors: the fused round with the in-kernel actor branch against the
    torch bookkeeping of the same module (NeuRADHashEncoding._split_static_vs_actors + per-actor grids + zero padding,
    neurad_encoding.py:160-187), forward and every gradient; and no host synchronisation on the kernel route."""
    import neuradar_b200 as pkg
    from neuradar_b200.synthetic import SyntheticActors, synthetic_rays

    n, S = 384, 96
    actors = SyntheticActors(16, device=DEV)
    pcfg = pkg.NeuRADProposalFieldConfig()
    pcfg.grid.static.log2_hashmap_size = 13
    pcfg.grid.actor.log2_hashmap_size = 9
    pcfg.grid.actor.flip_prob = 0.25
    prop = pkg.NeuRADProposalField(pcfg, actors=actors, static_scale=100.0).to(DEV)
    prop.train()
    with torch.no_grad():
        prop.hashgrid.static_grid.hash_table.mul_(2000.0)
        for g in prop.hashgrid.actor_grids:
            g.hash_table.mul_(2000.0)
    r = synthetic_rays(n, seed=4)
    centres = actors.centres[torch.arange(n // 2) % 16].cpu()
    d = centres - r["origins"][: n // 2]
    r["directions"][: n // 2] = d / d.norm(dim=-1, keepdim=True)
    rb = nb.RayBundle(origins=r["origins"].to(DEV), directions=r["directions"].to(DEV), pixel_area=r["pixel_area"].to(DEV),
                      times=r["times"].to(DEV), metadata={})
    bins = (torch.linspace(0.5, 60.0, S + 1)[None, :].repeat(n, 1)).to(DEV)
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    prop.hashgrid.ray_flip_override = (torch.rand(n, device=DEV) < 0.25).float() * -2 + 1
    assert prop.hashgrid.can_assign_in_kernel(proposal=True)
    gw = torch.randn((n, S, 1), device=DEV)
    gd = torch.randn((n, S, 1), device=DEV) * 1e-3

    def run():
        for p in prop.parameters():
            p.grad = None
        dens, w = prop.density_and_weights(rs)
        ((w * gw).sum() + (dens * gd).sum()).backward()
        return dens.detach(), w.detach(), {k: p.grad.clone() for k, p in prop.named_parameters() if p.grad is not None}

    run()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        dens_k, w_k, grads_k = run()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    rays, iv = rs.per_ray()
    inside = int((prop.hashgrid.assign_actors(rays, iv, rs.times.reshape(n, -1)[:, 0]).grid_id >= 0).sum())
    assert inside > 100, inside
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
    assert nonzero_actor_tables >= 4
