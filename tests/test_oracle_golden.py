"""Pin the CPU oracle against vectors produced by the reference itself (tests/golden/make_golden.py)
and against the reference's own known-answer tests.  CPU only."""
import pytest
import torch

from oracle import neuradar_oracle as O


def params_from_golden(g, prefix=""):
    main = O.GridParams(g[prefix + "main_table"], O.level_scalings(16, 16, 1024), 10)
    fld = O.FieldParams(
        grid=main,
        geo_w=[g[f"{prefix}geo_w{k}"] for k in range(2)],
        geo_b=[g[f"{prefix}geo_b{k}"] for k in range(2)],
        feat_w=[g[f"{prefix}feat_w{k}"] for k in range(3)],
        feat_b=[g[f"{prefix}feat_b{k}"] for k in range(3)],
        beta=g[prefix + "beta"],
    )
    props = [
        O.ProposalParams(O.GridParams(g[f"{prefix}prop{i}_table"], O.level_scalings(6, 128, 4096), 10), g[f"{prefix}prop{i}_w"])
        for i in range(2)
    ]
    return fld, props


def test_level_scalings(golden):
    g = golden("hash")
    assert torch.equal(O.level_scalings(16, 16, 1024), g["scalings_A"])
    assert torch.equal(O.level_scalings(8, 32, 8192), g["scalings_B"])
    assert torch.equal(O.level_scalings(6, 128, 4096), g["scalings_P"])
    assert torch.equal(O.level_scalings(4, 64, 1024), g["scalings_actor"])
    assert g["scalings_B"][-1].item() == 8191.0  # SURVEY.md section 0, trap 2
    assert g["scalings_A"].tolist() == [16, 21, 27, 36, 48, 64, 84, 111, 147, 194, 256, 337, 445, 588, 776, 1024]


def test_hash_known_answers(golden):
    g = golden("hash")
    coords = g["kat_coords"][:, None, :].expand(-1, 16, -1)
    got = O.hash_coords(coords, 19)
    assert got.dtype == torch.int64 and torch.equal(got, g["kat_hash"])
    # values recorded in SURVEY.md 8c (level 0 / level 15)
    want = {(0, 0, 0): (0, 7864320), (1, 0, 0): (1, 7864321), (0, 1, 0): (489905, 8354225), (0, 0, 1): (153493, 8017813),
            (1, 1, 1): (339493, 8203813), (15, 16, 17): (19450, 7883770), (1023, 1024, 1): (299114, 8163434),
            (-1, -2, 3): (128478, 7992798)}
    for row, c in enumerate(g["kat_coords"].tolist()):
        if tuple(c) in want:
            assert (got[row, 0].item(), got[row, 15].item()) == want[tuple(c)]
    # uint32 wrap-around formulation used by the CUDA kernels is bit-identical
    c = g["kat_coords"].to(torch.int64) & 0xFFFFFFFF
    h32 = (c[:, 0] ^ ((c[:, 1] * O.PRIME_Y) & 0xFFFFFFFF) ^ ((c[:, 2] * O.PRIME_Z) & 0xFFFFFFFF)) & ((1 << 19) - 1)
    assert torch.equal(h32, g["kat_hash"][:, 0])


@pytest.mark.parametrize("F", [1, 2, 4])
def test_hash_encode_forward_backward(golden, F):
    g = golden("hash")
    table = g[f"F{F}_table"].clone().requires_grad_(True)
    x = g["x"].clone().requires_grad_(True)
    y = O.hash_encode(x, table, g["scalings_A"], 10)
    assert torch.equal(y, g[f"F{F}_y"])
    (y * g[f"F{F}_dy"]).sum().backward()
    torch.testing.assert_close(table.grad, g[f"F{F}_dtable"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(x.grad, g[f"F{F}_dx"], rtol=1e-5, atol=1e-5)


def test_reference_known_answer_tests(golden):
    g = golden("kats")
    # reference tests/cameras/test_rays.py:11-30
    assert torch.equal(g["frustum_positions"], torch.tensor([1.0, 3.5, 1.0]).expand(5, 3))
    # SURVEY.md 8c vectors
    w, T = O.alpha_weights(g["alpha_in"][..., 0], eps=1e-7)
    assert torch.equal(w, g["alpha_w"][..., 0]) and torch.equal(T, g["alpha_T"][..., 0])
    torch.testing.assert_close(w[0], torch.tensor([0.1, 0.45000005, 0.40500015, 0.0090000136]), rtol=1e-6, atol=0)
    torch.testing.assert_close(g["gw_kat"].flatten(), torch.tensor([0.39346933, 0.3834005, 0.08779488, 0.12859733]), rtol=1e-6, atol=0)
    # reference tests/utils/test_math.py:8-16: SH basis is orthonormal over the sphere
    gen = torch.Generator().manual_seed(0)
    d = torch.randn((200000, 3), generator=gen)
    d = d / d.norm(dim=-1, keepdim=True)
    sh = O.sh16(d)
    gram = 4 * torch.pi * (sh.T @ sh) / d.shape[0]
    torch.testing.assert_close(gram, torch.eye(16), rtol=0, atol=3e-2)


def test_weights_and_renderers(golden):
    g = golden("kats")
    w, T = O.alpha_weights(g["alpha2_in"][..., 0], eps=1e-7)
    torch.testing.assert_close(w, g["alpha2_w"][..., 0], rtol=1e-5, atol=1e-9)
    torch.testing.assert_close(T, g["alpha2_T"][..., 0], rtol=1e-5, atol=1e-9)
    w0, _ = O.alpha_weights(g["alpha2_in"][..., 0], eps=0.0)  # nerfacc contract vs in-tree twin (SURVEY 8a C3)
    torch.testing.assert_close(w0, w, rtol=1e-4, atol=1e-6)
    bins = g["gw_bins"]
    dens = g["gw_dens"].clone().requires_grad_(True)
    gw = O.density_weights(dens, (bins[:, 1:] - bins[:, :-1])[..., None])
    torch.testing.assert_close(gw, g["gw_w"], rtol=1e-5, atol=1e-9)
    (gw * g["gw_dw"]).sum().backward()
    torch.testing.assert_close(dens.grad, g["gw_ddens"], rtol=1e-5, atol=1e-9, equal_nan=True)
    starts, ends = bins[:, :-1], bins[:, 1:]
    # float reductions: torch's CPU kernels may split them differently from run to run (thread count), so these
    # are held to 1e-6 instead of bit equality; integer outputs and bins stay bit-exact elsewhere in this file
    torch.testing.assert_close(torch.sum(g["rend_feats"] * g["rend_w"], dim=-2), g["rend_feature"], rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(O.expected_depth(g["rend_w"], starts, ends), g["rend_depth_expected"], rtol=1e-5, atol=1e-9)
    assert torch.equal(O.median_depth(g["rend_w"] * 3, starts, ends), g["rend_depth_median"])
    torch.testing.assert_close(O.sh16((g["sh_dirs"] + 1.0) / 2.0), g["sh_out"], rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(O.sh16(g["sh_dirs"]), g["sh_enc"], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("tag,n", [("geo", 2), ("feat", 3), ("lidar", 3), ("radar", 3)])
def test_mlp(golden, tag, n):
    g = golden("kats")
    ws = [g[f"mlp_{tag}_w{k}"].clone().requires_grad_(True) for k in range(n)]
    bs = [g[f"mlp_{tag}_b{k}"].clone().requires_grad_(True) for k in range(n)]
    x = g[f"mlp_{tag}_x"].clone().requires_grad_(True)
    y = O.mlp(x, ws, bs)
    assert torch.equal(y, g[f"mlp_{tag}_y"])
    (y * g[f"mlp_{tag}_dy"]).sum().backward()
    torch.testing.assert_close(x.grad, g[f"mlp_{tag}_dx"], rtol=1e-6, atol=1e-7)
    for k in range(n):
        torch.testing.assert_close(ws[k].grad, g[f"mlp_{tag}_dw{k}"], rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(bs[k].grad, g[f"mlp_{tag}_db{k}"], rtol=1e-6, atol=1e-7)


def test_pdf_sampler_known_answer(golden):
    g = golden("samplers")
    bins, inds, cdf, u = O.pdf_sample(g["kat_w"][..., 0], g["kat_in_sbins"], 4, None)
    assert torch.equal(bins, g["kat_sbins"])
    torch.testing.assert_close(bins[0], torch.tensor([0.33514851, 0.40910226, 0.45324191, 0.49738157, 0.58283591]), rtol=1e-6, atol=0)
    torch.testing.assert_close(bins[1], torch.tensor([0.1, 0.3, 0.5, 0.7, 0.9]), rtol=1e-6, atol=0)
    torch.testing.assert_close(2.0 + 4.0 * bins[0, :4], torch.tensor([3.3405938, 3.6364093, 3.8129675, 3.9895263]), rtol=1e-6, atol=0)
    assert torch.equal(2.0 + (6.0 - 2.0) * bins[:, :4], g["kat_starts"]) or torch.allclose(
        bins[:, :4] * 6.0 + (1 - bins[:, :4]) * 2.0, g["kat_starts"], rtol=1e-6
    )


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_samplers(golden, mode):
    g = golden("samplers")
    j0 = g[f"{mode}_j0"] if mode == "train" else None
    j1 = g[f"{mode}_j1"] if mode == "train" else None
    sb0, eb0, sp = O.spaced_bins(g["nears"], g["fars"], 64, j0)
    assert torch.equal(sb0.expand(96, -1), g[f"{mode}_sbins0"])
    assert torch.equal(eb0, g[f"{mode}_ebins0"])
    sb1, inds, cdf, u = O.pdf_sample(g[f"{mode}_w"][..., 0], sb0.expand(96, -1), 48, j1)
    assert torch.equal(sb1, g[f"{mode}_sbins1"])
    assert torch.equal(sp.to_euclidean(sb1), g[f"{mode}_ebins1"])
    assert inds.dtype == torch.int64 and inds.min() >= 1 and inds.max() <= 64


@pytest.mark.parametrize("mode", ["train", "eval"])
def test_whole_path(golden, mode):
    g = golden("path")
    fld, props = params_from_golden(g)
    leaves = [fld.grid.table, *fld.geo_w, *fld.geo_b, *fld.feat_w, *fld.feat_b, fld.beta] + [p.grid.table for p in props] + [p.decoder_w for p in props]
    for t in leaves:
        t.requires_grad_(True)
    cfg = O.PathConfig(num_proposal_samples=(64, 48), num_nerf_samples=48)
    jit = [g[f"{mode}_jitter{i}"] for i in range(3)] if mode == "train" else None
    out = O.nff_forward(fld, props, g["origins"], g["directions"], g["pixel_area"], g["nears"], g["fars"], cfg, jit, composite_eps=1e-7)
    pre = mode + "_"
    for i in range(2):
        assert torch.equal(out.sbins_list[i], g[f"{pre}sbins{i}"])
        assert torch.equal(out.ebins_list[i], g[f"{pre}ebins{i}"])
        torch.testing.assert_close(out.weights_list[i], g[f"{pre}prop_w{i}"], rtol=1e-6, atol=1e-9)
    assert torch.equal(out.sbins_list[2], g[f"{pre}sbins2"][:, :-1])
    assert torch.equal(out.ebins_list[2], g[f"{pre}ebins2"][:, :-1])
    torch.testing.assert_close(out.features, g[f"{pre}features"], rtol=1e-6, atol=1e-8)
    torch.testing.assert_close(out.depth, g[f"{pre}depth"], rtol=1e-6, atol=1e-8)
    torch.testing.assert_close(out.accumulation, g[f"{pre}accumulation"], rtol=1e-6, atol=1e-8)
    torch.testing.assert_close(out.weights_list[2], g[f"{pre}weights"], rtol=1e-6, atol=1e-9)
    loss = O.bench_loss(out)
    torch.testing.assert_close(loss, g[f"{pre}loss"], rtol=1e-6, atol=0)
    if mode == "train":
        loss.backward()
        names = (["d_main_table"] + [f"d_geo_w{k}" for k in range(2)] + [f"d_geo_b{k}" for k in range(2)]
                 + [f"d_feat_w{k}" for k in range(3)] + [f"d_feat_b{k}" for k in range(3)] + ["d_beta"]
                 + [f"d_prop{i}_table" for i in range(2)] + [f"d_prop{i}_w" for i in range(2)])
        for t, n in zip(leaves, names):
            ref = g[pre + n]
            scale = ref.abs().max().item() + 1e-30
            assert (t.grad - ref).abs().max().item() <= 1e-5 * scale, n


def _actor_setup(g):
    sd = {k[2:].replace("__", "."): v for k, v in g.items() if k.startswith("p_")}
    static = O.GridParams(sd["hashgrid.static_grid.hash_table"].clone().requires_grad_(True), O.level_scalings(16, 16, 1024), 10)
    actor_grids = [O.GridParams(sd[f"hashgrid.actor_grids.{i}.hash_table"].clone().requires_grad_(True),
                                O.level_scalings(4, 64, 1024), 9) for i in range(3)]
    fld = O.FieldParams(
        grid=static,
        geo_w=[sd[f"mlp_geo.layers.{k}.weight"].clone().requires_grad_(True) for k in range(2)],
        geo_b=[sd[f"mlp_geo.layers.{k}.bias"] for k in range(2)],
        feat_w=[sd[f"mlp_feature.layers.{k}.weight"] for k in range(3)],
        feat_b=[sd[f"mlp_feature.layers.{k}.bias"] for k in range(3)],
        beta=sd["sdf_to_density.beta"],
    )
    return fld, actor_grids


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_dynamic_actor_branch(golden, mode):
    """H8: NeuRADHashEncoding / NeuRADField with per-actor grids against the reference run on the same scene."""
    g = golden("actors")
    fld, actor_grids = _actor_setup(g)
    bins = g["bins"]
    flip = g["train_ray_flip"] if mode == "train" else None
    out = O.field_forward_with_actors(fld, actor_grids, 10.0, g["origins"], g["directions"], g["pixel_area"], bins[:, :-1],
                                      bins[:, 1:], g[f"{mode}_boxes2world"], g[f"{mode}_valid"], g["actor_bounds"],
                                      g["actor_to_id"], flip)
    ref_feats = g[f"{mode}_grid_features"]
    inside = (ref_feats[:, 16:] == 0).all(dim=-1)
    assert int(inside.sum()) > 100, "the golden scene must put samples inside actor boxes"
    assert torch.equal((out["grid_features"][:, 16:] == 0).all(dim=-1), inside), "same samples must be claimed by actors"
    torch.testing.assert_close(out["grid_features"], ref_feats, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out["directions"], g[f"{mode}_grid_directions"], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(out["feature"], g[f"{mode}_feature"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(out["alpha"], g[f"{mode}_alpha"], rtol=1e-4, atol=1e-5)
    if mode == "train":
        ((out["feature"] * g["train_gf"]).sum() + (out["alpha"] * g["train_ga"]).sum()).backward()
        scale = g["train_d_static_table"].abs().max()
        assert float((fld.grid.table.grad - g["train_d_static_table"]).abs().max()) <= 1e-4 * float(scale)
        for i, ag in enumerate(actor_grids):
            ref = g[f"train_d_actor_table{i}"]
            got = ag.table.grad if ag.table.grad is not None else torch.zeros_like(ref)
            assert float((got - ref).abs().max()) <= 1e-4 * float(ref.abs().max() + 1e-12), i
        assert float((fld.geo_w[0].grad - g["train_d_geo_w0"]).abs().max()) <= 1e-4 * float(g["train_d_geo_w0"].abs().max())


def test_losses(golden):
    """SURVEY.md 8f next-1: interlevel and distortion losses against the reference functions run on path.npz."""
    g = golden("losses")
    ws = [g[f"w{i}"].clone().requires_grad_(True) for i in range(3)]
    li = O.zipnerf_interlevel_loss(g["sbins2"], ws[2][..., 0], [(g["sbins0"], ws[0][..., 0]), (g["sbins1"], ws[1][..., 0])])
    ld = O.distortion_loss(g["sbins2"], ws[2][..., 0])
    torch.testing.assert_close(li, g["interlevel"], rtol=1e-5, atol=1e-9)
    torch.testing.assert_close(ld, g["distortion"], rtol=1e-5, atol=1e-9)
    (li + ld).backward()
    for i in range(3):
        scale = float(g[f"dw{i}"].abs().max()) + 1e-30
        assert float((ws[i].grad - g[f"dw{i}"]).abs().max()) <= 1e-5 * scale, i


@pytest.mark.parametrize("decoupled,wd", [(False, 0.0), (False, 1e-3), (True, 1e-7), (True, 1e-2)])
def test_adam_step_matches_torch_optim(decoupled, wd):
    """SURVEY 8f next-2: the oracle's Adam / AdamW restatement against torch.optim itself (the reference uses
    torch.optim.Adam / AdamW directly, configs/method_configs.py:393-400)."""
    gen = torch.Generator().manual_seed(3)
    p0 = torch.randn((257,), generator=gen) * 1e-2
    ref_p = p0.clone().requires_grad_(True)
    cls = torch.optim.AdamW if decoupled else torch.optim.Adam
    opt = cls([ref_p], lr=1e-2, eps=1e-15, weight_decay=wd, foreach=False, fused=False)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for step in range(1, 8):
        g = torch.randn((257,), generator=gen) * (10.0 ** float(torch.randint(-6, 1, (1,), generator=gen)))
        ref_p.grad = g.clone()
        opt.step()
        O.adam_step(p, g, m, v, step, lr=1e-2, eps=1e-15, weight_decay=wd, decoupled=decoupled)
        torch.testing.assert_close(p, ref_p.detach(), rtol=1e-6, atol=1e-9)
    st = opt.state[ref_p]
    torch.testing.assert_close(m, st["exp_avg"], rtol=1e-6, atol=1e-12)
    torch.testing.assert_close(v, st["exp_avg_sq"], rtol=1e-6, atol=1e-20)


def test_is_close_to_lidar_matches_reference_method():
    """oracle.is_close_to_lidar against the reference's own NeuRadarModel._compute_is_close_to_lidar (executed from
    oracle/_ref or the checkout; skipped where neither exists)."""
    import types

    from oracle import ref_shim

    if not ref_shim.available():
        pytest.skip("reference modules not available")
    ref_shim.install()
    from nerfstudio.cameras.rays import Frustums, RaySamples
    from nerfstudio.models.neuradar import NeuRadarModel

    g = torch.Generator().manual_seed(11)
    n, S = 40, 16
    bins = torch.cumsum(torch.rand((n, S + 1), generator=g) * 20, dim=-1)
    is_lidar = (torch.arange(n) % 2 == 0)[:, None]
    dnorm = torch.rand((n, 1), generator=g) * float(bins.max())
    dnorm[::4] = ((bins[::4, 3] + bins[::4, 4]) * 0.5 + 0.05)[:, None]
    did_return = torch.rand((n, 1), generator=g) > 0.3
    for use_return in (True, False):
        md = {"is_lidar": is_lidar[:, None, :].expand(n, S, 1), "directions_norm": dnorm[:, None, :].expand(n, S, 1)}
        if use_return:
            md["did_return"] = did_return[:, None, :].expand(n, S, 1)
        fr = Frustums(origins=torch.zeros((n, S, 3)), directions=torch.zeros((n, S, 3)), starts=bins[:, :-1, None].clone(),
                      ends=bins[:, 1:, None].clone(), pixel_area=torch.ones((n, S, 1)))
        rs = RaySamples(frustums=fr, metadata=md)
        fake_self = types.SimpleNamespace(config=types.SimpleNamespace(loss=types.SimpleNamespace(
            carving_epsilon=0.1, non_return_lidar_distance=150.0)))
        NeuRadarModel._compute_is_close_to_lidar(fake_self, rs)
        want = rs.metadata["is_close_to_lidar"][..., 0]
        got = O.is_close_to_lidar(bins[:, :-1], bins[:, 1:], is_lidar, dnorm, did_return if use_return else None)
        assert torch.equal(got, want)
        assert bool(want.any()) and not bool(want.all())


def test_is_close_to_lidar_golden(golden):
    """oracle.is_close_to_lidar against the stored masks (tests/golden/lidar_close.npz, gen_lidar_close), on the inputs of
    the test above and of tests/test_gpu_ray_tail.py, with and without did_return."""
    g = golden("lidar_close")
    for case in ("a", "b"):
        bins, is_lidar, dnorm, did_return = (g[f"{case}_{k}"] for k in ("bins", "is_lidar", "dnorm", "did_return"))
        for want, ret in ((g[f"{case}_close"], did_return), (g[f"{case}_close_no_return"], None)):
            got = O.is_close_to_lidar(bins[:, :-1], bins[:, 1:], is_lidar, dnorm, ret)
            assert torch.equal(got, want), case
            assert bool(want.any()) and not bool(want.all())


def test_radar_rays(golden):
    """Radar ray generation (SURVEY.md 8f next-4) against Radars._generate_rays_from_fov of the reference."""
    g = golden("radar_rays")
    out = O.radar_rays(g["radar_to_worlds"], g["min_azimuth"].reshape(-1), g["max_azimuth"].reshape(-1),
                       g["radar_azimuth_ray_divergence"].reshape(-1), g["min_elevation"].reshape(-1),
                       g["max_elevation"].reshape(-1), g["radar_elevation_ray_divergence"].reshape(-1), g["scan_indices"])
    assert torch.equal(out["ray_scan"], g["camera_indices"][:, 0])
    assert torch.equal(out["origins"], g["origins"])
    assert torch.equal(out["directions_spher"], g["directions_spher"])
    assert torch.equal(out["pixel_area"], g["pixel_area"])
    assert float((out["directions"] - g["directions"]).abs().max()) <= 1e-7
    assert float((out["directions_norm"] - g["directions_norm"]).abs().max()) <= 1e-7
    assert out["directions"].shape[0] == 1232  # six scans with ragged fields of view (two of them the default 16 x 16)
