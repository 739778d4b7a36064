"""Generate golden vectors by EXECUTING the reference's own fp32 torch path (container only).

Usage:  python tests/golden/make_golden.py      (needs the reference modules: oracle/_ref or $NEURADAR_REFERENCE)
        python tests/golden/make_golden.py --lidar-close-only   (runs without them, see gen_lidar_close)

Writes tests/golden/*.npz.  The vectors pin `oracle/neuradar_oracle.py` (tests/test_oracle_golden.py)
and are compared with the CUDA path on the GPU box, where the reference itself does not exist.
Every array is produced by reference code; this script only builds inputs and records outputs.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _ref_shim  # noqa: E402

HAVE_REFERENCE = _ref_shim.available()
if HAVE_REFERENCE:  # every generator except gen_lidar_close needs the reference
    _ref_shim.install()
    from nerfstudio.cameras.rays import Frustums, RayBundle, RaySamples  # noqa: E402
    from nerfstudio.field_components.encodings import HashEncoding, SHEncoding  # noqa: E402
    from nerfstudio.field_components.field_heads import FieldHeadNames  # noqa: E402
    from nerfstudio.field_components.mlp import MLP  # noqa: E402
    from nerfstudio.field_components.neurad_encoding import (  # noqa: E402
        ActorSettings,
        NeuRADHashEncodingConfig,
        StaticSettings,
    )
    from nerfstudio.fields.neurad_field import (  # noqa: E402
        NeuRADField,
        NeuRADFieldConfig,
        NeuRADProposalField,
        NeuRADProposalFieldConfig,
    )
    from nerfstudio.model_components.dynamic_actors import DynamicActors, DynamicActorsConfig  # noqa: E402
    from nerfstudio.model_components.ray_samplers import (  # noqa: E402
        PDFSampler,
        PowerSampler,
        ProposalNetworkSampler,
        UniformSampler,
    )
    from nerfstudio.model_components.renderers import (  # noqa: E402
        AccumulationRenderer,
        DepthRenderer,
        FeatureRenderer,
    )
    from nerfstudio.utils.math import components_from_spherical_harmonics  # noqa: E402

torch.set_grad_enabled(True)


def npy(t):
    return t.detach().cpu().numpy()


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **{k: (npy(v) if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in arrays.items()})
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB, {len(arrays)} arrays")


def synth_rays(n, seed):
    """Mixed camera/lidar/radar-like rays (SURVEY.md 8d), small n."""
    g = torch.Generator().manual_seed(seed)
    origins = torch.rand((n, 3), generator=g) * torch.tensor([40.0, 40.0, 3.0]) - torch.tensor([20.0, 20.0, 0.0])
    d = torch.randn((n, 3), generator=g)
    directions = d / d.norm(dim=-1, keepdim=True)
    kinds = torch.arange(n) % 3
    pixel_area = torch.where(kinds == 0, 2.25e-6, torch.where(kinds == 1, 4.5e-6, 1.5625e-4))[:, None].float()
    nears = torch.zeros((n, 1))
    fars = torch.full((n, 1), 1e6)
    times = torch.rand((n, 1), generator=g) * 20
    return origins, directions, pixel_area, nears, fars, times


# ---------------------------------------------------------------------------------------------
def gen_hash():
    out = {}
    # H1: level resolutions of every grid configuration on the path
    for tag, kw in {
        "A": dict(num_levels=16, min_res=16, max_res=1024, log2_hashmap_size=4),
        "B": dict(num_levels=8, min_res=32, max_res=8192, log2_hashmap_size=4),
        "P": dict(num_levels=6, min_res=128, max_res=4096, log2_hashmap_size=4),
        "actor": dict(num_levels=4, min_res=64, max_res=1024, log2_hashmap_size=4),
    }.items():
        out[f"scalings_{tag}"] = HashEncoding(implementation="torch", **kw).scalings

    # H2: hash_fn known answers, T = 2^19, 16 levels (includes negative coordinates)
    enc = HashEncoding(implementation="torch", log2_hashmap_size=19, num_levels=16, features_per_level=1)
    coords = torch.tensor(
        [[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1, 1], [15, 16, 17], [1023, 1024, 1], [-1, -2, 3],
         [8191, 8191, 8191], [4096, 0, 4095], [2147483647, 1, 1]],
        dtype=torch.int32,
    )
    out["kat_coords"] = coords
    out["kat_hash"] = enc.hash_fn(coords[:, None, :].expand(-1, 16, -1).contiguous())
    del enc

    # H3/H4: forward, table gradient, input gradient on a small grid for F in {1, 2, 4}
    g = torch.Generator().manual_seed(7)
    x = torch.rand((253, 3), generator=g)
    x[0] = 0.0
    x[1] = 1.0
    x[2] = torch.tensor([0.5, 0.25, 0.125])  # integral after scaling at several levels: ceil == floor
    x[3] = torch.tensor([1.0, 0.0, 0.5])
    out["x"] = x
    for F in (1, 2, 4):
        enc = HashEncoding(
            implementation="torch", num_levels=16, min_res=16, max_res=1024, log2_hashmap_size=10, features_per_level=F
        )
        with torch.no_grad():
            enc.hash_table.copy_((torch.rand(enc.hash_table.shape, generator=g) * 2 - 1) * 0.1)
        xr = x.clone().requires_grad_(True)
        y = enc(xr)
        dy = torch.randn(y.shape, generator=g)
        (y * dy).sum().backward()
        out[f"F{F}_table"] = enc.hash_table
        out[f"F{F}_y"] = y
        out[f"F{F}_dy"] = dy
        out[f"F{F}_dtable"] = enc.hash_table.grad
        out[f"F{F}_dx"] = xr.grad
    save("hash", **out)


def gen_small_kats():
    out = {}
    # the reference's own known-answer test: tests/cameras/test_rays.py:11-30
    fr = Frustums(
        origins=torch.ones((5, 3)), directions=torch.tensor([0.0, 1.0, 0.0]).expand(5, 3).contiguous() * 0 + torch.tensor([[0.0, 1.0, 0.0]]),
        starts=torch.ones((5, 1)) * 2, ends=torch.ones((5, 1)) * 3, pixel_area=torch.ones((5, 1)),
    )
    out["frustum_positions"] = fr.get_positions()
    # weights from alphas / densities (cameras/rays.py:188-248)
    a = torch.tensor([[0.1, 0.5, 0.9, 0.2]])[..., None]
    w, T = RaySamples.get_weights_and_transmittance_from_alphas(a)
    out["alpha_in"], out["alpha_w"], out["alpha_T"] = a, w, T
    g = torch.Generator().manual_seed(3)
    a2 = torch.rand((37, 48, 1), generator=g)
    a2[0] = 0.0
    a2[1] = 1.0
    w2, T2 = RaySamples.get_weights_and_transmittance_from_alphas(a2)
    out["alpha2_in"], out["alpha2_w"], out["alpha2_T"] = a2, w2, T2
    # get_weights
    N, S = 37, 64
    ends = torch.cumsum(torch.rand((N, S + 1), generator=g) * 2, dim=-1)
    rb = RayBundle(origins=torch.zeros((N, 3)), directions=torch.ones((N, 3)), pixel_area=torch.ones((N, 1)))
    rs = rb.get_ray_samples(bin_starts=ends[:, :-1, None], bin_ends=ends[:, 1:, None])
    dens = torch.exp(torch.randn((N, S, 1), generator=g) * 3)
    dens[0] = 0.0
    dens[1] = 1e30  # overflow path -> nan_to_num
    dens.requires_grad_(True)
    gw = rs.get_weights(dens)
    dgw = torch.randn(gw.shape, generator=g)
    (gw * dgw).sum().backward()
    out["gw_bins"], out["gw_dens"], out["gw_w"], out["gw_dw"], out["gw_ddens"] = ends, dens, gw, dgw, dens.grad
    kat = rb[:1].get_ray_samples(
        bin_starts=torch.tensor([[0.0, 0.5, 1.0, 2.0]])[..., None], bin_ends=torch.tensor([[0.5, 1.0, 2.0, 3.0]])[..., None]
    ).get_weights(torch.tensor([[1.0, 2.0, 0.5, 3.0]])[..., None])
    out["gw_kat"] = kat
    # renderers (model_components/renderers.py)
    feats = torch.randn((N, S, 32), generator=g)
    wts = torch.rand((N, S, 1), generator=g) / S
    out["rend_feats"], out["rend_w"] = feats, wts
    out["rend_feature"] = FeatureRenderer()(features=feats, weights=wts)
    out["rend_acc"] = AccumulationRenderer()(weights=wts)
    out["rend_depth_expected"] = DepthRenderer(method="expected")(weights=wts, ray_samples=rs)
    out["rend_depth_median"] = DepthRenderer(method="median")(weights=wts * 3, ray_samples=rs)
    # SH basis (utils/math.py:31-94) evaluated the way NeuRADField does: on (d+1)/2
    d = torch.randn((101, 3), generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    out["sh_dirs"] = d
    out["sh_out"] = components_from_spherical_harmonics(4, (d + 1.0) / 2.0)
    out["sh_enc"] = SHEncoding(levels=4, implementation="torch")(d)
    # MLP (field_components/mlp.py)
    torch.manual_seed(11)
    for tag, (i, n, w, o) in {"geo": (32, 2, 32, 33), "feat": (48, 3, 32, 32), "lidar": (48, 3, 32, 2), "radar": (48, 3, 16, 3)}.items():
        m = MLP(in_dim=i, num_layers=n, layer_width=w, out_dim=o, implementation="torch")
        xin = torch.randn((77, i), generator=g).requires_grad_(True)
        y = m(xin)
        dy = torch.randn(y.shape, generator=g)
        (y * dy).sum().backward()
        out[f"mlp_{tag}_x"], out[f"mlp_{tag}_y"], out[f"mlp_{tag}_dy"], out[f"mlp_{tag}_dx"] = xin, y, dy, xin.grad
        for k, layer in enumerate(m.layers):
            out[f"mlp_{tag}_w{k}"], out[f"mlp_{tag}_b{k}"] = layer.weight, layer.bias
            out[f"mlp_{tag}_dw{k}"], out[f"mlp_{tag}_db{k}"] = layer.weight.grad, layer.bias.grad
    save("kats", **out)


def gen_samplers():
    out = {}
    # PDFSampler known answer of SURVEY.md 8c: eval mode, uniform bins over [2, 6]
    N = 2
    rb = RayBundle(origins=torch.zeros((N, 3)), directions=torch.ones((N, 3)), pixel_area=torch.ones((N, 1)),
                   nears=torch.full((N, 1), 2.0), fars=torch.full((N, 1), 6.0))
    uni = UniformSampler(num_samples=8)
    uni.eval()
    rs = uni(rb)
    pdf = PDFSampler(num_samples=4, include_original=False, single_jitter=True)
    pdf.eval()
    w = torch.tensor([[0, 0, 1, 4, 2, 0, 0, 0], [1, 1, 1, 1, 1, 1, 1, 1]], dtype=torch.float32)[..., None]
    new = pdf(rb, rs, w, num_samples=4)
    out["kat_w"] = w
    out["kat_in_sbins"] = torch.cat([rs.spacing_starts[..., 0], rs.spacing_ends[..., -1:, 0]], -1)
    out["kat_sbins"] = torch.cat([new.spacing_starts[..., 0], new.spacing_ends[..., -1:, 0]], -1)
    out["kat_starts"] = new.frustums.starts[..., 0]

    # PowerSampler + PDFSampler, training (jittered) and eval, mixed near/far
    N = 96
    origins, directions, pixel_area, nears, fars, _ = synth_rays(N, 5)
    fars = fars.clamp_max(20000.0)
    nears = nears.clone()
    nears[::7] = 0.5
    fars = fars.clone()
    fars[::5] = 150.0
    rb = RayBundle(origins=origins, directions=directions, pixel_area=pixel_area, nears=nears, fars=fars)
    out["nears"], out["fars"] = nears, fars
    g = torch.Generator().manual_seed(9)
    for mode in ("train", "eval"):
        ps = PowerSampler(lambda_=-1.0, scaling=0.1, single_jitter=True)
        pdf = PDFSampler(include_original=False, single_jitter=True)
        ps.train(mode == "train")
        pdf.train(mode == "train")
        torch.manual_seed(123)
        j0 = torch.rand((N, 1))
        j1 = torch.rand((N, 1))
        torch.manual_seed(123)
        rs = ps(rb, num_samples=64)
        out[f"{mode}_j0"], out[f"{mode}_j1"] = j0, j1
        sb0 = torch.cat([rs.spacing_starts[..., 0], rs.spacing_ends[..., -1:, 0]], -1)
        out[f"{mode}_sbins0"] = sb0.expand(N, -1)
        out[f"{mode}_ebins0"] = torch.cat([rs.frustums.starts[..., 0], rs.frustums.ends[..., -1:, 0]], -1)
        w = torch.rand((N, 64, 1), generator=g) ** 8
        w[0] = 0.0  # zero-weight ray
        w[1, :, 0] = torch.zeros(64).index_fill_(0, torch.tensor([17]), 1.0)  # delta
        new = pdf(rb, rs, w, num_samples=48)
        out[f"{mode}_w"] = w
        out[f"{mode}_sbins1"] = torch.cat([new.spacing_starts[..., 0], new.spacing_ends[..., -1:, 0]], -1)
        out[f"{mode}_ebins1"] = torch.cat([new.frustums.starts[..., 0], new.frustums.ends[..., -1:, 0]], -1)
    save("samplers", **out)


def build_fields(log2_main=10, log2_prop=10, seed=21):
    torch.manual_seed(seed)
    actors = DynamicActors(DynamicActorsConfig(), trajectories=[])
    fcfg = NeuRADFieldConfig(
        grid=NeuRADHashEncodingConfig(
            static=StaticSettings(hashgrid_dim=2, num_levels=16, base_res=16, max_res=1024, log2_hashmap_size=log2_main),
            actor=ActorSettings(flip_prob=0.25),
        )
    )
    fld = NeuRADField(fcfg, actors, static_scale=100.0, implementation="torch")
    props = []
    for _ in range(2):
        pcfg = NeuRADProposalFieldConfig()
        pcfg.grid.static.log2_hashmap_size = log2_prop
        props.append(NeuRADProposalField(pcfg, actors, 100.0, implementation="torch"))
    with torch.no_grad():
        # default init (+-1e-3 tables) gives near-constant outputs; scale up so that parity is meaningful
        fld.hashgrid.static_grid.hash_table.mul_(300.0)
        for p in props:
            p.hashgrid.static_grid.hash_table.mul_(2000.0)
        fld.sdf_to_density.beta.fill_(20.0)
    return fld, props


def field_arrays(prefix, fld, props):
    out = {}
    out[f"{prefix}main_table"] = fld.hashgrid.static_grid.hash_table
    for k, layer in enumerate(fld.mlp_geo.layers):
        out[f"{prefix}geo_w{k}"], out[f"{prefix}geo_b{k}"] = layer.weight, layer.bias
    for k, layer in enumerate(fld.mlp_feature.layers):
        out[f"{prefix}feat_w{k}"], out[f"{prefix}feat_b{k}"] = layer.weight, layer.bias
    out[f"{prefix}beta"] = fld.sdf_to_density.beta
    for i, p in enumerate(props):
        out[f"{prefix}prop{i}_table"] = p.hashgrid.static_grid.hash_table
        out[f"{prefix}prop{i}_w"] = p.density_decoder.weight
    return out


def gen_path():
    """Fields + the whole sampled/composited path on 64 rays, forward and backward."""
    fld, props = build_fields()
    N = 64
    origins, directions, pixel_area, nears, fars, times = synth_rays(N, 42)
    out = dict(origins=origins, directions=directions, pixel_area=pixel_area, nears=nears, fars=fars, times=times)
    out.update(field_arrays("", fld, props))

    for mode in ("train", "eval"):
        fld.train(mode == "train")
        fld.zero_grad()
        for p in props:
            p.train(mode == "train")
            p.zero_grad()
        rb = RayBundle(origins=origins.clone(), directions=directions.clone(), pixel_area=pixel_area.clone(),
                       nears=nears.clone(), fars=fars.clone().clamp_max(20000.0), times=times.clone(), metadata={})
        sampler = ProposalNetworkSampler(
            num_proposal_samples_per_ray=(64, 48), num_nerf_samples_per_ray=48, num_proposal_network_iterations=2,
            single_jitter=True, initial_sampler=PowerSampler(lambda_=-1.0, scaling=0.1), update_sched=lambda x: 0,
        )
        sampler.train(mode == "train")
        torch.manual_seed(77)
        # the model builds PowerSampler WITHOUT single_jitter (models/neuradar.py:288-291): round 0 draws one
        # jitter per bin edge, the PDF rounds (single_jitter=True) one per ray
        jit = [torch.rand((N, 65)), torch.rand((N, 1)), torch.rand((N, 1))]
        torch.manual_seed(77)
        density_fns = [lambda rs, f=f: f.get_density(rs)[0] for f in props]
        ray_samples, weights_list, rs_list = sampler(rb, density_fns, pass_ray_samples=True)
        # sky sample (models/neuradar.py:578-582)
        dist = 20000.0 - ray_samples.frustums.ends[..., -1, 0]
        ray_samples.frustums.ends[..., -1, 0] += dist
        ray_samples.deltas[..., -1, 0] += dist
        ray_samples.spacing_ends[..., -1, 0] = 1 - 1e-7
        fo = fld(ray_samples)
        alpha = fo[FieldHeadNames.ALPHA]
        # compositing through the in-tree formula (the CPU branch of _render_weights is a 0.5 stub)
        w = RaySamples.get_weights_and_transmittance_from_alphas(alpha, weights_only=True)[..., 0]
        acc = AccumulationRenderer()(weights=w[..., None])
        w = torch.cat((w[..., :-1], w[..., -1:] + 1 - acc), dim=-1).unsqueeze(-1)
        feats = FeatureRenderer()(features=fo[FieldHeadNames.FEATURE], weights=w)
        w, rs_ns = w[..., :-1, :], ray_samples[..., :-1]
        steps = (rs_ns.frustums.starts + rs_ns.frustums.ends) / 2
        depth = torch.sum(w * steps, dim=-2)
        loss = feats.pow(2).mean() + 1e-3 * depth.mean() + sum(pw.pow(2).mean() for pw in weights_list)
        o = {}
        for i in range(3):
            o[f"jitter{i}"] = jit[i]
        for i, (pw, prs) in enumerate(zip(weights_list, rs_list)):
            o[f"prop_w{i}"] = pw
            o[f"sbins{i}"] = torch.cat([prs.spacing_starts[..., 0], prs.spacing_ends[..., -1:, 0]], -1).expand(N, -1)
            o[f"ebins{i}"] = torch.cat([prs.frustums.starts[..., 0], prs.frustums.ends[..., -1:, 0]], -1)
        o["sbins2"] = torch.cat([ray_samples.spacing_starts[..., 0], ray_samples.spacing_ends[..., -1:, 0]], -1)
        o["ebins2"] = torch.cat([ray_samples.frustums.starts[..., 0], ray_samples.frustums.ends[..., -1:, 0]], -1)
        o["field_feature"], o["field_sdf"], o["field_alpha"] = fo[FieldHeadNames.FEATURE], fo[FieldHeadNames.SDF], alpha
        o["features"], o["depth"], o["accumulation"], o["weights"], o["loss"] = feats, depth, acc, w, loss
        if mode == "train":
            loss.backward()
            o["d_main_table"] = fld.hashgrid.static_grid.hash_table.grad
            for k, layer in enumerate(fld.mlp_geo.layers):
                o[f"d_geo_w{k}"], o[f"d_geo_b{k}"] = layer.weight.grad, layer.bias.grad
            for k, layer in enumerate(fld.mlp_feature.layers):
                o[f"d_feat_w{k}"], o[f"d_feat_b{k}"] = layer.weight.grad, layer.bias.grad
            o["d_beta"] = fld.sdf_to_density.beta.grad
            for i, p in enumerate(props):
                o[f"d_prop{i}_table"] = p.hashgrid.static_grid.hash_table.grad
                o[f"d_prop{i}_w"] = p.density_decoder.weight.grad
        out.update({f"{mode}_{k}": v for k, v in o.items()})
    save("path", **out)


def _main_all():
    gen_hash()
    gen_small_kats()
    gen_samplers()
    gen_path()


def synth_trajectories(n_actors=3, n_times=6):
    """Non-overlapping boxes moving on straight lines with a slow yaw (SURVEY.md 8d, config 4)."""
    import math

    trajs = []
    ts = torch.linspace(0.0, 2.0, n_times)
    for a in range(n_actors):
        poses = torch.eye(4).repeat(n_times, 1, 1)
        for i, t in enumerate(ts):
            yaw = 0.3 * a + 0.1 * float(t)
            c, s = math.cos(yaw), math.sin(yaw)
            poses[i, :3, :3] = torch.tensor([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
            poses[i, :3, 3] = torch.tensor([8.0 + 9.0 * a + 1.5 * float(t), -6.0 + 6.0 * a, 0.9])
        trajs.append({"poses": poses, "timestamps": ts.clone(), "dims": torch.tensor([2.0, 4.6, 1.7]),
                      "symmetric": True, "deformable": False})
    return trajs


def gen_actors():
    """NeuRADHashEncoding / NeuRADField with dynamic actors (neurad_encoding.py:152-307), eval and training mode."""
    torch.manual_seed(31)
    trajs = synth_trajectories()
    actors = DynamicActors(DynamicActorsConfig(), trajectories=trajs)
    fcfg = NeuRADFieldConfig(
        grid=NeuRADHashEncodingConfig(
            static=StaticSettings(hashgrid_dim=2, num_levels=16, base_res=16, max_res=1024, log2_hashmap_size=10),
            actor=ActorSettings(flip_prob=0.25, log2_hashmap_size=9),
        )
    )
    fld = NeuRADField(fcfg, actors, static_scale=100.0, implementation="torch")
    with torch.no_grad():
        fld.hashgrid.static_grid.hash_table.mul_(300.0)
        for g_ in fld.hashgrid.actor_grids:
            g_.hash_table.mul_(300.0)
    N, S = 96, 32
    g = torch.Generator().manual_seed(32)
    origins = torch.tensor([0.0, 0.0, 1.5]) + torch.randn((N, 3), generator=g) * torch.tensor([1.0, 1.0, 0.2])
    times = torch.rand((N, 1), generator=g) * 2.0
    # aim most rays at an actor (position at the ray's time, roughly), the rest anywhere
    target = torch.stack([torch.tensor([8.0 + 9.0 * (i % 3) + 1.5, -6.0 + 6.0 * (i % 3), 0.9]) for i in range(N)])
    target = target + torch.randn((N, 3), generator=g) * torch.tensor([1.5, 0.8, 0.5])
    d = target - origins
    d[::5] = torch.randn((len(d[::5]), 3), generator=g)
    directions = d / d.norm(dim=-1, keepdim=True)
    pixel_area = torch.full((N, 1), 4.5e-6)
    bins = torch.linspace(0.0, 40.0, S + 1).expand(N, S + 1).contiguous() + torch.rand((N, 1), generator=g) * 0.3
    rb = RayBundle(origins=origins, directions=directions, pixel_area=pixel_area, times=times, metadata={})
    rs = rb.get_ray_samples(bin_starts=bins[:, :-1, None], bin_ends=bins[:, 1:, None])
    out = dict(origins=origins, directions=directions, pixel_area=pixel_area, times=times, bins=bins,
               actor_bounds=actors.actor_bounds(), actor_to_id=actors.actor_to_id)
    out.update({f"p_{k.replace('.', '__')}": v for k, v in fld.state_dict().items() if "actors" not in k})
    for mode in ("eval", "train"):
        fld.train(mode == "train")
        actors.train(mode == "train")
        fld.zero_grad()
        boxes2world, valid = actors.get_boxes2world(times[:, 0], flatten=False)
        out[f"{mode}_boxes2world"], out[f"{mode}_valid"] = boxes2world, valid
        torch.manual_seed(5)
        flips = torch.bernoulli(torch.full((N,), 0.25)) * -2 + 1
        torch.manual_seed(5)
        gaussians = rs.frustums.get_fast_isotropic_gaussian(1)
        feats, dirs = fld.hashgrid(gaussians, rs.times, rs.frustums.directions)
        out[f"{mode}_grid_features"], out[f"{mode}_grid_directions"] = feats, dirs
        if mode == "train":
            out["train_ray_flip"] = flips
        torch.manual_seed(5)
        fo = fld(rs)
        out[f"{mode}_feature"], out[f"{mode}_sdf"], out[f"{mode}_alpha"] = (
            fo[FieldHeadNames.FEATURE], fo[FieldHeadNames.SDF], fo[FieldHeadNames.ALPHA])
        if mode == "train":
            gf = torch.randn(fo[FieldHeadNames.FEATURE].shape, generator=g)
            ga = torch.randn(fo[FieldHeadNames.ALPHA].shape, generator=g)
            out["train_gf"], out["train_ga"] = gf, ga
            ((fo[FieldHeadNames.FEATURE] * gf).sum() + (fo[FieldHeadNames.ALPHA] * ga).sum()).backward()
            out["train_d_static_table"] = fld.hashgrid.static_grid.hash_table.grad
            for i, g_ in enumerate(fld.hashgrid.actor_grids):
                out[f"train_d_actor_table{i}"] = g_.hash_table.grad if g_.hash_table.grad is not None else torch.zeros_like(g_.hash_table)
            out["train_d_geo_w0"] = fld.mlp_geo.layers[0].weight.grad
    n_inside = int((out["eval_grid_features"][:, 16:] == 0).all(dim=-1).sum())
    print("samples inside actor boxes:", n_inside, "of", N * S)
    save("actors", **out)





def gen_losses():
    """zipnerf_interlevel_loss / distortion_loss (model_components/losses.py:137-156,648-705) on the golden path run."""
    from nerfstudio.model_components.losses import distortion_loss, zipnerf_interlevel_loss

    g = np.load(os.path.join(HERE, "path.npz"))
    N = 64
    rb = RayBundle(origins=torch.zeros((N, 3)), directions=torch.ones((N, 3)), pixel_area=torch.ones((N, 1)))
    out = {}
    rs_list, w_list = [], []
    for i in range(3):
        sb = torch.from_numpy(g[f"train_sbins{i}"])
        if i == 2:
            sb = sb[:, :-1]  # the sky sample is dropped before the losses (models/neuradar.py:515-516)
        eb = sb.clone()
        rs = rb.get_ray_samples(bin_starts=eb[:, :-1, None], bin_ends=eb[:, 1:, None], spacing_starts=sb[:, :-1, None],
                                spacing_ends=sb[:, 1:, None])
        rs_list.append(rs)
        w = torch.from_numpy(g[f"train_prop_w{i}"] if i < 2 else g["train_weights"]).clone().requires_grad_(True)
        w_list.append(w)
        out[f"sbins{i}"], out[f"w{i}"] = sb, w
    li = zipnerf_interlevel_loss(w_list, rs_list)
    ld = distortion_loss(w_list, rs_list)
    (li + ld).backward()
    out["interlevel"], out["distortion"] = li, ld
    for i in range(3):
        out[f"dw{i}"] = w_list[i].grad
    save("losses", **out)


def gen_radar_rays():
    """Radars._generate_rays_from_fov (cameras/radars.py:268-357) for poses with the default and with non-dyadic fields of
    view (SURVEY.md 8f next-4)."""
    import math

    from nerfstudio.cameras.radars import Radars

    g = torch.Generator().manual_seed(17)
    n = 6
    yaw, pitch = torch.rand(n, generator=g) * 2 * math.pi, (torch.rand(n, generator=g) - 0.5) * 0.2
    cy, sy, cp, sp = torch.cos(yaw), torch.sin(yaw), torch.cos(pitch), torch.sin(pitch)
    z, o = torch.zeros(n), torch.ones(n)
    Rz = torch.stack([torch.stack([cy, -sy, z], -1), torch.stack([sy, cy, z], -1), torch.stack([z, z, o], -1)], -2)
    Ry = torch.stack([torch.stack([cp, z, sp], -1), torch.stack([z, o, z], -1), torch.stack([-sp, z, cp], -1)], -2)
    t = (torch.rand((n, 3, 1), generator=g) - 0.5) * torch.tensor([200.0, 200.0, 4.0]).reshape(1, 3, 1)
    r2w = torch.cat([Rz @ Ry, t], -1)
    fov = dict(radar_azimuth_ray_divergence=torch.tensor([0.0625, 0.0625, 0.05, 0.03, 0.0625, 0.11]).reshape(n, 1),
               radar_elevation_ray_divergence=torch.tensor([0.0625, 0.0625, 0.07, 0.0625, 0.02, 0.13]).reshape(n, 1),
               min_azimuth=torch.tensor([-0.5, -0.5, -0.6, -0.31, -0.5, -0.9]).reshape(n, 1),
               max_azimuth=torch.tensor([0.5, 0.5, 0.55, 0.33, 0.5, 0.85]).reshape(n, 1),
               min_elevation=torch.tensor([-0.5, -0.5, -0.2, -0.5, -0.11, -0.3]).reshape(n, 1),
               max_elevation=torch.tensor([0.5, 0.5, 0.27, 0.5, 0.12, 0.35]).reshape(n, 1))
    radars = Radars(radar_to_worlds=r2w, times=torch.arange(n).float() * 0.1, **fov)
    scans = torch.tensor([4, 0, 5, 2, 2, 3])
    rb = radars._generate_rays_from_fov(scans)
    out = dict(radar_to_worlds=r2w, scan_indices=scans, times_in=radars.times, **fov)
    out.update(origins=rb.origins, directions=rb.directions, pixel_area=rb.pixel_area, camera_indices=rb.camera_indices,
               times=rb.times, fars=rb.fars, directions_norm=rb.metadata["directions_norm"],
               did_return=rb.metadata["did_return"], directions_spher=rb.metadata["directions_spher"])
    print("radar rays:", rb.origins.shape[0])
    save("radar_rays", **out)


def _close_inputs(n, S, seed, scale):
    """Sorted sample bins, lidar flags, hit distances (a quarter of them inside a sample) and return flags."""
    g = torch.Generator().manual_seed(seed)
    bins = torch.cumsum(torch.rand((n, S + 1), generator=g) * scale, dim=-1)
    is_lidar = (torch.arange(n) % 2 == 0)[:, None]
    dnorm = torch.rand((n, 1), generator=g) * float(bins.max())
    dnorm[::4] = ((bins[::4, 3] + bins[::4, 4]) * 0.5 + 0.05)[:, None]
    did_return = torch.rand((n, 1), generator=g) > 0.3
    return bins, is_lidar, dnorm, did_return


def _reference_is_close_to_lidar(bins, is_lidar, dnorm, did_return):
    """NeuRadarModel._compute_is_close_to_lidar (models/neuradar.py:971-994) on its own RaySamples."""
    import types

    from nerfstudio.cameras.rays import Frustums, RaySamples
    from nerfstudio.models.neuradar import NeuRadarModel

    n, S = bins.shape[0], bins.shape[1] - 1
    md = {"is_lidar": is_lidar[:, None, :].expand(n, S, 1), "directions_norm": dnorm[:, None, :].expand(n, S, 1)}
    if did_return is not None:
        md["did_return"] = did_return[:, None, :].expand(n, S, 1)
    fr = Frustums(origins=torch.zeros((n, S, 3)), directions=torch.zeros((n, S, 3)), starts=bins[:, :-1, None].clone(),
                  ends=bins[:, 1:, None].clone(), pixel_area=torch.ones((n, S, 1)))
    rs = RaySamples(frustums=fr, metadata=md)
    fake_self = types.SimpleNamespace(config=types.SimpleNamespace(loss=types.SimpleNamespace(
        carving_epsilon=0.1, non_return_lidar_distance=150.0)))
    NeuRadarModel._compute_is_close_to_lidar(fake_self, rs)
    return rs.metadata["is_close_to_lidar"][..., 0]


def gen_lidar_close():
    """is_close_to_lidar masks of the carving loss: case a (40 x 16, with and without did_return), case b (64 x 32).
    Recorded from the reference's own method where the reference modules exist; otherwise from oracle.is_close_to_lidar
    (which tests/test_oracle_golden.py compares with that method wherever the reference is present).  `source` says
    which one produced the file (UTF-8 bytes: `bytes(z["source"]).decode()`)."""
    if HAVE_REFERENCE:
        close, source = _reference_is_close_to_lidar, "reference: NeuRadarModel._compute_is_close_to_lidar"
    else:
        sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
        from oracle import neuradar_oracle as O

        def close(bins, is_lidar, dnorm, did_return):
            return O.is_close_to_lidar(bins[:, :-1], bins[:, 1:], is_lidar, dnorm, did_return)

        source = "oracle: neuradar_oracle.is_close_to_lidar (reference modules absent)"
    out = {"source": np.frombuffer(source.encode(), dtype=np.uint8)}
    for case, (n, S, seed, scale) in {"a": (40, 16, 11, 20.0), "b": (64, 32, 9, 4.0)}.items():
        bins, is_lidar, dnorm, did_return = _close_inputs(n, S, seed, scale)
        out.update({f"{case}_bins": bins, f"{case}_is_lidar": is_lidar, f"{case}_dnorm": dnorm, f"{case}_did_return": did_return})
        out[f"{case}_close"] = close(bins, is_lidar, dnorm, did_return)
        out[f"{case}_close_no_return"] = close(bins, is_lidar, dnorm, None)
    save("lidar_close", **out)


if __name__ == "__main__":
    if "--lidar-close-only" in sys.argv:
        gen_lidar_close()
        sys.exit(0)
    if "--radar-rays-only" in sys.argv:
        gen_radar_rays()
        sys.exit(0)
    if "--losses-only" in sys.argv:
        gen_losses()
    elif "--actors-only" in sys.argv:
        gen_actors()
    else:
        _main_all()
        gen_actors()
        gen_losses()
        gen_radar_rays()
        gen_lidar_close()
