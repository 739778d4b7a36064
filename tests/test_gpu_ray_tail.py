"""GPU tests of the per-ray tail (SURVEY.md 8a C6, appendix A7): point heads and the lidar carving terms, against the
oracle and - where oracle/_ref is materialised - against the reference's own `_compute_is_close_to_lidar`."""
import types

import pytest
import torch

from oracle import neuradar_oracle as O
from oracle import ref_shim
from tests.parity_utils import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rays(n, seed):
    g = torch.Generator().manual_seed(seed)
    o = torch.randn((n, 3), generator=g) * 10
    d = torch.randn((n, 3), generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    depth = torch.rand((n, 1), generator=g) * 80 + 0.5
    spher = (torch.rand((n, 2), generator=g) - 0.5)  # (phi, theta)
    return o, d, depth, spher


@pytest.mark.parametrize("n", [1, 257, 5000])
def test_point_heads_forward_backward(n):
    from neuradar_b200 import functional as Fn

    o, d, depth, spher = _rays(n, n)
    is_radar = (torch.arange(n) % 3 == 0)[:, None]
    w2l = torch.eye(4)
    w2l[:3, :3] = torch.linalg.qr(torch.randn(3, 3, generator=torch.Generator().manual_seed(1)))[0]
    w2l[:3, 3] = torch.tensor([1.0, -2.0, 0.5])
    dr = depth.clone().requires_grad_(True)
    lid = O.lidar_points(o, d, dr)
    lid = (w2l[:3, :3] @ lid.T).T + w2l[:3, 3]
    rad = O.radar_points(dr, spher[:, 1:2], spher[:, 0:1])
    ref = torch.where(is_radar, rad, lid)
    gp = torch.randn((n, 3), generator=torch.Generator().manual_seed(2))
    (ref * gp).sum().backward()
    dd = depth.to(DEV).requires_grad_(True)
    pts = Fn.point_heads(dd, o.to(DEV), d.to(DEV), is_radar.to(DEV), spher.to(DEV), w2l.to(DEV))
    assert rel_err(pts, ref) <= 2e-6
    (pts * gp.to(DEV)).sum().backward()
    assert rel_err(dd.grad, dr.grad) <= 2e-6
    # no radar flags, no sensor frame: the plain lidar head of ad_model.py:105
    pts2 = Fn.point_heads(depth.to(DEV), o.to(DEV), d.to(DEV))
    assert rel_err(pts2, O.lidar_points(o, d, depth)) <= 1e-6


def _carving_inputs(n, S, seed):
    g = torch.Generator().manual_seed(seed)
    bins = torch.cumsum(torch.rand((n, S + 1), generator=g) * 4, dim=-1)
    is_lidar = (torch.arange(n) % 2 == 0)[:, None]
    dnorm = torch.rand((n, 1), generator=g) * float(bins.max())
    # put some hits exactly inside a sample
    dnorm[::4] = ((bins[::4, 3] + bins[::4, 4]) * 0.5 + 0.05)[:, None]
    did_return = (torch.rand((n, 1), generator=g) > 0.3)
    w = torch.rand((n, S), generator=g)
    return bins, is_lidar, dnorm, did_return, w


@pytest.mark.parametrize("with_return", [True, False])
def test_carving_vs_oracle(with_return):
    from neuradar_b200 import functional as Fn

    n, S = 301, 48
    bins, is_lidar, dnorm, did_return, w = _carving_inputs(n, S, 5)
    dr = did_return if with_return else None
    close_ref = O.is_close_to_lidar(bins[:, :-1], bins[:, 1:], is_lidar, dnorm, dr)
    wr = w.clone().requires_grad_(True)
    loss_ref = O.carving_loss(wr, close_ref, is_lidar)
    loss_ref.backward()
    iv = Fn.SampleIntervals.from_bins(bins.to(DEV))
    close = Fn.is_close_to_lidar(iv, is_lidar.to(DEV), dnorm.to(DEV), None if dr is None else dr.to(DEV))
    assert torch.equal(close.cpu(), close_ref)
    wd = w.to(DEV).requires_grad_(True)
    loss = Fn.carving_loss(wd, iv, is_lidar.to(DEV), dnorm.to(DEV), None if dr is None else dr.to(DEV))
    assert abs(float(loss) - float(loss_ref)) <= 1e-5 * abs(float(loss_ref))
    (loss * 3.0).backward()
    assert rel_err(wd.grad, wr.grad * 3.0) <= 1e-6


@pytest.mark.skipif(not ref_shim.available(), reason="reference modules not materialised (oracle/build_ref.py)")
def test_carving_vs_reference_model_method():
    """The reference's own NeuRadarModel._compute_is_close_to_lidar, run on its own RaySamples."""
    from neuradar_b200 import functional as Fn

    ref_shim.install()
    from nerfstudio.cameras.rays import Frustums, RaySamples
    from nerfstudio.models.neuradar import NeuRadarModel

    n, S = 64, 32
    bins, is_lidar, dnorm, did_return, _ = _carving_inputs(n, S, 9)
    fr = Frustums(origins=torch.zeros((n, S, 3)), directions=torch.zeros((n, S, 3)), starts=bins[:, :-1, None].clone(),
                  ends=bins[:, 1:, None].clone(), pixel_area=torch.ones((n, S, 1)))
    rs = RaySamples(frustums=fr, metadata={"is_lidar": is_lidar[:, None, :].expand(n, S, 1),
                                           "directions_norm": dnorm[:, None, :].expand(n, S, 1),
                                           "did_return": did_return[:, None, :].expand(n, S, 1)})
    fake_self = types.SimpleNamespace(config=types.SimpleNamespace(loss=types.SimpleNamespace(
        carving_epsilon=0.1, non_return_lidar_distance=150.0)))
    NeuRadarModel._compute_is_close_to_lidar(fake_self, rs)
    want = rs.metadata["is_close_to_lidar"][..., 0]
    iv = Fn.SampleIntervals.from_bins(bins.to(DEV))
    got = Fn.is_close_to_lidar(iv, is_lidar.to(DEV), dnorm.to(DEV), did_return.to(DEV))
    assert torch.equal(got.cpu(), want)


def test_carving_mask_golden(golden):
    """The kernel's is_close_to_lidar against the stored masks (tests/golden/lidar_close.npz, gen_lidar_close)."""
    from neuradar_b200 import functional as Fn

    g = golden("lidar_close")
    for case in ("a", "b"):
        bins, is_lidar, dnorm, did_return = (g[f"{case}_{k}"].to(DEV) for k in ("bins", "is_lidar", "dnorm", "did_return"))
        iv = Fn.SampleIntervals.from_bins(bins)
        for want, ret in ((g[f"{case}_close"], did_return), (g[f"{case}_close_no_return"], None)):
            assert torch.equal(Fn.is_close_to_lidar(iv, is_lidar, dnorm, ret).cpu(), want), case


def test_nff_outputs_training_extras():
    """get_nff_outputs(calc_lidar_losses=True) emits the training-only outputs of models/neuradar.py:527-546."""
    import neuradar_b200 as nb
    from neuradar_b200.synthetic import build_hot_path, synthetic_rays

    n = 512
    model = build_hot_path(log2_main=12, log2_prop=12, table_gain=(300.0, 2000.0), device=DEV)
    model.config.gather_non_nearby = True
    model.train()
    rays = synthetic_rays(n, seed=4)
    dn = torch.rand((n, 1)) * 60 + 1
    md = {"is_lidar": rays["is_lidar"].to(DEV), "is_radar": rays["is_radar"].to(DEV), "directions_norm": dn.to(DEV),
          "did_return": (torch.rand((n, 1)) > 0.2).to(DEV), "directions_spher": torch.rand((n, 2)).to(DEV) - 0.5}
    rb = nb.RayBundle(origins=rays["origins"].to(DEV), directions=rays["directions"].to(DEV), pixel_area=rays["pixel_area"].to(DEV),
                      nears=rays["nears"].to(DEV), fars=rays["fars"].to(DEV), times=rays["times"].to(DEV), metadata=md)
    out = model.get_nff_outputs(rb, calc_lidar_losses=True)
    for key in ("prop_weights_loss_0", "prop_weights_loss_1", "non_nearby_mask", "non_nearby_weights_sq_sum", "non_nearby_weights",
                "non_nearby_lidar_ray_indices", "prop_depth_0", "prop_depth_1", "weights_list", "ray_samples_list"):
        assert key in out, key
    w = out["weights_list"][-1][..., 0]
    assert out["non_nearby_mask"].shape == w.shape
    assert abs(float(out["non_nearby_weights"].pow(2).sum()) - float(out["non_nearby_weights_sq_sum"])) <= 1e-5 * float(
        out["non_nearby_weights_sq_sum"]) + 1e-12
    # proposal carving loss against the dense formula on the same weights / samples
    for i in range(2):
        pw, prs = out["weights_list"][i][..., 0], out["ray_samples_list"][i]
        close = O.is_close_to_lidar(prs.frustums.starts[..., 0].cpu(), prs.frustums.ends[..., 0].cpu(), rays["is_lidar"],
                                    dn, md["did_return"].cpu())
        ref = O.carving_loss(pw.detach().cpu(), close, rays["is_lidar"])
        assert abs(float(out[f"prop_weights_loss_{i}"]) - float(ref)) <= 1e-5 * abs(float(ref)) + 1e-12
    # gradients flow from the extras to the proposal table
    (out["prop_weights_loss_0"] + out["non_nearby_weights_sq_sum"]).backward()
    assert float(model.proposal_fields[1].hashgrid.static_grid.hash_table.grad.abs().sum()) > 0
    assert float(model.field.hashgrid.static_grid.hash_table.grad.abs().sum()) > 0
    heads = model.point_heads(rb, out["depth"].detach())
    assert heads["points"].shape == (n, 3) and heads["radar_xyz"].shape[0] == int(rays["is_radar"].sum())


@pytest.mark.parametrize("n,S", [(1, 48), (300, 64), (77, 33)])
def test_weighted_depth_forward_backward(n, S):
    """render_depth_simple (models/neurad.py:721-728) with the midpoints formed in-kernel, against torch."""
    from neuradar_b200 import functional as Fn

    g = torch.Generator().manual_seed(n + S)
    bins = torch.cumsum(torch.rand((n, S + 1), generator=g) + 0.01, dim=-1)
    w = torch.rand((n, S), generator=g)
    go = torch.randn((n, 1), generator=g)
    wr = w.clone().requires_grad_(True)
    ref = (wr * (bins[:, :-1] + bins[:, 1:]) / 2).sum(-1, keepdim=True)
    (ref * go).sum().backward()
    wd = w.to(DEV).requires_grad_(True)
    out = Fn.weighted_depth(wd, Fn.SampleIntervals.from_bins(bins.to(DEV)))
    assert out.shape == (n, 1)
    assert rel_err(out, ref) <= 1e-6
    (out * go.to(DEV)).sum().backward()
    assert rel_err(wd.grad, wr.grad) <= 1e-6
