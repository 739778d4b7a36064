"""Synthetic workloads of the BASELINE configurations (SURVEY.md 8d): rays, actors and ready-built hot paths.

Used by bench.py, `__graft_entry__.smoke()` and the tests.  Nothing here touches the oracle or the reference: the
generators only reproduce the *shapes and value ranges* the reference's data pipeline feeds the hot path with
(ray origins / directions / pixel areas of cameras, lidars and radars: nerfstudio/cameras/radars.py:38-44,279-328,
nerfstudio/cameras/lidars.py:41-42,389-391, nerfstudio/models/neuradar.py:996-1008).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor


@dataclass(frozen=True)
class Workload:
    """One BASELINE.json configuration."""

    key: int
    name: str
    rays: int                                   # rays per GPU per step
    mix: str = "mixed"                          # "mixed" (camera / lidar / radar) or "radar"
    main: Tuple[int, int, int, int, int] = (16, 2, 19, 16, 1024)   # levels, features, log2 T, base res, max res
    prop_log2: int = 20
    proposal_samples: Tuple[int, ...] = (64, 48)
    nerf_samples: int = 48
    train: bool = True
    actors: int = 0
    chunk: int = 0                              # inference: rays per chunk (0 = one pass)

    @property
    def description(self) -> str:
        L, F, T, r0, r1 = self.main
        acts = f", {self.actors} dynamic actors (L4/F4/T2^17 grids)" if self.actors else ""
        mode = "fwd+bwd" if self.train else "inference, fwd only"
        return (f"config{self.key}: {self.rays} {self.mix} rays per GPU, main grid L{L}/F{F}/T2^{T} (res {r0}..{r1}), "
                f"proposals {self.proposal_samples} on L6/F1/T2^{self.prop_log2}, {self.nerf_samples} samples/ray{acts}, {mode}")

    # ---- algorithmic work per ray (SURVEY.md 8d / BASELINE.md section 3)
    def bytes_per_ray(self) -> float:
        L, F, *_ = self.main
        gathers = sum(self.proposal_samples) * 8 * 6 * 1 * 4 + self.nerf_samples * 8 * L * F * 4
        if self.actors:  # ~10 % of the samples fall into actor boxes: actor grid L4/F4, proposal-actor grid L4/F1
            gathers += 0.1 * (self.nerf_samples * 8 * 4 * 4 * 4 + sum(self.proposal_samples) * 8 * 4 * 1 * 4)
        io = 40 + 136 + (sum(self.proposal_samples) + self.nerf_samples + len(self.proposal_samples) + 1 +
                         sum(self.proposal_samples) + self.nerf_samples) * 4
        return (2 * gathers + io) if self.train else (gathers + 176)

    def mlp_flop_per_ray(self) -> float:
        fwd = 2 * (32 * 32 + 32 * 33 + 48 * 32 + 32 * 32 + 32 * 32) * self.nerf_samples
        return 3 * fwd if self.train else fwd


WORKLOADS: Dict[int, Workload] = {
    1: Workload(1, "cpu-runnable", 4096, mix="radar"),
    2: Workload(2, "single-gpu", 65536),
    3: Workload(3, "8-gpu shard", 32768),
    4: Workload(4, "large scene", 65536, main=(8, 4, 22, 32, 8192), proposal_samples=(128, 64), nerf_samples=128, actors=16),
    5: Workload(5, "inference sweep", 1 << 20, mix="radar", train=False, chunk=1 << 15),
}


def synthetic_rays(num_rays: int, seed: int = 42, mix: str = "mixed", device: str = "cpu") -> Dict[str, Tensor]:
    """Synthetic rays (SURVEY.md 8d).  mix="mixed": 62.5% camera, 31.25% lidar, 6.25% radar (the reference batch
    40960/20480/4096 of config 2); mix="radar": 16x16 azimuth x elevation scans of 256 rays."""
    g = torch.Generator().manual_seed(seed)
    n = num_rays
    origins = torch.rand((n, 3), generator=g) * torch.tensor([40.0, 40.0, 3.0]) - torch.tensor([20.0, 20.0, 0.0])
    d = torch.randn((n, 3), generator=g)
    directions = d / d.norm(dim=-1, keepdim=True)
    if mix == "radar":
        n_radar = n
    else:
        n_radar = max((n // 16 // 256) * 256, 0)
    n_lidar = 0 if mix == "radar" else (n * 5) // 16
    n_cam = n - n_lidar - n_radar
    is_lidar = torch.zeros((n, 1), dtype=torch.bool)
    is_radar = torch.zeros((n, 1), dtype=torch.bool)
    is_lidar[n_cam : n_cam + n_lidar] = True
    is_radar[n_cam + n_lidar :] = True
    if n_radar > 0:
        scans = n_radar // 256
        az = torch.arange(16) * 0.0625 - 0.5
        el = torch.arange(16) * 0.0625 - 0.5
        azg, elg = torch.meshgrid(az, el, indexing="ij")
        yaw = torch.rand((max(scans, 1), 1), generator=g) * 2 * math.pi
        phi = (azg.reshape(1, -1) + yaw).reshape(-1)[:n_radar]
        theta = elg.reshape(1, -1).expand(max(scans, 1), -1).reshape(-1)[:n_radar]
        rd = torch.stack([torch.cos(phi) * torch.cos(theta), torch.sin(phi) * torch.cos(theta), torch.sin(theta)], -1)
        directions[n - n_radar :] = rd
        origins[n - n_radar :] = origins[n - n_radar :: 256][: max(scans, 1)].repeat_interleave(256, 0)[:n_radar]
    pixel_area = torch.full((n, 1), 1.0 / 2000.0**2)  # camera; x9 is applied by _scale_pixel_area
    pixel_area[is_lidar] = 3e-3 * 1.5e-3
    pixel_area[is_radar] = (0.0625 / 5) ** 2
    out = dict(
        origins=origins,
        directions=directions,
        pixel_area=pixel_area,
        nears=torch.zeros((n, 1)),
        fars=torch.full((n, 1), 1e6),
        times=torch.rand((n, 1), generator=g) * 20,
        is_lidar=is_lidar,
        is_radar=is_radar,
    )
    return {k: v.to(device) for k, v in out.items()}


def scaled_pixel_area(rays: Dict[str, Tensor], upsample: int = 3) -> Tensor:
    """pixel_area after NeuRadarModel._scale_pixel_area (models/neuradar.py:996-1008)."""
    scaling = torch.ones_like(rays["pixel_area"])
    scaling[~(rays["is_lidar"] | rays["is_radar"])] = upsample**2
    return rays["pixel_area"] * scaling


class SyntheticActors(torch.nn.Module):
    """Stand-in for the reference's DynamicActors (model_components/dynamic_actors.py:183-197) with the interface
    NeuRADHashEncoding uses: `n_actors`, `get_boxes2world(times, flatten=False) -> ([N,A,4,4], valid [N,A])`,
    `actor_bounds() -> [A,3]`, `actor_to_id [A]`.  Actors are non-overlapping boxes on a grid around the origin that move on
    straight lines with a slow yaw (SURVEY.md 8d, config 4); poses are closed-form in time, as trajectory interpolation is
    outside the hot path.  With `trainable` the trajectory (`centres`, `velocity`, `yaw0`, `yaw_rate`) is made of
    parameters under the same state-dict names, as the reference optimises its actor trajectories."""

    def __init__(self, n_actors: int = 16, device: str = "cpu", seed: int = 5, trainable: bool = False):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.n_actors = n_actors
        side = int(math.ceil(math.sqrt(n_actors)))
        idx = torch.arange(n_actors)
        # centres on a 12 m lattice inside the +-20 m area the synthetic rays start in; half extents of a car
        centres = torch.stack([(idx % side).float() * 12.0 - 6.0 * (side - 1), (idx // side).float() * 12.0 - 6.0 * (side - 1),
                               torch.full((n_actors,), 0.9)], -1)
        trajectory = dict(
            centres=centres,
            velocity=(torch.rand((n_actors, 3), generator=g) - 0.5) * torch.tensor([0.2, 0.2, 0.0]),
            yaw0=torch.rand((n_actors,), generator=g) * 2 * math.pi,
            yaw_rate=(torch.rand((n_actors,), generator=g) - 0.5) * 0.02,
        )
        for name, value in trajectory.items():
            if trainable:
                self.register_parameter(name, torch.nn.Parameter(value.to(device)))
            else:
                self.register_buffer(name, value.to(device))
        self.register_buffer("bounds", torch.tensor([1.0, 2.3, 0.85]).repeat(n_actors, 1).to(device))
        self.register_buffer("actor_to_id", torch.arange(n_actors).to(device))
        self.register_buffer("bottom_row", torch.tensor([0.0, 0.0, 0.0, 1.0]).to(device))

    def actor_bounds(self) -> Tensor:
        return self.bounds

    def get_boxes2world(self, times: Tensor, flatten: bool = False):
        t = times.reshape(-1, 1).float()
        yaw = self.yaw0[None, :] + self.yaw_rate[None, :] * t                      # [N, A]
        c, s = torch.cos(yaw), torch.sin(yaw)
        pos = self.centres[None] + self.velocity[None] * t[..., None]              # [N, A, 3]
        z, o = torch.zeros_like(c), torch.ones_like(c)
        rot = torch.stack([torch.stack([c, -s, z], -1), torch.stack([s, c, z], -1), torch.stack([z, z, o], -1)], -2)
        top = torch.cat([rot, pos[..., None]], -1)                                 # [N, A, 3, 4]
        bottom = self.bottom_row.expand(*top.shape[:2], 1, 4)
        b2w = torch.cat([top, bottom], -2)
        valid = torch.ones(b2w.shape[:2], dtype=torch.bool, device=t.device)
        if flatten:
            return b2w.reshape(-1, 4, 4), valid.reshape(-1)
        return b2w, valid


def build_hot_path(
    log2_main: int = 19,
    log2_prop: int = 20,
    num_proposal_samples: Tuple[int, ...] = (64, 48),
    num_nerf_samples: int = 48,
    main_levels: int = 16,
    main_features: int = 2,
    main_res: Tuple[int, int] = (16, 1024),
    late_binding: bool = True,
    table_gain: Tuple[float, float] = (1.0, 1.0),
    seed: int = 42,
    device: str = "cuda",
    actors=None,
):
    """NeuRadarHotPath in the configuration BASELINE.json names (cfg-A main grid, cfg-P proposal grids)."""
    import neuradar_b200 as nb

    torch.manual_seed(seed)
    cfg = nb.NeuRadarHotPathConfig()
    cfg.late_binding_density_fns = late_binding
    cfg.sampling.num_proposal_samples = tuple(num_proposal_samples)
    cfg.sampling.num_nerf_samples = num_nerf_samples
    cfg.field.grid.static = nb.StaticSettings(
        hashgrid_dim=main_features, num_levels=main_levels, base_res=main_res[0], max_res=main_res[1],
        log2_hashmap_size=log2_main,
    )
    for p in (cfg.sampling.proposal_field_1, cfg.sampling.proposal_field_2):
        p.grid.static.log2_hashmap_size = log2_prop
    model = nb.NeuRadarHotPath(cfg, actors=actors)
    with torch.no_grad():
        model.field.hashgrid.static_grid.hash_table.mul_(table_gain[0])
        for p in model.proposal_fields:
            p.hashgrid.static_grid.hash_table.mul_(table_gain[1])
    return model.to(device)


def build_workload(w: Workload, seed: int = 42, device: str = "cuda"):
    """The hot path of a BASELINE configuration (random-init tables and MLPs of that architecture)."""
    actors = SyntheticActors(w.actors, device=device) if w.actors else None
    L, F, T, r0, r1 = w.main
    return build_hot_path(log2_main=T, log2_prop=w.prop_log2, num_proposal_samples=w.proposal_samples,
                          num_nerf_samples=w.nerf_samples, main_levels=L, main_features=F, main_res=(r0, r1), seed=seed,
                          device=device, actors=actors)
