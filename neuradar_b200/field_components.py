"""Field components of the hot path with the reference's constructor signatures and parameter names.

HashEncoding   <- nerfstudio/field_components/encodings.py:311-471
SHEncoding     <- nerfstudio/field_components/encodings.py:760-805
MLP            <- nerfstudio/field_components/mlp.py:60-183
NeuRADHashEncoding (+ StaticSettings / ActorSettings / NeuRADHashEncodingConfig)
               <- nerfstudio/field_components/neurad_encoding.py:36-316
trunc_exp, SigmoidDensity <- field_components/activations.py:28-52, model_components/utils.py:21-41

State-dict keys match the reference's torch path (`hash_table`, `scalings`, `layers.{i}.weight|bias`, `beta`), so
checkpoints are interchangeable with it.  `implementation` is accepted for signature compatibility; there is one
implementation here: the CUDA kernels.
"""
from __future__ import annotations

import contextlib
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Set, Tuple, Type

import numpy as np
import torch
from torch import Tensor, nn

from . import _lib
from . import functional as F
from .rays import GaussiansStd


def _warn_impl(implementation: str) -> None:
    if implementation not in ("tcnn", "torch", "b200"):
        raise ValueError(f"unknown implementation {implementation!r}")


class HashEncoding(nn.Module):
    """Multiresolution hash grid; forward = gather-bound CUDA kernel, backward = atomic scatter kernel."""

    def __init__(
        self,
        num_levels: int = 16,
        min_res: int = 16,
        max_res: int = 1024,
        log2_hashmap_size: int = 19,
        features_per_level: int = 2,
        hash_init_scale: float = 0.001,
        implementation: str = "b200",
        interpolation: Optional[str] = None,
        n_input_dims: int = 3,
    ) -> None:
        super().__init__()
        _warn_impl(implementation)
        assert interpolation is None or interpolation == "Linear", f"interpolation '{interpolation}' is not supported"
        if n_input_dims != 3:
            raise NotImplementedError("only 3-D hash grids are on the NeuRadar torch path")
        if features_per_level not in (1, 2, 4):
            raise NotImplementedError("features_per_level must be 1, 2 or 4")
        self.in_dim = 3
        self.num_levels = num_levels
        self.min_res = min_res
        self.max_res = max_res
        self.features_per_level = features_per_level
        self.hash_init_scale = hash_init_scale
        self.log2_hashmap_size = log2_hashmap_size
        self.hash_table_size = 2**log2_hashmap_size

        # identical expressions to encodings.py:348-352 so that the fp32 level resolutions agree bit for bit
        levels = torch.arange(num_levels)
        self.growth_factor = np.exp((np.log(max_res) - np.log(min_res)) / (num_levels - 1)) if num_levels > 1 else 1.0
        self.register_buffer("scalings", torch.floor(min_res * self.growth_factor**levels))
        self.hash_offset = levels * self.hash_table_size
        self.tcnn_encoding = None

        table = torch.rand(size=(self.hash_table_size * num_levels, features_per_level)) * 2 - 1
        self.hash_table = nn.Parameter(table * hash_init_scale)
        self._spec = F.GridSpec(num_levels, features_per_level, log2_hashmap_size, tuple(float(s) for s in self.scalings))

    @property
    def spec(self) -> F.GridSpec:
        return self._spec

    def get_out_dim(self) -> int:
        return self.num_levels * self.features_per_level

    def hash_fn(self, in_tensor: Tensor) -> Tensor:
        """Rows of integer grid coordinates [..., L, 3] -> [..., L] int64 (encodings.py:406-423), for inspection."""
        c = in_tensor.to(torch.int64)
        h = c[..., 0] ^ (c[..., 1] * 2654435761) ^ (c[..., 2] * 805459861)
        return torch.remainder(h, self.hash_table_size) + self.hash_offset.to(h.device)

    def corner_indices(self, in_tensor: Tensor) -> Tensor:
        """Rows gathered for each point: [*bs, L, 8] int64, computed by the CUDA kernel."""
        flat = in_tensor.reshape(-1, 3)
        return F.hash_indices(flat, self._spec).view(*in_tensor.shape[:-1], self.num_levels, 8)

    def forward(self, in_tensor: Tensor, std: Optional[Tensor] = None) -> Tensor:
        assert in_tensor.shape[-1] == 3
        flat = in_tensor.reshape(-1, 3)
        out = F.hash_encode(flat, self.hash_table, self._spec, None if std is None else std.reshape(-1))
        return out.view(*in_tensor.shape[:-1], self.get_out_dim())


class SHEncoding(nn.Module):
    """Degree-4 spherical harmonics (16 components); no gradient, like the reference's torch path."""

    def __init__(self, levels: int = 4, implementation: str = "b200") -> None:
        super().__init__()
        _warn_impl(implementation)
        if levels != 4:
            raise NotImplementedError("the B200 kernel implements the 4-level encoding NeuRadar uses")
        self.in_dim = 3
        self.levels = levels

    def get_out_dim(self) -> int:
        return self.levels**2

    @torch.no_grad()
    def forward(self, in_tensor: Tensor) -> Tensor:
        out = F.sh16(in_tensor.reshape(-1, 3), normalize_to_unit_cube=False)
        return out.view(*in_tensor.shape[:-1], 16)


class MLP(nn.Module):
    """Linear+ReLU chain evaluated by the fused MLP kernels (ReLU hidden activation, no output activation)."""

    def __init__(
        self,
        in_dim: int,
        num_layers: int,
        layer_width: int,
        out_dim: Optional[int] = None,
        skip_connections: Optional[Tuple[int]] = None,
        activation: Optional[nn.Module] = nn.ReLU(),
        out_activation: Optional[nn.Module] = None,
        implementation: str = "b200",
    ) -> None:
        super().__init__()
        _warn_impl(implementation)
        assert in_dim > 0
        if skip_connections:
            raise NotImplementedError("skip connections are not used on the NeuRadar path")
        if not isinstance(activation, nn.ReLU):
            raise NotImplementedError("hidden activation must be ReLU")
        self.in_dim = in_dim
        self.out_dim = out_dim if out_dim is not None else layer_width
        self.num_layers = num_layers
        self.layer_width = layer_width
        self.skip_connections = skip_connections
        self._skip_connections: Set[int] = set()
        self.activation = activation
        self.out_activation = out_activation
        self.tcnn_encoding = None
        dims = [in_dim] + [layer_width] * (num_layers - 1) + [self.out_dim]
        self.layers = nn.ModuleList([nn.Linear(dims[i], dims[i + 1]) for i in range(num_layers)])

    def get_out_dim(self) -> int:
        return self.out_dim

    def forward(self, in_tensor: Tensor) -> Tensor:
        flat = in_tensor.reshape(-1, self.in_dim)
        y = F.mlp_forward(flat, [l.weight for l in self.layers], [l.bias for l in self.layers])
        y = y.view(*in_tensor.shape[:-1], self.out_dim)
        if self.out_activation is not None:
            y = self.out_activation(y)
        return y


class _TruncExp(torch.autograd.Function):
    """exp with the backward exponent clamped to [-15, 15] (activations.py:28-41)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g):
        return g * torch.exp(ctx.saved_tensors[0].clamp(-15, 15))


trunc_exp = _TruncExp.apply


class SigmoidDensity(nn.Module):
    """alpha = sigmoid(-sdf * (|beta| + beta_min)) (model_components/utils.py:21-41)."""

    def __init__(self, init_val, beta_min=0.0001, learnable_beta=False):
        super().__init__()
        self.register_buffer("beta_min", torch.tensor(beta_min))
        self.register_parameter("beta", nn.Parameter(init_val * torch.ones(1), requires_grad=learnable_beta))
        self.beta_min_value = float(beta_min)  # host copy: the kernels take it by value, reading the buffer would synchronise

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        key = prefix + "beta_min"
        if key in state_dict:
            self.beta_min_value = float(state_dict[key])
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    def forward(self, sdf: Tensor, beta: Optional[Tensor] = None) -> Tensor:
        if beta is None:
            beta = self.get_beta()
        return torch.sigmoid(-sdf * beta)

    def get_beta(self):
        return self.beta.abs() + self.beta_min


# ------------------------------------------------------------------------------------------------
@dataclass
class StaticSettings:
    hashgrid_dim: int = 4
    num_levels: int = 8
    base_res: int = 32
    max_res: int = 8192
    log2_hashmap_size: int = 22


@dataclass
class ActorSettings:
    flip_prob: float = 0.5
    actor_scale: float = 10.0
    hashgrid_dim: int = 4
    num_levels: int = 4
    base_res: int = 64
    max_res: int = 1024
    log2_hashmap_size: int = 17
    use_4d_hashgrid: bool = True


@dataclass
class NeuRADHashEncodingConfig:
    _target: Type = field(default_factory=lambda: NeuRADHashEncoding)
    static: StaticSettings = field(default_factory=StaticSettings)
    actor: ActorSettings = field(default_factory=ActorSettings)
    disable_actors: bool = False
    require_actor_grad: bool = True

    def setup(self, **kwargs):
        return self._target(self, **kwargs)


class NoActors:
    """Stand-in for DynamicActors with zero trajectories (model_components/dynamic_actors.py): static scenes."""

    n_actors = 0


def _pose_inverse(pose: Tensor) -> Tensor:
    """[..., 3|4, 4] -> [..., 3, 4] (utils/poses.py:42-55)."""
    Ri = pose[..., :3, :3].transpose(-2, -1)
    return torch.cat([Ri, -Ri.matmul(pose[..., :3, 3:])], dim=-1)


def _transform(points: Tensor, transforms: Tensor, with_translation: bool = True) -> Tensor:
    """cameras/lidars.py:507-519"""
    out = (points.unsqueeze(-2) @ transforms[..., :3, :3].swapaxes(-2, -1)).squeeze(-2)
    return out + transforms[..., :3, 3] if with_translation else out


class NeuRADHashEncoding(nn.Module):
    """Static-world hash grid plus per-actor grids with contraction and per-level anti-alias weights
    (neurad_encoding.py:87-316, the torch path: one 3-D grid per actor).

    `dynamic_actors` is the reference's `DynamicActors` (or anything with `n_actors`, `get_boxes2world(times,
    flatten=False) -> (boxes2world [N,A,4,4], valid [N,A])`, `actor_bounds() -> [A,3]` and `actor_to_id [A]`); its
    trajectory interpolation is outside the hot path and is used as is.  The static grid runs through the
    gaussian+contraction and hash kernels; the actor branch keeps the reference's bookkeeping (which samples fall
    into which box) in PyTorch index ops and evaluates the per-actor grids with the same hash kernels."""

    def __init__(self, config: NeuRADHashEncodingConfig, dynamic_actors=None, static_scale: float = 1.0,
                 implementation: str = "b200") -> None:
        super().__init__()
        _warn_impl(implementation)
        self.config = config
        self.implementation = implementation
        self.actors = dynamic_actors if dynamic_actors is not None else NoActors()
        self.static_scale = float(static_scale)
        self.actor_scale = float(config.actor.actor_scale)
        self.static_grid = HashEncoding(
            features_per_level=config.static.hashgrid_dim,
            num_levels=config.static.num_levels,
            min_res=config.static.base_res,
            max_res=config.static.max_res,
            log2_hashmap_size=config.static.log2_hashmap_size,
        )
        n_grids = int(getattr(self.actors, "n_actors", 0))
        self.actor_grids = nn.ModuleList(
            [
                HashEncoding(
                    features_per_level=config.actor.hashgrid_dim,
                    num_levels=config.actor.num_levels,
                    min_res=config.actor.base_res,
                    max_res=config.actor.max_res,
                    log2_hashmap_size=config.actor.log2_hashmap_size,
                )
                for _ in range(n_grids)
            ]
        )
        self.scene_repr_dim = self.static_grid.get_out_dim()

    def get_out_dim(self) -> int:
        return self.scene_repr_dim

    def get_param_groups(self, param_groups: Dict):
        param_groups["hashgrids"] += list(self.static_grid.parameters()) + list(self.actor_grids.parameters())

    @property
    def has_actors(self) -> bool:
        return int(getattr(self.actors, "n_actors", 0)) > 0 and not self.config.disable_actors

    def forward(self, positions: GaussiansStd, times: Optional[Tensor] = None, directions: Optional[Tensor] = None):
        """World-space gaussians (mean [N,S,1,3], std [N,S,1,1]) -> (features [N*S, L*F], directions)."""
        mean = positions.mean.reshape(-1, 3)
        std = positions.std.reshape(-1, 1)
        feats = self.static_grid(*self._contract(mean, std, self.static_scale))
        if not self.has_actors or times is None:
            return feats, directions
        n, s = positions.mean.shape[0], positions.mean.shape[1]
        dirs = None if directions is None else directions.reshape(n, s, 3)
        feats, dirs = self._apply_actors(feats, positions.mean.reshape(n, s, 3), positions.std.reshape(n, s, 1), dirs,
                                         times.reshape(n, -1)[:, 0])
        return feats, (None if dirs is None else dirs.reshape(directions.shape))

    @staticmethod
    def _contract(mean: Tensor, std: Tensor, scale: float) -> Tuple[Tensor, Tensor]:
        """ScaledSceneContraction(order=inf, scale) on GaussiansStd, spatial_distortions.py:103-113,132-136."""
        mean = mean / scale
        std = std / scale
        mag = mean.abs().amax(dim=-1, keepdim=True)
        cm = mag.clamp_min(1.0)
        inside = mag < 1
        mean = torch.where(inside, mean, (2 - (1 / cm)) * (mean / cm))
        std = torch.where(inside, std, std * ((2 * cm - 1).pow(1 / 3) / cm) ** 2)
        return (mean + 2.0) / 4.0, std / 4.0

    def encode_samples(self, rays: F.RayData, iv: F.SampleIntervals, times: Optional[Tensor] = None):
        """Fast path from per-ray data.  Returns (features [N*S, L*F], per-sample directions [N,S,3] or None when no
        sample was claimed by an actor and the per-ray directions still apply)."""
        x, std = F.frustum_gaussians(rays, iv, self.static_scale)
        feats = F.hash_encode(x, self.static_grid.hash_table, self.static_grid.spec, std, samples_per_ray=iv.num_samples)
        if not self.has_actors or times is None:
            return feats, None
        # world-space gaussians of cameras/rays.py:109-124 for the actor bookkeeping
        starts, ends = iv.starts, iv.ends
        dist = (ends - starts) / 2
        t = starts + dist
        mean = rays.origins[:, None, :] + rays.directions[:, None, :] * t[..., None]
        wstd = (rays.pixel_area[:, None, None] * t[..., None].pow(2) * dist[..., None]).pow(1 / 3)
        dirs = rays.directions[:, None, :].expand(-1, iv.num_samples, -1)
        return self._apply_actors(feats, mean, wstd, dirs, times.reshape(-1))

    pose_cache: Optional[dict] = None
    """Set by the owner of several encodings that see the same rays within one step (NeuRadarHotPath: the field and the
    proposal networks): the actor poses at the rays' times are then computed once per step instead of once per encoding."""

    ray_flip_override: Optional[Tensor] = None
    """Tests: replay a recorded per-ray mirror draw ([N] of +1 / -1) instead of drawing one."""

    def _draw_flip(self, n: int, device) -> Optional[Tensor]:
        """-1 with probability flip_prob, per ray, in training (neurad_encoding.py:218-225)."""
        if not (self.training and self.config.actor.flip_prob > 1.0e-7):
            return None
        if self.ray_flip_override is not None:
            return self.ray_flip_override
        return torch.bernoulli(torch.full((n,), self.config.actor.flip_prob, device=device)) * -2 + 1

    def _poses_trainable(self) -> bool:
        return any(p.requires_grad for p in getattr(self.actors, "parameters", lambda: [])())

    def can_assign_in_kernel(self, proposal: bool = False) -> bool:
        """The actor kernels cover the reference's default actor grids (4 levels, one table shape; 4 features in the field,
        the static grid's feature count in a proposal network) for up to _lib.MAX_ACTORS (256) actor grids.  Trained
        actor poses stay on them: the field takes their gradient in CUDA (nrb_actor_pose_grad), and an encoding with
        require_actor_grad=False (the proposal networks' default) treats them as constants, as the reference does.  A
        proposal network configured with require_actor_grad=True and trained poses takes the torch bookkeeping below."""
        if not self.has_actors or len(self.actor_grids) == 0 or len(self.actor_grids) > _lib.MAX_ACTORS:
            return False
        a = self.config.actor
        dim = self.config.static.hashgrid_dim if proposal else 4
        if proposal and self.config.static.num_levels < a.num_levels:
            return False
        return a.num_levels == 4 and a.hashgrid_dim == dim and not (
            proposal and self.config.require_actor_grad and self._poses_trainable())

    def assign_actors(self, rays: F.RayData, iv: F.SampleIntervals, times: Tensor) -> "F.ActorBatch":
        """Which samples fall into which actor box, in one kernel (csrc/actors.cu): no nonzero(), no host synchronisation.
        With trained poses, grad mode and require_actor_grad the batch carries the pose context (F.ActorPose), through
        which the field differentiates with respect to the actor trajectories."""
        track = torch.is_grad_enabled() and self._poses_trainable()
        key = (times.data_ptr(), times._version, tuple(times.shape))
        cached = None if self.pose_cache is None else self.pose_cache.get(key)
        # The encodings of one step share the cache and the proposal rounds fill it first: an entry always carries the
        # graph when poses are trained, and an encoding that does not differentiate by them only reads it detached.
        if cached is None or (track and not cached[0].requires_grad):
            with torch.set_grad_enabled(track):
                boxes2world, valid = self.actors.get_boxes2world(times.reshape(-1), flatten=False)
                # (R^T | -R^T t) element-wise: a matmul over [N, A] 3x3 blocks becomes A batched cuBLAS gemv launches
                Ri = boxes2world[..., :3, :3].transpose(-2, -1)
                world2boxes = torch.cat([Ri, -(Ri * boxes2world[..., None, :3, 3]).sum(-1, keepdim=True)], dim=-1).contiguous()
            cached = (world2boxes, valid.detach(), times)  # (times is held so that its address cannot be recycled under the key)
            if self.pose_cache is not None:
                self.pose_cache[key] = cached
        world2boxes, valid = cached[0], cached[1]
        pose_grad = track and self.config.require_actor_grad
        flip = self._draw_flip(rays.num_rays, rays.origins.device)
        index = torch.empty((rays.num_rays * iv.num_samples,), device=rays.origins.device, dtype=torch.int32) if pose_grad else None
        with torch.no_grad():
            grid_id, pos, std, dirs = F.actor_assign(rays, iv, world2boxes, valid, self.actors.actor_bounds(),
                                                     self.actors.actor_to_id, flip, self.actor_scale, index)
        pose = F.ActorPose(world2boxes, index, flip, self.actor_scale, rays, iv) if pose_grad else None
        return F.ActorBatch(grid_id, pos, std, dirs, [g.hash_table for g in self.actor_grids], self.actor_grids[0].spec, pose)

    @torch.no_grad()
    def _actor_indices(self, mean: Tensor, boxes2world: Tensor, valid: Tensor, world2boxes: Tensor, bounds: Tensor):
        """(ray, sample, actor) of the samples inside actor boxes: ray line vs bounding sphere, sample vs sphere, then
        the exact box test (neurad_encoding.py:231-275)."""
        eps = 1.0e-7
        radii = bounds.norm(dim=-1)
        p0 = mean[:, 0, :]
        line = mean[:, -1, :] - p0
        line = (line / (torch.linalg.norm(line, dim=-1, keepdim=True) + eps)).unsqueeze(-2)
        centers = boxes2world[..., :3, 3]
        dist = torch.linalg.norm(torch.cross(centers - p0.unsqueeze(-2), line.expand_as(centers), dim=-1), dim=-1)
        r, a = ((dist < radii) & valid).nonzero(as_tuple=False).T
        if r.shape[0] == 0:
            return r, r, r
        within = torch.linalg.norm(mean[r] - centers[r, a].unsqueeze(-2), dim=-1) < radii[a].unsqueeze(-1)
        k, s = within.nonzero(as_tuple=False).T
        ri, ai = r[k], a[k]
        inside = (_transform(mean[ri, s], world2boxes[ri, ai]).abs() < bounds[ai]).all(dim=-1)
        return ri[inside], s[inside], ai[inside]

    def _apply_actors(self, feats: Tensor, mean: Tensor, std: Tensor, dirs: Optional[Tensor], times: Tensor,
                      ray_flip: Optional[Tensor] = None):
        """Overwrite the features (and directions) of the samples that fall into an actor box
        (neurad_encoding.py:176-229,295-316).  mean [N,S,3], std [N,S,1] in world units."""
        n, s, _ = mean.shape
        # the reference keeps the ambient grad mode when the actor poses are trainable (neurad_encoding.py:177)
        grad_ctx = contextlib.nullcontext() if self.config.require_actor_grad else torch.no_grad()
        with grad_ctx:
            boxes2world, valid = self.actors.get_boxes2world(times, flatten=False)
            world2boxes = _pose_inverse(boxes2world)
            ri, si, ai = self._actor_indices(mean.detach(), boxes2world.detach(), valid, world2boxes.detach(),
                                             self.actors.actor_bounds())
            if ri.shape[0] == 0:
                return feats, None
            w2b = world2boxes[ri, ai]
            pos = _transform(mean[ri, si], w2b)
            new_dirs = None
            if dirs is not None:
                d = _transform(dirs[ri, si], w2b, with_translation=False)
                d = d / (torch.linalg.norm(d, dim=-1, keepdim=True) + 1.0e-7)
            if self.training and self.config.actor.flip_prob > 1.0e-7:
                if ray_flip is None:
                    ray_flip = self._draw_flip(n, mean.device)
                f = ray_flip.to(pos.dtype)[ri][:, None]
                pos = torch.cat([pos[:, :1] * f, pos[:, 1:]], dim=-1)
                if dirs is not None:
                    d = torch.cat([d[:, :1] * f, d[:, 1:]], dim=-1)
            if dirs is not None:
                new_dirs = dirs.clone()
                new_dirs[ri, si] = d
        cpos, cstd = self._contract(pos, std[ri, si], self.actor_scale)
        grid_id = self.actors.actor_to_id[ai]
        out_dim = self.scene_repr_dim
        actor_feats = torch.zeros((ri.shape[0], out_dim), device=feats.device, dtype=feats.dtype)
        for gid in grid_id.unique().tolist():  # per-actor grids, as the reference's torch path (neurad_encoding.py:295-307)
            grid = self.actor_grids[gid]
            sel = (grid_id == gid).nonzero(as_tuple=True)[0]
            f = grid(cpos[sel], std=cstd[sel])
            actor_feats = actor_feats.index_put((sel,), torch.nn.functional.pad(f, (0, out_dim - f.shape[-1])))
        feats = feats.view(n, s, out_dim).index_put((ri, si), actor_feats).view(n * s, out_dim)
        return feats, new_dirs
