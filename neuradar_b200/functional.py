"""Autograd-aware wrappers around the C ABI.  Every function here launches hand-written sm_100a kernels from
libneuradar_b200.so on the current CUDA stream; none has a PyTorch or CPU implementation.

Shapes follow the reference: N rays, S samples per ray, M = N*S points, L levels, F features per level.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, replace
from types import SimpleNamespace
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor
from torch.amp import custom_bwd, custom_fwd

from . import _lib
from ._lib import Grid, Intervals, Mlp, MlpGrad, Rays, Spacing, check, f32c, ptr, stream_ptr
from .dist import padded_numel


# ------------------------------------------------------------------------------------------------
# plain-data descriptors
# ------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class GridSpec:
    """Static description of one HashEncoding (reference: field_components/encodings.py:326-352)."""

    num_levels: int
    features_per_level: int
    log2_hashmap_size: int
    scalings: Tuple[float, ...]

    @property
    def out_dim(self) -> int:
        return self.num_levels * self.features_per_level

    @property
    def rows(self) -> int:
        return self.num_levels << self.log2_hashmap_size

    @property
    def tag(self) -> str:
        return f"L{self.num_levels}F{self.features_per_level}T{self.log2_hashmap_size}"

    def struct(self, table: Tensor) -> Grid:
        if table.shape != (self.rows, self.features_per_level):
            raise ValueError(f"hash_table has shape {tuple(table.shape)}, expected {(self.rows, self.features_per_level)}")
        g = Grid()
        g.table = ptr(table)
        for i, s in enumerate(self.scalings):
            g.scalings[i] = s
        g.num_levels = self.num_levels
        g.features_per_level = self.features_per_level
        g.log2_hashmap_size = self.log2_hashmap_size
        return g


@dataclass
class RayData:
    """Per-ray tensors of a RayBundle, un-broadcast and contiguous: origins/directions [N,3], the rest [N]."""

    origins: Tensor
    directions: Tensor
    pixel_area: Tensor
    nears: Optional[Tensor] = None
    fars: Optional[Tensor] = None

    def __post_init__(self):
        self.origins = f32c(self.origins)
        self.directions = f32c(self.directions)
        self.pixel_area = f32c(self.pixel_area.reshape(-1))
        if self.nears is not None:
            self.nears = f32c(self.nears.reshape(-1))
        if self.fars is not None:
            self.fars = f32c(self.fars.reshape(-1))

    @property
    def num_rays(self) -> int:
        return self.origins.shape[0]

    def struct(self) -> Rays:
        r = Rays()
        r.origins, r.directions, r.pixel_area = ptr(self.origins), ptr(self.directions), ptr(self.pixel_area)
        r.nears, r.fars = ptr(self.nears), ptr(self.fars)
        r.num_rays = self.num_rays
        return r


class SampleIntervals:
    """starts/ends [N,S] of the samples along each ray.  Views of one [N,S+1] bin tensor are passed through
    without a copy (row stride S+1), which is how every sampler on the path produces them."""

    def __init__(self, starts: Tensor, ends: Tensor):
        if starts.dim() == 3:
            starts, ends = starts[..., 0], ends[..., 0]
        if starts.shape != ends.shape or starts.dim() != 2:
            raise ValueError("starts/ends must both be [N,S] (or [N,S,1])")
        ok = (
            starts.dtype == torch.float32
            and ends.dtype == torch.float32
            and starts.stride(1) == 1
            and ends.stride(1) == 1
            and starts.stride(0) == ends.stride(0)
            and starts.stride(0) >= starts.shape[1]
        )
        if not ok:
            starts, ends = f32c(starts), f32c(ends)
        self.starts, self.ends = starts, ends

    @classmethod
    def from_bins(cls, bins: Tensor) -> "SampleIntervals":
        bins = f32c(bins)
        return cls(bins[:, :-1], bins[:, 1:])

    @property
    def num_samples(self) -> int:
        return self.starts.shape[1]

    def struct(self) -> Intervals:
        if not self.starts.is_cuda:
            raise _lib.NeuradarB200Error("neuradar_b200 ops need CUDA tensors; there is no CPU path")
        iv = Intervals()
        # (views of a bins tensor are not contiguous, so no ptr(); empty tensors have a null data_ptr: see _lib.ptr)
        empty = self.starts.numel() == 0
        iv.starts = _lib._EMPTY_SENTINEL if empty else self.starts.data_ptr()
        iv.ends = _lib._EMPTY_SENTINEL if empty else self.ends.data_ptr()
        iv.row_stride = self.starts.stride(0) if self.starts.shape[0] > 1 else max(self.starts.stride(0), self.num_samples)
        iv.num_samples = self.num_samples
        return iv


def _lib_():
    return _lib.load()


_WORKSPACES = {}


def _workspace(nbytes: int, device):
    """Scratch memory for kernels that want it: one buffer per (device, stream), grown on demand.  Calls on one stream
    are ordered, so they can share a buffer; calls on different streams (the path overlaps its backward branches on
    side streams) must not."""
    if nbytes <= 0:
        return None, 0
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty((nbytes,), device=device, dtype=torch.uint8)
        _WORKSPACES[key] = buf
    return buf.data_ptr(), nbytes


def _scatter_workspace(grid_struct: Grid, M: int, device):
    """Workspace of a hash-table gradient scatter over M samples (the lattice replicas of its coarse levels)."""
    return _workspace(int(_lib_().nrb_hash_bwd_workspace_bytes(C.byref(grid_struct), M)), device)


_SIDE_STREAMS = {}


def side_stream(device, index: int = 0) -> "torch.cuda.Stream":
    """Per-device auxiliary streams.  Autograd replays every backward node on the stream its forward ran on, so
    running independent branches of the forward on side streams is what lets their backward kernels overlap (the
    latency-bound tensor-core MLP backward with the L2-reduction-bound table scatters)."""
    key = (torch.device(device), index)
    s = _SIDE_STREAMS.get(key)
    if s is None:
        s = torch.cuda.Stream(device=device)
        _SIDE_STREAMS[key] = s
    return s


# ------------------------------------------------------------------------------------------------
# hash grid
# ------------------------------------------------------------------------------------------------
def grad_sink_of(table: Optional[Tensor]) -> Optional[Tensor]:
    """Opt-in direct gradient accumulation: when the owner of the flat gradient buffer (dist.GradArena, optim.FusedAdam)
    marked a parameter with `_nrb_grad_sink` (a view with the parameter's shape), the backward kernels add straight
    into it and the autograd Function returns no gradient for it.  For a hash table this skips a zero-fill of a
    table-sized temporary and AccumulateGrad's read-add-write of it (3 x 64 MiB of traffic for the main grid) per
    backward; for the small MLP parameters it removes a zero-fill and an add launch each."""
    if table is None:
        return None
    sink = getattr(table, "_nrb_grad_sink", None)
    if sink is None or sink.shape != table.shape or sink.dtype != torch.float32 or not sink.is_contiguous():
        return None
    return sink


_CONSUMER_STREAMS = {}


def note_consumer_stream(device) -> None:
    """Called where a branch of the forward is moved to a side stream: the current stream is the one the training loop
    runs on, i.e. the one that will read the gradient sinks after `backward()`."""
    device = torch.device(device)
    _CONSUMER_STREAMS[device] = torch.cuda.current_stream(device)


def _sink_written(params: Sequence[Tensor]) -> None:
    """Called once by a backward that added straight into the gradient sinks of `params` (no tensor is returned to
    autograd for them, so autograd's own stream bookkeeping does not cover the writes).  (1) If the backward ran on a
    side stream - autograd replays a node on the stream its forward ran on - the default stream is made to wait for it,
    so that an all-reduce or optimiser step issued after `loss.backward()` cannot race with the scatter.  (2) The owner of
    a sink may have registered a callback (dist.OverlappedReduce.start_early) to start reducing that gradient right away."""
    dev = params[0].device
    cur = torch.cuda.current_stream(dev)
    if not torch.cuda.is_current_stream_capturing():  # (a graph capture orders its own streams)
        # the default stream and the stream the forward was issued from (`note_consumer_stream`): whoever reads the sink next
        waiters = {torch.cuda.default_stream(dev), _CONSUMER_STREAMS.get(dev, cur)} - {cur}
        if waiters:
            ev = cur.record_event()
            for s in waiters:
                s.wait_event(ev)
    for p in params:
        ready = getattr(p, "_nrb_grad_ready", None)
        if ready is not None:
            ready()


class _GradSinks:
    """The gradient sinks (`grad_sink_of`) of an autograd node's parameters, looked up by its forward.  The backward takes
    each gradient buffer from `dest()` / `packed_dests()` (the sink, or zeroed memory whose content goes back to autograd),
    launches, and returns what `written()` gives back."""

    def __init__(self, params: Sequence[Optional[Tensor]]):
        self.params = list(params)
        self.sinks = [grad_sink_of(p) for p in self.params]

    def dest(self, i: int) -> Tensor:
        p = self.params[i]
        return self.sinks[i] if self.sinks[i] is not None else torch.zeros(p.shape, device=p.device, dtype=torch.float32)

    def packed_dests(self, idx: range) -> List[Optional[Tensor]]:
        """`dest()` of the parameters `idx` (None for a None parameter), with the zeroed ones packed into ONE scratch
        buffer: one memset instead of one per parameter."""
        need = [self.params[i] for i in idx if self.params[i] is not None and self.sinks[i] is None]
        scratch = torch.zeros((sum(padded_numel(p.numel()) for p in need),), device=need[0].device,
                              dtype=torch.float32) if need else None
        out, off = [], 0
        for i in idx:
            p, sink = self.params[i], self.sinks[i]
            if p is None or sink is not None:
                out.append(sink)
            else:
                out.append(scratch[off : off + p.numel()].view(p.shape))
                off += padded_numel(p.numel())
        return out

    def written(self, grads: Sequence[Optional[Tensor]]) -> List[Optional[Tensor]]:
        """Called once after the launches with one buffer per parameter: orders and signals every sink (`_sink_written`);
        returns `grads` with None where a sink took the gradient."""
        written = [p for p, sink in zip(self.params, self.sinks) if sink is not None]
        if written:
            _sink_written(written)
        return [None if sink is not None else g for g, sink in zip(grads, self.sinks)]


def _save(ctx, **named) -> None:
    """ctx.save_for_backward, once, under names; a value is a tensor, None or a list of them.  `_saved(ctx)` gives them
    back as attributes."""
    ctx.saved_layout = [(k, len(v) if isinstance(v, list) else -1) for k, v in named.items()]
    ctx.save_for_backward(*[t for v in named.values() for t in (v if isinstance(v, list) else [v])])


def _saved(ctx) -> SimpleNamespace:
    it = iter(ctx.saved_tensors)
    return SimpleNamespace(**{k: next(it) if n < 0 else [next(it) for _ in range(n)] for k, n in ctx.saved_layout})


class _HashEncode(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, table, std, spec: GridSpec, samples_per_ray: int = 0):
        ctx.sinks = _GradSinks([table])
        x = f32c(x)
        table = f32c(table)
        std = None if std is None else f32c(std.reshape(-1))
        M = x.shape[0]
        out = torch.empty((M, spec.out_dim), device=x.device, dtype=torch.float32)
        g = spec.struct(table)
        _lib.call("nrb_hash_fwd", C.byref(g), ptr(x), ptr(std), ptr(out), M, stream_ptr(), tag="nrb_hash_fwd:" + spec.tag)
        ctx.save_for_backward(x, table, std)
        ctx.spec = spec
        ctx.samples_per_ray = int(samples_per_ray)
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dy):
        x, table, std = ctx.saved_tensors
        spec = ctx.spec
        dy = f32c(dy)
        need_dx = ctx.needs_input_grad[0]
        dtable = ctx.sinks.dest(0)
        dx = torch.empty_like(x) if need_dx else None
        g = spec.struct(table)
        ws, ws_bytes = _scatter_workspace(g, x.shape[0], x.device)
        _lib.call("nrb_hash_bwd", C.byref(g), ptr(x), ptr(std), ptr(dy), ptr(dtable), ptr(dx), x.shape[0], ws, ws_bytes,
                  stream_ptr(), tag="nrb_hash_bwd:" + spec.tag)
        return dx, *ctx.sinks.written([dtable]), None, None, None


def hash_encode(x: Tensor, table: Tensor, spec: GridSpec, std: Optional[Tensor] = None, samples_per_ray: int = 0) -> Tensor:
    """HashEncoding.forward on points x [M,3]; with `std` [M] also applies the per-level anti-alias weights.
    `samples_per_ray` is a layout hint for the backward kernel (runs of consecutive samples of one ray)."""
    return _HashEncode.apply(x, table, std, spec, samples_per_ray)


def hash_indices(x: Tensor, spec: GridSpec) -> Tensor:
    """Table rows of the 8 cell corners, [M, L, 8] int64 (corner order of encodings.py:436-443)."""
    x = f32c(x)
    M = x.shape[0]
    idx = torch.empty((M, spec.num_levels, 8), device=x.device, dtype=torch.int64)
    g = Grid()
    g.table = ptr(x)  # unused by the kernel, must be non-null and aligned
    for i, s in enumerate(spec.scalings):
        g.scalings[i] = s
    g.num_levels, g.features_per_level, g.log2_hashmap_size = spec.num_levels, spec.features_per_level, spec.log2_hashmap_size
    _lib.call("nrb_hash_indices", C.byref(g), ptr(x), ptr(idx), M, stream_ptr())
    return idx


def frustum_gaussians(rays: RayData, iv: SampleIntervals, scale: float) -> Tuple[Tensor, Tensor]:
    """Contracted sample means [N*S,3] and stds [N*S] (get_fast_isotropic_gaussian(1) + ScaledSceneContraction)."""
    N, S = rays.num_rays, iv.num_samples
    x = torch.empty((N * S, 3), device=rays.origins.device, dtype=torch.float32)
    std = torch.empty((N * S,), device=rays.origins.device, dtype=torch.float32)
    r, i = rays.struct(), iv.struct()
    _lib.call("nrb_frustum_gaussians", C.byref(r), C.byref(i), float(scale), ptr(x), ptr(std), stream_ptr())
    return x, std


# ------------------------------------------------------------------------------------------------
# tiny MLP
# ------------------------------------------------------------------------------------------------
def _mlp_struct(dims: Sequence[int], weights: Sequence[Tensor], biases: Sequence[Optional[Tensor]]) -> Mlp:
    m = Mlp()
    m.num_layers = len(weights)
    for i, d in enumerate(dims):
        m.dims[i] = d
    for i, (w, b) in enumerate(zip(weights, biases)):
        m.weights[i] = ptr(w)
        m.biases[i] = ptr(b)
    return m


class _MlpForward(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, n_layers: int, *params):
        weights = [f32c(w) for w in params[:n_layers]]
        biases = [None if b is None else f32c(b) for b in params[n_layers:]]
        x = f32c(x)
        dims = [weights[0].shape[1]] + [w.shape[0] for w in weights]
        if x.shape[-1] != dims[0]:
            raise ValueError(f"MLP input has {x.shape[-1]} features, expected {dims[0]}")
        M = x.shape[0]
        y = torch.empty((M, dims[-1]), device=x.device, dtype=torch.float32)
        n_hidden = sum(dims[1:-1])
        keep = any(ctx.needs_input_grad) and n_hidden > 0
        hidden = torch.empty((n_hidden, M), device=x.device, dtype=torch.float32) if keep else None
        m = _mlp_struct(dims, weights, biases)
        _lib.call("nrb_mlp_fwd", C.byref(m), ptr(x), ptr(y), ptr(hidden), M, stream_ptr(), tag="nrb_mlp_fwd:" + "x".join(map(str, dims)))
        _save(ctx, x=x, hidden=hidden, weights=weights, biases=biases)
        ctx.dims = dims
        return y

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dy):
        s = _saved(ctx)
        x, hidden, weights, biases, n = s.x, s.hidden, s.weights, s.biases, len(ctx.dims) - 1
        dy = f32c(dy)
        M = x.shape[0]
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dws = [torch.zeros_like(w) for w in weights]
        dbs = [None if b is None else torch.zeros_like(b) for b in biases]
        m = _mlp_struct(ctx.dims, weights, biases)
        g = MlpGrad()
        for i in range(n):
            g.weights[i] = ptr(dws[i])
            g.biases[i] = ptr(dbs[i])
        _lib.call("nrb_mlp_bwd", C.byref(m), ptr(x), ptr(hidden), ptr(dy), ptr(dx), C.byref(g), M, stream_ptr(),
                  tag="nrb_mlp_bwd:" + "x".join(map(str, ctx.dims)))
        return (dx, None, *dws, *dbs)


def mlp_forward(x: Tensor, weights: Sequence[Tensor], biases: Sequence[Optional[Tensor]]) -> Tensor:
    """Linear+ReLU chain on x [M, in] (no output activation), MLP.pytorch_fwd semantics."""
    return _MlpForward.apply(x, len(weights), *weights, *biases)


def tc_linear(x: Tensor, weight: Tensor, bias: Optional[Tensor], relu: bool = False) -> Tensor:
    """y = x W^T + b through the tcgen05 building blocks (K in {32, 48}, out <= 48); forward only, for testing."""
    x, weight = f32c(x), f32c(weight)
    bias = None if bias is None else f32c(bias)
    M, K = x.shape
    y = torch.empty((M, weight.shape[0]), device=x.device, dtype=torch.float32)
    _lib.call("nrb_tc_linear", ptr(x), ptr(weight), ptr(bias), K, weight.shape[0], int(relu), M, ptr(y), stream_ptr())
    return y


def _field_struct(weights: Sequence[Tensor], biases: Sequence[Optional[Tensor]], beta: Tensor, beta_min: float):
    m = _lib.FieldMlp()
    for i in range(5):
        m.weights[i] = ptr(weights[i])
        m.biases[i] = ptr(biases[i])
    m.beta = ptr(beta)
    m.beta_min = float(beta_min)
    return m


# ------------------------------------------------------------------------------------------------
# dynamic actors: per-sample assignment (no compaction, no host synchronisation)
# ------------------------------------------------------------------------------------------------
@dataclass
class ActorBatch:
    """Which samples of a [N,S] batch fall into which actor box (csrc/actors.cu): grid_id [M] int32 (-1 = static world),
    pos [M,3] in the actor grid's unit cube, std [M], dirs [M,3] in the actor frame; plus the per-actor tables."""

    grid_id: Tensor
    pos: Tensor
    std: Tensor
    dirs: Tensor
    tables: List[Tensor]
    spec: GridSpec  # of ONE actor grid

    def grids_struct(self) -> "_lib.ActorGrids":
        g = _lib.ActorGrids()
        for i, t in enumerate(self.tables):
            g.tables[i] = ptr(t)
        for i, sc in enumerate(self.spec.scalings):
            g.scalings[i] = sc
        g.num_levels, g.features_per_level = self.spec.num_levels, self.spec.features_per_level
        g.log2_hashmap_size, g.num_grids = self.spec.log2_hashmap_size, len(self.tables)
        return g

    def samples_struct(self) -> "_lib.ActorSamples":
        a = _lib.ActorSamples()
        a.grid_id, a.pos, a.std, a.dirs = ptr(self.grid_id), ptr(self.pos), ptr(self.std), ptr(self.dirs)
        return a

    def with_tables(self, tables: Sequence[Tensor]) -> "ActorBatch":
        return replace(self, tables=list(tables))

    def to_save(self) -> List[Tensor]:  # what `from_saved` rebuilds the batch from
        return [self.grid_id, self.pos, self.std, self.dirs, *self.tables]

    @classmethod
    def from_saved(cls, saved: Sequence[Tensor], spec: GridSpec) -> "ActorBatch":
        return cls(*saved[:4], list(saved[4:]), spec)


def actor_assign(rays: RayData, iv: SampleIntervals, world2boxes: Tensor, valid: Tensor, bounds: Tensor, actor_to_id: Tensor,
                 flip: Optional[Tensor], actor_scale: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """NeuRADHashEncoding._split_static_vs_actors as one kernel: (grid_id [M] int32, pos [M,3], std [M], dirs [M,3]) of the
    M = N*S samples; world2boxes [N,A,3,4], valid [N,A], bounds [A,3], actor_to_id [A], flip [N] (+1 / -1) or None."""
    N, S = rays.num_rays, iv.num_samples
    dev = rays.origins.device
    w2b = f32c(world2boxes.detach()[..., :3, :4])
    A = w2b.shape[1]
    val, bnd = _u8(valid), f32c(bounds.detach())
    a2i = actor_to_id.to(device=dev, dtype=torch.int32).contiguous()
    flp = None if flip is None else f32c(flip.reshape(-1))
    grid_id = torch.empty((N * S,), device=dev, dtype=torch.int32)
    pos = torch.zeros((N * S, 3), device=dev, dtype=torch.float32)
    std = torch.zeros((N * S,), device=dev, dtype=torch.float32)
    dirs = torch.zeros((N * S, 3), device=dev, dtype=torch.float32)
    r, i = rays.struct(), iv.struct()
    _lib.call("nrb_actor_assign", C.byref(r), C.byref(i), ptr(w2b), ptr(val), ptr(bnd), ptr(a2i), A, ptr(flp), float(actor_scale),
              ptr(grid_id), ptr(pos), ptr(std), ptr(dirs), None, stream_ptr())
    return grid_id, pos, std, dirs


# ------------------------------------------------------------------------------------------------
# fused field: hash gather + both MLPs in one kernel; backward recomputes the activations
# ------------------------------------------------------------------------------------------------
def _field_fused_backward(ctx, s: SimpleNamespace, dfeature, dfeat_ray, weights, dsdf, dalpha):
    """Shared by the two autograd Functions that end in the fused field kernel; `s` is `_saved(ctx)`.  Returns (dx or None,
    the gradients of [table, beta, w0..w4, b0..b4, *actor tables] for autograd); in gather mode the hash-table gradient
    is scattered here too."""
    actors = None if ctx.actor_spec is None else ActorBatch.from_saved(s.actors, ctx.actor_spec)
    M, dev = s.sdf.shape[0], s.sdf.device
    need_dx = ctx.gather or ctx.needs_x_grad
    dximg = torch.empty((int(_lib_().nrb_field_fused_image_bytes(M)) // 4,), device=dev, dtype=torch.float32) if need_dx else None
    sinks = ctx.sinks  # [table, beta, w0..w4, b0..b4, *actor tables]
    dmlp = sinks.packed_dests(range(1, 12))
    dbeta, dws, dbs = dmlp[0], dmlp[1:6], dmlp[6:11]
    m = _field_struct(s.weights, s.biases, s.beta, ctx.beta_min)
    bi = _lib.FieldFusedBwdIn()
    bi.saved.ximg, bi.saved.masks, bi.saved.ld = ptr(s.ximg), ptr(s.masks), s.masks.shape[1]
    bi.sh, bi.sdf, bi.alpha = ptr(s.sh), ptr(s.sdf), ptr(s.alpha)
    bi.dfeature, bi.dfeat_ray, bi.weights = ptr(dfeature), ptr(dfeat_ray), ptr(weights)
    bi.dsdf, bi.dalpha = ptr(dsdf), ptr(dalpha)
    if actors is not None:
        bi.actor_grid_id, bi.actor_dirs = ptr(actors.grid_id), ptr(actors.dirs)
    bo = _lib.FieldFusedBwdOut()
    bo.dximg = ptr(dximg)
    for i in range(5):
        bo.dweights[i] = ptr(dws[i])
        bo.dbiases[i] = ptr(dbs[i])
    bo.dbeta = ptr(dbeta)
    _lib.call("nrb_field_fused_bwd", C.byref(m), C.byref(bi), C.byref(bo), ctx.samples_per_ray, M, stream_ptr())
    dx = dtable = None
    if ctx.gather:
        spec = ctx.spec
        dtable = sinks.dest(0)
        g = spec.struct(s.table)
        ws, ws_bytes = _scatter_workspace(g, M, dev)
        _lib.call("nrb_hash_bwd_image", C.byref(g), ptr(s.x3), ptr(s.std), ptr(dximg), ptr(dtable),
                  None if actors is None else ptr(actors.grid_id), M, ws, ws_bytes, stream_ptr(), tag="nrb_hash_bwd:" + spec.tag)
    elif ctx.needs_x_grad:
        dx = dximg.view(-1, 8, 128, 4).permute(0, 2, 1, 3).reshape(-1, 32)[:M]
    dactor = []
    if actors is not None:  # the actor samples' gradient goes to their own tables
        dactor = [sinks.dest(i) for i in range(12, len(sinks.params))]
        arr = (C.c_void_p * len(dactor))(*[ptr(t) for t in dactor])
        ag, asmp = actors.grids_struct(), actors.samples_struct()
        _lib.call("nrb_actor_scatter", C.byref(ag), arr, C.byref(asmp), ptr(dximg), None, M, stream_ptr())
    return dx, sinks.written([dtable, *dmlp, *dactor])


def _field_fused_forward(ctx, table, x, x3, std, sh, samples_per_ray, beta_min, spec, beta, params, train,
                         actors: Optional[ActorBatch] = None):
    """Launch nrb_field_fused_fwd and set on ctx what the backward needs besides tensors.  Returns (feature, sdf, alpha,
    the tensors to save by name or None when not training)."""
    gather = table is not None
    ctx.sinks = _GradSinks([table, beta, *params])
    sh, beta = f32c(sh.detach()), f32c(beta)
    weights = [f32c(w) for w in params[:5]]
    biases = [None if b is None else f32c(b) for b in params[5:10]]
    ag = asmp = None
    if actors is not None:
        actors = actors.with_tables([f32c(t) for t in params[10:]])
        ag, asmp = actors.grids_struct(), actors.samples_struct()
    if gather:
        table, x3 = f32c(table), f32c(x3)
        std = None if std is None else f32c(std.reshape(-1))
        M, dev = x3.shape[0], x3.device
        g = spec.struct(table)
    else:
        x = f32c(x)
        M, dev = x.shape[0], x.device
    feature = torch.empty((M, 32), device=dev, dtype=torch.float32)
    sdf = torch.empty((M,), device=dev, dtype=torch.float32)
    alpha = torch.empty((M,), device=dev, dtype=torch.float32)
    sv = _lib.FieldFusedSaved()
    ximg = masks = None
    if train:
        ximg = torch.empty((int(_lib_().nrb_field_fused_image_bytes(M)),), device=dev, dtype=torch.uint8)
        masks = torch.empty((3, int(_lib_().nrb_field_saved_ld(M))), device=dev, dtype=torch.int32)
        sv.ximg, sv.masks, sv.ld = ptr(ximg), ptr(masks), masks.shape[1]
    m = _field_struct(weights, biases, beta, beta_min)
    _lib.call("nrb_field_fused_fwd", C.byref(m), C.byref(g) if gather else None, ptr(x3) if gather else None,
              ptr(std) if gather else None, None if gather else ptr(x), ptr(sh), int(samples_per_ray), M, ptr(feature),
              ptr(sdf), ptr(alpha), C.byref(sv), None if ag is None else C.byref(ag), None if asmp is None else C.byref(asmp),
              stream_ptr())
    ctx.actor_spec = None if actors is None else actors.spec
    ctx.samples_per_ray, ctx.beta_min, ctx.gather, ctx.spec = int(samples_per_ray), float(beta_min), gather, spec
    saved = None if not train else dict(
        table=table if gather else None, x3=x3 if gather else None, std=std if gather else None, ximg=ximg, masks=masks,
        sh=sh, beta=beta, sdf=sdf, alpha=alpha, weights=weights, biases=biases, actors=[] if actors is None else actors.to_save())
    return feature, sdf, alpha, saved


class _FieldFused(torch.autograd.Function):
    """NeuRADField on (table, sample means x3 [M,3], stds [M]) or on given hash features x [M,32]: one forward kernel,
    one backward kernel (+ the table scatter).  Outputs feature [M,32], sdf [M], alpha [M]."""

    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, table, x, x3, std, sh, samples_per_ray: int, beta_min: float, spec, actors, beta, *params):
        train = any(ctx.needs_input_grad)
        ctx.needs_x_grad = x is not None and ctx.needs_input_grad[1]
        feature, sdf, alpha, saved = _field_fused_forward(ctx, table, x, x3, std, sh, samples_per_ray, beta_min, spec, beta,
                                                          params, train, actors)
        if train:
            _save(ctx, **saved)
        return feature, sdf, alpha

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dfeature, dsdf, dalpha):
        s = _saved(ctx)
        dfeature = torch.zeros((s.sdf.shape[0], 32), device=s.sdf.device) if dfeature is None else f32c(dfeature)
        dsdf = None if dsdf is None else f32c(dsdf)
        dalpha = None if dalpha is None else f32c(dalpha)
        dx, grads = _field_fused_backward(ctx, s, dfeature, None, None, dsdf, dalpha)
        return (grads[0], dx, None, None, None, None, None, None, None, *grads[1:])


def field_fused(table: Optional[Tensor], x: Optional[Tensor], x3: Optional[Tensor], std: Optional[Tensor], sh: Tensor,
                samples_per_ray: int, spec: Optional[GridSpec], weights: Sequence[Tensor],
                biases: Sequence[Optional[Tensor]], beta: Tensor, beta_min: float,
                actors: Optional[ActorBatch] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """Fused field.  Gather mode: `table` + sample means `x3` [M,3] + `std` [M] (+ `actors`: the samples inside actor boxes
    read their actor's grid instead); otherwise hash features `x` [M,32]."""
    extra = [] if actors is None else list(actors.tables)
    return _FieldFused.apply(table, x, x3, std, sh, samples_per_ray, beta_min, spec, actors, beta, *weights, *biases, *extra)


class _FieldRender(torch.autograd.Function):
    """Fused field + alpha compositing tail of NeuRadarModel.get_nff_outputs (models/neuradar.py:500-517) on
    (table, sample means, stds, intervals): outputs weights [N,S] (after the sky fix-up), features [N,32], depth [N],
    accumulation [N].  Forward = the fused field kernel + the compositor; the per-sample [M,32] feature gradient is
    never formed in the backward: it is weights[m] * dfeatures[ray] and the field's backward kernel takes the factors."""

    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, table, x3, std, sh, iv: "SampleIntervals", beta_min: float, spec, trans_eps: float, actors, beta, *params):
        train = any(ctx.needs_input_grad)
        ctx.needs_x_grad = False
        S = iv.num_samples
        feature, sdf, alpha, saved = _field_fused_forward(ctx, table, None, x3, std, sh, S, beta_min, spec, beta, params, train,
                                                          actors)
        N, dev = alpha.shape[0] // S, alpha.device
        weights = torch.empty((N, S), device=dev, dtype=torch.float32)
        features = torch.empty((N, 32), device=dev, dtype=torch.float32)
        depth = torch.empty((N,), device=dev, dtype=torch.float32)
        acc = torch.empty((N,), device=dev, dtype=torch.float32)
        i = iv.struct()
        _lib.call("nrb_alpha_composite_fwd", ptr(alpha), ptr(feature), C.byref(i), N, 32, float(trans_eps), 1, ptr(weights),
                  ptr(features), ptr(depth), ptr(acc), None, stream_ptr())
        if train:  # (`weights` is an output: saved, not kept on ctx, so that output -> graph -> output is no cycle)
            _save(ctx, **saved, feature=feature, render_weights=weights)
            ctx.iv, ctx.trans_eps = iv, float(trans_eps)
        return weights, features, depth, acc

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dweights, dfeatures, ddepth, dacc):
        s = _saved(ctx)
        N, S = s.render_weights.shape
        dev = s.render_weights.device
        dweights = None if dweights is None else f32c(dweights)
        dfeatures = torch.zeros((N, 32), device=dev) if dfeatures is None else f32c(dfeatures)
        ddepth = None if ddepth is None else f32c(ddepth)
        dacc = None if dacc is None else f32c(dacc)
        dalphas = torch.empty((N * S,), device=dev, dtype=torch.float32)
        i = ctx.iv.struct()
        _lib.call("nrb_alpha_composite_bwd", ptr(s.alpha), ptr(s.feature), C.byref(i), N, 32, ctx.trans_eps, 1, ptr(dweights),
                  ptr(dfeatures), ptr(ddepth), ptr(dacc), ptr(dalphas), None, stream_ptr())
        _, grads = _field_fused_backward(ctx, s, None, dfeatures, s.render_weights.reshape(-1), None, dalphas)
        return (grads[0], None, None, None, None, None, None, None, None, *grads[1:])


def field_render(table: Tensor, x3: Tensor, std: Optional[Tensor], sh: Tensor, iv: SampleIntervals, spec: GridSpec,
                 weights: Sequence[Tensor], biases: Sequence[Optional[Tensor]], beta: Tensor, beta_min: float,
                 trans_eps: float = 0.0, actors: Optional[ActorBatch] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """(weights [N,S], features [N,32], depth [N], accumulation [N]) of the rays whose samples are (x3, std, iv)."""
    extra = [] if actors is None else list(actors.tables)
    return _FieldRender.apply(table, x3, std, sh, iv, beta_min, spec, trans_eps, actors, beta, *weights, *biases, *extra)


def sh16(directions: Tensor, normalize_to_unit_cube: bool = False) -> Tensor:
    """16 real SH basis values of directions [M,3]; no gradient (reference: torch.no_grad)."""
    d = f32c(directions.detach())
    out = torch.empty((d.shape[0], 16), device=d.device, dtype=torch.float32)
    _lib.call("nrb_sh16", ptr(d), ptr(out), d.shape[0], int(normalize_to_unit_cube), stream_ptr())
    return out


# ------------------------------------------------------------------------------------------------
# samplers (no gradients: bins are detached in the reference, ray_samplers.py:364)
# ------------------------------------------------------------------------------------------------
_LINSPACE_CACHE = {}


def _linspace(start: float, end: float, steps: int, device) -> Tensor:
    """torch.linspace evaluated on the CPU exactly like the reference does, cached per device."""
    key = (start, end, steps, str(device))
    t = _LINSPACE_CACHE.get(key)
    if t is None:
        t = torch.linspace(start, end, steps).to(device)
        _LINSPACE_CACHE[key] = t
    return t


def spaced_bins(rays: RayData, num_samples: int, jitter: Optional[Tensor], lam: float, scaling: float) -> Tuple[Tensor, Tensor]:
    """PowerSampler bins: spacing bins and euclidean bins, both [N, S+1].  jitter: [N,1]/[N] or [N,S+1] or None."""
    N = rays.num_rays
    dev = rays.origins.device
    base = _linspace(0.0, 1.0, num_samples + 1, dev)
    sbins = torch.empty((N, num_samples + 1), device=dev, dtype=torch.float32)
    ebins = torch.empty_like(sbins)
    per_bin = 0
    if jitter is not None:
        jitter = f32c(jitter)
        if jitter.numel() == N * (num_samples + 1) and num_samples > 0 and jitter.dim() == 2 and jitter.shape[1] == num_samples + 1:
            per_bin = 1
        elif jitter.numel() != N:
            raise ValueError("jitter must be [N,1] or [N,S+1]")
    r = rays.struct()
    _lib.call("nrb_spaced_bins", C.byref(r), Spacing(lam, scaling), ptr(base), ptr(jitter), per_bin, num_samples,
                                ptr(sbins), ptr(ebins), stream_ptr())
    return sbins, ebins


def pdf_sample(
    rays: RayData,
    weights: Tensor,
    sbins_in: Tensor,
    num_samples: int,
    jitter: Optional[Tensor],
    lam: float,
    scaling: float,
    histogram_padding: float = 0.01,
    eps: float = 1e-5,
    return_debug: bool = False,
):
    """PDFSampler (include_original=False): new spacing/euclidean bins [N, S_out+1] from weights [N,S_in]."""
    weights = f32c(weights.detach())
    sbins_in = f32c(sbins_in)
    N, S_in = weights.shape
    if sbins_in.shape != (N, S_in + 1):
        raise ValueError(f"existing bins have shape {tuple(sbins_in.shape)}, expected {(N, S_in + 1)}")
    dev = weights.device
    nb = num_samples + 1
    u_base = _linspace(0.0, 1.0 - (1.0 / nb), nb, dev)
    if jitter is not None:
        jitter = f32c(jitter.reshape(-1))
        if jitter.numel() != N:
            raise ValueError("jitter must hold one value per ray (single_jitter)")
    sb = torch.empty((N, nb), device=dev, dtype=torch.float32)
    eb = torch.empty_like(sb)
    inds = torch.empty((N, nb), device=dev, dtype=torch.int64) if return_debug else None
    cdf = torch.empty((N, S_in + 1), device=dev, dtype=torch.float32) if return_debug else None
    r = rays.struct()
    _lib.call("nrb_pdf_sample", C.byref(r), Spacing(lam, scaling), ptr(weights), ptr(sbins_in), S_in, ptr(u_base),
                               ptr(jitter), num_samples, float(histogram_padding), float(eps), ptr(sb), ptr(eb),
                               ptr(inds), ptr(cdf), stream_ptr())
    if return_debug:
        return sb, eb, inds, cdf
    return sb, eb


# ------------------------------------------------------------------------------------------------
# compositing
# ------------------------------------------------------------------------------------------------
class _DensityWeights(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, densities, iv: SampleIntervals):
        dens = f32c(densities)
        N, S = dens.shape
        w = torch.empty_like(dens)
        i = iv.struct()
        _lib.call("nrb_density_weights_fwd", ptr(dens), C.byref(i), N, ptr(w), stream_ptr())
        ctx.save_for_backward(dens)
        ctx.iv = iv
        return w

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dw):
        (dens,) = ctx.saved_tensors
        dw = f32c(dw)
        dd = torch.empty_like(dens)
        i = ctx.iv.struct()
        _lib.call("nrb_density_weights_bwd", ptr(dens), C.byref(i), ptr(dw), dens.shape[0], ptr(dd), stream_ptr())
        return dd, None


def density_weights(densities: Tensor, iv: SampleIntervals) -> Tensor:
    """RaySamples.get_weights: densities [N,S] -> weights [N,S]."""
    return _DensityWeights.apply(densities, iv)


class _AlphaComposite(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, alphas, feats, iv: SampleIntervals, trans_eps: float, sky: bool):
        alphas = f32c(alphas)
        N, S = alphas.shape
        dev = alphas.device
        feats = None if feats is None else f32c(feats)
        Cn = 0 if feats is None else feats.shape[-1]
        weights = torch.empty_like(alphas)
        trans = torch.empty_like(alphas)
        features = torch.empty((N, Cn), device=dev, dtype=torch.float32) if feats is not None else None
        depth = torch.empty((N,), device=dev, dtype=torch.float32)
        acc = torch.empty((N,), device=dev, dtype=torch.float32)
        i = iv.struct()
        _lib.call("nrb_alpha_composite_fwd", ptr(alphas), ptr(feats), C.byref(i), N, Cn, float(trans_eps), int(sky),
                                            ptr(weights), ptr(features), ptr(depth), ptr(acc), ptr(trans),
                                            stream_ptr())
        ctx.save_for_backward(alphas, feats)
        ctx.iv, ctx.eps, ctx.sky, ctx.C = iv, float(trans_eps), int(sky), Cn
        if features is None:
            features = torch.empty((N, 0), device=dev, dtype=torch.float32)
        ctx.mark_non_differentiable(trans)
        return weights, features, depth, acc, trans

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dweights, dfeatures, ddepth, dacc, _dtrans):
        alphas, feats = ctx.saved_tensors
        N, S = alphas.shape
        dalphas = torch.empty_like(alphas)
        need_df = feats is not None and ctx.needs_input_grad[1]
        dfeats = torch.empty_like(feats) if need_df else None
        dweights = None if dweights is None else f32c(dweights)
        dfeatures = None if (dfeatures is None or feats is None) else f32c(dfeatures)
        ddepth = None if ddepth is None else f32c(ddepth)
        dacc = None if dacc is None else f32c(dacc)
        i = ctx.iv.struct()
        _lib.call("nrb_alpha_composite_bwd", ptr(alphas), ptr(feats), C.byref(i), N, ctx.C, ctx.eps, ctx.sky,
                                            ptr(dweights), ptr(dfeatures), ptr(ddepth), ptr(dacc), ptr(dalphas),
                                            ptr(dfeats), stream_ptr())
        return dalphas, dfeats, None, None, None


def alpha_composite(
    alphas: Tensor, feats: Optional[Tensor], iv: SampleIntervals, trans_eps: float = 0.0, sky_sample: bool = False
) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """alphas [N,S], feats [N,S,C] -> (weights [N,S], features [N,C], depth [N], accumulation [N])."""
    return _AlphaComposite.apply(alphas, feats, iv, trans_eps, sky_sample)[:4]


def alpha_weights(alphas: Tensor, trans_eps: float = 0.0) -> Tuple[Tensor, Tensor]:
    """(weights [N,S], transmittance [N,S]) with T_i = prod_{j<i} (1 - alpha_j + eps)."""
    zeros = torch.zeros((alphas.shape[0], alphas.shape[1] + 1), device=alphas.device, dtype=torch.float32)
    out = _AlphaComposite.apply(alphas, None, SampleIntervals.from_bins(zeros), trans_eps, False)
    return out[0], out[4]


class _Accumulate(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, weights, values):
        w = f32c(weights)
        N, S = w.shape
        v = None if values is None else f32c(values)
        Cn = 0 if v is None else v.shape[-1]
        out = torch.empty((N, max(Cn, 1)), device=w.device, dtype=torch.float32)
        _lib.call("nrb_accumulate_fwd", ptr(w), ptr(v), N, S, Cn, ptr(out), stream_ptr())
        ctx.save_for_backward(w, v)
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        w, v = ctx.saved_tensors
        N, S = w.shape
        dout = f32c(dout)
        dw = torch.empty_like(w) if ctx.needs_input_grad[0] else None
        dv = torch.empty_like(v) if (v is not None and ctx.needs_input_grad[1]) else None
        Cn = 0 if v is None else v.shape[-1]
        _lib.call("nrb_accumulate_bwd", ptr(w), ptr(v), ptr(dout), N, S, Cn, ptr(dw), ptr(dv), stream_ptr())
        return dw, dv


class _WeightedDepth(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, weights, iv: SampleIntervals):
        w = f32c(weights)
        N = w.shape[0]
        out = torch.empty((N, 1), device=w.device, dtype=torch.float32)
        i = iv.struct()
        _lib.call("nrb_weighted_depth_fwd", ptr(w), C.byref(i), N, ptr(out), stream_ptr())
        ctx.iv, ctx.shape = iv, w.shape
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dout):
        dout = f32c(dout)
        dw = torch.empty(ctx.shape, device=dout.device, dtype=torch.float32)
        i = ctx.iv.struct()
        _lib.call("nrb_weighted_depth_bwd", C.byref(i), ptr(dout), ctx.shape[0], ptr(dw), stream_ptr())
        return dw, None


def weighted_depth(weights: Tensor, iv: SampleIntervals) -> Tensor:
    """render_depth_simple (models/neurad.py:721-728): sum_s weights[N,S] (start + end) / 2 -> [N,1], midpoints in-kernel."""
    return _WeightedDepth.apply(weights, iv)


def accumulate(weights: Tensor, values: Optional[Tensor]) -> Tensor:
    """sum_s weights[N,S] * values[N,S,C] -> [N,C]  (values None -> [N,1])."""
    return _Accumulate.apply(weights, values)


# ------------------------------------------------------------------------------------------------
# per-ray tail: point heads, lidar carving
# ------------------------------------------------------------------------------------------------
def _u8(t: Optional[Tensor]) -> Optional[Tensor]:
    return None if t is None else t.reshape(-1).to(torch.uint8).contiguous()


class _PointHeads(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, depth, origins, directions, is_radar, spher, world2sensor):
        ctx.depth_shape = depth.shape
        depth, origins, directions = f32c(depth.reshape(-1)), f32c(origins), f32c(directions)
        spher = None if spher is None else f32c(spher.reshape(-1, 2))
        w2s = None if world2sensor is None else f32c(world2sensor[..., :3, :4].reshape(3, 4))
        N = depth.shape[0]
        pts = torch.empty((N, 3), device=depth.device, dtype=torch.float32)
        _lib.call("nrb_point_heads_fwd", ptr(origins), ptr(directions), ptr(depth), ptr(is_radar), ptr(spher), ptr(w2s), ptr(pts), N,
                  stream_ptr())
        ctx.save_for_backward(directions, is_radar, spher, w2s)
        return pts

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dpts):
        directions, is_radar, spher, w2s = ctx.saved_tensors
        dpts = f32c(dpts)
        dd = torch.empty((dpts.shape[0],), device=dpts.device, dtype=torch.float32)
        _lib.call("nrb_point_heads_bwd", ptr(directions), ptr(is_radar), ptr(spher), ptr(w2s), ptr(dpts), ptr(dd), dpts.shape[0],
                  stream_ptr())
        return dd.view(ctx.depth_shape), None, None, None, None, None


def point_heads(depth: Tensor, origins: Tensor, directions: Tensor, is_radar: Optional[Tensor] = None,
                directions_spher: Optional[Tensor] = None, world2sensor: Optional[Tensor] = None) -> Tensor:
    """Rendered depth [N] / [N,1] -> points [N,3]: lidar / camera rays o + d * depth (optionally in the sensor frame given by
    world2sensor [3,4] or [4,4]), radar rays depth * unit(phi, theta) from directions_spher [N,2].  Differentiable in depth."""
    return _PointHeads.apply(depth, origins, directions, _u8(is_radar), directions_spher, world2sensor)


class _CarvingLoss(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, weights, iv: SampleIntervals, is_lidar, dir_norm, did_return, eps: float, max_dist: float):
        w = f32c(weights)
        N, S = w.shape
        out = torch.empty_like(w)
        i = iv.struct()
        _lib.call("nrb_lidar_carving", C.byref(i), N, ptr(is_lidar), ptr(dir_norm), ptr(did_return), float(eps), float(max_dist),
                  ptr(w), None, None, ptr(out), stream_ptr())
        ctx.save_for_backward(w, is_lidar, dir_norm, did_return)
        ctx.iv, ctx.eps, ctx.max_dist = iv, float(eps), float(max_dist)
        return out.sum()

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dloss):
        w, is_lidar, dir_norm, did_return = ctx.saved_tensors
        dw = torch.empty_like(w)
        i = ctx.iv.struct()
        dl = f32c(dloss.reshape(1))
        _lib.call("nrb_lidar_carving", C.byref(i), w.shape[0], ptr(is_lidar), ptr(dir_norm), ptr(did_return), ctx.eps, ctx.max_dist,
                  ptr(w), ptr(dl), None, ptr(dw), stream_ptr())
        return dw, None, None, None, None, None, None


def is_close_to_lidar(iv: SampleIntervals, is_lidar: Tensor, directions_norm: Tensor, did_return: Optional[Tensor] = None,
                      carving_epsilon: float = 0.1, non_return_lidar_distance: float = 150.0) -> Tensor:
    """NeuRadarModel._compute_is_close_to_lidar for the samples `iv` of N rays: bool [N,S]."""
    N, S = iv.starts.shape[0], iv.num_samples
    out = torch.empty((N, S), device=iv.starts.device, dtype=torch.uint8)
    i = iv.struct()
    lid, dn, ret = _u8(is_lidar), f32c(directions_norm.reshape(-1)), _u8(did_return)  # kept alive across the launch
    _lib.call("nrb_lidar_carving", C.byref(i), N, ptr(lid), ptr(dn), ptr(ret), float(carving_epsilon),
              float(non_return_lidar_distance), None, None, ptr(out), None, stream_ptr())
    return out.bool()


def carving_loss(weights: Tensor, iv: SampleIntervals, is_lidar: Tensor, directions_norm: Tensor,
                 did_return: Optional[Tensor] = None, carving_epsilon: float = 0.1,
                 non_return_lidar_distance: float = 150.0) -> Tensor:
    """sum((weights * (is_lidar & ~is_close_to_lidar))^2) over weights [N,S] (models/neuradar.py:527-531), one kernel each way."""
    return _CarvingLoss.apply(weights, iv, _u8(is_lidar), f32c(directions_norm.reshape(-1)), _u8(did_return), carving_epsilon,
                              non_return_lidar_distance)


# ------------------------------------------------------------------------------------------------
# fused proposal round
# ------------------------------------------------------------------------------------------------
class _ProposalRound(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, table, decoder_w, rays: RayData, iv: SampleIntervals, spec: GridSpec, scale: float, actors, *actor_tables):
        ctx.sinks = _GradSinks([table, decoder_w, *actor_tables])
        table = f32c(table)
        dec = f32c(decoder_w.reshape(-1))
        N, S = rays.num_rays, iv.num_samples
        dev = table.device
        density = torch.empty((N, S), device=dev, dtype=torch.float32)
        weights = torch.empty_like(density)
        train = any(ctx.needs_input_grad[:2]) or any(ctx.needs_input_grad[7:])
        feats = torch.empty((N, S, spec.out_dim), device=dev, dtype=torch.float32) if train else None
        pre = torch.empty((N, S), device=dev, dtype=torch.float32) if train else None
        g, r, i = spec.struct(table), rays.struct(), iv.struct()
        ag = asmp = None
        if actors is not None:
            actors = actors.with_tables([f32c(t) for t in actor_tables])
            ag, asmp = actors.grids_struct(), actors.samples_struct()
        _lib.call("nrb_proposal_fwd", C.byref(r), C.byref(g), ptr(dec), float(scale), C.byref(i), ptr(density),
                  ptr(weights), ptr(feats), ptr(pre), None if ag is None else C.byref(ag),
                  None if asmp is None else C.byref(asmp), stream_ptr())
        _save(ctx, table=table, dec=dec, feats=feats, pre=pre, actors=[] if actors is None else actors.to_save())
        ctx.rays, ctx.iv, ctx.spec, ctx.scale = rays, iv, spec, float(scale)
        ctx.actor_spec = None if actors is None else actors.spec
        return density, weights

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, ddensity, dweights):
        s, sinks = _saved(ctx), ctx.sinks
        dtable, ddec = sinks.dest(0), sinks.dest(1)  # (ddec has the decoder's shape; the kernel reads it flat)
        ddensity = None if ddensity is None else f32c(ddensity)
        dweights = None if dweights is None else f32c(dweights)
        g, r, i = ctx.spec.struct(s.table), ctx.rays.struct(), ctx.iv.struct()
        ws, ws_bytes = _scatter_workspace(g, ctx.rays.num_rays * ctx.iv.num_samples, s.table.device)
        ag = asmp = dptrs = None
        dactor: List[Tensor] = []
        if ctx.actor_spec is not None:
            actors = ActorBatch.from_saved(s.actors, ctx.actor_spec)
            ag, asmp = actors.grids_struct(), actors.samples_struct()
            dactor = [sinks.dest(i) for i in range(2, len(sinks.params))]
            dptrs = (C.c_void_p * len(dactor))(*[d.data_ptr() for d in dactor])
        _lib.call("nrb_proposal_bwd", C.byref(r), C.byref(g), ptr(s.dec), ctx.scale, C.byref(i), ptr(s.feats), ptr(s.pre),
                  ptr(dweights), ptr(ddensity), ptr(dtable), ptr(ddec), ws, ws_bytes, None if ag is None else C.byref(ag),
                  None if asmp is None else C.byref(asmp), dptrs, stream_ptr())
        grads = sinks.written([dtable, ddec, *dactor])
        return (grads[0], grads[1], None, None, None, None, None, *grads[2:])


def proposal_round(
    table: Tensor, decoder_w: Tensor, rays: RayData, iv: SampleIntervals, spec: GridSpec, static_scale: float,
    actors: Optional[ActorBatch] = None,
) -> Tuple[Tensor, Tensor]:
    """One fused proposal round: (density [N,S], weights [N,S]).  `actors` (from `actor_assign`): the samples inside actor
    boxes read their actor's 4-level grid instead."""
    extra = [] if actors is None else list(actors.tables)
    return _ProposalRound.apply(table, decoder_w, rays, iv, spec, static_scale, actors, *extra)
