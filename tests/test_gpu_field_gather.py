"""The gather mode of the fused field kernels (csrc/field_fused.cu, nrb_hash_bwd_image, nrb_actor_scatter) and the
anti-alias level weights of the hash-grid kernels (csrc/hash_grid.cu) against a float64 reference of the same operation.

* The reference locates cells exactly like the kernels (fp32 `x * scal`, floor / ceil hashed by the oracle, which is
  bit-exact with them: test_hash_indices_bit_exact) and does everything after that in float64 on the GPU: trilinear
  interpolation, level weights 1 / max(2 scal std, 1), both MLPs, the SH concatenation, the SDF head, compositing.
  It calls no neuradar_b200 kernel.
* Table gradients are compared level by level (`per_level`): a bar over the whole table is set by its largest level and
  would not see a fine or down-weighted level that is wrong or missing.
* The multi-tile sample counts (`tiles_for`) make every group of both persistent kernels run several tiles, so the
  steady state of their pipelines (mbarrier parities, TMEM reuse, the next tile's prefetch) is what is compared.

Error model of the bars: the forward evaluates every product as 3xTF32 with fp32 accumulation (~1e-7 relative), the
backward as bf16 hi / mid operand pairs (16 mantissa bits each, ~2^-17 per product) with fp32 accumulation, and the
table scatters add in fp32 in any order.
"""
import math

import pytest
import torch
import torch.nn.functional as TF

from oracle import neuradar_oracle as O
from tests.parity_utils import outside_bar, rel_err, scaled_pixel_area, synthetic_rays

pytestmark = pytest.mark.gpu

DEV = "cuda"
BETA_MIN = 1e-4
SKY = 20000.0
KINK = 1e-5  # |float64 pre-activation| below which a ReLU may switch sides between two fp32 evaluation orders
# levels, features, log2 rows per level, base and max resolution (the field grids of BASELINE configs 2 and 4)
GRIDS = {"L16F2": (16, 2, 16, 16, 1024), "L8F4": (8, 4, 16, 32, 8192)}


@pytest.fixture(scope="module")
def nb():
    import neuradar_b200

    assert torch.cuda.is_available()
    return neuradar_b200


# ------------------------------------------------------------------------------------------------ float64 reference
def ref_cells(x, scal, log2T):
    """Rows [M, L, 8] (corner order of O.hash_encode) and in-cell offsets [M, L, 3] in float64, located as the kernels do:
    fp32 x * scal (torch's fp32 multiply is correctly rounded, like __fmul_rn), floor / ceil hashed by the oracle.
    x * scal - floor(x * scal) is exact in fp32, so the float64 offsets are the kernel's offsets."""
    idx, off = O.hash_corner_indices(x.detach().float().cpu(), scal.float().cpu(), log2T)
    return idx.to(DEV), off.to(DEV, torch.float64)


def ref_encode(x, std, table, scal, log2T, x_leaf=None):
    """Anti-aliased hash encoding [M, L*F] in float64 of the fp32 points x and stds std (or None: weights 1) on the float64
    table.  With x_leaf (a float64 copy of x that requires grad) the result is differentiable in the point: the offsets keep
    their exact fp32 values and get the derivative scal."""
    L = scal.numel()
    idx, o = ref_cells(x, scal, log2T)
    s64 = scal.to(DEV, torch.float64)
    if x_leaf is not None:
        o = o + (x_leaf - x_leaf.detach())[:, None, :] * s64[None, :, None]
    f = [table[idx[..., k]] for k in range(8)]  # [M, L, F] each
    ox, oy, oz = o[..., 0:1], o[..., 1:2], o[..., 2:3]
    f03 = f[0] * ox + f[3] * (1 - ox)
    f12 = f[1] * ox + f[2] * (1 - ox)
    f56 = f[5] * ox + f[6] * (1 - ox)
    f47 = f[4] * ox + f[7] * (1 - ox)
    out = (f03 * oy + f12 * (1 - oy)) * oz + (f47 * oy + f56 * (1 - oy)) * (1 - oz)
    if std is not None:
        out = out * (1.0 / (2.0 * s64[None, :] * std.to(DEV, torch.float64)[:, None]).clamp_min(1.0))[..., None]
    return out.reshape(x.shape[0], L * table.shape[1])


def ref_sh(dirs):
    """SH basis of unit directions, the convention of sh16_of_direction (actor_grid.cuh) and SHEncoding: sh16((d + 1) / 2).
    O.sh16 evaluates in float64 but stores fp32 (its output buffer is float32): the basis values carry a rounding of
    <= 6e-8 relative, as an input would; the kernel rounds to fp32 too."""
    return O.sh16((dirs.detach().double().cpu() + 1.0) / 2.0).to(DEV, torch.float64)


def ref_field(feats, sh_rows, w, b, beta):
    """NeuRADField after the encoding (O.field_forward): feature [M,32], sdf [M], alpha [M]."""
    geo = O.mlp(feats, w[:2], b[:2])
    sdf, emb = geo[:, 0], geo[:, 1:]
    feature = emb + O.mlp(torch.cat([emb, sh_rows], -1), w[2:], b[2:])
    return feature, sdf, torch.sigmoid(-sdf * (beta.abs() + BETA_MIN))


def near_kink(feats, sh_rows, w, b):
    """Samples with a hidden unit whose float64 pre-activation is within KINK of zero (test_field_fused_backward_rows)."""
    with torch.no_grad():
        p0 = O.mlp(feats, w[:1], b[:1])
        inp = torch.cat([O.mlp(feats, w[:2], b[:2])[:, 1:], sh_rows], -1)
        p2, p3 = O.mlp(inp, w[2:3], b[2:3]), O.mlp(inp, w[2:4], b[2:4])
        return torch.cat([p0, p2, p3], -1).abs().min(dim=-1).values < KINK


def per_level(got, want, L, T, F, rel=1e-3):
    """Per level of a table gradient [L * 2^T, F]: (max |got - want| over the level / the level's own max |want|, number of
    elements outside the element-wise bar |got - want| <= rel |want| + rel rms(level))."""
    g, w = got.detach().double().reshape(L, 1 << T, F), want.detach().double().reshape(L, 1 << T, F)
    out = []
    for l in range(L):
        err, top = float((g[l] - w[l]).abs().max()), float(w[l].abs().max())
        out.append((err / top if top > 0 else (0.0 if err == 0 else math.inf), outside_bar(g[l], w[l], rel)))
    return out


def check_table(what, got, want, L, T, F, tol, rel=1e-3):
    levels = per_level(got, want, L, T, F, rel)
    worst = max(range(L), key=lambda l: levels[l][0])
    print(f"[measured] {what}: worst per-level max-rel {levels[worst][0]:.3e} at level {worst}")
    assert float(want.detach().reshape(L, -1).abs().amax(dim=1).min()) > 0, f"{what}: a level received no gradient"
    for l, (e, n) in enumerate(levels):
        assert e <= tol and n == 0, (what, l, e, n)


def check(what, got, want, tol, bar=True):
    e = rel_err(got, want)
    print(f"[measured] {what}: max-rel {e:.3e}")
    assert e <= tol, (what, e)
    if bar:
        assert outside_bar(got, want) == 0, what


def tiles_for(min_tiles_per_group, S=1):
    """A sample count M, a multiple of S, at which every group of the fused backward runs at least `min_tiles_per_group`
    tiles (3: both groups go through mbarrier parities 0 -> 1 -> 0) and every group of the fused forward at least 2; the
    last tile of 128 samples is partial unless S is a multiple of 128.  Returns (M, backward tiles per CTA)."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count

    def counts(tiles):
        # nrb_field_fused_fwd: `nblk = min((tiles + kFGroups - 1) / kFGroups, sm_count())`, kFGroups = 3; group g of CTA b
        # runs tiles b + g * gridDim.x + k * 3 * gridDim.x (the tile loop of field_fused_fwd_kernel)
        fb = min((tiles + 2) // 3, sm)
        fwd = [len(range(b + g * fb, tiles, 3 * fb)) for b in range(fb) for g in range(3)]
        # nrb_field_fused_bwd: `nblk = min((tiles + 1) / 2, sm_count())`; CTA b owns `mine` tiles b + k * gridDim.x and
        # group g takes k = g, g + 2, ... (field_fused_bwd_kernel: `mine`, the workers' loop over k)
        bb = min((tiles + 1) // 2, sm)
        mine = [len(range(b, tiles, bb)) for b in range(bb)]
        return fwd, mine, [(c + 1) // 2 for c in mine] + [c // 2 for c in mine]

    tiles = 1
    while True:
        fwd, _, bwd = counts(tiles)
        if min(fwd) >= 2 and min(bwd) >= min_tiles_per_group:
            break
        tiles += 1
    M = -(-((tiles - 1) * 128 + 1) // S) * S
    while M % 128 == 0 and S % 128 != 0:
        M += S
    fwd, mine, bwd = counts(-(-M // 128))
    assert M % 128 != 0 or S % 128 == 0
    assert min(fwd) >= 2 and min(bwd) >= min_tiles_per_group and min(mine) >= 2 * min_tiles_per_group - 1, (fwd, mine)
    return M, mine


# ------------------------------------------------------------------------------------------------ inputs
def make_grid(name, seed, log2T=None):
    from neuradar_b200.functional import GridSpec

    L, F, T, lo, hi = GRIDS[name]
    T = log2T or T
    scal = O.level_scalings(L, lo, hi)
    g = torch.Generator().manual_seed(seed)
    table = torch.rand((L << T, F), generator=g) * 2 - 1
    return GridSpec(L, F, T, tuple(float(s) for s in scal)), scal, table.to(DEV)


def synthetic_std(M, scal, g):
    """Log-uniform over [1e-5, 1e-1], where the cut-over 2 scal std = 1 of every level of these grids lies; 5 % zeros, and
    5 % exactly 1 / (2 scal) of a power-of-two level (2 scal std == 1 in fp32 and float64: the clamp's edge)."""
    std = torch.empty(M).uniform_(math.log(1e-5), math.log(1e-1), generator=g).exp()
    k = torch.randint(0, 20, (M,), generator=g)
    std[k == 0] = 0.0
    p2 = [float(s) for s in scal if int(s) & (int(s) - 1) == 0]
    assert p2
    edge = k == 1
    std[edge] = torch.tensor([0.5 / s for s in p2])[torch.randint(0, len(p2), (int(edge.sum()),), generator=g)]
    return std


def synthetic_points(N, S, g):
    """Ray-ordered clustered points [N*S, 3]: each ray walks a short segment from a random anchor, and every 37th sample
    starts a run of 4 identical points (the run merging adds their lanes, whose stds differ)."""
    anchor = torch.rand((N, 1, 3), generator=g) * 0.8 + 0.1
    d = torch.randn((N, 1, 3), generator=g)
    d = d / d.norm(dim=-1, keepdim=True)
    t = torch.sort(torch.rand((N, S, 1), generator=g), dim=1).values * torch.rand((N, 1, 1), generator=g).pow(2) * 0.05
    x = (anchor + d * t).reshape(-1, 3).clamp(0, 1)
    head = torch.arange(0, x.shape[0] - 4, 37)
    for j in range(1, 4):
        x[head + j] = x[head]
    return x


def make_samples(N, S, scal, seed):
    """N rays of S samples: even rays are camera / lidar / radar rays through Fn.frustum_gaussians (power-spaced bins with
    the sky sample of nff_forward), odd rays get synthetic points and stds.  Returns x3 [N*S,3], std [N*S], sh [N,16] (fp32,
    on the device) and the bins [N,S+1]."""
    from neuradar_b200 import functional as Fn

    g = torch.Generator().manual_seed(seed)
    rays = synthetic_rays(N, seed=seed)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(SKY), S, torch.rand((N, S + 1), generator=g))
    last = eb[:, -1:]
    eb = torch.cat([eb[:, :-1], last + (SKY - last)], dim=-1).contiguous()  # the sky sample (neuradar.py:578-582)
    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), scaled_pixel_area(rays).to(DEV))
    x3, std = Fn.frustum_gaussians(rd, Fn.SampleIntervals.from_bins(eb.to(DEV)), 100.0)
    x3, std = x3.cpu().view(N, S, 3), std.cpu().view(N, S)
    odd = torch.arange(N) % 2 == 1
    n_odd = int(odd.sum())
    if n_odd:
        x3[odd] = synthetic_points(n_odd, S, g).view(n_odd, S, 3)
        std[odd] = synthetic_std(n_odd * S, scal, g).view(n_odd, S)
    d = rays["directions"] / rays["directions"].norm(dim=-1, keepdim=True)
    sh = O.sh16((d + 1.0) / 2.0)
    return x3.reshape(-1, 3).to(DEV), std.reshape(-1).to(DEV), sh.to(DEV), eb.to(DEV)


def mlp_params(seed, beta=-8.0):
    """The field's five layers (default init) and a negative beta (d|beta| / d beta = -1)."""
    torch.manual_seed(seed)
    layers = [torch.nn.Linear(i, o) for i, o in [(32, 32), (32, 33), (48, 32), (32, 32), (32, 32)]]
    return [l.weight.detach().clone() for l in layers], [l.bias.detach().clone() for l in layers], torch.tensor([beta])


def leaves(ts, dtype):
    return [t.detach().to(DEV, dtype).clone().requires_grad_(True) for t in ts]


def sample_kind(kind, S):
    """'ray': one ray; 'tile': one partial tile; 'multi': several tiles per group of both persistent kernels."""
    return {"ray": S, "tile": 77, "multi": tiles_for(3)[0]}[kind]


# ------------------------------------------------------------------------------------------------ 1. hash_encode + std
@pytest.mark.parametrize(
    "L,F,M,log2T,need_dx",
    # hash_fwd_rows_kernel + the run-merging backward (L*F a power of two, M >= 32)
    [(16, 2, 4000, 12, False), (8, 4, 4000, 12, False), (4, 1, 4000, 12, False),
     # the level-major forward and backward: M < 32, L*F not a power of two; hash_bwd_kernel's dx branch
     (16, 2, 31, 12, False), (6, 1, 3000, 12, False), (12, 2, 3000, 12, True),
     # T = 2^19 and M >= 2^16: the coarse levels scatter into dense-lattice replicas
     (16, 2, 70000, 19, False), (6, 1, 65600, 19, False), (12, 2, 65600, 19, True)],
)
def test_hash_encode_level_weights(nb, L, F, M, log2T, need_dx):
    """nrb_hash_fwd / nrb_hash_bwd with per-sample stds against float64, level by level."""
    import ctypes as C

    from neuradar_b200 import _lib
    from neuradar_b200 import functional as Fn
    from neuradar_b200.functional import GridSpec

    g = torch.Generator().manual_seed(M + 7 * L)
    scal = O.level_scalings(L, 16, 1024)
    spec = GridSpec(L, F, log2T, tuple(float(s) for s in scal))
    x = synthetic_points(-(-M // 40), 40, g)[:M].contiguous()
    std = synthetic_std(M, scal, g)
    table = torch.rand((L << log2T, F), generator=g) * 2 - 1
    dy = torch.randn((M, L * F), generator=g)
    if log2T == 19:
        assert _lib.load().nrb_hash_bwd_workspace_bytes(C.byref(spec.struct(table.to(DEV))), M) > 0
    t_ref = table.to(DEV, torch.float64).requires_grad_(True)
    x_ref = x.to(DEV, torch.float64).requires_grad_(True) if need_dx else None
    y_ref = ref_encode(x.to(DEV), std, t_ref, scal, log2T, x_ref)
    (y_ref * dy.to(DEV, torch.float64)).sum().backward()
    t_dev = table.to(DEV).requires_grad_(True)
    x_dev = x.to(DEV).requires_grad_(need_dx)
    y = Fn.hash_encode(x_dev, t_dev, spec, std.to(DEV))
    # forward: seven fp32 lerps and the weight, a few ulp of the level's largest feature
    yl, rl = y.detach().double().view(M, L, F), y_ref.detach().view(M, L, F)
    for l in range(L):
        e = float((yl[:, l] - rl[:, l]).abs().max() / rl[:, l].abs().max())
        assert e <= 1e-6, ("forward", l, e)
    (y * dy.to(DEV)).sum().backward()
    # table: a few ulp per contribution, fp32 sums in any order; 1e-5 element-wise is >= 100x that at these sizes
    check_table(f"hash L{L}F{F} M{M} T{log2T} dtable", t_dev.grad, t_ref.grad, L, log2T, F, 1e-5, rel=1e-5)
    if need_dx:
        check("hash dx", x_dev.grad, x_ref.grad, 1e-5, bar=False)


# ------------------------------------------------------------------------------------------------ 2. fused forward
@pytest.mark.parametrize("with_std", [True, False])
@pytest.mark.parametrize("S", [33, 48, 128])
@pytest.mark.parametrize("kind", ["ray", "tile", "multi"])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_gather_forward(nb, grid, kind, S, with_std):
    from neuradar_b200 import functional as Fn

    spec, scal, table = make_grid(grid, seed=S)
    w, b, beta = mlp_params(seed=3)
    M = sample_kind(kind, S)
    N = -(-M // S)
    x3, std, sh, _ = make_samples(N, S, scal, seed=M + S)
    x3, std = x3[:M].contiguous(), std[:M].contiguous() if with_std else None
    # eval forward: no input requires grad, so nothing is saved (`train` is any(ctx.needs_input_grad), which follows the
    # inputs' requires_grad even under no_grad); no grad_fn on the outputs is the proof
    we, be, betae = [t.to(DEV) for t in w], [t.to(DEV) for t in b], beta.to(DEV)
    f, s, a = Fn.field_fused(table, None, x3, std, sh, S, spec, we, be, betae, BETA_MIN)
    assert f.grad_fn is None and s.grad_fn is None and a.grad_fn is None
    with torch.no_grad():
        w64, b64, (beta64,) = leaves(w, torch.float64), leaves(b, torch.float64), leaves([beta], torch.float64)
        feats = ref_encode(x3, std, table.double(), scal, spec.log2_hashmap_size)
        rf, rs, ra = ref_field(feats, sh.double()[torch.arange(M, device=DEV) // S], w64, b64, beta64)
    for what, got, want in (("feature", f, rf), ("sdf", s, rs), ("alpha", a, ra)):
        check(f"forward {grid} {kind} S{S} std={with_std} {what}", got, want, 1e-5)
    if kind != "multi":
        return
    # the training forward (it writes the saved image and ReLU masks) computes the same bits as the eval forward
    wk, bk, (betak,) = leaves(w, torch.float32), leaves(b, torch.float32), leaves([beta], torch.float32)
    ft, st, at = Fn.field_fused(table.clone().requires_grad_(True), None, x3, std, sh, S, spec, wk, bk, betak, BETA_MIN)
    assert ft.grad_fn is not None
    assert torch.equal(ft.detach(), f) and torch.equal(st.detach(), s) and torch.equal(at.detach(), a)
    # the first M0 samples on their own (eval forward): another tile -> CTA -> group mapping, the same bits
    M0 = 40 * 128 + 45
    f0, s0, a0 = Fn.field_fused(table, None, x3[:M0].contiguous(), None if std is None else std[:M0].contiguous(),
                                sh[: -(-M0 // S)].contiguous(), S, spec, we, be, betae, BETA_MIN)
    assert torch.equal(f0, f[:M0]) and torch.equal(s0, s[:M0]) and torch.equal(a0, a[:M0])


# ------------------------------------------------------------------------------------------------ 3. fused backward
@pytest.mark.parametrize("S,kind", [(33, "multi"), (128, "multi"), (33, "tile"), (48, "tile")])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_gather_backward_dfeature(nb, grid, S, kind):
    """Field backward on a [M,32] feature gradient + sdf and alpha gradients, then nrb_hash_bwd_image."""
    from neuradar_b200 import functional as Fn

    spec, scal, table = make_grid(grid, seed=11 + S)
    L, F, T = spec.num_levels, spec.features_per_level, spec.log2_hashmap_size
    w, b, beta = mlp_params(seed=5)
    M = sample_kind(kind, S)
    if kind == "multi":
        mine = tiles_for(3)[1]  # (from the mirrored launcher formulas, not counted in the kernel)
        print(f"[tiles_for] backward tiles per CTA: {min(mine)}..{max(mine)}")
    N = -(-M // S)
    x3, std, sh, _ = make_samples(N, S, scal, seed=2 * M + S)
    x3, std = x3[:M].contiguous(), std[:M].contiguous()
    sh_rows = sh.double()[torch.arange(M, device=DEV) // S]
    g = torch.Generator(device=DEV).manual_seed(S)
    gf, gs, ga = (torch.randn((M, 32), device=DEV, generator=g), torch.randn((M,), device=DEV, generator=g),
                  torch.randn((M,), device=DEV, generator=g))
    w64, b64, (beta64,) = leaves(w, torch.float64), leaves(b, torch.float64), leaves([beta], torch.float64)
    t64 = table.double().requires_grad_(True)
    feats = ref_encode(x3, std, t64, scal, T)
    kink = near_kink(feats, sh_rows, w64, b64)
    gf[kink], gs[kink], ga[kink] = 0, 0, 0
    rf, rs, ra = ref_field(feats, sh_rows, w64, b64, beta64)
    ((rf * gf.double()).sum() + (rs * gs.double()).sum() + (ra * ga.double()).sum()).backward()
    tk = table.clone().requires_grad_(True)
    wk, bk, (betak,) = leaves(w, torch.float32), leaves(b, torch.float32), leaves([beta], torch.float32)
    f, s, a = Fn.field_fused(tk, None, x3, std, sh, S, spec, wk, bk, betak, BETA_MIN)
    check(f"backward {grid} {kind} S{S} feature", f, rf, 1e-5)
    ((f * gf).sum() + (s * gs).sum() + (a * ga).sum()).backward()
    tag = f"dfeature {grid} {kind} S{S}"
    check_table(f"{tag} dtable", tk.grad, t64.grad, L, T, F, 1e-4)
    for k in range(5):
        check(f"{tag} dW{k}", wk[k].grad, w64[k].grad, 1e-4)
        check(f"{tag} db{k}", bk[k].grad, b64[k].grad, 1e-4)
    check(f"{tag} dbeta", betak.grad, beta64.grad, 1e-4)


# ------------------------------------------------------------------------------------------------ 4. field + compositing
@pytest.mark.parametrize("S,kind", [(33, "multi"), (128, "multi"), (33, "few")])
@pytest.mark.parametrize("grid", list(GRIDS))
def test_gather_backward_render(nb, grid, S, kind):
    """Fn.field_render: the backward takes dfeature = weights * dfeat_ray in factored form."""
    from neuradar_b200 import functional as Fn

    spec, scal, table = make_grid(grid, seed=23 + S)
    L, F, T = spec.num_levels, spec.features_per_level, spec.log2_hashmap_size
    w, b, beta = mlp_params(seed=9)
    # compositing needs whole rays, M = N * S: at S = 128 the last tile is full (S = 33 keeps a partial one)
    N = -(-tiles_for(3)[0] // S) if kind == "multi" else 3
    M = N * S
    x3, std, sh, bins = make_samples(N, S, scal, seed=3 * N + S)
    sh_rows = sh.double()[torch.arange(M, device=DEV) // S]
    w64, b64, (beta64,) = leaves(w, torch.float64), leaves(b, torch.float64), leaves([beta], torch.float64)
    # the per-sample feature gradient is a product of the compositing weights here, so no upstream value can be zeroed
    # at a ReLU kink: samples near one are moved instead (a fixed, seeded step)
    g = torch.Generator(device=DEV).manual_seed(N)
    for _ in range(10):
        kink = near_kink(ref_encode(x3, std, table.double(), scal, T), sh_rows, w64, b64)
        if not bool(kink.any()):
            break
        x3[kink] = (x3[kink] + 1e-3 * torch.randn(x3[kink].shape, device=DEV, generator=g)).clamp(0, 1)
    assert not bool(kink.any())
    iv = Fn.SampleIntervals.from_bins(bins)
    gw, gfe = torch.randn((N, S), device=DEV, generator=g), torch.randn((N, 32), device=DEV, generator=g)
    gd, ga = torch.randn((N,), device=DEV, generator=g) * 1e-3, torch.randn((N,), device=DEV, generator=g)
    # reference: the oracle's compositing (sky sample included) in float64
    t64 = table.double().requires_grad_(True)
    rf, _, ra = ref_field(ref_encode(x3, std, t64, scal, T), sh_rows, w64, b64, beta64)
    starts, ends = bins[:, :-1].double().cpu(), bins[:, 1:].double().cpu()
    alpha, feats = ra.view(N, S).cpu(), rf.view(N, S, 32).cpu()
    comp = O.composite(alpha, feats, starts, ends, 0.0)
    raw, _ = O.alpha_weights(alpha, 0.0)
    r_w = torch.cat([comp["weights"][..., 0], raw[:, -1:] + 1 - comp["accumulation"]], dim=-1)  # the sky fix-up
    r_feat, r_depth, r_acc = comp["features"], comp["depth"][:, 0], comp["accumulation"][:, 0]
    ((r_w * gw.double().cpu()).sum() + (r_feat * gfe.double().cpu()).sum() + (r_depth * gd.double().cpu()).sum()
     + (r_acc * ga.double().cpu()).sum()).backward()
    tk = table.clone().requires_grad_(True)
    wk, bk, (betak,) = leaves(w, torch.float32), leaves(b, torch.float32), leaves([beta], torch.float32)
    kw, kf, kd, ka = Fn.field_render(tk, x3, std, sh, iv, spec, wk, bk, betak, BETA_MIN)
    tag = f"render {grid} {kind} S{S}"
    for what, got, want in (("weights", kw, r_w), ("features", kf, r_feat), ("depth", kd, r_depth), ("accumulation", ka, r_acc)):
        check(f"{tag} {what}", got, want, 1e-5)
    ((kw * gw).sum() + (kf * gfe).sum() + (kd * gd).sum() + (ka * ga).sum()).backward()
    check_table(f"{tag} dtable", tk.grad, t64.grad, L, T, F, 1e-4)
    for k in range(5):
        check(f"{tag} dW{k}", wk[k].grad, w64[k].grad, 1e-4)
        check(f"{tag} db{k}", bk[k].grad, b64[k].grad, 1e-4)
    check(f"{tag} dbeta", betak.grad, beta64.grad, 1e-4)


# ------------------------------------------------------------------------------------------------ 5. actors
@pytest.mark.parametrize("grid", list(GRIDS))
def test_gather_actors(nb, grid):
    """A hand-built ActorBatch (no nrb_actor_assign): actor samples read their actor's 4x4 grid with its level weights,
    zero-padded to 32 features, and the SH of their own direction; their gradient goes to that actor's table
    (nrb_actor_scatter) and none of it to the static table (the actor mask of nrb_hash_bwd_image)."""
    from neuradar_b200 import functional as Fn
    from neuradar_b200.functional import GridSpec

    S = 48
    spec, scal, table = make_grid(grid, seed=31, log2T=18)
    L, F, T = spec.num_levels, spec.features_per_level, spec.log2_hashmap_size
    M, _ = tiles_for(3, S)
    N = M // S
    x3, std, sh, _ = make_samples(N, S, scal, seed=77)
    g = torch.Generator().manual_seed(5)
    # which samples belong to which actor: scattered single samples, whole warps, one whole tile, runs across 32-lane and
    # 128-sample boundaries, in early and late tiles; actors 0, 1, 3 are used, actor 2 is not
    used = torch.tensor([0, 1, 3], dtype=torch.int32)
    gid = torch.full((M,), -1, dtype=torch.int32)
    r = torch.rand((M,), generator=g) < 0.08
    gid[r] = used[torch.randint(0, 3, (int(r.sum()),), generator=g)]
    for wp in (3, 10, 11, 57, 2001):
        gid[32 * wp : 32 * wp + 32] = 1
    gid[5 * 128 : 6 * 128] = used[torch.arange(128) % 3]
    gid[20 * 128 - 45 : 20 * 128 + 50] = 3
    gid[600 * 128 - 20 : 601 * 128 + 70] = 0
    gid[M - 100 : M - 60] = 0
    A, Ta = 4, 12
    ascal = O.level_scalings(4, 64, 1024)
    aspec = GridSpec(4, 4, Ta, tuple(float(s) for s in ascal))
    atables = [(torch.rand((4 << Ta, 4), generator=g) * 2 - 1) for _ in range(A)]
    pos = synthetic_points(N, S, g)
    astd = synthetic_std(M, ascal, g)
    d = torch.randn((M, 3), generator=g)
    dirs = d / d.norm(dim=-1, keepdim=True)
    gid_d, pos_d, astd_d, dirs_d = gid.to(DEV), pos.to(DEV), astd.to(DEV), dirs.to(DEV)
    act = gid_d >= 0
    # the static positions of actor samples are never read by the forward; spread over the cube, they hash to many static
    # rows that no static sample touches
    x3[act] = torch.rand((int(act.sum()), 3), generator=g).to(DEV)
    sh_rows = torch.where(act[:, None], ref_sh(dirs), sh.double()[torch.arange(M, device=DEV) // S])
    w, b, beta = mlp_params(seed=13)
    w64, b64, (beta64,) = leaves(w, torch.float64), leaves(b, torch.float64), leaves([beta], torch.float64)
    t64 = table.double().requires_grad_(True)
    a64 = leaves(atables, torch.float64)

    def ref_feats():
        static = ref_encode(x3, std, t64, scal, T)
        afeat = torch.zeros_like(static)
        for i in range(A):
            sel = (gid_d == i).nonzero()[:, 0]
            if sel.numel():
                f16 = ref_encode(pos_d[sel], astd_d[sel], a64[i], ascal, Ta)
                afeat = afeat.index_put((sel,), TF.pad(f16, (0, 16)))
        return torch.where(act[:, None], afeat, static)

    feats = ref_feats()
    gd = torch.Generator(device=DEV).manual_seed(1)
    gf, gs, ga = (torch.randn((M, 32), device=DEV, generator=gd), torch.randn((M,), device=DEV, generator=gd),
                  torch.randn((M,), device=DEV, generator=gd))
    kink = near_kink(feats, sh_rows, w64, b64)
    gf[kink], gs[kink], ga[kink] = 0, 0, 0
    rf, rs, ra = ref_field(feats, sh_rows, w64, b64, beta64)
    ((rf * gf.double()).sum() + (rs * gs.double()).sum() + (ra * ga.double()).sum()).backward()
    tk = table.clone().requires_grad_(True)
    ak = leaves(atables, torch.float32)
    wk, bk, (betak,) = leaves(w, torch.float32), leaves(b, torch.float32), leaves([beta], torch.float32)
    batch = Fn.ActorBatch(gid_d, pos_d, astd_d, dirs_d, ak, aspec)
    f, s, a = Fn.field_fused(tk, None, x3, std, sh, S, spec, wk, bk, betak, BETA_MIN, batch)
    tag = f"actors {grid}"
    for what, got, want in (("feature", f, rf), ("sdf", s, rs), ("alpha", a, ra)):
        check(f"{tag} {what}", got, want, 1e-5)
    ((f * gf).sum() + (s * gs).sum() + (a * ga).sum()).backward()
    check_table(f"{tag} static dtable", tk.grad, t64.grad, L, T, F, 1e-4)
    for i in range(A):
        if i == 2:
            assert a64[i].grad is None and float(ak[i].grad.abs().max()) == 0.0
            continue
        check_table(f"{tag} actor {i} dtable", ak[i].grad, a64[i].grad, 4, Ta, 4, 1e-4)
    for k in range(5):
        check(f"{tag} dW{k}", wk[k].grad, w64[k].grad, 1e-4)
        check(f"{tag} db{k}", bk[k].grad, b64[k].grad, 1e-4)
    check(f"{tag} dbeta", betak.grad, beta64.grad, 1e-4)
    # static rows that only actor samples' positions hash to receive exactly nothing
    idx, _ = ref_cells(x3, scal, T)
    static_rows = torch.unique(idx[~act].reshape(-1))
    actor_rows = torch.unique(idx[act].reshape(-1))
    only = actor_rows[~torch.isin(actor_rows, static_rows)]
    assert only.numel() > 1000, only.numel()
    assert float(tk.grad[only].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ 6. row mode, many tiles
def test_rows_backward_multi_tile(nb):
    """Row mode (hash features given) with x.grad at the multi-tile M: against float64, and the first M0 rows bit for bit
    against a run on those rows alone (a row's dx depends on that row only)."""
    from neuradar_b200 import functional as Fn

    S = 48
    M, mine = tiles_for(3, S)
    print(f"[tiles_for] rows backward tiles per CTA: {min(mine)}..{max(mine)}")  # (mirrored launcher formulas)
    N = M // S
    g = torch.Generator().manual_seed(17)
    x = torch.randn((M, 32), generator=g) * 0.5
    d = torch.randn((N, 3), generator=g)
    sh = O.sh16((d / d.norm(dim=-1, keepdim=True) + 1.0) / 2.0).to(DEV)
    x = x.to(DEV)
    w, b, beta = mlp_params(seed=21)
    sh_rows = sh.double()[torch.arange(M, device=DEV) // S]
    gd = torch.Generator(device=DEV).manual_seed(2)
    gf, gs, ga = (torch.randn((M, 32), device=DEV, generator=gd), torch.randn((M,), device=DEV, generator=gd),
                  torch.randn((M,), device=DEV, generator=gd))
    w64, b64, (beta64,) = leaves(w, torch.float64), leaves(b, torch.float64), leaves([beta], torch.float64)
    x64 = x.double().requires_grad_(True)
    kink = near_kink(x64, sh_rows, w64, b64)
    gf[kink], gs[kink], ga[kink] = 0, 0, 0
    rf, rs, ra = ref_field(x64, sh_rows, w64, b64, beta64)
    ((rf * gf.double()).sum() + (rs * gs.double()).sum() + (ra * ga.double()).sum()).backward()

    def run(n):
        xk = x[:n].clone().requires_grad_(True)
        wk, bk, (betak,) = leaves(w, torch.float32), leaves(b, torch.float32), leaves([beta], torch.float32)
        f, s, a = Fn.field_fused(None, xk, None, None, sh[: -(-n // S)].contiguous(), S, None, wk, bk, betak, BETA_MIN)
        ((f * gf[:n]).sum() + (s * gs[:n]).sum() + (a * ga[:n]).sum()).backward()
        return xk.grad, wk, bk, betak

    dx, wk, bk, betak = run(M)
    check("rows dx", dx, x64.grad, 1e-4)
    for k in range(5):
        check(f"rows dW{k}", wk[k].grad, w64[k].grad, 1e-4)
        check(f"rows db{k}", bk[k].grad, b64[k].grad, 1e-4)
    check("rows dbeta", betak.grad, beta64.grad, 1e-4)
    M0 = 40 * 128 + 45
    assert torch.equal(run(M0)[0], dx[:M0])
