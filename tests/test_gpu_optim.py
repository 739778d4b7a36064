"""GPU parity of the fused Adam / AdamW step (SURVEY.md 8f next-2) against the CPU oracle (itself pinned against
torch.optim in tests/test_oracle_golden.py) and against torch.optim + GradScaler run on the same gradients."""
import ctypes as C

import pytest
import torch

from oracle import neuradar_oracle as O
from tests.parity_utils import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _params(gen, shapes):
    return [torch.randn(s, generator=gen) * 1e-2 for s in shapes]


@pytest.mark.parametrize("decoupled,wd", [(False, 0.0), (True, 1e-7), (False, 1e-3)])
def test_fused_adam_vs_oracle(decoupled, wd):
    from neuradar_b200.optim import FusedAdam, FusedAdamW

    gen = torch.Generator().manual_seed(11)
    shapes = [(1 << 12, 2), (33, 32), (33,), (1,), (7, 3)]  # odd sizes: every view is padded to 16 bytes
    host = _params(gen, shapes)
    dev = [torch.nn.Parameter(h.clone().to(DEV)) for h in host]
    opt = (FusedAdamW if decoupled else FusedAdam)(dev, lr=1e-2, eps=1e-15, weight_decay=wd)
    ms, vs = [torch.zeros_like(h) for h in host], [torch.zeros_like(h) for h in host]
    for step in range(1, 6):
        grads = [torch.randn(h.shape, generator=gen) * 10.0 ** (-step) for h in host]
        for d, g in zip(dev, grads):
            d.grad.copy_(g.to(DEV))  # .grad is a view of the flat gradient buffer
        opt.step(grad_mult=0.25, zero_grad=True)
        for h, g, m, v in zip(host, grads, ms, vs):
            O.adam_step(h, g, m, v, step, lr=1e-2, eps=1e-15, weight_decay=wd, decoupled=decoupled, grad_mult=0.25)
        for d, h in zip(dev, host):
            assert rel_err(d, h) < 1e-6  # fp32 elementwise chain, fused multiply-adds on the device
            assert float(d.grad.abs().max()) == 0.0  # fused zero_grad
    sd = opt.state_dict()
    assert rel_err(sd["state"][1]["exp_avg"], ms[1]) < 1e-6 and rel_err(sd["state"][1]["exp_avg_sq"], vs[1]) < 1e-6
    assert float(sd["state"][0]["step"]) == 5.0


def test_fused_adam_with_grad_scaler_matches_torch():
    """Same gradients through torch.amp.GradScaler: torch.optim.Adam (unscale + foreach kernels) vs FusedAdam (scale
    and found_inf consumed inside the one kernel); an inf gradient skips the step in both."""
    from neuradar_b200.optim import FusedAdam

    gen = torch.Generator().manual_seed(5)
    w0 = torch.randn((5000,), generator=gen) * 1e-2
    a = torch.nn.Parameter(w0.clone().to(DEV))
    b = torch.nn.Parameter(w0.clone().to(DEV))
    opt_a = torch.optim.Adam([a], lr=1e-2, eps=1e-15)
    opt_b = FusedAdam([b], lr=1e-2, eps=1e-15)
    sc_a = torch.amp.GradScaler("cuda", init_scale=1024.0, growth_interval=3)
    sc_b = torch.amp.GradScaler("cuda", init_scale=1024.0, growth_interval=3)
    for step in range(8):
        x = torch.randn((5000,), generator=gen).to(DEV)
        bad = step == 4
        for p, opt, sc in ((a, opt_a, sc_a), (b, opt_b, sc_b)):
            opt.zero_grad()
            loss = (p * x).sum() * (float("inf") if bad else 1.0) + (p * p).sum()
            sc.scale(loss).backward()
            sc.step(opt)
            sc.update()
        assert rel_err(b, a) < 1e-6, step
        assert sc_a.get_scale() == sc_b.get_scale()


def test_adam_c_abi_tail_and_skip():
    """Segment lengths that are not a multiple of four, and the found_inf skip, straight through the C ABI."""
    from neuradar_b200 import _lib
    from neuradar_b200._lib import AdamCfg, ptr, stream_ptr

    gen = torch.Generator().manual_seed(1)
    for n in (1, 3, 4, 7, 1026):
        p = torch.randn((n + 8,), generator=gen)
        g = torch.randn((n + 8,), generator=gen)
        pd, gd = p.to(DEV), g.to(DEV)
        md, vd = torch.zeros_like(pd), torch.zeros_like(pd)
        cfg = AdamCfg(1e-2, 0.9, 0.999, 1e-15, 0.0, 0, 1, 1.0, 0)
        _lib.call("nrb_adam_step", ptr(pd), ptr(gd), ptr(md), ptr(vd), n, C.byref(cfg), None, None, None, stream_ptr())
        ph, m, v = p.clone(), torch.zeros_like(p), torch.zeros_like(p)
        O.adam_step(ph[:n], g[:n], m[:n], v[:n], 1, lr=1e-2)
        assert rel_err(pd[:n], ph[:n]) < 1e-6
        assert torch.equal(pd[n:].cpu(), p[n:])  # nothing beyond n is touched
        flag = torch.ones((1,), device=DEV)
        before = pd.clone()
        cfg.step = 2
        cfg.zero_grad = 1
        _lib.call("nrb_adam_step", ptr(pd), ptr(gd), ptr(md), ptr(vd), n, C.byref(cfg), None, ptr(flag), None, stream_ptr())
        assert torch.equal(pd, before) and float(gd[:n].abs().max()) == 0.0 and torch.equal(gd[n:].cpu(), g[n:])
    # non-finite detection
    gbad = torch.zeros((1001,), device=DEV)
    flag = torch.zeros((1,), device=DEV)
    _lib.call("nrb_grad_check", ptr(gbad), 1001, ptr(flag), stream_ptr())
    assert float(flag) == 0.0
    gbad[1000] = float("nan")
    _lib.call("nrb_grad_check", ptr(gbad), 1001, ptr(flag), stream_ptr())
    assert float(flag) == 1.0
    gbad[1000] = 0.0
    gbad[17] = float("-inf")
    flag.zero_()
    _lib.call("nrb_grad_check", ptr(gbad), 1001, ptr(flag), stream_ptr())
    assert float(flag) == 1.0


def test_adam_full_size_streaming_properties():
    """Arena size of config 2 (22 M parameters): zero gradients leave parameters untouched for Adam (m = v = 0 ->
    update 0 / eps-guarded), and one step with g = sign pattern moves every parameter by exactly lr (|m|/sqrt(v) = 1)."""
    from neuradar_b200.optim import FusedAdam

    n = 22_000_000
    q = torch.nn.Parameter(torch.zeros((1 << 20,), device=DEV))
    opt_q = FusedAdam([q], lr=1e-2, eps=1e-15)
    opt_q.step()
    assert float(q.detach().abs().max()) == 0.0
    p = torch.nn.Parameter(torch.zeros((n,), device=DEV))
    opt = FusedAdam([p], lr=1e-2, eps=1e-15)
    sign = (torch.arange(n, device=DEV) % 2).float() * 2 - 1
    p.grad.copy_(sign * 3.0)
    opt.step()  # first step: m / (1 - beta1) = g, sqrt(v / (1 - beta2)) = |g|
    assert rel_err(p, -1e-2 * sign) < 1e-6


def test_direct_scatter_into_arena_matches_autograd_accumulation():
    """GradArena(direct_scatter=True): the hash-grid backward kernels add straight into the arena views; gradients
    must equal the ordinary autograd accumulation (also when a table is used twice, as the late-binding proposal
    field is) and accumulate over two backward passes."""
    import neuradar_b200 as nb
    from neuradar_b200.dist import GradArena
    from tests.parity_utils import FixedJitter, build_hot_path, make_ray_bundle, synthetic_rays

    n = 512
    rays = synthetic_rays(n, seed=9)
    gen = torch.Generator().manual_seed(10)
    jit = [torch.rand((n, 65), generator=gen), torch.rand((n, 1), generator=gen), torch.rand((n, 1), generator=gen)]
    grads = []
    for direct in (False, True):
        model = build_hot_path(log2_main=14, log2_prop=14, num_proposal_samples=(64, 48), num_nerf_samples=48,
                               late_binding=True, table_gain=(300.0, 2000.0), seed=4, device=DEV)
        model.train()
        used = [p for name, p in model.named_parameters() if not name.startswith("proposal_fields.0")]
        arena = GradArena(used, direct_scatter=direct)
        assert any(getattr(p, "_nrb_grad_sink", None) is not None for p in used) == direct
        for _ in range(2):  # gradients accumulate across backward passes, like .grad does
            with FixedJitter(jit):
                out = model(make_ray_bundle(rays, DEV))
            nb.bench_loss(out).backward()
        grads.append(arena.flat.clone())
    scale = float(grads[0].abs().max())
    assert scale > 0
    assert float((grads[0] - grads[1]).abs().max()) <= 1e-5 * scale  # atomics: last-bit differences only


def test_direct_scatter_from_a_side_stream_is_ordered_before_the_default_stream():
    """A backward that ran on a side stream (autograd replays a node on its forward's stream) and added straight into a
    gradient sink must be visible to work queued on the default stream right after `backward()` - an all-reduce or an
    optimiser step (ADVICE round 1: functional._sink_written makes the default stream wait)."""
    import neuradar_b200 as nb
    from neuradar_b200 import functional as Fn
    from neuradar_b200.dist import GradArena

    spec = nb.HashEncoding(num_levels=16, features_per_level=2, log2_hashmap_size=17, min_res=16, max_res=1024).spec
    g = torch.Generator().manual_seed(3)
    M = 1 << 20  # ~1 ms of scatter: long enough for a missing dependency to show
    x = torch.rand((M, 3), generator=g).to(DEV)
    dy = torch.randn((M, 32), generator=g).to(DEV)
    table = torch.nn.Parameter((torch.rand((spec.rows, 2), generator=g) * 2e-4 - 1e-4).to(DEV))
    # expected: ordinary autograd accumulation on the default stream
    (Fn.hash_encode(x, table, spec) * dy).sum().backward()
    want = table.grad.clone()
    table.grad = None
    arena = GradArena([table], direct_scatter=True)
    side = torch.cuda.Stream()
    for _ in range(3):
        arena.zero()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            loss = (Fn.hash_encode(x, table, spec) * dy).sum()
        torch.cuda.current_stream().wait_stream(side)
        loss.backward()
        got = arena.flat[: want.numel()].clone()  # queued on the default stream immediately after backward()
        assert rel_err(got.view_as(want), want) <= 1e-5


def test_decoder_only_sink_from_a_side_stream_is_ordered_before_the_default_stream():
    """A proposal round on a side stream whose only gradient sink is its density decoder's (the "fields" optimiser
    scatters directly, the "hashgrids" one does not): no gradient goes back to autograd, so only the sink bookkeeping
    orders the decoder's gradient before work queued on the default stream right after `backward()`."""
    from neuradar_b200 import functional as Fn
    from neuradar_b200.dist import GradArena
    from tests.parity_utils import build_hot_path, scaled_pixel_area, synthetic_rays

    N, S = 16384, 64  # ~1 M samples: a backward long enough for a missing dependency to show
    model = build_hot_path(log2_main=12, log2_prop=17, table_gain=(300.0, 2000.0), seed=4, device=DEV)
    pf = model.proposal_fields[1]
    table, dec = pf.hashgrid.static_grid.hash_table, pf.density_decoder.weight
    table.requires_grad_(False)
    rays = synthetic_rays(N, seed=6)
    g = torch.Generator().manual_seed(3)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), S, torch.rand((N, S + 1), generator=g))
    rd = Fn.RayData(rays["origins"].to(DEV), rays["directions"].to(DEV), scaled_pixel_area(rays).to(DEV))
    iv = Fn.SampleIntervals.from_bins(eb.contiguous().to(DEV))
    gw = torch.randn((N, S), generator=g).to(DEV)

    def loss():
        _, w = Fn.proposal_round(table, dec, rd, iv, pf.hashgrid.static_grid.spec, 100.0)
        return (w * gw).sum()

    loss().backward()  # expected: ordinary autograd accumulation on the default stream
    want = dec.grad.clone()
    dec.grad = None
    arena = GradArena([dec], direct_scatter=True)
    side = torch.cuda.Stream()
    for _ in range(3):
        arena.zero()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            l = loss()
        torch.cuda.current_stream().wait_stream(side)
        l.backward()
        got = arena.flat[: want.numel()].clone()  # queued on the default stream immediately after backward()
        assert rel_err(got.view_as(want), want) <= 1e-4


def test_field_render_keeps_no_reference_cycle():
    """The outputs of `field_render` are saved for its backward, not kept on ctx: with the cyclic garbage collector off,
    dropping the outputs after backward frees them (and the [M,32] feature buffer the node holds)."""
    import gc
    import weakref

    from tests.parity_utils import build_hot_path, make_ray_bundle, synthetic_rays

    model = build_hot_path(log2_main=12, log2_prop=12, table_gain=(300.0, 2000.0), seed=9, device=DEV)
    rays = synthetic_rays(256, seed=10)
    _, eb, _ = O.spaced_bins(rays["nears"], rays["fars"].clamp_max(20000.0), 48, torch.rand((256, 49)))
    rs = make_ray_bundle(rays, DEV).get_ray_samples(bin_starts=eb[:, :-1, None].to(DEV), bin_ends=eb[:, 1:, None].to(DEV))
    gc.disable()
    try:
        weights, features, depth, acc = model.field.render(rs)
        alive = weakref.ref(weights)
        (weights.sum() + features.sum() + depth.sum()).backward()
        del weights, features, depth, acc
        assert alive() is None
    finally:
        gc.enable()
