#!/usr/bin/env python
"""Benchmark of the NeuRadar per-ray hot path (BASELINE.json: train-step rays/sec at 1/2/4/8 B200).

  python bench.py --gpus N --steps K --warmup W [--config C]     # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...        # the reference's own torch path on the host CPU

A step = one pass of the hot path (proposal sampling -> hash encode -> MLPs -> compositing; training configs add the
loss of SURVEY.md 8d, the backward pass and the gradient all-reduce) over one batch of synthetic rays.  `--config`
selects a BASELINE.json configuration (default 2: 65536 mixed camera/lidar/radar rays per GPU, 16-level 2^19 main
grid, 48 samples per ray, proposal rounds of 64 and 48 samples on the 6-level 2^20 grid):
    1  4096 radar rays (the reference's CPU-runnable case)          4  large scene: 2^22 tables, 128 samples, 16 actors
    3  the 8-GPU shard of the 262144-ray step: 32768 rays per GPU   5  inference sweep: 1 M radar rays, chunks of 32768
For N > 1 each rank owns its own rays (weak scaling) and the step ends with the all-reduce of the flat gradient arena:
the main table's 64 MiB start reducing as soon as the field's backward is enqueued, hidden behind the proposal rounds'.
The step is captured ONCE in a CUDA graph (fwd + bwd + collectives) and replayed; the timed loop rotates through four
resident ray batches.  Prints ONE JSON line.

  --optimizer      adds the fused Adam / AdamW update (SURVEY.md 8f next-2) to the step of both arms
  --regularisers   adds the interlevel + distortion losses (SURVEY.md 8f next-1) to the step of both arms
  --no-graph       launch the step eagerly (what a plain training loop does)
  --dump-outputs DIR   after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32): the
                   path's outputs and, for training configs, the loss and every gradient (the updated parameters with
                   --optimizer).  Arrays beyond the 64 MB budget are replaced by a fixed, seeded sample of their
                   elements; the inputs are seeded, so two builds can be compared output for output.

`roofline` = the kernel with the largest share of the step (`rooflines` has every major kernel): algorithmic bytes or
FLOPs per launch (DESIGN.md section 4) / CUDA-event duration, against MEASURED_PEAKS.json; `traffic` = DRAM bytes per
launch from the committed ncu capture (profiles/r2_traffic.json).  `path_roofline` = the whole step against the HBM
roofline of SURVEY.md 8d (algorithmic bytes per ray).  `parity_at_config` = the CUDA path against the reference's torch
path on 4096 of the benchmark's own rays with the benchmark's own tables.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "train_step_rays_per_sec"
UNIT = "rays/s"
N_BATCHES = 4
DUMP_BYTES = 60_000_000  # --dump-outputs budget: 64 MB with room for the .npy headers


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "tflops": p.get("bf16_tflops_sustained", p.get("bf16_tflops")), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "source": "fallback"}


class ClockSampler:
    """Samples SM clocks and throttle reasons with NVML while the timed region runs."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        return False

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own torch path (oracle/_ref, materialised by oracle/build_ref.py), or the
# oracle port of it when the reference modules are not there
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_run(w, sample: int, steps: int, warmup: int, seed: int = 42, regularisers: bool = False,
                      optimizer: bool = False):
    """fwd(+bwd) of the reference algorithm on `sample` rays of workload `w` on the host CPU.
    Returns (rays/s, ms/step, threads, kind, cpu model)."""
    from neuradar_b200.synthetic import scaled_pixel_area, synthetic_rays
    from oracle import ref_runner as R

    rays = synthetic_rays(sample, seed=seed, mix=w.mix)
    pa = scaled_pixel_area(rays)
    if R.available() and not regularisers and not optimizer:
        path = R.ReferencePath(main=w.main, prop_log2=w.prop_log2, proposal_samples=w.proposal_samples,
                               nerf_samples=w.nerf_samples, seed=seed)
        value, ms, cores = R.time_reference(rays, pa, path, steps, warmup, train=w.train)
        return value, ms, cores, "reference", R.cpu_model_name()
    value, ms, cores = cpu_port_run(w, rays, pa, steps, warmup, seed, regularisers, optimizer)
    return value, ms, cores, "port", R.cpu_model_name()


def cpu_port_run(w, rays, pa, steps, warmup, seed, regularisers, optimizer):
    from oracle import neuradar_oracle as O

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(seed)
    L, F, T, r0, r1 = w.main
    main = O.GridParams(((torch.rand((L << T, F)) * 2 - 1) * 1e-3).requires_grad_(True), O.level_scalings(L, r0, r1), T)
    lin = torch.nn.Linear

    def wb(i, o):
        layer = lin(i, o)
        return layer.weight.detach().requires_grad_(True), layer.bias.detach().requires_grad_(True)

    g0, g1 = wb(32, 32), wb(32, 33)
    f0, f1, f2 = wb(48, 32), wb(32, 32), wb(32, 32)
    fld = O.FieldParams(main, [g0[0], g1[0]], [g0[1], g1[1]], [f0[0], f1[0], f2[0]], [f0[1], f1[1], f2[1]],
                        torch.full((1,), 20.0, requires_grad=True))
    prop = O.ProposalParams(
        O.GridParams(((torch.rand((6 << w.prop_log2, 1)) * 2 - 1) * 1e-3).requires_grad_(True), O.level_scalings(6, 128, 4096),
                     w.prop_log2),
        lin(6, 1, bias=False).weight.detach().requires_grad_(True),
    )
    num_rays = rays["origins"].shape[0]
    cfg = O.PathConfig(num_proposal_samples=w.proposal_samples, num_nerf_samples=w.nerf_samples)
    leaves = [main.table, *fld.geo_w, *fld.geo_b, *fld.feat_w, *fld.feat_b, fld.beta, prop.grid.table, prop.decoder_w]
    opts = []
    if optimizer:  # the reference's parameter groups (configs/method_configs.py:393-400)
        opts = [torch.optim.Adam([main.table, prop.grid.table], lr=1e-2, eps=1e-15),
                torch.optim.AdamW([t for t in leaves if t is not main.table and t is not prop.grid.table], lr=1e-2, eps=1e-15,
                                  weight_decay=1e-7)]

    def step():
        for t in leaves:
            t.grad = None
        jit = [torch.rand((num_rays, w.proposal_samples[0] + 1)), torch.rand((num_rays, 1)), torch.rand((num_rays, 1))]
        if not w.train:
            with torch.no_grad():
                O.nff_forward(fld, [prop, prop], rays["origins"], rays["directions"], pa, rays["nears"], rays["fars"], cfg, None)
            return
        out = O.nff_forward(fld, [prop, prop], rays["origins"], rays["directions"], pa, rays["nears"], rays["fars"], cfg, jit)
        loss = O.bench_loss(out)
        if regularisers:
            loss = loss + O.training_losses(out)
        loss.backward()
        for o in opts:
            o.step()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return num_rays / dt, dt * 1e3, cores


def run_reference(args, rank):
    if rank != 0:
        return
    from neuradar_b200.synthetic import WORKLOADS

    w = WORKLOADS[args.config]
    sample = min(4096, w.rays)
    steps, warmup = args.steps, args.warmup
    value, ms, cores, kind, cpu = cpu_reference_run(w, sample, steps, warmup, regularisers=args.regularisers,
                                                    optimizer=args.optimizer)
    what = ("the reference's own modules (oracle/_ref, unmodified) on its fp32 torch path" if kind == "reference"
            else "the oracle port of the reference's torch path (oracle/_ref not materialised)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.description, "note": f"host CPU, {what}; autocast off; compositing through "
                   "RaySamples.get_weights_and_transmittance_from_alphas (the model's CPU branch is a 0.5 stub)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu,
                         "sample": f"{sample} {w.mix} rays of the workload per step, {warmup} warm-up + {steps} timed steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------
def parity_at_config(model, w, rays_cpu, n_check: int = 4096):
    """The CUDA path against the reference torch path (oracle/_ref; else the oracle port) on `n_check` of the benchmark's
    rays with the benchmark's parameters: outputs and every parameter gradient.  Element-wise bar of north_star:
    |a - b| <= 1e-3 |b| + 1e-3 rms(b)."""
    import neuradar_b200 as nb
    from neuradar_b200.synthetic import scaled_pixel_area
    from oracle import ref_runner as R
    from tests.parity_utils import FixedJitter

    dev = next(model.parameters()).device
    n = min(n_check, rays_cpu["origins"].shape[0])
    sub = {k: v[:n].clone() for k, v in rays_cpu.items()}
    g = torch.Generator().manual_seed(7)
    jit = [torch.rand((n, w.proposal_samples[0] + 1), generator=g), torch.rand((n, 1), generator=g), torch.rand((n, 1), generator=g)]
    # CUDA path (eager, its gradients go to fresh tensors: detach the flat-buffer plumbing for this one call)
    saved = [(p, p.grad, getattr(p, "_nrb_grad_sink", None), getattr(p, "_nrb_grad_ready", None)) for p in model.parameters()]
    for p, *_ in saved:
        p.grad = None
        p._nrb_grad_sink = None
        p._nrb_grad_ready = None
    model.train(w.train)
    grids = [model.field.hashgrid] + [p.hashgrid for p in model.proposal_fields]
    flips = None
    if w.actors and w.train:  # the per-ray mirror draw of the actor branch (neurad_encoding.py:218-225), replayed on both sides
        flips = (torch.rand((n,), generator=g) < 0.25).float() * -2 + 1
        for h in grids:
            h.ray_flip_override = flips.to(dev)
    rb = nb.RayBundle(origins=sub["origins"].to(dev), directions=sub["directions"].to(dev), pixel_area=sub["pixel_area"].to(dev),
                      nears=sub["nears"].to(dev), fars=sub["fars"].to(dev), times=sub["times"].to(dev),
                      metadata={"is_lidar": sub["is_lidar"].to(dev), "is_radar": sub["is_radar"].to(dev)})
    if w.train:
        with FixedJitter(jit):
            out = model(rb)
        nb.bench_loss(out).backward()
    else:
        with torch.no_grad():
            out = model(rb)
    torch.cuda.synchronize()
    got_out = {k: out[k].detach().cpu() for k in ("features", "depth", "accumulation")}
    got_grad = {name: (None if p.grad is None else p.grad.detach().cpu()) for name, p in model.named_parameters()}
    for p, gr, sk, rd in saved:
        p.grad, p._nrb_grad_sink, p._nrb_grad_ready = gr, sk, rd
    for h in grids:
        h.ray_flip_override = None
    # reference
    kind = "reference" if R.available() else "port"
    if kind != "reference":
        return {"kind": "port", "note": "oracle/_ref not materialised; run tests/ for the oracle-port parity"}
    from neuradar_b200.synthetic import SyntheticActors
    path = R.ReferencePath(main=w.main, prop_log2=w.prop_log2, proposal_samples=w.proposal_samples, nerf_samples=w.nerf_samples,
                           actors=SyntheticActors(w.actors) if w.actors else None)
    path.load_from(model.state_dict())
    path.train(w.train)
    torch.set_num_threads(os.cpu_count() or 1)
    if w.train:
        draw = torch.bernoulli
        if flips is not None:
            torch.bernoulli = lambda probs, *a, **k: (flips < 0).to(probs.dtype)
        try:
            with FixedJitter(jit):
                ref = path.forward(sub, scaled_pixel_area(sub))
        finally:
            torch.bernoulli = draw
        R.bench_loss(ref).backward()
    else:
        with torch.no_grad():
            ref = path.forward(sub, scaled_pixel_area(sub))

    def err(a, b):
        a, b = a.float().reshape(-1), b.detach().float().reshape(-1)
        rms = float(b.pow(2).mean().sqrt())
        outside = int(((a - b).abs() > (1e-3 * b.abs() + 1e-3 * rms)).sum())
        return {"max_abs_over_max": float((a - b).abs().max() / (b.abs().max() + 1e-30)), "within_bar": outside == 0,
                "outside": outside, "elements": a.numel()}

    report = {"kind": kind, "rays": n, "outputs": {}, "grads": {}}
    for k, v in got_out.items():
        report["outputs"][k] = err(v, ref[k])
    if w.train:
        refp = path.named_parameters()
        for name, gr in got_grad.items():
            rg = refp[name].grad if name in refp else None
            if rg is None:
                continue
            report["grads"][name] = err(gr if gr is not None else torch.zeros_like(rg), rg)
    everything = list(report["outputs"].values()) + list(report["grads"].values())
    report["worst"] = max(e["max_abs_over_max"] for e in everything)
    # A sample that sits on a bin edge or an actor-box face within one ulp can be claimed differently by the two
    # implementations (CPU vs GPU rounding of the poses), which moves that one sample's gradient between table rows:
    # the same 1e-5 allowance as for PDF indices, counted in elements, and nothing may be off by more than 1e-3 of the
    # tensor's largest entry.
    report["ok"] = all(e["outside"] <= 1e-5 * e["elements"] and e["max_abs_over_max"] <= 1e-3 for e in everything)
    report["strict_ok"] = all(e["within_bar"] for e in everything)
    return report


def step_outputs(out):
    """The arrays of one forward's output dict, detached (holding them must not keep the autograd graph alive)."""
    arrays = {k: v.detach() for k, v in out.items() if torch.is_tensor(v)}
    arrays.update({f"weights_{i}": t.detach() for i, t in enumerate(out.get("weights_list", []))})
    return arrays


def dump_outputs(directory, arrays, seed: int = 0):
    """Write {name: tensor} as directory/<name>.npy in float32, DUMP_BYTES in all.  The budget is shared smallest array
    first; an array that gets k < numel elements is written as a seeded stratified sample of its flattened elements: one
    element from each of k equal strides, in index order, so the same arguments always select the same elements."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    budget = DUMP_BYTES // 4
    names = sorted(arrays, key=lambda k: arrays[k].numel())
    for i, name in enumerate(names):
        t = arrays[name].detach().float()
        keep = min(t.numel(), budget // (len(names) - i))
        budget -= keep
        if keep < t.numel():
            edges = torch.arange(keep + 1, dtype=torch.int64) * t.numel() // keep
            u = torch.rand(keep, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
            idx = edges[:-1] + (u * (edges[1:] - edges[:-1])).long()
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    import neuradar_b200 as nb
    from neuradar_b200 import _lib
    from neuradar_b200.dist import GradArena
    from neuradar_b200.synthetic import WORKLOADS, build_workload, synthetic_rays

    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    w = WORKLOADS[args.config]
    n = args.rays or w.rays
    model = build_workload(w, seed=42, device=dev)
    model.train(w.train)
    used = [(name, p) for name, p in model.named_parameters() if not name.startswith("proposal_fields.0")]
    main_table = model.field.hashgrid.static_grid.hash_table
    opts, arena, arena_bytes = None, None, 0
    if w.train:
        if args.optimizer:
            # the reference's "hashgrids" (Adam) and "fields" (AdamW) groups, each one flat buffer and one fused kernel
            from neuradar_b200.optim import FusedAdam, FusedAdamW

            tables = [p for name, p in used if name.endswith("hash_table")]
            others = [p for name, p in used if not name.endswith("hash_table")]
            opts = [FusedAdam(tables, lr=1e-2, eps=1e-15, direct_scatter=True, early=[main_table]),
                    FusedAdamW(others, lr=1e-2, eps=1e-15, weight_decay=1e-7, direct_scatter=True)]
            arena_bytes = sum(g.numel() * 4 for o in opts for g in o.flat_grads())
        else:
            arena = GradArena([p for _, p in used], direct_scatter=True, early=[main_table])
            arena_bytes = arena.nbytes
    # ray batches: each rank draws its own (train.py:104 seeds seed+rank); the timed loop rotates through them
    keys = ["origins", "directions", "pixel_area", "nears", "fars", "times", "is_lidar", "is_radar"]
    n_batches = N_BATCHES if n <= (1 << 17) else 1
    batches_cpu = [synthetic_rays(n, seed=42 + rank + 1000 * b, mix=w.mix) for b in range(n_batches)]
    # one flat byte buffer per batch (fields at 256-byte aligned offsets): a step's rays move host -> device in ONE copy
    offsets, total_bytes = {}, 0
    for k in keys:
        offsets[k] = total_bytes
        total_bytes += (batches_cpu[0][k].numel() * batches_cpu[0][k].element_size() + 255) // 256 * 256

    def views(flat):
        return {k: flat[offsets[k]: offsets[k] + batches_cpu[0][k].numel() * batches_cpu[0][k].element_size()]
                .view(batches_cpu[0][k].dtype).view(batches_cpu[0][k].shape) for k in keys}

    host_flat = [torch.zeros((total_bytes,), dtype=torch.uint8).pin_memory() for _ in batches_cpu]
    for hf, b in zip(host_flat, batches_cpu):
        for k, v in views(hf).items():
            v.copy_(b[k])
    resident_flat = [hf.to(dev) for hf in host_flat]
    cur_flat = torch.empty((total_bytes,), dtype=torch.uint8, device=dev)
    cur = views(cur_flat)  # the step's (static) inputs
    staging = [torch.empty_like(cur_flat) for _ in range(2)]  # landing buffers of the prefetching host -> device copies
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event() for _ in range(2)]
    h2d_bytes = sum(batches_cpu[0][k].numel() * batches_cpu[0][k].element_size() for k in keys)

    def bundle(src, lo=0, hi=None):
        sl = slice(lo, hi)
        return nb.RayBundle(origins=src["origins"][sl].clone(), directions=src["directions"][sl].clone(),
                            pixel_area=src["pixel_area"][sl].clone(), nears=src["nears"][sl].clone(), fars=src["fars"][sl].clone(),
                            times=src["times"][sl], metadata={"is_lidar": src["is_lidar"][sl], "is_radar": src["is_radar"][sl]})

    result = {}

    def step():
        """One step on the rays in `cur`; leaves the step's scalar result in result['loss'] (device)."""
        kept = result["outs"] = [] if args.dump_outputs else None  # the step's outputs, for --dump-outputs
        if not w.train:
            chunk = w.chunk or n
            acc = None
            with torch.no_grad():
                for lo in range(0, n, chunk):
                    out = model(bundle(cur, lo, min(lo + chunk, n)))
                    s = out["depth"].sum()
                    acc = s if acc is None else acc + s
                    if kept is not None:
                        kept.append(step_outputs(out))
            result["loss"] = acc
            return
        if opts is None:
            arena.zero()
        out = model(bundle(cur))
        loss = nb.bench_loss(out)
        if args.regularisers:
            loss = loss + nb.training_losses(out)
        loss.backward()
        if opts is not None:
            for o in opts:  # sum over ranks; the average and zero_grad ride inside the fused update
                o.step(grad_mult=o.all_reduce_grads(), zero_grad=True)
        else:
            arena.all_reduce()
        result["loss"] = loss.detach()
        if kept is not None:
            kept.append(step_outputs(out))

    def load_resident(i):
        cur_flat.copy_(resident_flat[i % n_batches], non_blocking=True)

    def prefetch_host(i):
        """Host -> device copy of step i's rays (pinned memory) on the copy stream, into staging buffer i % 2."""
        with torch.cuda.stream(copy_stream):
            staging[i % 2].copy_(host_flat[i % n_batches], non_blocking=True)
            copied[i % 2].record(copy_stream)

    def load_host(i):
        """Step i's rays are on their way (prefetch_host(i)); the step waits for them and takes them over."""
        torch.cuda.current_stream(dev).wait_event(copied[i % 2])
        cur_flat.copy_(staging[i % 2], non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (eager), then capture the step in a CUDA graph
    # (on a side stream, as torch's whole-network capture recipe prescribes: autograd's gradient-accumulation nodes stay
    # bound to the stream they were first used on, and that must be the capturing stream)
    side = torch.cuda.Stream(device=dev, priority=-1)  # above the side streams independent backward branches run on
    load_resident(0)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for i in range(args.warmup):
            step()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    graph, graph_note, launches_per_step = None, "eager launches (--no-graph)", None
    if not args.no_graph:
        try:
            l0 = _lib.launch_count()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                step()
            launches_per_step = _lib.launch_count() - l0
            graph.replay()
            torch.cuda.synchronize()
            graph_note = "one CUDA graph per step (fwd + bwd + collectives), replayed"
        except Exception as e:  # noqa: BLE001 - a capture problem must not cost the measurement
            # a failed capture leaves the CUDA generator and the allocator pool in capture mode: start over without it
            sys.stderr.write(f"bench.py: CUDA graph capture failed ({type(e).__name__}: {str(e)[:200]}); re-running with --no-graph\n")
            sys.stderr.flush()
            if world == 1:
                os.execv(sys.executable, [sys.executable] + sys.argv + ["--no-graph"])
            raise

    def run_step():
        if graph is not None:
            graph.replay()
        else:
            step()

    def timed(loader, steps, read_back):
        """read_back=False: rays resident in HBM.  read_back=True: the end-to-end loop of a training process with a
        prefetching loader - every step's rays are copied from pinned host memory inside the timed region (the copy of
        step i+1 is in flight while step i computes, like a data loader's prefetch), every step's loss is read back."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if read_back:
            prefetch_host(0)
        for i in range(steps):
            loader(i)
            run_step()
            if read_back:
                if i + 1 < steps:
                    prefetch_host(i + 1)
                result["loss"].item()  # device -> host read of the step's result
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    for i in range(2):
        load_resident(i)
        run_step()
    l0 = _lib.launch_count()
    with ClockSampler(local_rank) as clocks:
        ms = timed(load_resident, args.steps, False)
    launches = _lib.launch_count() - l0 if graph is None else launches_per_step * args.steps
    for i in range(2):
        prefetch_host(i)
        load_host(i)
        run_step()
    torch.cuda.synchronize()
    ms_e2e = timed(load_host, args.steps, True)
    if args.dump_outputs and rank == 0:
        # what a caller of the step receives from the last timed one (inference: every chunk's outputs, in ray order)
        outs = result["outs"]
        arrays = {k: torch.cat([o[k] for o in outs]) for k in outs[0]}
        if w.train:
            arrays["loss"] = result["loss"]
            for name, p in used:
                t = p if args.optimizer else p.grad
                if t is not None:
                    arrays[("param." if args.optimizer else "grad.") + name] = t
        dump_outputs(args.dump_outputs, arrays)

    # ---- per-kernel durations from CUDA events on the launching stream (separate eager pass: the events add launch gaps)
    # (the two backward branches are serialised for this pass: overlapped kernels would time each other's contention)
    reps = max(3, min(args.steps, 10))
    overlap, model.sampler.overlap_backward = model.sampler.overlap_backward, False
    _lib.TIMER = _lib.KernelTimer()
    for i in range(reps):
        load_resident(i)
        step()
    kernels = _lib.TIMER.summary()
    _lib.TIMER = None
    model.sampler.overlap_backward = overlap

    peaks = load_peaks()
    total_rays = n * world
    per_step = {name: {"launches_per_step": count / reps, "mean_ms": mean_ms} for name, (count, mean_ms) in kernels.items()}
    # Roofline of every major kernel: algorithmic work per launch (DESIGN.md section 4) / CUDA-event duration.
    #   gathers / scatters: 8 corners x L x F x 4 B per sample, counted once                              -> HBM GB/s
    #   fused field kernels: the gather bytes (fwd) resp. the saved image + masks + d x image streams (bwd) -> HBM GB/s,
    #   and their MLP FLOPs against the tensor peak (reported as `tensor_frac`)
    L, F, T, _, _ = w.main
    S = w.nerf_samples
    passes = (n // (w.chunk or n)) if not w.train else 1
    n_main = n * S / passes
    grid_tag = f"L{L}F{F}T{T}"
    mlp_flop = 2 * (32 * 32 + 32 * 33 + 48 * 32 + 32 * 32 + 32 * 32)
    prop_mean = sum(w.proposal_samples) / len(w.proposal_samples)
    work = {
        "nrb_field_fused_fwd": ("hbm", n_main * 8.0 * L * F * 4, n_main * float(mlp_flop)),
        "nrb_field_fused_bwd": ("hbm", n_main * (128.0 + 12.0 + 128.0 + 4 * 4), n_main * float(mlp_flop) * 2.6),
        f"nrb_hash_bwd:{grid_tag}": ("hbm", n_main * 8.0 * L * F * 4, 0.0),
        f"nrb_hash_fwd:{grid_tag}": ("hbm", n_main * 8.0 * L * F * 4, 0.0),
        "nrb_proposal_fwd": ("hbm", n / passes * prop_mean * 192.0, 0.0),
        "nrb_proposal_bwd": ("hbm", n / passes * prop_mean * 192.0, 0.0),
        "nrb_alpha_composite_fwd": ("hbm", n_main * 32 * 4.0, 0.0),
        "nrb_alpha_composite_bwd": ("hbm", n_main * 32 * 4.0, 0.0),
    }
    if args.optimizer:  # read p, g, m, v + write p, m, v, g = 32 B per parameter, averaged over the two groups' launches
        work["nrb_adam_step"] = ("hbm", arena_bytes / 4 * 32.0 / 2, 0.0)
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            captured = json.load(fh)["kernels"] if args.config == 2 and n == w.rays else {}
    except (OSError, ValueError, KeyError):
        captured = {}
    rooflines = {}
    for name, (bound, amount, flops) in work.items():
        if name not in kernels:
            continue
        mean_ms = kernels[name][1]
        if bound == "hbm":
            achieved, peak, unit = amount / (mean_ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s"
        else:
            achieved, peak, unit = amount / (mean_ms * 1e-3) / 1e12, peaks["tflops"], "TFLOP/s"
        entry = {"kernel": name, "bound": bound, "achieved": achieved, "peak": peak, "unit": unit,
                 "frac": achieved / peak, "traffic": captured.get(name, {}).get("dram_bytes_per_launch"),
                 "traffic_unit": "B (ncu dram read+write per launch, profiles/r2_traffic.json)",
                 "peak_source": peaks["source"], "algorithmic_per_launch": amount, "mean_launch_ms": mean_ms,
                 "ms_per_step": mean_ms * per_step[name]["launches_per_step"]}
        if flops:
            entry["tensor_tflops"] = flops / (mean_ms * 1e-3) / 1e12
            entry["tensor_frac"] = entry["tensor_tflops"] / peaks["tflops"]
        rooflines[name] = entry
    roofline = max(rooflines.values(), key=lambda r: r["ms_per_step"]) if rooflines else None
    path_gbs = n * w.bytes_per_ray() / (ms * 1e-3) / 1e9
    kernel_ms = sum(v["mean_ms"] * v["launches_per_step"] for v in per_step.values())

    line = {
        "metric": METRIC if w.train else "inference_rays_per_sec", "value": total_rays / (ms * 1e-3), "unit": UNIT,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.description, "rays_per_gpu": n, "global_rays": total_rays,
                   "parallelism": (f"ray-sharded dp{world}, all-reduce of a {arena_bytes / 2**20:.0f} MiB gradient arena in two "
                                   "pieces (main table overlapped with the proposal backward); see `collective`") if w.train else f"replicas x{world}",
                   "launch": graph_note,
                   "backward": ("proposal and field backward on two streams" if w.train and model.sampler.overlap_backward and world == 1
                                else "single stream"),
                   "l2": f"{n_batches} resident ray batches rotated; per-step working set (tables 64-512 MiB, saved images, gradient "
                         "arena, > 0.7 GB) exceeds the 126 MB L2; no explicit flush",
                   "optimizer": ("fused Adam (hash grids) + AdamW (MLPs) inside the step" if args.optimizer
                                 else "not part of the path (SURVEY.md 8f next-2; --optimizer adds it)") if w.train else "n/a",
                   "regularisers": bool(args.regularisers)},
        "e2e": {"value": total_rays / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e,
                "note": "per step: one pinned host -> device copy of the rays (prefetched on a copy stream while the previous step "
                        "computes, as a data loader does), the step, loss.item()"},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roofline,
        "rooflines": rooflines,
        "path_roofline": {"bound": "hbm", "bytes_per_ray": w.bytes_per_ray(), "achieved": path_gbs, "peak": peaks["hbm_gbs"],
                          "unit": "GB/s", "frac": path_gbs / peaks["hbm_gbs"],
                          "roofline_rays_per_sec": peaks["hbm_gbs"] * 1e9 / w.bytes_per_ray()},
        "kernels": per_step,
        "kernel_ms_per_step": kernel_ms,
    }
    if world > 1 and arena is not None:
        # the exchange step against NCCL on the same data: fill the arena with a per-rank pattern, reduce it the way the
        # step does (early piece + tail), compare with NCCL's all-reduce of a copy
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        pattern = torch.randn((arena.flat.numel(),), device=dev, generator=gen)
        want = pattern.clone()
        dist.all_reduce(want)
        want /= world
        arena.flat.copy_(pattern)
        torch.cuda.synchronize()
        dist.barrier()
        arena.reducer.start_early()
        arena.all_reduce()
        torch.cuda.synchronize()
        diff = (arena.flat - want).abs().max()
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        kind = "NCCL all-reduce (two communicators)"
        if arena.peer is not None:
            kind = ("own kernel over NVLink peer memory, " +
                    ("in-switch reduction (NVLS multimem)" if arena.peer.multicast_ptr else "unicast two-shot") + ", x 1/world fused")
        line["collective"] = {"kind": kind, "bytes": arena.nbytes, "early_bytes": arena.reducer.n_early * 4,
                              "max_abs_diff_vs_nccl": float(diff)}
    if w.actors:  # how many field samples the actor boxes claimed on this batch (bytes_per_ray assumes ~10 %)
        with torch.no_grad():
            rs = model(bundle(cur))["ray_samples_list"][-1]
            rays_, iv_ = rs.per_ray()
            inside = model.field.hashgrid.assign_actors(rays_, iv_, rs.times.reshape(rays_.num_rays, -1)[:, 0]).grid_id >= 0
        line["config"]["actor_sample_fraction"] = float(inside.float().mean())
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["parity_at_config"] = parity_at_config(model, w, batches_cpu[0])
            except Exception as e:  # noqa: BLE001
                line["parity_at_config"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
            from neuradar_b200.synthetic import WORKLOADS as WL

            # BASELINE.md section 4: the reference torch path on config 1 (4096 radar rays), all host cores
            big = (os.cpu_count() or 1) >= 12
            v, cms, cores, kind, cpu = cpu_reference_run(WL[1] if w.train else w, 4096, 10 if big else 3, 3 if big else 1,
                                                         regularisers=args.regularisers, optimizer=args.optimizer)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu, "ms_per_step": cms,
                                    "sample": (f"BASELINE config 1: 4096 radar rays, {3 if big else 1} warm-up + "
                                               f"{10 if big else 3} timed {'fwd+bwd' if w.train else 'fwd'} iterations")}
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="BASELINE.json configuration")
    ap.add_argument("--rays", type=int, default=0, help="rays per GPU per step (default: the configuration's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--optimizer", action="store_true",
                    help="add the fused Adam / AdamW update (SURVEY.md 8f next-2) to the step of both arms")
    ap.add_argument("--regularisers", action="store_true",
                    help="add the interlevel + distortion losses (SURVEY.md 8f next-1) to the step of both arms")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (and gradients or updated parameters) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of this repo's CUDA path (--impl b200)")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: neuradar_b200 has no CPU path (use --impl reference for the CPU arm)")
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # NCCL prints its version banner on stdout; stdout carries ONE JSON line
        torch.cuda.set_device(local_rank)
        dist.init_process_group(backend="nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
