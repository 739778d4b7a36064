"""Step time of the config-4 workload (65 536 rays, 128 field samples, 2^22 main table, --actors dynamic actors, 16 by
default) when the actor trajectories are trained, on three routes:
  kernel  trained poses on the actor kernels (nrb_actor_assign, the fused kernels, nrb_actor_scatter, nrb_actor_pose_grad)
  torch   trained poses on the torch bookkeeping (`can_assign_in_kernel` forced False in all three encodings), which is
          where trained poses ran before the pose gradient kernel existed
  fixed   fixed poses on the actor kernels (what bench.py --config 4 measures)
One step = forward + bench_loss + backward.  Eager for all three, and replayed as one CUDA graph for the two kernel
routes (the torch route synchronises the host and cannot be captured).  CUDA events, `--warmup` steps per measurement,
`--steps` timed steps, `--runs` runs with the routes alternating.  Also recorded, because SyntheticActors spreads its boxes
on a 12 m lattice and at large --actors most of them are far from the synthetic rays: the fraction of the field's samples
inside a box, and the mean time of one nrb_actor_assign launch (torch.profiler, in a pass of its own after the timings).
Writes `actor_pose_step.json` (`actor_pose_step_A<actors>.json` for other counts than 16) to --out.
Usage: python tools/actor_pose_step.py --out /tmp/actor_pose [--actors 64]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuradar_b200 as nb  # noqa: E402
from neuradar_b200.synthetic import WORKLOADS, SyntheticActors, build_hot_path, scaled_pixel_area, synthetic_rays  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True, help="directory that receives actor_pose_step.json")
ap.add_argument("--rays", type=int, default=0)
ap.add_argument("--warmup", type=int, default=10)
ap.add_argument("--steps", type=int, default=50)
ap.add_argument("--runs", type=int, default=3)
ap.add_argument("--actors", type=int, default=16, help="dynamic actors (one grid each)")
args = ap.parse_args()
assert torch.cuda.is_available(), "this measurement needs a CUDA device"
w = WORKLOADS[4]
n = args.rays or w.rays
dev = "cuda"


def build(trainable: bool, torch_route: bool):
    L, F, T, r0, r1 = w.main
    model = build_hot_path(log2_main=T, log2_prop=w.prop_log2, num_proposal_samples=w.proposal_samples,
                           num_nerf_samples=w.nerf_samples, main_levels=L, main_features=F, main_res=(r0, r1), seed=42,
                           device=dev, actors=SyntheticActors(args.actors, device=dev, trainable=trainable))
    model.train()
    if torch_route:
        for h in [model.field.hashgrid] + [p.hashgrid for p in model.proposal_fields]:
            h.can_assign_in_kernel = lambda proposal=False: False
    return model


r = synthetic_rays(n, seed=42, mix=w.mix, device=dev)
r["pixel_area"] = scaled_pixel_area(r)


def make_step(model):
    def step():
        rb = nb.RayBundle(origins=r["origins"].clone(), directions=r["directions"].clone(), pixel_area=r["pixel_area"].clone(),
                          nears=r["nears"].clone(), fars=r["fars"].clone(), times=r["times"],
                          metadata={"is_lidar": r["is_lidar"], "is_radar": r["is_radar"]})
        nb.bench_loss(model(rb)).backward()
    return step


routes = {"kernel": build(True, False), "torch": build(True, True), "fixed": build(False, False)}
steps, graphs = {}, {}
for name, model in routes.items():
    step = make_step(model)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            model.zero_grad(set_to_none=True)
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()

    def eager(model=model, step=step):
        model.zero_grad(set_to_none=True)
        step()

    steps[name] = eager
    if name != "torch":
        model.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            step()
        graphs[name] = g
torch.cuda.synchronize()
# the trained routes compute pose gradients; the kernel route's agree with the torch route's (on the same jitter and
# mirror draws: both routes draw them in the same order)
pose = {}
for name in ("kernel", "torch"):
    torch.manual_seed(1234)
    steps[name]()
    pose[name] = [p.grad.detach().clone() for p in routes[name].field.hashgrid.actors.parameters()]
pose_rel = [float((a - b).abs().max() / b.abs().max()) for a, b in zip(pose["kernel"], pose["torch"])]


def timed(fn):
    for _ in range(args.warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.steps


cases = [(f"{k} eager", steps[k]) for k in routes] + [(f"{k} graph", graphs[k].replay) for k in graphs]
result = {k: [] for k, _ in cases}
for run in range(args.runs):
    order = cases if run % 2 == 0 else cases[::-1]
    for k, fn in order:
        result[k].append(round(timed(fn), 4))
# samples of the field inside actor boxes: the field's own assignment of one kernel-route forward
inside = {}
field = routes["kernel"].field.hashgrid
assign = field.assign_actors


def counting_assign(rays, iv, times):
    batch = assign(rays, iv, times)
    inside["fraction"] = float((batch.grid_id >= 0).float().mean())
    return batch


field.assign_actors = counting_assign
torch.manual_seed(1234)
steps["kernel"]()
field.assign_actors = assign
# per-launch time of the assignment kernel (all three encodings' launches of a kernel-route step)
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(5):
        steps["kernel"]()
    torch.cuda.synchronize()
assign_us = [e for e in prof.key_averages() if "actor_assign_kernel" in e.key]
assign_launch_us = round(assign_us[0].device_time_total / assign_us[0].count, 2) if assign_us else None
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
line = {
    "workload": (w.description.replace(f"{w.actors} dynamic actors", f"{args.actors} dynamic actors")
                 + ", actor trajectories trained (SyntheticActors(trainable=True))"),
    "actors": args.actors,
    "field_samples_in_boxes": round(inside.get("fraction", float("nan")), 5),
    "nrb_actor_assign_us_per_launch": assign_launch_us,
    "card": q[0] if q else torch.cuda.get_device_name(),
    "ms_per_step": {k: v for k, v in result.items()},
    "pose_grad_kernel_vs_torch_route_max_rel": pose_rel,
    "timing": f"CUDA events, {args.warmup} warm-up + {args.steps} timed steps per measurement, {args.runs} runs alternating",
}
os.makedirs(args.out, exist_ok=True)
name = "actor_pose_step.json" if args.actors == 16 else f"actor_pose_step_A{args.actors}.json"
with open(os.path.join(args.out, name), "w") as fh:
    json.dump(line, fh, indent=1)
print(json.dumps(line))
