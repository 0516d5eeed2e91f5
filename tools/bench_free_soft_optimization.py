#!/usr/bin/env python3
"""Device-resident descent on the free derivatives against the collision cost plus the soft velocity and
acceleration limits (minsnap_optimize_free_constraints_soft), next to the collision-only driver
(minsnap_optimize_free_constraints): milliseconds per iteration from CUDA events, the per-kernel split of an
iteration from a torch.profiler run of its own, and, after the iterations, the share of trajectories in collision and
the share within 1.05x of both limits.
    python tools/bench_free_soft_optimization.py [--B 8192 65536] [--iterations 20] [--steps 8] [--out FILE]

Workload: that of tools/bench_free_constraint_optimization.py (K = 10, the standard mask started at the QP optimum,
the sphere of radius 3 at (1, -2, 0.5) on a 48 x 88 x 48 grid of 0.5 m, w_d = 0.1, w_c = 10, w_t = 1, times fixed),
with two soft limits, velocity 3 m/s and acceleration 5 m/s^2, the reference's weight 100 and maximum cost 1e12, and
w_sc = 1."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mav_trajectory_generation_cmake_b200 as ms  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, nargs="+", default=[8192, 65536])
ap.add_argument("--K", type=int, default=10)
ap.add_argument("--iterations", type=int, default=20)
ap.add_argument("--steps", type=int, default=8)
ap.add_argument("--out", default=None)
a = ap.parse_args()

lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()
say("card: %s" % (card[torch.cuda.current_device()] if card else "unknown"))

ORIGIN, RES, DIMS = np.array([-12.0, -22.0, -12.0]), 0.5, (48, 88, 48)
ax = [ORIGIN[k] + (np.arange(DIMS[k]) + 0.5) * RES for k in range(3)]
X, Y, Z = np.meshgrid(*ax, indexing="ij")
sdf = torch.from_numpy(np.sqrt((X - 1.0) ** 2 + (Y + 2.0) ** 2 + (Z - 0.5) ** 2) - 3.0).cuda()
MAP = dict(origin=ORIGIN, resolution=RES, min_bound=[-10.0, -20.0, -10.0], max_bound=[10.0, 20.0, 10.0], dt=0.1,
           map_resolution=RES, epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.5, oob_value=10.0)
W = dict(w_c=10.0, w_d=0.1, w_t=1.0)
CONS = [(1, 3.0), (2, 5.0)]
W_SC = 1.0


def workload(B, K):
    mask = ms.standard_mask(K)
    pos = ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 12345)
    vals = np.zeros((B, K + 1, 5, 3))
    vals[:, :, 0] = pos
    fixed = torch.from_numpy(np.ascontiguousarray(vals[:, mask.astype(bool)])).cuda()
    times = ms.estimate_segment_times(torch.from_numpy(pos).cuda(), 3.0, 5.0)
    free = ms.solve(mask, fixed, times)["free_values"]
    return mask, fixed, free, times


def run(args, iterations, soft):
    kw = dict(iterations=iterations, n_steps=a.steps, **W, **MAP)
    if soft:
        return ms.optimize_free_constraints_soft(*args, sdf, constraints=CONS, w_sc=W_SC, **kw)
    return ms.optimize_free_constraints(*args, sdf, **kw)


def timed(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


lim = torch.tensor([v for _, v in CONS], dtype=torch.float64, device="cuda")
for B in a.B:
    args = workload(B, a.K)
    c0 = ms.coeffs_from_constraints(args[0], args[1], args[2], args[3])
    peak0 = ms.soft_constraint_cost(c0, args[3], CONS, want_terms=True)[1]["max_value"]
    hit0 = ms.collision_cost(c0, args[3], sdf, **MAP)["is_collision"]
    say("B=%d K=%d S=%d: at the start %.3f in collision, %.3f within 1.05x of both limits"
        % (B, a.K, a.steps, float(hit0.double().mean()), float((peak0 <= 1.05 * lim).all(1).double().mean())))
    for soft in (False, True):
        t0, _ = timed(lambda: run(args, 0, soft))
        t1, out = timed(lambda: run(args, a.iterations, soft))
        free, times, hist, hit = out[:4]
        per_it = (t1 - t0) / a.iterations
        peak = ms.soft_constraint_cost(ms.coeffs_from_constraints(args[0], args[1], free, times), times, CONS,
                                       want_terms=True)[1]["max_value"]
        say("  %-15s %.3f ms per iteration; after %d iterations %.3f in collision, %.3f within 1.05x of both limits"
            % ("soft + collision" if soft else "collision only", per_it, a.iterations, float(hit.double().mean()),
               float((peak <= 1.05 * lim).all(1).double().mean())))

    # per-kernel split of one call of 5 iterations of the new driver, in a run of its own
    n_it = 5
    run(args, n_it, True)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(args, n_it, True)
        torch.cuda.synchronize()
    rows = []
    for ev in prof.key_averages():
        t = getattr(ev, "self_device_time_total", None)
        if t is None:
            t = ev.self_cuda_time_total
        if t > 0:
            rows.append((t, ev.count, ev.key))
    rows.sort(reverse=True)
    total = sum(r[0] for r in rows)
    say("  per-kernel split, B=%d, soft + collision, one call of %d iterations and the initial objective (profiler, "
        "us per iteration):" % (B, n_it))
    for t, count, key in rows[:14]:
        say("    %9.1f us  %5.1f%%  x%-4d %s" % (t / n_it, 100.0 * t / total, count, key[:110]))

if a.out:
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
