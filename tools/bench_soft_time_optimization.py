#!/usr/bin/env python3
"""Device-resident time descent with the reference's soft limits on max |velocity| and |acceleration|
(minsnap_optimize_segment_times_soft): milliseconds per iteration from CUDA events, the per-kernel split of an
iteration from a torch.profiler run of its own, the torch-glue driver for comparison, and the rate of
minsnap_time_objective_soft.
    python tools/bench_soft_time_optimization.py [--B 8192 65536] [--iterations 10] [--steps 16] [--out FILE]

Workload: K = 10 (createRandomVertices in the box +-(10, 20, 10), estimateSegmentTimes with v_max 3, a_max 5), the
standard mask, constraints (1, 3.0) and (2, 5.0) (the limits the times were estimated for), the reference's
soft_constraint_weight 100 and maximum cost 1e12, time_penalty 0.05."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mav_trajectory_generation_cmake_b200 as ms  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--B", type=int, nargs="+", default=[8192, 65536])
ap.add_argument("--K", type=int, default=10)
ap.add_argument("--iterations", type=int, default=10)
ap.add_argument("--steps", type=int, default=16)
ap.add_argument("--glue-B", type=int, default=8192)
ap.add_argument("--out", default=None)
a = ap.parse_args()

LIMITS = [(1, 3.0), (2, 5.0)]
PENALTY = 0.05
lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()
say("card: %s" % (card[torch.cuda.current_device()] if card else "unknown"))


def workload(B, K):
    pos = torch.from_numpy(ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 12345)).cuda()
    return pos, ms.estimate_segment_times(pos, 3.0, 5.0)


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


def run(pos, times, iterations):
    return ms.optimize_segment_times_soft(pos, times, LIMITS, iterations=iterations, time_penalty=PENALTY,
                                          n_steps=a.steps)


for B in a.B:
    pos, times = workload(B, a.K)
    t0, _ = timed(lambda: run(pos, times, 0))
    t1, (t_out, hist, peak) = timed(lambda: run(pos, times, a.iterations))
    per_it = (t1 - t0) / a.iterations
    say("B=%d K=%d S=%d: %.3f ms per iteration (%.2f M trajectory-iterations/s); %d iterations %.3f ms, initial "
        "objective and final maxima alone %.3f ms" % (B, a.K, a.steps, per_it, B / per_it / 1e3, a.iterations, t1, t0))
    _, _, peak0 = run(pos, times, 0)
    within = lambda p: float(((p[:, 0] <= 1.05 * LIMITS[0][1]) & (p[:, 1] <= 1.05 * LIMITS[1][1])).double().mean())
    say("    objective mean %.6g -> %.6g; within 1.05x of both limits %.1f%% -> %.1f%%"
        % (float(hist[0].mean()), float(hist[-1].mean()), 100.0 * within(peak0), 100.0 * within(peak)))

    if B == a.glue_B:
        g0, _ = timed(lambda: ms.api.optimize_segment_times_soft_reference_glue(pos, times, LIMITS, iterations=0,
                                                                              time_penalty=PENALTY, n_steps=a.steps), 2)
        g1, _ = timed(lambda: ms.api.optimize_segment_times_soft_reference_glue(pos, times, LIMITS,
                                                                              iterations=a.iterations,
                                                                              time_penalty=PENALTY, n_steps=a.steps), 2)
        say("    torch-glue driver: %.3f ms per iteration" % ((g1 - g0) / a.iterations))

    # per-kernel split of one call of n_it iterations, in a run of its own
    n_it = 5
    run(pos, times, n_it)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(pos, times, n_it)
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
    say("  per-kernel split, B=%d, one call of %d iterations with the initial objective and the final maxima "
        "(profiler, us per iteration):" % (B, n_it))
    for t, count, key in rows[:14]:
        say("    %9.1f us  %5.1f%%  x%-4d %s" % (t / n_it, 100.0 * t / total, count, key[:110]))

# minsnap_time_objective_soft on B x S candidate allocations
B = max(a.B)
pos, times = workload(B, a.K)
scale = torch.linspace(0.8, 1.2, a.steps, dtype=torch.float64, device="cuda")
cand = (times[:, None, :] * scale[None, :, None]).contiguous()
t_obj, obj = timed(lambda: ms.time_objective_soft(pos, cand, PENALTY, LIMITS), 5)
say("time_objective_soft %d x %d: %.3f ms per call = %.1f M objective evaluations/s (%d finite)"
    % (B, a.steps, t_obj, B * a.steps / t_obj / 1e3, int(torch.isfinite(obj).sum())))

if a.out:
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
