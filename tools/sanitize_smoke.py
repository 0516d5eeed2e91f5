#!/usr/bin/env python3
"""Small end-to-end pass over every kernel family, sized for compute-sanitizer
(memcheck / racecheck):  compute-sanitizer --tool racecheck python tools/sanitize_smoke.py"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mav_trajectory_generation_cmake_b200 as ms  # noqa: E402

rng = np.random.default_rng(1)
for K, B in ((10, 40), (9, 37), (5, 20), (3, 5), (33, 6), (64, 3), (100, 2)):
    pos = torch.from_numpy(ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 7)).cuda()
    times = ms.estimate_segment_times(pos, 3.0, 5.0)
    ends = torch.from_numpy(rng.normal(size=(B, 2, 4, 3))).cuda()
    out = ms.solve_standard(pos, times, end_derivatives=ends, want_free=True, want_cost=True)
    assert int((out["status"] != 0).sum()) == 0
    if K > 24:
        for which in ("pair_long", "bcr", "chunked"):
            if which == "chunked" and K not in (64,):
                continue
            os.environ["MINSNAP_STANDARD_ROUTE"] = which
            o2 = ms.solve_standard(pos, None, v_max=3.0, a_max=5.0, want_times=True)
            assert torch.isfinite(o2["coeffs"]).all()
        del os.environ["MINSNAP_STANDARD_ROUTE"]
    s = ms.sample_uniform(out["coeffs"], times, 50, 5)
    e = ms.extrema(out["coeffs"], times, 1, mode=1, want_roots=True)
    g = ms.time_gradient(out["coeffs"], times)
    assert torch.isfinite(s).all() and torch.isfinite(e["max_value"]).all() and torch.isfinite(g).all()
    if K == 10:
        sw = ms.cost_sweep(pos, times[:, None, :].repeat(1, 4, 1).contiguous())
        ob = ms.time_objective(pos, times[:, None, :].repeat(1, 4, 1).contiguous(), 500.0)
        mask = ms.standard_mask(K)
        fixed = torch.zeros((B, K + 9, 3), dtype=torch.float64, device="cuda")
        fixed[:, 0] = pos[:, 0]
        fixed[:, 5:5 + K - 1] = pos[:, 1:K]
        fixed[:, 5 + K - 1] = pos[:, K]
        gen = ms.solve(mask, fixed, times)
        assert torch.isfinite(sw).all() and torch.isfinite(ob).all() and torch.isfinite(gen["coeffs"]).all()
# the two-batches-per-warp path of the headline kernel (more than two waves of CTAs), even and odd K
for K in (4, 7):
    B = 2 * 296 * 64 + 70
    pos = torch.from_numpy(ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 9)).cuda()
    out = ms.solve_standard(pos, None, v_max=3.0, a_max=5.0, want_cost=True)
    assert int((out["status"] != 0).sum()) == 0 and torch.isfinite(out["coeffs"]).all()
torch.cuda.synchronize()
print("sanitize smoke OK")
