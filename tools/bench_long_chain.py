import os, sys, torch
sys.path.insert(0, os.getcwd())
import mav_trajectory_generation_cmake_b200 as ms
K = 256
for B in (296, 512, 1024, 4096, 16384):
    pos = torch.from_numpy(ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 12345)).cuda()
    times = ms.estimate_segment_times(pos, 3.0, 5.0)
    coeffs = torch.empty((B, K, 3, 10), dtype=torch.float64, device="cuda")
    for which in ("bcr", "pair_long", "chunked"):
        os.environ["MINSNAP_STANDARD_ROUTE"] = which
        for _ in range(3): ms.solve_standard(pos, times, coeffs=coeffs, want_status=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20): ms.solve_standard(pos, times, coeffs=coeffs, want_status=False)
        e1.record(); torch.cuda.synchronize()
        print("B=%6d %-8s %8.1f us" % (B, which, e0.elapsed_time(e1) / 20 * 1e3))
