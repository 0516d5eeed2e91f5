#!/usr/bin/env python3
"""bench.py -- headline benchmark: min-snap solves/s (3-D, N=10, 10 segments) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--skip-configs] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (setup + solveLinear, SURVEY.md section 8a rows a9-a13)
over one batch of 65,536 synthetic trajectories PER GPU (BASELINE.json configs[1]; weak
scaling, the batch shards by trajectory with no data-path collective).  Inputs (positions,
segment times) are resident in HBM when the timed region starts; coefficients land in HBM.

Timed region: after W eager warm-up steps the K steps are captured into ONE CUDA graph (K
launches of the solve kernel through the C ABI, rotating over buffer sets larger than L2),
the graph is replayed once untimed and once between two CUDA events.  The host therefore
issues one launch per timed region and a host hiccup on one of N ranks cannot stretch the
device time (round 1: 20 Python launches in a 1.2 ms window, MAX over 8 ranks -> 0.68
efficiency under the driver's --steps 20).  Every rank's time is gathered and reported.

Printed JSON line (rank 0): value = whole-job solves/s, roofline (HBM, algorithmic 2,744 B per
solve), cpu_baseline (the oracle port on this box's host cores, bounded sample), e2e (same
metric through the host-buffer C-ABI call with pinned host memory, copies inside, against the
box's measured concurrent pinned-copy rate), clocks, parity, and `configs`: BASELINE.json
configs[2..4] and the strong-scaling target at full size, sharded over the N ranks, each with
its own time, roofline fraction and oracle parity.

--impl reference: the reference's CPU path.  The reference itself cannot be compiled in this
image (Eigen3/glog/NLopt absent), so this arm times the oracle port of its algorithm (dense
Householder QR in place of Eigen::SparseQR) with all host threads.  It never imports the
product package.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "min-snap solves/sec (3D, N=10, 10 seg)"
UNIT = "solves/s"
B_PER_GPU = 65536
K_SEG, DIM, NCOEF, SNAP = 10, 3, 10, 4
V_MAX, A_MAX, MAGIC = 3.0, 5.0, 6.5
BOX_LO, BOX_HI = [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0]
BASE_SEED = 12345
L2_BYTES = 126e6
# --dump-outputs writes the coefficients of a fixed sample of the batch: 16,384 x 10 x 3 x 10 doubles = 39 MB
DUMP_ROWS, DUMP_SEED = 16384, 20261020


def bytes_in(K):
    return 8 * ((K + 1) * DIM + K)        # positions + segment times


def bytes_out(K):
    return 8 * K * DIM * NCOEF            # coefficients


def flops_solve(K, D=DIM):                # SURVEY 8(d): F_solve(K, D)
    return K * (95 + 132 * D) + (K - 1) * (160 + 96 * D)


def flops_cost(K, D=DIM):                 # SURVEY 8(d): F_cost(K, D)
    return K * (95 + 32 * D + 200 * D) + (K - 1) * (160 + 96 * D)


BYTES_IN, BYTES_OUT = bytes_in(K_SEG), bytes_out(K_SEG)            # 344 B, 2400 B
BYTES_PER_SOLVE = BYTES_IN + BYTES_OUT                             # 2744 B algorithmic HBM traffic
FLOPS_PER_SOLVE = flops_solve(K_SEG)                               # 8942
# identical in both arms (the driver compares the dicts)
CONFIG = {"workload": "configs[1]: batch of 65,536 independent 3-D N=10 min-snap problems, 10 segments each, per GPU",
          "batch_per_gpu": B_PER_GPU, "segments": K_SEG, "dimension": DIM, "N": NCOEF, "derivative": "snap",
          "inputs": "createRandomVertices(seed=12345+b, box +-(10,20,10)) + estimateSegmentTimes(3,5,6.5)",
          "l2": "GPU arm: inputs/outputs rotate over buffer sets whose cycle exceeds the 126 MB L2",
          "parallelism": "trajectory-sharded over the ranks, no data-path collective",
          "status_word": "the timed step does not store the per-problem status word (4 B/solve)"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class Clocks:
    """SM clock and throttle reasons through NVML, sampled from the calling thread only (no sampler
    thread competes with the launch path): one sample while the timed graph runs and a run of
    samples every 10 ms while the same graph is replayed as a load probe right after it."""

    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples, self.reasons, self.timed_samples, self.mem_mhz = [], set(), 0, None
        self.max_mhz, self.h, self.nv = None, None, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            # NVML indexes physical devices: honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    index = int(ids[index])
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as exc:  # NVML missing: report that instead of inventing numbers
            self.reasons.add("nvml_unavailable: %s" % type(exc).__name__)

    def sample(self, timed=False):
        if self.h is None:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.NAMES.items():
                if mask & bit:
                    self.reasons.add(name)
            if timed:
                self.timed_samples += 1
                try:
                    self.mem_mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_MEM)
                except Exception:
                    pass
        except Exception as exc:
            self.reasons.add("nvml_error: %s" % type(exc).__name__)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "mem_mhz_in_timed_region": self.mem_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "samples_inside_timed_region": self.timed_samples,
                "how": "NVML from the main thread: inside the timed graph replay and every 10 ms during a load probe "
                       "(the same graph replayed for >= 0.2 s) right after it"}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def dump_rows(batch):
    """The trajectories whose outputs --dump-outputs writes: a seeded sample of the batch, in increasing order."""
    rng = np.random.default_rng(DUMP_SEED)
    return np.sort(rng.choice(batch, size=min(DUMP_ROWS, batch), replace=False))


def coeff_rel_err(c, ref):
    """Per-polynomial max-norm relative error (SURVEY 8d ii), worst polynomial."""
    ref = np.asarray(ref, np.float64)
    num = np.abs(np.asarray(c, np.float64) - ref).max(axis=-1)
    den = np.abs(ref).max(axis=-1)
    return float((num / np.where(den == 0, 1.0, den)).max())


# ------------------------------------------------------------------------------------------
# CPU arm: oracle port of the reference algorithm (test infrastructure used as the baseline)
# ------------------------------------------------------------------------------------------
def oracle_inputs(orc, B, K, seed_base):
    pos = np.stack([orc.create_random_positions(K, BOX_LO, BOX_HI, seed_base + b) for b in range(B)])
    times = np.stack([orc.estimate_segment_times(pos[b], V_MAX, A_MAX, MAGIC) for b in range(B)])
    return pos, times


def cpu_solves_per_s(positions, times, n_threads, budget_s):
    """Times the oracle on a bounded sample of the workload; returns (solves/s, sample size, 1-thread solves/s)."""
    from oracle.oracle_py import Oracle
    orc = Oracle("f64")
    probe = 256
    t0 = time.perf_counter()
    orc.solve_batch_standard(positions[:probe], times[:probe], NCOEF, SNAP, 4, 1, want_coeffs=True)
    per_solve_1t = (time.perf_counter() - t0) / probe
    sample = int(min(len(positions), max(1024, budget_s / per_solve_1t)))
    orc.solve_batch_standard(positions[:n_threads * 64], times[:n_threads * 64], NCOEF, SNAP, 4, n_threads)
    best = 0.0
    for _ in range(3):
        t0 = time.perf_counter()
        _, _, st = orc.solve_batch_standard(positions[:sample], times[:sample], NCOEF, SNAP, 4, n_threads)
        dt = time.perf_counter() - t0
        best = max(best, sample / dt)
        assert st == 0
    return best, sample, 1.0 / per_solve_1t


def ld_truth_coeffs(pos, times, K):
    """Long-double build of the same oracle: the extended-precision truth for a few problems."""
    from oracle.oracle_py import Oracle, standard_mask, vertex_values_from_positions
    ld = Oracle("ld")
    mask = standard_mask(K, NCOEF)
    out = []
    for b in range(len(pos)):
        r = ld.solve(NCOEF, K, DIM, SNAP, mask, vertex_values_from_positions(pos[b], NCOEF), times[b])
        out.append((np.asarray(r["coeffs"], np.float64), float(r["cost"])))
    return out


def parity_block(ms, torch, pos_h, times_h, n_threads, n_check=4096, n_truth=256):
    """SURVEY 8(d): parity checks run with every benchmark -- the CUDA path against the oracle on a
    random subset of the benchmark batch (coefficients, cost, sampled derivatives, index map), and both
    against the long-double build of the oracle on a smaller subset (which side owns the distance)."""
    from oracle.oracle_py import Oracle, standard_mask
    orc = Oracle("f64")
    rng = np.random.default_rng(20261018)
    idx = np.sort(rng.choice(len(pos_h), size=min(n_check, len(pos_h)), replace=False))
    p, t = np.ascontiguousarray(pos_h[idx]), np.ascontiguousarray(times_h[idx])
    ref_c, ref_cost, st = orc.solve_batch_standard(p, t, NCOEF, SNAP, 4, n_threads)
    out = ms.solve_standard(torch.from_numpy(p).cuda(), torch.from_numpy(t).cuda(), want_cost=True)
    c = out["coeffs"].cpu().numpy()
    coeff_err = coeff_rel_err(c, ref_c)
    cost_err = float(np.abs(out["cost"].cpu().numpy() / ref_cost - 1.0).max())
    n_s = 64
    samples, ts = ms.sample_uniform(out["coeffs"][:n_s], torch.from_numpy(t[:n_s]).cuda(), 128, 5, want_times=True)
    samples, ts = samples.cpu().numpy(), ts.cpu().numpy()
    sample_err = max(float(np.abs(samples[b] - orc.trajectory_sample(ref_c[b], t[b], ts[b], 5)).max())
                     for b in range(n_s))
    mask = standard_mask(K_SEG, NCOEF)
    col_ref, nf, npf = orc.reorder(NCOEF, K_SEG, mask)
    col, counts = ms.reorder(torch.from_numpy(mask.reshape(1, -1)).cuda(), NCOEF, K_SEG)
    index_ok = bool(np.array_equal(col.cpu().numpy()[0], col_ref)) and tuple(counts.cpu().numpy()[0]) == (nf, npf)
    truth = ld_truth_coeffs(p[:n_truth], t[:n_truth], K_SEG)
    truth_c = np.stack([x[0] for x in truth])
    gpu_vs_truth = coeff_rel_err(c[:n_truth], truth_c)
    oracle_vs_truth = coeff_rel_err(ref_c[:n_truth], truth_c)
    ok = st == 0 and int((out["status"] != 0).sum()) == 0 and coeff_err <= 1e-8 and cost_err <= 1e-8 and \
        sample_err <= 1e-6 and index_ok
    return {"ok": bool(ok), "n_checked": int(len(idx)), "coeff_rel_err": coeff_err, "cost_rel_err": cost_err,
            "sample_abs_err": sample_err, "index_map_bit_exact": index_ok,
            "long_double_truth": {"n": int(len(truth)), "gpu_coeff_rel_err": gpu_vs_truth,
                                  "f64_oracle_coeff_rel_err": oracle_vs_truth,
                                  "note": "distance of each side from the long-double build of the oracle: the "
                                          "reference-order f64 arithmetic (A^-T Q A^-1) owns the GPU-vs-oracle gap"},
            "bars": {"coeff_rel_err": 1e-8, "cost_rel_err": 1e-8, "sample_abs_err": 1e-6}}


def run_reference_arm(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    from oracle.oracle_py import Oracle   # the oracle has its own bit-identical input generator
    cores = os.cpu_count() or 1
    orc = Oracle("f64")
    # size one step so that warmup + steps finish within a few minutes
    probe = 256
    pos, times = oracle_inputs(orc, probe, K_SEG, BASE_SEED)
    t0 = time.perf_counter()
    orc.solve_batch_standard(pos, times, NCOEF, SNAP, 4, 1)
    per_solve = (time.perf_counter() - t0) / probe
    budget_per_step = min(10.0, 120.0 / max(1, args.steps + args.warmup))
    sample = int(min(B_PER_GPU, max(512, budget_per_step * cores / per_solve)))
    pos, times = oracle_inputs(orc, sample, K_SEG, BASE_SEED)
    for _ in range(args.warmup):
        orc.solve_batch_standard(pos, times, NCOEF, SNAP, 4, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.solve_batch_standard(pos, times, NCOEF, SNAP, 4, cores)
    elapsed = time.perf_counter() - t0
    value = sample * args.steps / elapsed
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": CONFIG,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d of the 65,536 problems per step; oracle port of the reference algorithm "
                                   "(dense Householder QR for Eigen::SparseQR), OpenMP over problems" % sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference needs Eigen3/glog/NLopt, absent from this image: its algorithm is timed through the oracle port",
    }
    emit(line)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def bind_to_gpu_cpus(local):
    """Run this rank on the host cores (and so allocate its pinned buffers on the NUMA node) next to
    its GPU: with 8 ranks on a two-socket host the e2e copies otherwise cross the socket link."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + bit for w, mask in enumerate(words) for bit in range(64) if (mask >> bit) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class Ranks:
    """The torch.distributed plumbing of the bench: barrier, max over ranks, gather of per-rank times."""

    def __init__(self, torch, dist, world):
        self.torch, self.dist, self.world = torch, dist, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def all_ms(self, ms_local):
        if self.world == 1:
            return [float(ms_local)]
        t = self.torch.tensor([ms_local], dtype=self.torch.float64, device="cuda")
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x.item()) for x in out]

    @staticmethod
    def spread(all_ms, per=1.0):
        a = np.asarray(all_ms, np.float64) / per
        return {"min": float(a.min()), "median": float(np.median(a)), "max": float(a.max())}


def timed_steps(torch, ranks, launch, steps, warmup, clocks=None, probe_s=0.0):
    """W eager warm-up launches, then `steps` launches timed as ONE CUDA-graph replay between two CUDA
    events (an untimed replay first).  Falls back to an eager loop when capture is not possible (a path
    that allocates stream-ordered scratch).  Returns (per-rank elapsed ms list, mode)."""
    for i in range(warmup):
        launch(i)
    torch.cuda.synchronize()
    graph, mode = None, "cuda_graph"
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for i in range(steps):
                launch(warmup + i)
        # Untimed replays for ~8 ms (at least one).  This is a burst measurement, like the driver-written peaks it is
        # compared with, taken on a GPU that is awake: after an idle second the first replay can still read 42.3 us per
        # step, 5-50 ms of work later a step takes 41.3-41.5 us every time, from ~100 ms of continuous load on 42.4 us
        # and under seconds of it 44 us at the 1 kW power cap (tools/warmup_curve.py, tools/sustained_load.py).
        t_w = time.perf_counter()
        g.replay()
        torch.cuda.synchronize()
        while time.perf_counter() - t_w < 0.008:
            g.replay()
            if clocks is not None:
                # the first NVML clock / event-reason reads of a process take milliseconds and cost the kernels
                # running beside them ~1 us per step (tools/nvml_perturbation.py); later reads do not: they are made
                # here, under the same load, so that the read inside the timed window is not the first one
                clocks.sample()
            torch.cuda.synchronize()
        graph = g
    except Exception as exc:
        mode = "eager (graph capture failed: %s)" % type(exc).__name__
        torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ranks.barrier()
    torch.cuda.synchronize()
    # A spin kernel of ~0.3 ms goes first: while it runs the host enqueues the start event, the graph and the stop
    # event, so that the first timed kernel starts right behind the start event.  Without it the window opened on an
    # idle GPU and contained the host's graph-submission latency (10-40 us, more with several ranks sharing the
    # host: 41.4 us per step at N = 1 against 43.1 us per rank at N = 2 on the same box).
    torch.cuda._sleep(600_000)
    ev0.record()
    if graph is not None:
        graph.replay()
    else:
        for i in range(steps):
            launch(warmup + i)
    ev1.record()
    if clocks is not None:
        # the read is made once the start event has fired (the host polls it through the spin kernel) and counts
        # as inside the window only if the stop event has not fired when it returns
        while not ev0.query():
            pass
        clocks.sample(timed=True)
        if ev1.query():
            clocks.timed_samples -= 1
    torch.cuda.synchronize()
    elapsed = ev0.elapsed_time(ev1)
    ranks.barrier()
    if clocks is not None and probe_s > 0:
        # load probe: the same work, untimed, with the clocks sampled every 10 ms from this thread
        t_end = time.perf_counter() + probe_s
        while time.perf_counter() < t_end:
            if graph is not None:
                graph.replay()
            else:
                for i in range(steps):
                    launch(i)
            time.sleep(0.01)
            clocks.sample()
        torch.cuda.synchronize()
    return ranks.all_ms(elapsed), mode


def n_buffer_sets(bytes_per_set):
    """Rotate over enough buffer sets that a step never finds its inputs (or its previous outputs) in L2."""
    return max(2, int(np.ceil(2.1 * L2_BYTES / max(1, bytes_per_set))))


def solve_workload(ms, torch, pos_h, K, n_sets):
    pos_d = [torch.from_numpy(pos_h).cuda() for _ in range(n_sets)]
    times_d = [ms.estimate_segment_times(p, V_MAX, A_MAX, MAGIC) for p in pos_d]
    coeffs_d = [torch.empty((pos_h.shape[0], K, DIM, NCOEF), dtype=torch.float64, device="cuda") for _ in range(n_sets)]
    torch.cuda.synchronize()

    def launch(i):
        s = i % n_sets
        ms.solve_standard(pos_d[s], times_d[s], coeffs=coeffs_d[s], want_status=False)

    return pos_d, times_d, coeffs_d, launch


def config_target(ms, torch, ranks, rank, world, args, hbm_peak, fp64_peak, cores):
    """north_star Target: 65,536 problems IN TOTAL on the N GPUs (strong scaling: 65,536 / N per rank)."""
    total = B_PER_GPU
    b = total // world
    pos_h = ms.random_positions_host(b, K_SEG, BOX_LO, BOX_HI, BASE_SEED + rank * b)
    n_sets = n_buffer_sets(b * BYTES_PER_SOLVE)
    pos_d, times_d, coeffs_d, launch = solve_workload(ms, torch, pos_h, K_SEG, n_sets)
    all_ms, mode = timed_steps(torch, ranks, launch, args.steps, args.warmup)
    ms_step = max(all_ms) / args.steps
    out = {"shape": "65,536 problems in total, %d per GPU (strong scaling)" % b, "scaling": "strong",
           "ms": ms_step, "value": total / (ms_step * 1e-3), "unit": UNIT, "timed_loop": mode, "buffer_sets": n_sets,
           "per_rank_ms": Ranks.spread(all_ms, args.steps),
           "roofline": {"bound": "hbm", "achieved": BYTES_PER_SOLVE * b / (ms_step * 1e-3) / 1e9, "peak": hbm_peak,
                        "unit": "GB/s", "frac": BYTES_PER_SOLVE * b / (ms_step * 1e-3) / 1e9 / hbm_peak,
                        "fp64_frac": FLOPS_PER_SOLVE * b / (ms_step * 1e-3) / 1e12 / fp64_peak,
                        "note": "per GPU; %d trajectories = %d warps of 16 on 148 SMs" % (b, (b + 15) // 16)}}
    if rank == 0:
        from oracle.oracle_py import Oracle
        n = min(256, b)
        ref_c, _, st = Oracle("f64").solve_batch_standard(pos_h[:n], times_d[0][:n].cpu().numpy(), NCOEF, SNAP, 4, cores)
        launch(0)
        err = coeff_rel_err(coeffs_d[0][:n].cpu().numpy(), ref_c)
        out["parity"] = {"ok": bool(st == 0 and err <= 1e-8), "n_checked": n, "coeff_rel_err": err}
    return out


def config_sampling(ms, torch, ranks, rank, world, hbm_peak, cores):
    """configs[2]: 1M solved 10-segment trajectories x 1,000 instants, position..snap, sharded by trajectory;
    the 120 GB of samples do not stay: each rank streams them through two rotating 7.9 GB chunk buffers."""
    total, M, chunk = 1 << 20, 1000, 65536
    b = total // world
    pos_h = ms.random_positions_host(b, K_SEG, BOX_LO, BOX_HI, BASE_SEED + rank * b)
    pos_d = torch.from_numpy(pos_h).cuda()
    times_d = ms.estimate_segment_times(pos_d, V_MAX, A_MAX, MAGIC)
    coeffs_d = ms.solve_standard(pos_d, times_d, want_status=False)["coeffs"]
    bufs = [torch.empty((chunk, M, 5, DIM), dtype=torch.float64, device="cuda") for _ in range(2)]
    n_chunks = (b + chunk - 1) // chunk

    def one_pass():
        for c in range(n_chunks):
            lo, hi = c * chunk, min(b, (c + 1) * chunk)
            ms.sample_uniform(coeffs_d[lo:hi], times_d[lo:hi], M, 5, out=bufs[c % 2][: hi - lo])

    one_pass()
    torch.cuda.synchronize()
    reps = 3
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ranks.barrier()
    ev0.record()
    for _ in range(reps):
        one_pass()
    ev1.record()
    torch.cuda.synchronize()
    all_ms = ranks.all_ms(ev0.elapsed_time(ev1))
    ms_pass = max(all_ms) / reps
    sps = total * M / (ms_pass * 1e-3)
    out = {"shape": "1,048,576 trajectories x 1,000 instants x (pos..snap) x 3 in total, %d trajectories per GPU, "
                    "%d chunks of <= 65,536 per pass" % (b, n_chunks),
           "ms": ms_pass, "value": sps, "unit": "samples/s", "launches_per_pass": n_chunks,
           "per_rank_ms": Ranks.spread(all_ms, reps),
           "roofline": {"bound": "hbm", "achieved": sps / world * 120.0 / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": sps / world * 120.0 / 1e9 / hbm_peak,
                        "note": "per GPU; 120 B written per sample (15 doubles), coefficient reads negligible"}}
    if rank == 0:
        from oracle.oracle_py import Oracle
        orc = Oracle("f64")
        n = min(256, b)
        t_h = times_d[:n].cpu().numpy()
        ref_c, _, st = orc.solve_batch_standard(pos_h[:n], t_h, NCOEF, SNAP, 4, cores)
        smp, ts = ms.sample_uniform(coeffs_d[:n], times_d[:n], M, 5, want_times=True)
        smp, ts, c_gpu = smp.cpu().numpy(), ts.cpu().numpy(), coeffs_d[:n].cpu().numpy()
        same_c = max(float(np.abs(smp[i] - orc.trajectory_sample(c_gpu[i], t_h[i], ts[i], 5)).max()) for i in range(n))
        e2e = max(float(np.abs(smp[i] - orc.trajectory_sample(ref_c[i], t_h[i], ts[i], 5)).max()) for i in range(n))
        out["parity"] = {"ok": bool(st == 0 and same_c <= 1e-6 and e2e <= 1e-6), "n_checked": n, "instants": M,
                         "sample_abs_err_same_coefficients": same_c, "sample_abs_err_oracle_solve_and_sample": e2e,
                         "bar": 1e-6}
    del bufs, coeffs_d
    return out


def config_long_horizon(ms, torch, ranks, rank, world, args, hbm_peak, fp64_peak, cores):
    """configs[3]: 4,096 trajectories x 256 segments, 4,096 / N per rank."""
    total, K = 4096, 256
    b = total // world
    pos_h = ms.random_positions_host(b, K, BOX_LO, BOX_HI, BASE_SEED + rank * b)
    per = bytes_in(K) + bytes_out(K)
    n_sets = n_buffer_sets(b * per)
    pos_d, times_d, coeffs_d, launch = solve_workload(ms, torch, pos_h, K, n_sets)
    all_ms, mode = timed_steps(torch, ranks, launch, args.steps, args.warmup)
    ms_step = max(all_ms) / args.steps
    out = {"shape": "4,096 trajectories x 256 segments in total, %d per GPU" % b, "ms": ms_step,
           "value": total / (ms_step * 1e-3), "unit": UNIT, "timed_loop": mode, "buffer_sets": n_sets,
           "per_rank_ms": Ranks.spread(all_ms, args.steps),
           "roofline": {"bound": "hbm", "achieved": per * b / (ms_step * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": per * b / (ms_step * 1e-3) / 1e9 / hbm_peak,
                        "fp64_frac": flops_solve(K) * b / (ms_step * 1e-3) / 1e12 / fp64_peak,
                        "note": "per GPU; dependency-chain bound (255 block rows): both fractions reported"}}
    if rank == 0:
        from oracle.oracle_py import Oracle
        n = min(max(16, 2 * cores), b, 64)   # the dense-QR oracle needs ~1.6 core-seconds per K=256 problem
        t_h = times_d[0][:n].cpu().numpy()
        ref_c, ref_cost, st = Oracle("f64").solve_batch_standard(pos_h[:n], t_h, NCOEF, SNAP, 4, cores)
        launch(0)
        err = coeff_rel_err(coeffs_d[0][:n].cpu().numpy(), ref_c)
        out["parity"] = {"ok": bool(st == 0 and err <= 1e-8), "n_checked": n, "coeff_rel_err": err,
                         "note": "n bounded by the oracle's dense 1020 x 1020 QR (1.6 core-seconds per problem)"}
    return out


def config_time_sweep(ms, torch, ranks, rank, world, args, hbm_peak, fp64_peak, cores):
    """configs[4]: 8,192 trajectories x 64 perturbed segment-time allocations, cost only, split by trajectory."""
    total, S = 8192, 64
    b = total // world
    pos_h = ms.random_positions_host(b, K_SEG, BOX_LO, BOX_HI, BASE_SEED + rank * b)
    pos_d = torch.from_numpy(pos_h).cuda()
    base = ms.estimate_segment_times(pos_d, V_MAX, A_MAX, MAGIC)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(977 + rank)
    factor = 0.75 + 0.5 * torch.rand((b, S, K_SEG), dtype=torch.float64, device="cuda", generator=gen)
    factor[:, 0, :] = 1.0
    times_d = (base[:, None, :] * factor).contiguous()
    cost_d = torch.empty((b, S), dtype=torch.float64, device="cuda")
    lib, api = ms.capi.load(), ms.api

    def launch(i):
        ms.capi.check(lib.minsnap_cost_sweep(b, S, K_SEG, DIM, NCOEF, SNAP, api._dptr(pos_d), None, api._dptr(times_d),
                                             api._dptr(cost_d), None, api._stream()), "minsnap_cost_sweep")

    all_ms, mode = timed_steps(torch, ranks, launch, args.steps, args.warmup)
    ms_step = max(all_ms) / args.steps
    evals = total * S
    out = {"shape": "8,192 trajectories x 64 time allocations in total, %d trajectories per GPU, cost only" % b,
           "ms": ms_step, "value": evals / (ms_step * 1e-3), "unit": "cost evaluations/s", "timed_loop": mode,
           "per_rank_ms": Ranks.spread(all_ms, args.steps),
           "roofline": {"bound": "fp64", "achieved": flops_cost(K_SEG) * b * S / (ms_step * 1e-3) / 1e12,
                        "peak": fp64_peak, "unit": "TFLOP/s",
                        "frac": flops_cost(K_SEG) * b * S / (ms_step * 1e-3) / 1e12 / fp64_peak,
                        "note": "per GPU; 11,942 flop per evaluation (SURVEY 8d); peak = measured DFMA loop; the "
                                "working set (%.1f MB) is L2-resident by construction" % (b * S * 88 / 1e6)}}
    if rank == 0:
        from oracle.oracle_py import Oracle
        n_t, n_s = min(32, b), 8       # 256 (trajectory, allocation) pairs
        t_h = times_d[:n_t, :n_s].cpu().numpy()
        p_rep = np.repeat(pos_h[:n_t], n_s, axis=0)
        _, ref_cost, st = Oracle("f64").solve_batch_standard(p_rep, t_h.reshape(n_t * n_s, K_SEG), NCOEF, SNAP, 4, cores)
        err = float(np.abs(cost_d[:n_t, :n_s].cpu().numpy().reshape(-1) / ref_cost - 1.0).max())
        out["parity"] = {"ok": bool(st == 0 and err <= 1e-8), "n_checked": n_t * n_s, "cost_rel_err": err, "bar": 1e-8}
    return out


def pinned_copy_ceiling(torch, ranks, h2d_pairs, d2h_pairs, reps=5):
    """The box's concurrent pinned-copy rate for exactly the e2e step's bytes: plain cudaMemcpyAsync of the
    inputs (host->device) and the coefficients (device->host) on two streams at once, all ranks together."""
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def go():
        with torch.cuda.stream(s_in):
            for dst, src in h2d_pairs:
                dst.copy_(src, non_blocking=True)
        with torch.cuda.stream(s_out):
            for dst, src in d2h_pairs:
                dst.copy_(src, non_blocking=True)

    go()
    torch.cuda.synchronize()
    ranks.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        go()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ranks.barrier()
    return max(ranks.all_ms(dt * 1e3)) * 1e-3 / reps


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    import mav_trajectory_generation_cmake_b200 as ms

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the GPU arm has no CPU fallback")
    torch.cuda.set_device(local)
    n_local_cpus = bind_to_gpu_cpus(local)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ranks = Ranks(torch, dist, world)
    barrier = ranks.barrier

    ms.load()
    B = B_PER_GPU
    cores = os.cpu_count() or 1
    hbm_peak, peak_src = measured_peaks()
    # each rank owns a contiguous slice of the global batch: seeds 12345 + rank*B + b
    from mav_trajectory_generation_cmake_b200.sharding import gather_to_rank0, weak_scaling_seed_base
    pos_h = ms.random_positions_host(B, K_SEG, BOX_LO, BOX_HI, weak_scaling_seed_base(BASE_SEED, B, rank))
    n_sets = n_buffer_sets(B * BYTES_PER_SOLVE)   # 2 x 180 MB > 126 MB L2
    pos_d, times_d, coeffs_d, step = solve_workload(ms, torch, pos_h, K_SEG, n_sets)

    clocks = Clocks(local)
    # A rehearsal of the whole procedure, discarded: the FIRST timed window of a process read 42.2-42.4 us per step on
    # every fresh box, whatever real warm-up preceded it, and the same work timed a moment later 41.1-41.5 us
    # (profiles/r2_warmup_curve.txt, first trial; the other configurations below, timed later in the process, never
    # showed it).
    timed_steps(torch, ranks, step, args.steps, args.warmup)
    all_ms, timed_mode = timed_steps(torch, ranks, step, args.steps, args.warmup, clocks=clocks, probe_s=0.25)
    elapsed_ms = max(all_ms)
    ms_per_step = elapsed_ms / args.steps
    value = world * B * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # The buffer set the last timed step wrote.  Every set is solved from the same pos_h, so any set holds the same
        # answer; this one is taken so that the file shows what the last step returned.
        last = coeffs_d[(args.warmup + args.steps - 1) % n_sets]
        rows = torch.from_numpy(dump_rows(B)).cuda()
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "coeffs.npy"), last.index_select(0, rows).cpu().numpy())

    # ---- e2e: host buffers through the C-ABI host entry point, copies inside the timed region
    pos_pin = torch.from_numpy(pos_h).pin_memory()
    times_pin = times_d[0].cpu().pin_memory()
    coeffs_pin = torch.empty((B, K_SEG, DIM, NCOEF), dtype=torch.float64).pin_memory()
    e2e_steps = max(3, min(args.steps, 20))
    for _ in range(3):
        ms.solve_standard_host(pos_pin, times_pin, coeffs=coeffs_pin)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ms.solve_standard_host(pos_pin, times_pin, coeffs=coeffs_pin)
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_all = ranks.all_ms(e2e_s * 1e3)
    e2e_s = max(e2e_all) * 1e-3
    e2e_value = world * B * e2e_steps / e2e_s
    ceiling_s = pinned_copy_ceiling(torch, ranks, [(pos_d[0], pos_pin), (times_d[0], times_pin)],
                                    [(coeffs_pin, coeffs_d[0])])
    e2e_bytes = (BYTES_IN + BYTES_OUT) * B
    e2e_ceiling = world * B / ceiling_s

    # ---- optional: one NCCL gather of the coefficient blocks (reported separately) ------------
    gather_ms = None
    if distributed:
        gather_to_rank0(coeffs_d[0], world * B, dist)
        torch.cuda.synchronize()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gathered = gather_to_rank0(coeffs_d[0], world * B, dist)
        g1.record()
        del gathered
        torch.cuda.synchronize()
        gather_ms = max(ranks.all_ms(g0.elapsed_time(g1)))

    # the same collection through a CUDA-IPC peer buffer on rank 0: one device-to-peer copy per rank
    peer_gather_ms = None
    if distributed:
        from mav_trajectory_generation_cmake_b200.sharding import PeerGatherBuffer
        buf, ok = None, 1
        try:
            buf = PeerGatherBuffer(dist, B, (K_SEG, DIM, NCOEF), torch.float64, dst=0)
        except Exception:
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        all_ok = int(flag.item()) == 1
        if all_ok:
            buf.push(coeffs_d[0])
            torch.cuda.synchronize()
            barrier()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            buf.push(coeffs_d[0])
            q1.record()
            torch.cuda.synchronize()
            barrier()
            peer_gather_ms = max(ranks.all_ms(q0.elapsed_time(q1)))
        if buf is not None:
            buf.close(barrier=all_ok)

    fp64_peak = ms.fp64_peak(5)
    if distributed:   # every rank uses rank 0's figure in the fractions below
        t = torch.tensor([fp64_peak], dtype=torch.float64, device="cuda")
        dist.broadcast(t, 0)
        fp64_peak = t.item()

    # extrema of |velocity| over every trajectory (SURVEY 8(f)1: computeMaximumOfMagnitude), rank 0's batch
    extrema_ms = None
    if rank == 0:
        reps = 5
        for _ in range(2):
            ms.extrema(coeffs_d[0], times_d[0], 1)
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record()
        for _ in range(reps):
            ms.extrema(coeffs_d[0], times_d[0], 1)
        x1.record()
        torch.cuda.synchronize()
        extrema_ms = x0.elapsed_time(x1) / reps

    parity = cpu = None
    if rank == 0:
        cpu = cpu_solves_per_s(pos_h, times_pin.numpy(), cores, budget_s=15.0)
        parity = parity_block(ms, torch, pos_h, times_pin.numpy(), cores)
    del pos_d, times_d, coeffs_d, coeffs_pin
    torch.cuda.empty_cache()

    # ---- BASELINE.json configs[2..4] and the strong-scaling target, every rank takes its share --------
    configs = {}
    if not args.skip_configs:
        for key, fn, extra in (("target_65536_total", config_target, (args, hbm_peak, fp64_peak, cores)),
                               ("2_sampling_1M_x_1000", config_sampling, (hbm_peak, cores)),
                               ("3_long_horizon_4096_x_256", config_long_horizon, (args, hbm_peak, fp64_peak, cores)),
                               ("4_time_sweep_8192_x_64", config_time_sweep, (args, hbm_peak, fp64_peak, cores))):
            try:
                configs[key] = fn(ms, torch, ranks, rank, world, *extra)
            except Exception as exc:   # a failing side config must not take the headline line down
                configs[key] = {"error": "%s: %s" % (type(exc).__name__, exc)}
                if distributed:
                    raise
            torch.cuda.empty_cache()

    if rank == 0:
        achieved = BYTES_PER_SOLVE * B / (ms_per_step * 1e-3) / 1e9          # GB/s, one rank's kernel
        fp64_achieved = FLOPS_PER_SOLVE * B / (ms_per_step * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "solve_standard_traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = "static, from profiles/solve_standard_traffic.json (%s)" % tj.get("source", "ncu --set full")
            except Exception:
                traffic = None
        cpu_value, cpu_sample, cpu_1t = cpu
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": CONFIG,
            "run": {"timed_loop": timed_mode, "buffer_sets": n_sets,
                    "extra_warmup": "a discarded rehearsal of the whole timed procedure (the first timed window of a process reads ~1 us per step high), then the %d eager steps and untimed replays of the %d-step graph for ~8 ms (burst measurement on an awake GPU: tools/warmup_curve.py; sustained load: tools/sustained_load.py)" % (args.warmup, args.steps),
                    "window": "start event behind a ~0.3 ms spin kernel: events, graph and stop event are enqueued while "
                              "it runs, so the window holds the K steps and no host submission latency"},
            "per_rank_ms": Ranks.spread(all_ms, args.steps),
            "gpu_launches": args.steps * ms_launches_per_step(ms),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_solve": BYTES_PER_SOLVE, "kernel": "solve_standard",
                         "fp64_tflops_achieved": fp64_achieved, "fp64_tflops_peak_measured": fp64_peak,
                         "fp64_frac": fp64_achieved / fp64_peak, "flops_per_solve": FLOPS_PER_SOLVE},
            "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d of the 65,536 problems, best of 3; oracle port of the reference "
                                       "algorithm (dense QR stands in for Eigen::SparseQR); 1 thread: %.0f solves/s"
                                       % (cpu_sample, cpu_1t)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": BYTES_IN * B,
                    "d2h_bytes_per_step": BYTES_OUT * B, "steps": e2e_steps,
                    "api": "minsnap_solve_standard_host (pinned host buffers, chunked pipelined copies)",
                    "host_cpus_bound": n_local_cpus,
                    "per_rank_ms": Ranks.spread(e2e_all, e2e_steps),
                    "gb_per_s_per_gpu": e2e_bytes * e2e_steps / e2e_s / 1e9,
                    "ceiling": {"value": e2e_ceiling, "unit": UNIT, "gb_per_s_per_gpu": e2e_bytes / ceiling_s / 1e9,
                                "how": "plain pinned cudaMemcpyAsync of the step's inputs (H2D) and coefficients "
                                       "(D2H) on two streams at once, all %d ranks together, no kernel" % world},
                    "frac": e2e_value / e2e_ceiling},
            "clocks": clocks.summary(),
            "parity": parity,
            "configs": configs,
            "extra": {"extrema_ms": extrema_ms, "extrema_trajectories_per_s": B / (extrema_ms * 1e-3),
                      "extrema_shape": "max |velocity| of %d trajectories x %d segments "
                                       "(computeMaximumOfMagnitude)" % (B, K_SEG),
                      "nccl_gather_ms": gather_ms, "peer_copy_gather_ms": peer_gather_ms},
        }
        emit(line)
    if distributed:
        dist.destroy_process_group()


def ms_launches_per_step(ms):
    """Kernels one solve_standard call launches: 1 on the fast route, 4 on the generic route
    (mask, reorder, pack, general solve)."""
    return 1 if getattr(ms.api, "STANDARD_FAST_ROUTE", False) else 4


_RESULT_FD = None


def emit(line):
    """The one JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    # Libraries print to the C-level stdout behind Python's back (NCCL announces its version there):
    # keep the original stdout for the JSON line only and send everything else to stderr.
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--skip-configs", action="store_true", help="headline only (no configs[2..4] / target)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the coefficients the last headline step computed for a fixed, "
                         "seeded sample of %d of rank 0's trajectories to DIR/coeffs.npy (float64)" % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native arm")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
