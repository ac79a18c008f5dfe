"""
Pipe-Menon density compensation (indigo_b200.sense.pipe_menon_dcf, csrc/dcf.cu) on bench.py's full-size
trajectories, one GPU, one process.  Prints one JSON line per workload:
  setup seconds and peak memory (DensityDevice: sample order, records, windows, 4x4x4 block entries, grid), ms per
  iteration (CUDA events around `--steps` iterations without residual), ms per kernel (events around each launch)
  with compulsory bytes and fraction of the copy peak, for the update kernel also the L1-path figure (bench.py's
  model for kb_gather), the fixed-point residual after `--iters` iterations of pipe_menon_dcf and its wall time;
  GPU name and power limit read in the same run.

    python tools/bench_dcf.py                    # cfg3 (kooshball, 6.8 M samples) and cfg5 (stack of spirals, 12.6 M)
    python tools/bench_dcf.py --only cfg5 --steps 50
"""
import argparse
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))

import bench                                                     # noqa: E402  (KernelTimer, peaks, workloads)
from bench_toeplitz import gpu_info                              # noqa: E402


def kernel_bytes(d):
    """Compulsory HBM bytes of one launch of each kernel of an iteration."""
    t, M = d.tiles, d.M
    split = 2 * t['nslot'] * 64 * 4                                  # partial sums written and read back by the fold
    return {"kb_density_spread": t['bytes'] + 16 * t['nwork'] + 4 * M + 4 * d.inside + split,
            "kb_density_update": 96 * M + 4 * d.inside + 8 * M}


def run(name, wl, steps, iters, torch):
    from indigo_b200 import B200Backend
    from indigo_b200.sense import DensityDevice, pipe_menon_dcf
    B = B200Backend(0)
    N = wl["N"]
    coord = bench.make_traj(wl["traj"])
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    d = DensityDevice(B, N, coord, wl["oversamp"])
    torch.cuda.synchronize()
    setup = time.perf_counter() - t0
    line = dict(workload=name, N=list(N), oN=list(d.oN), M=d.M, setup_s=round(setup, 3),
                setup_peak_gb=round((torch.cuda.max_memory_allocated() - base) / 1e9, 3),
                resident_gb=round((torch.cuda.memory_allocated() - base) / 1e9, 3),
                entries_gb=round(d.tiles['bytes'] / 1e9, 3), grid_gb=round(4 * int(np.prod(d.oN)) / 1e9, 3),
                inside_fraction=round(d.inside / float(np.prod(d.oN)), 3), work_items=d.tiles['nwork'],
                split_blocks=d.tiles['nsplit'])
    line.update(gpu_info())
    for _ in range(3):                                           # warm-up
        d.iterate()
    # whole iterations, no probe: alternate two blocks of `steps` to see the spread
    per_it = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            d.iterate()
        e1.record(); e1.synchronize()
        per_it.append(e0.elapsed_time(e1) / steps)
    line["ms_per_iteration"] = round(float(np.median(per_it)), 4)
    line["ms_per_iteration_blocks"] = [round(v, 4) for v in per_it]
    # per kernel
    kt = bench.KernelTimer(B, torch)
    d.probe = kt.probe
    cs = bench.ClockSampler(torch.cuda.current_device())
    cs.start()
    for _ in range(steps):
        d.iterate()
    torch.cuda.synchronize()
    clocks = cs.stop()
    if cs.proc is not None:
        cs.proc.wait()
    d.probe = None
    line["sm_clock"] = clocks
    per = {}
    for label, e0, e1, _, _ in kt.rec:
        per.setdefault(label, []).append(e0.elapsed_time(e1))
    peak_gbs, peak_src = bench.peaks()
    nbytes = kernel_bytes(d)
    line["copy_peak_gbs"], line["copy_peak_source"] = peak_gbs, peak_src
    line["kernels"] = {k: dict(ms=round(float(np.median(v)), 4), gb=round(nbytes[k] / 1e9, 3),
                               frac_copy_peak=round(nbytes[k] / (float(np.median(v)) / 1e3) / (peak_gbs * 1e9), 3))
                       for k, v in per.items()}
    # the update has kb_gather's tap structure (125 taps per sample for width 3); with one float per tap a lane's
    # load is one 32-byte sector unless neighbouring samples of the warp share it: sector requests at most 125 M
    prop = torch.cuda.get_device_properties(torch.cuda.current_device())
    clk = clocks["sm_mhz"]
    l1_peak = 128.0 * prop.multi_processor_count * (clk or 1965.0) * 1e6 / 1e9
    ms_u = float(np.median(per["kb_density_update"]))
    taps = 125.0 * d.M
    line["kernels"]["kb_density_update"]["l1_path"] = dict(
        tap_loads=int(taps), sector_gb=round(taps * 32 / 1e9, 3), achieved_gbs=round(taps * 32 / (ms_u / 1e3) / 1e9, 1),
        peak_gbs=round(l1_peak, 1), frac=round(taps * 32 / (ms_u / 1e3) / 1e9 / l1_peak, 3),
        note="125 taps per sample, at most one 32-byte sector each; 128 B/clk/SM x SMs x %s MHz" % (clk or "1965 (nominal)"))
    del d
    # the public entry point, with the residual history
    hist = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    w = pipe_menon_dcf(B, N, coord, wl["oversamp"], maxiter=iters, history=hist)
    torch.cuda.synchronize()
    line["pipe_menon_dcf_s"] = round(time.perf_counter() - t0, 3)
    line["iterations"] = iters
    line["residual_first"], line["residual_last"] = hist[0], hist[-1]
    line["residual_history"] = [float("%.4g" % v) for v in hist]
    line["weights_min_max"] = [float(w.min()), float(w.max())]
    line["weights_finite"] = bool(np.isfinite(w).all())
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--only", choices=["cfg3", "cfg5", "cfg1", "tiny"], default=None)
    ap.add_argument("--steps", type=int, default=20, help="iterations per timed block")
    ap.add_argument("--iters", type=int, default=30, help="iterations of the pipe_menon_dcf run (residual)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_dcf.py measures on a CUDA device; none is visible")
    for name in ([args.only] if args.only else ["cfg3", "cfg5"]):
        run(name, bench.WORKLOADS[name], args.steps, args.iters, torch)
        import gc
        gc.collect()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
