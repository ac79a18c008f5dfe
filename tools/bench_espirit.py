"""
ESPIRiT coil sensitivity estimation (indigo_b200.espirit) on bench.py's geometries, one GPU, one process.  The data
is simulated with the fused SENSE operator from synth.phantom and synth.birdcage_maps; the maps are then estimated
from it with calibration_kspace + espirit_maps (defaults: width 24, kernel 6, thresh 0.02, crop 0.95, 100 power
iterations).  Prints one JSON line per workload:
  - calibration seconds (DCF, gridding, FFT: host clock around the call, which ends in a device read-back);
  - per device step, CUDA-event milliseconds, the flop and byte counts of the model below and the achieved rates:
    ib200_espirit_calib_gram, the two lag passes, ib200_espirit_maps;
  - host seconds of eigh + threshold + lag form (float64, numpy);
  - total wall seconds of the two calls, peak torch-owned device memory, mean alignment
    |<m_est, m_true>| in the phantom's support;
  - GPU name and power limit, read in the same run.

    python tools/bench_espirit.py                       # cfg1, cfg3, cfg4
    python tools/bench_espirit.py --workload cfg3
"""
import argparse
import contextlib
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))

import bench                                                     # noqa: E402  (workloads)
from bench_toeplitz import gpu_info                              # noqa: E402


def step_model(N, C, k, R, lags, iters):
    """{step: (flop, bytes)}: complex multiply-add = 8 flop, complex64 = 8 bytes; compulsory traffic only."""
    nvox = int(np.prod(N))
    n = C * int(np.prod(k))
    CC = C * C
    q1 = N[2] * lags[1] * lags[0] * CC
    q2 = N[2] * N[1] * lags[0] * CC
    return {
        "espirit_calib_gram": (8.0 * n * (n + 1) / 2 * R, 8.0 * n * n),
        "espirit_lag_pass[z]": (8.0 * lags[2] * q1, 8.0 * (q1 + int(np.prod(lags)) * CC)),
        "espirit_lag_pass[y]": (8.0 * lags[1] * q2, 8.0 * (q2 + q1)),
        "espirit_maps": (8.0 * nvox * CC * (lags[0] + iters), 8.0 * (q2 + nvox * C) + 4.0 * nvox),
    }


def run(name, torch, width=24, kernel=6, iters=100):
    from indigo_b200 import B200Backend, synth, calibration_kspace, espirit_maps
    from indigo_b200 import espirit as E
    from indigo_b200.fused import sense_operator_fused
    wl = bench.WORKLOADS[name]
    N, C = tuple(wl["N"]), wl["C"]
    B = B200Backend(0)
    coord = bench.make_traj(wl["traj"])
    true = synth.birdcage_maps(N, C)
    ph = synth.phantom(N)
    A = sense_operator_fused(B, N, coord, true, wl["oversamp"])
    y = (A * ph.reshape(-1, 1, order='F')).reshape(-1, C, order='F')
    del A
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()

    events, host = {}, {}

    @contextlib.contextmanager
    def probe(label):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        yield
        e1.record()
        host[label] = time.perf_counter() - t0
        events[label] = (e0, e1)

    # warm-up at a small size: module load and first launches of every kernel
    E.probe = None
    small = tuple(16 if n > 1 else 1 for n in N)
    espirit_maps(B, synth.birdcage_maps(small, C)[:12, :12, :(12 if N[2] > 1 else 1)].copy(order='F'), small)
    torch.cuda.synchronize()

    t0 = time.perf_counter()
    calib = calibration_kspace(B, N, coord, y, width=width)
    t1 = time.perf_counter()
    E.probe = probe
    maps = espirit_maps(B, calib, N, kernel=kernel, max_iter=iters)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    E.probe = None
    peak = torch.cuda.max_memory_allocated()

    k = tuple(kernel if n > 1 else 1 for n in N)
    w = calib.shape[:3]
    R = int(np.prod([w[d] - k[d] + 1 for d in range(3)]))
    lags = tuple(2 * kd - 1 for kd in k)
    model = step_model(N, C, k, R, lags, iters)
    steps = {}
    for label, (flop, nbytes) in model.items():
        ms = events[label][0].elapsed_time(events[label][1])
        steps[label] = dict(ms=round(ms, 3), gflop=round(flop / 1e9, 3), mbytes=round(nbytes / 1e6, 3),
                            tflops=round(flop / ms / 1e9, 3), gbs=round(nbytes / ms / 1e6, 1))
    mask = np.abs(ph) > 0
    e, t = maps[mask], true[mask]
    align = np.abs((np.conj(e) * t).sum(axis=1)) / np.maximum(np.linalg.norm(e, axis=1) * np.linalg.norm(t, axis=1),
                                                              1e-30)
    out = dict(workload=name, N=list(N), coils=C, width=width, kernel=kernel, power_iters=iters,
               gram_n=C * int(np.prod(k)), calib_rows=R,
               calibration_s=round(t1 - t0, 3), host_eigh_lag_s=round(host["host_eigh_lag"], 3),
               steps=steps, total_s=round(t2 - t0, 3), espirit_maps_call_s=round(t2 - t1, 3),
               peak_torch_mem_gb=round(peak / 1e9, 3),
               alignment_mean=round(float(align.mean()), 6), alignment_min=round(float(align.min()), 6))
    out.update(gpu_info())
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[1])
    ap.add_argument("--workload", choices=["cfg1", "cfg3", "cfg4"], default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_espirit.py measures on a CUDA device; none is visible")
    for name in ([args.workload] if args.workload else ["cfg1", "cfg3", "cfg4"]):
        run(name, torch)
        import gc
        gc.collect()


if __name__ == "__main__":
    main()
