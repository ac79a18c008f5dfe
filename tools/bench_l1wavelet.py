"""
l1-wavelet FISTA (indigo_b200.wavelet.l1wavelet_recon) on bench.py's geometries, one GPU, one process.  Prints one
JSON line per workload:
  ms per FISTA iteration next to ms per B.cg iteration on the same normal operator (same run, same graph mode), the
  prox step's share of the iteration, per-kernel times of the prox step with compulsory bytes from the byte model
  below and the fraction of the copy peak, spectral_norm seconds, the extra device memory of the solver and, with
  --nrmse, the NRMSE to the synth.phantom truth after 50 iterations of l1-wavelet and of Tikhonov CG
  (lamda = 1e-2 ||A^H A||).  The data for the NRMSE is simulated with the same operator (an inverse crime).
  GPU name and power limit are read in the same run.

    python tools/bench_l1wavelet.py --workload cfg3 --normal gridded --nrmse
    python tools/bench_l1wavelet.py --workload cfg4 --normal toeplitz
    python tools/bench_l1wavelet.py --workload cfg1 --normal gridded --graph
    python tools/bench_l1wavelet.py --workload cfg5 --normal gridded

A workload the normal operator does not serve prints a line with "error".
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

import bench                                                     # noqa: E402  (workloads, peaks, power_norm)
from bench_toeplitz import gpu_info                              # noqa: E402


def prox_bytes(N, J):
    """Compulsory HBM bytes of one ib200_wavelet_fista_step, per kernel: {(axis, inverse): bytes}.  A pass of level j
    reads and writes the sub-box of nvox / 2^((j-1) d) points (d transformed axes, complex64); the first analysis
    pass also reads g and b, the last synthesis pass also reads x and writes z."""
    nvox = int(np.prod(N))
    axes = [a for a in range(3) if N[a] > 1]
    out = {}
    for inv in (False, True):
        for j in range(1, J + 1):
            sub = nvox // (1 << ((j - 1) * len(axes)))
            for a in axes:
                b = 16 * sub
                if j == 1 and a == 0:
                    b += 16 * nvox
                out[(a, inv)] = out.get((a, inv), 0) + b
    return out


def kernel_key(name):
    """(axis, inverse) of a wavelet_pass_kernel<LF, AXIS, INV> name, else None."""
    if "wavelet_pass_kernel<" not in name:
        return None
    args = name.split("wavelet_pass_kernel<")[1].split(">")[0].split(",")
    return int(args[1]), args[2].strip() == "true"


def iteration_ms(torch, fn, iters, reps=3):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(iters)
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3 / iters)
    return min(ts)


def run(args, torch):
    from indigo_b200 import B200Backend, synth
    from indigo_b200.fused import sense_operator_fused, toeplitz_normal
    from indigo_b200.sense import normal_operator, sqrt_dcf
    from indigo_b200 import wavelet as WV
    wl = bench.WORKLOADS[args.workload]
    B = B200Backend(0)
    rs = np.random.RandomState(0)
    N = wl["N"]
    C = args.coils or wl["C"]
    nvox = int(np.prod(N))
    coord = bench.make_traj(wl["traj"])
    w = sqrt_dcf(coord) if wl["kind"] == "cg" else None
    maps = synth.unit_rss_maps(rs, N, C)
    A = sense_operator_fused(B, N, coord, maps, wl["oversamp"], weights=w)
    AHA = normal_operator(A) if args.normal == "gridded" else toeplitz_normal(A)
    J = WV.wavelet_levels(N, args.wave)
    line = dict(workload=args.workload, normal=args.normal, coils=C, N=list(N), wave=args.wave, levels=J,
                graph=bool(args.graph))
    line.update(gpu_info())
    # data: y = A truth, b = A^H y
    truth = synth.phantom(N).reshape(-1, 1, order='F')
    xt = B.copy_array(truth)
    y = B.empty_array((A.shape[0], 1), bench.C64)
    A.eval(y, xt)
    bd = B.empty_array((nvox, 1), bench.C64)
    A.H.eval(bd, y)
    b_h = bd.to_host()
    del y, bd, xt
    # spectral norm
    torch.cuda.synchronize(); t0 = time.perf_counter()
    L = WV.spectral_norm(B, AHA)
    torch.cuda.synchronize()
    line["spectral_norm_s"] = round(time.perf_counter() - t0, 4)
    line["spectral_norm"] = L
    step, lam, lam_cg = 0.9 / L, args.lamda * L, 1e-2 * L
    # extra device memory of the solver (beyond the operator): peak of one short run
    x0 = np.zeros((nvox, 1), np.complex64, order='F')
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    WV.l1wavelet_recon(B, AHA, b_h, x0.copy(order='F'), N, lam, wave=args.wave, step=step, maxiter=3, graph=args.graph)
    torch.cuda.synchronize()
    line["extra_device_gb"] = round((torch.cuda.max_memory_allocated() - base) / 1e9, 3)
    # ms per iteration, FISTA and CG alternated; warm-up of both first
    B.cg(AHA, b_h, x0.copy(order='F'), lamda=lam_cg, maxiter=3, tol=0.0, graph=args.graph)
    it = args.iters
    fista = lambda n: WV.l1wavelet_recon(B, AHA, b_h, x0.copy(order='F'), N, lam, wave=args.wave, step=step,
                                         maxiter=n, graph=args.graph)
    cg = lambda n: B.cg(AHA, b_h, x0.copy(order='F'), lamda=lam_cg, maxiter=n, tol=0.0, graph=args.graph)
    f_ms, c_ms = [], []
    for _ in range(2):
        f_ms.append(iteration_ms(torch, fista, it, reps=1))
        c_ms.append(iteration_ms(torch, cg, it, reps=1))
    line["fista_ms_per_iter"] = round(min(f_ms), 3)
    line["cg_ms_per_iter"] = round(min(c_ms), 3)
    line["iters_timed"] = it
    # the prox step alone (CUDA events around repeated steps on the same buffers), and its kernels
    lib, s = B._lib, B._stream
    geom = WV._Geometry(N, args.wave, J)
    bufs = [B.copy_array(b_h) for _ in range(5)]
    g, b, z, x, work = bufs
    mom = torch.from_numpy(WV.fista_momentum(4096)).to(B._device)
    counter = torch.zeros(1, dtype=torch.int32, device=B._device)

    def prox():
        lib.wavelet_fista_step(s, geom.dims, len(geom.h), geom.hp, geom.J, step, step * lam, g.ptr, b.ptr, z.ptr,
                               x.ptr, work.ptr, mom.data_ptr(), counter.data_ptr(), None)

    for _ in range(3):
        prox()
    reps = 40
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        prox()
    e1.record(); e1.synchronize()
    prox_ms = e0.elapsed_time(e1) / reps
    line["prox_ms"] = round(prox_ms, 4)
    line["prox_share_of_iteration"] = round(prox_ms / line["fista_ms_per_iter"], 4)
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            prox()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        key = kernel_key(ev.name)
        if key is not None and ev.device_type.name == "CUDA":
            per[key] = per.get(key, 0.0) + ev.device_time / 1e3 / reps          # ms per step
    nbytes = prox_bytes(N, J)
    peak_gbs, peak_src = bench.peaks()
    line["copy_peak_gbs"], line["copy_peak_source"] = peak_gbs, peak_src
    line["prox_kernels"] = {"%s axis %d" % ("synthesis" if inv else "analysis", a):
                            dict(ms=round(ms, 4), gb=round(nbytes[(a, inv)] / 1e9, 4),
                                 frac_copy_peak=round(nbytes[(a, inv)] / (ms / 1e3) / (peak_gbs * 1e9), 3))
                            for (a, inv), ms in sorted(per.items())}
    line["prox_compulsory_gb"] = round(sum(nbytes.values()) / 1e9, 4)
    del bufs, g, b, z, x, work
    if args.nrmse:
        ref = np.ravel(truth)
        xs = x0.copy(order='F')
        WV.l1wavelet_recon(B, AHA, b_h, xs, N, lam, wave=args.wave, step=step, maxiter=50)
        line["nrmse_l1wavelet_50"] = float(np.linalg.norm(np.ravel(xs) - ref) / np.linalg.norm(ref))
        xc = x0.copy(order='F')
        B.cg(AHA, b_h, xc, lamda=lam_cg, maxiter=50, tol=0.0)
        line["nrmse_cg_50"] = float(np.linalg.norm(np.ravel(xc) - ref) / np.linalg.norm(ref))
        line["nrmse_note"] = "data simulated with the same operator (inverse crime)"
    line["lamda_over_norm"] = args.lamda
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workload", choices=["cfg3", "cfg4", "cfg1", "cfg5"], required=True)
    ap.add_argument("--normal", choices=["gridded", "toeplitz"], default="gridded")
    ap.add_argument("--coils", type=int, default=None, help="override the workload's coil count")
    ap.add_argument("--wave", default="db4")
    ap.add_argument("--lamda", type=float, default=1e-3, help="l1 weight as a fraction of ||A^H A||")
    ap.add_argument("--iters", type=int, default=20, help="iterations per timed solve")
    ap.add_argument("--graph", action="store_true", help="both solvers replay one iteration as a CUDA graph")
    ap.add_argument("--nrmse", action="store_true", help="also report NRMSE to the phantom after 50 iterations")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_l1wavelet.py measures on a CUDA device; none is visible")
    try:
        run(args, torch)
    except RuntimeError as e:                                     # e.g. no Toeplitz grid for this image
        print(json.dumps(dict(workload=args.workload, normal=args.normal, error=str(e))), flush=True)


if __name__ == "__main__":
    main()
