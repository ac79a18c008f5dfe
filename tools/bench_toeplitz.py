"""
Toeplitz-embedded normal operator (indigo_b200.fused.toeplitz_normal) against the gridded fused normal operator on
bench.py's workloads, one GPU, one process.  Prints one JSON line per workload:
  applies/s of both operators (alternated in the same run), per-pass times of T with compulsory bytes and fraction
  of the copy peak, setup seconds and peak memory of toeplitz_normal, ||Tx - A^H A x|| / ||A^H A x||, and for the
  CG workload the seconds per 50-iteration solve of both operators; GPU name and power limit read in the same run.

    python tools/bench_toeplitz.py                       # cfg3 16 coils, cfg3 2 coils, cfg1, cfg4 CG
    python tools/bench_toeplitz.py --only cfg3 --coils 2

A workload the operator does not serve prints a line with "error".
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import bench                                                     # noqa: E402  (KernelTimer, peaks, workloads)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [v.strip() for v in out.split(",")]
        return dict(gpu=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:                                       # the numbers are then unqualified: say so
        return dict(gpu="unknown (%s)" % e)


def t_pass_bytes(tdev):
    """Compulsory HBM bytes of every pass of one T apply (complex64 grid, coil-interleaved)."""
    N, L, C = tdev.N, tdev.L, tdev.C
    nvox = int(np.prod(N))
    if tdev.three:
        img_planes = L[0] * N[1] * N[2] * C * 8                     # x pass writes full x rows of the image window
        y_planes = L[0] * L[1] * N[2] * C * 8                       # y passes: all y for the z planes of the window
        return {"sense_expand_pk[x]": nvox * 8 + nvox * C * 8 + img_planes,
                "fft_pass[y fwd]": img_planes + y_planes,
                "toeplitz_pass[z]": 2 * y_planes + 4 * int(np.prod(L)),
                "fft_pass[y inv]": y_planes + img_planes,
                "sense_combine_pk[x]": img_planes + nvox * C * 8 + nvox * 8}
    rows = L[0] * N[1] * C * 8
    return {"sense_expand_pk[x]": nvox * 8 + nvox * C * 8 + rows,
            "toeplitz_pass[y]": 2 * rows + 4 * int(np.prod(L)),
            "sense_combine_pk[x]": rows + nvox * C * 8 + nvox * 8}


def run(name, wl, coils, steps, torch):
    from indigo_b200 import B200Backend, synth
    from indigo_b200.fused import sense_operator_fused, toeplitz_normal
    from indigo_b200.sense import normal_operator, sqrt_dcf
    B = B200Backend(0)
    rs = np.random.RandomState(0)
    N, C = wl["N"], coils or wl["C"]
    coord = bench.make_traj(wl["traj"])
    w = sqrt_dcf(coord) if wl["kind"] == "cg" else None
    maps = synth.unit_rss_maps(rs, N, C)
    nvox = int(np.prod(N))
    A = sense_operator_fused(B, N, coord, maps, wl["oversamp"], weights=w)
    AHA = normal_operator(A)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    T = toeplitz_normal(A)
    torch.cuda.synchronize()
    setup = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated() - base
    x_h = synth.rand64c(rs, nvox, 1)
    x, yt, yg = B.copy_array(x_h), B.empty_array((nvox, 1), bench.C64), B.empty_array((nvox, 1), bench.C64)
    T.eval(yt, x)
    AHA.eval(yg, x)
    err = float(np.linalg.norm(yt.to_host() - yg.to_host()) / np.linalg.norm(yg.to_host()))
    line = dict(workload=name, coils=C, N=list(N), L=list(T._tdev.L), s2=T._tdev.s2, setup_s=round(setup, 3),
                setup_peak_gb=round(peak / 1e9, 3), rel_err_vs_gridded=err)
    line.update(gpu_info())
    if wl["kind"] == "cg":
        y = B.empty_array((A.shape[0], 1), bench.C64)
        A.eval(y, x)
        b = B.empty_array((nvox, 1), bench.C64)
        A.H.eval(b, y)
        b_h = b.to_host()
        lam = 1e-2 * bench.power_norm(B, AHA, None, nvox, rs)
        for op, key in ((T, "toeplitz"), (AHA, "gridded")):
            xs = np.zeros_like(b_h, order='F')
            B.cg(op, b_h, xs, lamda=lam, maxiter=2, tol=0.0, graph=True)             # warm-up
            ts = []
            for _ in range(3):
                xs = np.zeros_like(b_h, order='F')
                torch.cuda.synchronize(); t0 = time.perf_counter()
                B.cg(op, b_h, xs, lamda=lam, maxiter=50, tol=0.0, graph=True)
                torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
            line["cg50_s_" + key] = round(min(ts), 4)
            line["cg_x_" + key] = xs
        xt, xg = line.pop("cg_x_toeplitz"), line.pop("cg_x_gridded")
        line["cg_solution_rel_diff"] = float(np.linalg.norm(xt - xg) / np.linalg.norm(xg))
        print(json.dumps(line), flush=True)
        return
    # applies/s, alternating blocks of `steps` applies of each operator
    for _ in range(3):
        T.eval(yt, x); AHA.eval(yg, x)
    rates = {"toeplitz": [], "gridded": []}
    for _ in range(4):
        for op, out, key in ((T, yt, "toeplitz"), (AHA, yg, "gridded")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                op.eval(out, x)
            e1.record(); e1.synchronize()
            rates[key].append(steps / (e0.elapsed_time(e1) / 1e3))
    line["applies_per_s_toeplitz"] = round(float(np.median(rates["toeplitz"])), 2)
    line["applies_per_s_gridded"] = round(float(np.median(rates["gridded"])), 2)
    line["speedup"] = round(line["applies_per_s_toeplitz"] / line["applies_per_s_gridded"], 3)
    # per pass
    kt = bench.KernelTimer(B, torch)
    T._tdev.probe = kt.probe
    for _ in range(steps):
        T.eval(yt, x)
    torch.cuda.synchronize()
    T._tdev.probe = None
    per = {}
    for label, e0, e1, _, _ in kt.rec:
        per.setdefault(label, []).append(e0.elapsed_time(e1))
    peak_gbs, peak_src = bench.peaks()
    nbytes = t_pass_bytes(T._tdev)
    line["copy_peak_gbs"], line["copy_peak_source"] = peak_gbs, peak_src
    line["passes"] = {k: dict(ms=round(float(np.median(v)), 4), gb=round(nbytes[k] / 1e9, 3),
                              frac_copy_peak=round(nbytes[k] / (float(np.median(v)) / 1e3) / (peak_gbs * 1e9), 3))
                      for k, v in per.items()}
    line["compulsory_gb_total"] = round(sum(nbytes.values()) / 1e9, 2)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--only", choices=["cfg3", "cfg1", "cfg4"], default=None)
    ap.add_argument("--coils", type=int, default=None, help="with --only: override the coil count")
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_toeplitz.py measures on a CUDA device; none is visible")
    runs = [("cfg3", None), ("cfg3", 2), ("cfg1", None), ("cfg4", None)]
    if args.only:
        runs = [(args.only, args.coils)]
    for name, coils in runs:
        try:
            run(name, bench.WORKLOADS[name], coils, args.steps, torch)
        except RuntimeError as e:                                   # e.g. no padded grid with fitting passes
            print(json.dumps(dict(workload=name, coils=coils, error=str(e))), flush=True)
        import gc
        gc.collect()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
