#!/usr/bin/env python
"""
bench.py -- BASELINE.json's headline metric on its headline configuration.

    metric   SENSE-NUFFT A^H A applies/sec (whole job), plus each kernel as a fraction of the HBM roofline
    workload cfg3 = BASELINE.json configs[2] (default): 3-D radial (kooshball) SENSE-NUFFT, image 208^3,
             2x oversampled grid 416^3, 16 coils, 16384 spokes x 416 samples (M = 6 815 744); the reference
             evaluates one apply as the six Backend calls of the -O3 tree of examples/pics.py
             ccsrmm(P^H,adj) -> fftn -> ccsrmm(G') -> ccsrmm(G',adj) -> ifftn -> ccsrmm(P^H)
             other workloads: cfg1 (configs[0]), cfg4 (configs[3]: 32 coils, 50 CG iterations), cfg5 (configs[4]:
             cgemm coil compression 48 -> 12 + stack-of-spirals NUFFT), tiny (development)
    step     one A^H A apply (AHA.eval(y, x)) on synthetic, seeded data (cfg4: one CG iteration = apply + the fused
             BLAS-1 updates; cfg5: one coil compression + one apply); with N > 1 GPUs the coils are sharded over
             the ranks (strong scaling) and each apply ends with one NCCL all-reduce of the image.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--check]
    torchrun ... bench.py --gpus N ...            (one rank per GPU; rank 0 prints ONE JSON line)

JSON line: the driver's contract (metric/value/unit/n_gpus/steps/warmup/ms_per_step/...), `e2e` (host buffers, H2D and
D2H inside the timed region), `kernels` (every kernel of the apply: CUDA-event time on the launching stream,
compulsory bytes of the formulation that runs, the bytes of the reference call it replaces (SURVEY.md 8d), ncu DRAM
traffic from the committed capture), `roofline` (the kernel with the largest time), `cpu_baseline`, `check`.

`--impl reference` times the reference's CPU implementation of the same apply on this box's host cores: SpMM through
the reference's own OpenMP kernel (oracle/_ref/_customcpu, all threads) and FFTs through scipy.fft with all workers,
next to the single-thread numpy/scipy numbers of indigo/backends/np.py; each step is a bounded sample of the apply
(`units_per_step` applies), see `cpu_baseline.sample`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

C64 = np.dtype("complex64")

WORKLOADS = {
    "cfg3": dict(N=(208, 208, 208), C=16, traj=("kooshball", 16384, 416), oversamp=2.0, kind="apply",
                 desc="cfg3: 3-D radial SENSE-NUFFT A^H A apply, image 208^3, grid 416^3 (2x oversampled), 16 coils, "
                      "16384 spokes x 416 samples (M=6815744), -O3 tree, 6 backend calls per apply"),
    "cfg1": dict(N=(256, 256, 1), C=8, traj=("radial2d", 402, 512), oversamp=2.0, kind="apply",
                 desc="cfg1: 2-D radial SENSE-NUFFT A^H A apply, image 256x256, grid 512x512x2, 8 coils, 402 spokes x 512"),
    "cfg4": dict(N=(208, 208, 208), C=32, traj=("kooshball", 16384, 416), oversamp=2.0, kind="cg",
                 desc="cfg4: pics.py-style CG reconstruction, cfg3 geometry, 32 coils, sqrt-DCF row weights, lamda via "
                      "cg(lamda=), 50 iterations (--steps 50); a step is one CG iteration (A^H A apply + fused BLAS-1 updates)"),
    "cfg5": dict(N=(256, 256, 128), C=12, traj=("spirals", 128, 48, 2048), oversamp=2.0, kind="cfg5", full_coils=48,
                 desc="cfg5: stack-of-spirals SENSE-NUFFT 256x256x128 (grid 512x512x256), 128 x 48 spirals x 2048 samples "
                      "(M=12582912), 48 coils compressed to 12 virtual coils by a DenseMatrix cgemm; a step is one coil "
                      "compression of the 48-coil data + one 12-coil A^H A apply"),
    "tiny": dict(N=(32, 32, 32), C=4, traj=("kooshball", 256, 64), oversamp=2.0, kind="apply",
                 desc="tiny: development smoke size (not a reportable workload)"),
}


def make_traj(spec):
    from indigo_b200 import synth
    if spec[0] == "kooshball":
        return synth.kooshball_3d(spec[1], spec[2])
    if spec[0] == "spirals":
        return synth.stack_of_spirals(nz=spec[1], nleaves=spec[2], nread=spec[3], turns=16.0)
    return synth.radial_2d(spec[1], spec[2])


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(workload, world, coils):
    """{kernel label: dram bytes per launch} from the committed `ncu --set full` capture of the same build, workload
    and per-GPU coil count (profiles/traffic.json, written by tools/make_traffic.py); {} when no capture matches."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(path):
        return {}, None
    table = json.load(open(path))
    entry = table.get("%s:coils%d" % (workload, coils))
    if not entry:
        return {}, None
    return entry["kernels"], entry["source"]


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks line of B200_PROFILING.md, sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([f.strip() for f in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- bytes per kernel
def fused_kernel_bytes(dev):
    """Per kernel of the fused recipe: (compulsory bytes of the formulation that runs, bytes of the reference call(s)
    it replaces per SURVEY.md 8(d), name of those calls).  Compulsory = every operand the kernel's formulation has to
    move, once: windows/pruning included, re-reads excluded; always <= the DRAM traffic ncu measures.  The six
    reference calls are spread over the kernels that replace them (a three-pass transform carries fftn's 2*8*points)."""
    N, oN, C, M = dev.N, dev.oN, dev.C, dev.M
    nvox, on = dev.nvox, dev.on
    inside = dev.support_fraction * on                       # grid points inside the k-space support windows
    px, py = oN[0] * N[1] * N[2], oN[0] * oN[1] * N[2]       # points per coil after the x pass / the y pass
    ent = dev.runs['entries'] * 20 if dev.runs is not None else dev.nnz * 8
    tiles = getattr(dev, 'tiles', None)
    tent = tiles['bytes'] if tiles is not None else 0
    nnzb = dev.nnz * 12
    ccs_G = nnzb + 4 * (M + 1) + 8 * C * (on + M)            # ccsrmm(G'), each operand once
    ccs_GH = nnzb + 4 * (M + 1) + 8 * C * (M + on)
    ccs_P = 12 * nvox * C + 4 * (nvox + 1) + 8 * (nvox + C * on)        # expand: beta = 0 writes the whole zero-padded grid
    ccs_PH = 12 * nvox * C + 4 * (nvox + 1) + 8 * (nvox * C + nvox)     # combine: reads only the image-sized part of it
    fft = 16 * on * C
    third = fft / 3.0
    return {
        "sense_expand_pk[x]": (8 * nvox + 8 * nvox * C + 8 * C * px, ccs_P + third, "ccsrmm(P^H,adj) + fftn/3"),
        "fft_pass[y fwd]": (8 * C * (px + py), third, "fftn/3"),
        "fft_pass[z fwd]": (8 * C * (py + inside), third, "fftn/3"),
        "kb_gather": (8 * C * inside + 96 * M + 8 * C * M, ccs_G, "ccsrmm(G')"),
        "csrmm_runs": (ent + 8 * C * M + 8 * C * inside, ccs_GH, "ccsrmm(G',adj)"),
        "kb_blocks": (tent + 8 * C * M + 8 * C * inside, ccs_GH, "ccsrmm(G',adj)"),
        "fft_pass[z inv]": (8 * C * (inside + py), third, "ifftn/3"),
        "fft_pass[y inv]": (8 * C * (py + px), third, "ifftn/3"),
        "sense_combine_pk[x]": (8 * C * px + 8 * nvox * C + 8 * nvox, ccs_PH + third, "ifftn/3 + ccsrmm(P^H)"),
    }


def reference_call_bytes(call):
    """SURVEY.md section 8(d): each operand of a reference Backend call counted once."""
    if call["op"] == "ccsrmm":
        # rows of X that can be read at all: no more than there are stored entries (the selection matrix P^H has
        # 1.15 G columns and 144 M entries; this is the reference's read_frac, operators.py:246-257)
        rd, wr = (call["m"], call["k"]) if call["adjoint"] else (call["k"], call["m"])
        rd = min(rd, call["nnz"])
        b = call["nnz"] * 12 + (call["m"] + 1) * 4 + 8 * call["ncols"] * (rd + wr)
        return b + (8 * call["ncols"] * wr if call["beta_nz"] else 0)
    return 16 * call["points"]


class KernelTimer(object):
    """CUDA events around every kernel-level call of the apply, on the launching stream.  The fused recipe is
    dissected through SenseDevice.probe (each pass of the two transforms is launched through ib200_sense_pass, same
    kernels and arguments as inside the fused calls); the six-call recipe through wrappers of the Backend methods."""

    def __init__(self, B, torch):
        self.B, self.torch, self.rec = B, torch, []

    def probe(self, label):
        timer = self

        class _Ctx(object):
            def __enter__(self):
                self.e0 = timer.torch.cuda.Event(enable_timing=True); self.e1 = timer.torch.cuda.Event(enable_timing=True)
                self.n0 = timer.B._lib.launch_count()
                self.e0.record()

            def __exit__(self, *exc):
                self.e1.record()
                timer.rec.append((label, self.e0, self.e1, timer.B._lib.launch_count() - self.n0, None))
        return _Ctx()

    def wrap_backend(self):
        B = self.B
        for name in ("ccsrmm", "ccsrmm_packed", "fftn", "ifftn"):
            setattr(B, name, self._wrap(name, getattr(B, name)))

    def _wrap(self, name, fn):
        def timed(*a, **k):
            e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
            n0 = self.B._lib.launch_count()
            e0.record(); out = fn(*a, **k); e1.record()
            if name == "ccsrmm_packed":
                y, shp, nnz, _, _, x = a[:6]
                beta = k.get("beta", a[7] if len(a) > 7 else 0)
                info = dict(op="ccsrmm", m=int(shp[0]), k=int(shp[1]), nnz=int(nnz), ncols=int(x.shape[1]),
                            adjoint=False, beta_nz=bool(beta != 0))
                key = "ccsrmm[packed real A %dx%d nnz/row=%.0f ncols=%d]" % (shp[0], shp[1], nnz / max(1, shp[0]), x.shape[1])
            elif name == "ccsrmm":
                y, shp, ind, ptr, vals, x = a[:6]
                adj = k.get("adjoint", a[8] if len(a) > 8 else False)
                beta = k.get("beta", a[7] if len(a) > 7 else 0)
                info = dict(op="ccsrmm", m=int(shp[0]), k=int(shp[1]), nnz=int(vals.size), ncols=int(x.shape[1]),
                            adjoint=bool(adj), beta_nz=bool(beta != 0))
                key = "ccsrmm[%s %dx%d nnz/row=%.0f ncols=%d]" % ("A^H" if adj else "A", shp[0], shp[1],
                                                                   vals.size / max(1, shp[0]), x.shape[1])
            else:
                x = a[1]
                info = dict(op=name, points=int(np.prod(x.shape)))
                key = "%s%s" % (name, tuple(int(s) for s in x.shape))
            self.rec.append((key, e0, e1, self.B._lib.launch_count() - n0, info))
            return out
        return timed

    def summary(self, peak, fused_bytes, traffic):
        agg = {}
        for label, e0, e1, nl, info in self.rec:
            d = agg.setdefault(label, dict(ms=[], launches=nl, info=info))
            d["ms"].append(e0.elapsed_time(e1))
        out = []
        for label, d in agg.items():
            ms = float(np.mean(d["ms"]))
            if d["info"] is not None:                              # a reference Backend call: 8(d) bytes are its own
                comp = ref_b = reference_call_bytes(d["info"]); what = d["info"]["op"]
            else:
                comp, ref_b, what = fused_bytes[label]
            dram = traffic.get(label)
            if dram and d["info"] is None:
                comp = min(comp, dram)          # never credit a kernel with more bytes than ncu saw it move (L2 carry-over
                                                # between consecutive kernels can shave a few percent off the reads)
            row = dict(kernel=label, ms=ms, launches=d["launches"], bytes=int(comp), gbs=comp / ms / 1e6,
                       frac=comp / ms / 1e6 / peak, replaces=what, replaced_call_bytes=int(ref_b),
                       frac_replaced_call=ref_b / ms / 1e6 / peak, dram_bytes=dram,
                       frac_dram=(dram / ms / 1e6 / peak) if dram else None)
            out.append(row)
        tot = sum(o["ms"] for o in out)
        for o in out:
            o["share"] = o["ms"] / tot if tot else 0.0
        return sorted(out, key=lambda o: -o["ms"])


# --------------------------------------------------------------------------- ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    from indigo_b200 import B200Backend, synth
    from indigo_b200.sense import sense_operator_device, normal_operator, sqrt_dcf
    from indigo_b200.fused import sense_operator_fused
    from indigo_b200.team import CoilTeam, coil_slice

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = WORKLOADS[args.workload]
    N, C, kind = wl["N"], wl["C"], wl["kind"]
    if getattr(args, "coils", 0):
        C = args.coils
        wl = dict(wl, desc=wl["desc"] + " [DEVELOPMENT RUN with %d coils, not the named configuration]" % C)
    if C % world:
        raise SystemExit("coil count %d not divisible by %d ranks" % (C, world))
    B = B200Backend(local)
    team = CoilTeam() if world > 1 else None
    rs = np.random.RandomState(2024)
    coord = make_traj(wl["traj"])
    maps = synth.unit_rss_maps(rs, N, C)
    mine = coil_slice(C, rank, world)
    weights = sqrt_dcf(coord) if kind == "cg" else None
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    my_maps = np.asfortranarray(maps[..., mine])
    tree = args.tree
    A = None
    if tree == "fused":
        try:
            A = sense_operator_fused(B, N, coord, my_maps, wl["oversamp"], weights=weights)
        except RuntimeError as e:                       # grid without specialised passes
            print("fused path unavailable (%s); using the six-call recipe" % e, file=sys.stderr)
            tree = "o3"
    if A is None:
        A = sense_operator_device(B, N, coord, my_maps, wl["oversamp"], weights=weights)
    AHA = normal_operator(A)
    B.barrier()
    setup_s = time.time() - t0
    setup_bytes = int(torch.cuda.max_memory_allocated())
    resident_bytes = int(torch.cuda.memory_allocated())
    dev = getattr(A, '_dev', None)
    nvox = int(np.prod(N))
    x_h = B.pinned_array((nvox, 1)); x_h[...] = synth.rand64c(rs, nvox, 1)
    y_h = B.pinned_array((nvox, 1))
    x_d = B.copy_array(np.asarray(x_h)); y_d = B.zero_array((nvox, 1), C64)
    lib = B._lib
    # cfg5: the 48-coil data set, coil-fastest, and the 12 x 48 compression matrix (SURVEY.md 8d)
    extra = None
    if kind == "cfg5":
        Cf, Msamp = wl["full_coils"], int(np.prod(coord.shape[1:]))
        calib = synth.rand64c(rs, Cf, 256)
        U = np.linalg.svd(calib.astype(np.complex128), full_matrices=False)[0][:, :C]
        Mc_d = B.copy_array(np.asfortranarray(U.conj().T.astype(C64)))
        ksp_t = torch.rand((Msamp * Cf * 2,), dtype=torch.float32, device=B._device)       # U[0,1) + i U[0,1), on the device
        from indigo_b200.backend import DevPtr
        ksp_d = B.dndarray(B, (Cf, Msamp), C64, own=False, data=DevPtr(ksp_t.data_ptr(), keep=ksp_t))
        comp_d = B.empty_array((C, Msamp), C64)
        extra = (Mc_d, ksp_d, comp_d)

    graph = None

    def apply_raw():
        if extra is not None:
            B.cgemm(extra[2], extra[0], extra[1], 1.0, 0.0, forward=True)
        AHA.eval(y_d, x_d)

    def apply():
        if graph is not None:
            graph.replay()
        else:
            apply_raw()
        if team is not None:
            team.allreduce_array(y_d)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 1)):
        apply()
    sync_all()
    if args.graph:
        # whole-apply CUDA graph (SURVEY 8f rank 3): every kernel of the apply is captured once and replayed with a
        # single launch; pays in the launch-bound regime (cfg1: ~13 launches around ~85 us of traffic)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            apply_raw()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                apply_raw()
        torch.cuda.current_stream().wait_stream(side)
        graph = g
        for _ in range(2):
            apply()
        sync_all()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    steps = args.steps
    cg_info = None
    if kind == "cg":
        # ---- timed region: a 50-iteration CG solve, device-resident scalars; a step = one iteration ----------
        want = np.asarray(x_h)
        b_h = np.asfortranarray(want / max(np.abs(want).max(), 1e-30)).astype(C64)
        nrm = power_norm(B, AHA, team, nvox, rs)
        lam = 1e-2 * nrm
        xs = np.zeros_like(b_h, order='F')
        B.cg(AHA, b_h, xs, lamda=lam, tol=0.0, maxiter=2, team=team)               # warm-up of the solver path
        sync_all()
        lib.launch_count_reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = steps
        e0.record()
        B.cg(AHA, b_h, xs, lamda=lam, tol=0.0, maxiter=iters, team=team)
        e1.record()
        sync_all()
        total_ms = e0.elapsed_time(e1)
        launches = lib.launch_count()
        applies = iters + 1                                                        # the iterations + the initial residual apply
        cg_info = {"iterations": iters, "applies": applies, "seconds_per_solve": total_ms * 1e-3, "lamda": lam,
                   "spectral_norm_estimate": nrm,
                   "note": "timed region includes the H2D of b and x0 and the D2H of the solution (Backend.cg's contract)"}
        outputs = {"solution": xs} if args.dump_outputs else None
    else:
        # ---- timed region: inputs resident in HBM --------------------------------------------------------
        lib.launch_count_reset()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sync_all()
        for a, b in ev:
            a.record(); apply(); b.record()
        sync_all()
        launches = lib.launch_count()
        total_ms = sum(a.elapsed_time(b) for a, b in ev)
        applies = steps
        outputs = None
        if args.dump_outputs and rank == 0:
            # what the last timed step handed back, read before anything else reuses the buffers
            outputs = {"image": y_d.to_host()}
            if extra is not None:
                outputs["compressed_kspace"] = extra[2].to_host()
    # ---- per-kernel timing (outside the headline region): the same kernels, each bracketed by events -----------
    timer = KernelTimer(B, torch)
    ksteps = max(3, min(steps, 10))
    if dev is not None:
        dev.probe = timer.probe
    else:
        timer.wrap_backend()
    sync_all()
    for _ in range(ksteps):
        if extra is not None:
            with timer.probe("cgemm_tc[12x48 coil compression]"):
                B.cgemm(extra[2], extra[0], extra[1], 1.0, 0.0, forward=True)
        AHA.eval(y_d, x_d)
    sync_all()
    if dev is not None:
        dev.probe = None
    # ---- end to end: host buffers, H2D + apply + D2H every step ----------------------------------------------
    def apply_on(y, x):
        if extra is not None:
            B.cgemm(extra[2], extra[0], extra[1], 1.0, 0.0, forward=True)
        AHA.eval(y, x)

    e2e = e2e_region(B, torch, dist, team, world, rank, AHA, apply, x_h, y_h, x_d, y_d, nvox, args.steps, sync_all,
                     apply_on=apply_on if (graph is None and kind != "cg") else None)
    clk = clocks.stop() if rank == 0 else None
    check = run_checks(B, A, AHA, team, world, rank, x_h, y_h, y_d, args) if args.check else None
    if world > 1:
        t = torch.tensor([total_ms, e2e["ms"], float(launches)], dtype=torch.float64, device="cuda")
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        total_ms, e2e["ms"], launches = float(tmax[0]), float(tmax[1]), int(tsum[2])
    peak, peak_src = peaks()
    fused_bytes = fused_kernel_bytes(dev) if dev is not None else {}
    if extra is not None:
        Cf, Msamp = wl["full_coils"], int(np.prod(coord.shape[1:]))
        gb = 8 * (C * Cf + Cf * Msamp + C * Msamp)
        fused_bytes["cgemm_tc[12x48 coil compression]"] = (gb, gb, "cgemm")
    traffic, traffic_src = measured_traffic(args.workload, world, C // world)
    kernels = timer.summary(peak, fused_bytes, traffic)
    if rank == 0:
        dom = kernels[0]
        line = {
            "metric": "SENSE-NUFFT A^H A applies/sec", "value": applies / (total_ms * 1e-3), "unit": "applies/s",
            "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": total_ms / applies,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "complex64 (fp32 accumulate)",
            "data": "synthetic (seeded trajectory, rand64c image and unit-RSS coil maps)",
            "config": {"workload": wl["desc"],
                       "tree": ("fused B200 recipe: expand+FFT (pruned, coil-interleaved, support windows) -> separable G' gather -> "
                                "matrix-free block G'^H gather -> IFFT+combine; 4 fused calls (8-9 kernels) replace the six calls of the -O3 tree"
                                if tree == "fused" else
                                "-O3 (examples/pics.py recipe), device-built CSR operands, six Backend calls"),
                       "parallelism": "coil-sharded x%d, NCCL all-reduce of the image" % world if world > 1 else "single GPU",
                       "cuda_graph": bool(args.graph),
                       "l2": "no explicit flush: every call streams operands far larger than L2 (grid %.1f GB)" %
                             (8.0 * np.prod([int(n * wl["oversamp"]) for n in N]) * C / world / 1e9)},
            "e2e": {"value": args.steps / (e2e["ms"] * 1e-3), "unit": "applies/s",
                    "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"], "path": e2e["path"],
                    "paths_timed": e2e["alt"]},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["gbs"], "peak": peak, "unit": "GB/s",
                         "frac": dom["frac"], "traffic": dom["dram_bytes"], "traffic_source": traffic_src,
                         "peak_source": peak_src, "share_of_step": dom["share"], "launches_per_call": dom["launches"],
                         "bytes_definition": "compulsory bytes of the formulation that runs (every operand once, windows and "
                                             "pruning included), capped at the DRAM traffic ncu measured for the kernel",
                         "frac_dram": dom["frac_dram"], "frac_replaced_call": dom["frac_replaced_call"],
                         "whole_apply": {"compulsory_bytes": int(sum(k["bytes"] for k in kernels)),
                                         "replaced_calls_bytes": int(sum(k["replaced_call_bytes"] for k in kernels)),
                                         "frac": sum(k["bytes"] for k in kernels) / (total_ms / applies) / 1e6 / peak}},
            "kernels": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in c.items()} for c in kernels],
            "clocks": clk,
            "setup": {"seconds": round(setup_s, 1), "peak_bytes_per_gpu": setup_bytes, "resident_bytes_per_gpu": resident_bytes},
        }
        try:
            # the forward gather is bound by the L1 data path, not by HBM (DESIGN.md section 4): one line request per tap,
            # 128 bytes per clock and SM; reported next to the HBM figures when it is the dominant kernel
            if dom["kernel"] == "kb_gather" and dev is not None and getattr(dev, "kb", None) is not None:
                import torch as _t
                prop = _t.cuda.get_device_properties(_t.cuda.current_device())
                taps = 125.0 * dev.M * max(1, (8 * dev.C + 127) // 128)
                l1_peak = 128.0 * prop.multi_processor_count * (clk["sm_mhz"] or 1965.0) * 1e6 / 1e9
                l1_gbs = taps * 128.0 / (dom["ms"] * 1e-3) / 1e9
                line["roofline"]["l1_path"] = {"line_requests": int(taps), "achieved": l1_gbs, "peak": l1_peak, "unit": "GB/s",
                                               "frac": l1_gbs / l1_peak,
                                               "note": "kb_gather: 125 taps per sample, one 128-byte line request each; "
                                                       "128 B/clk/SM x SMs x measured SM clock"}
        except Exception as exc:                        # never lose the line over an annotation
            line["roofline"]["l1_path"] = {"error": str(exc)[:120]}
        if cg_info:
            line["cg"] = cg_info
        if check is not None:
            line["check"] = check
        if outputs is not None:
            line["outputs"] = dump_outputs(args.dump_outputs, outputs)
        if world == 1 and not args.no_cpu_baseline and args.workload in ("cfg3", "cfg4", "cfg1", "tiny"):
            line["cpu_baseline"] = cpu_baseline("cfg3" if args.workload == "cfg4" else args.workload, steps=1)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(dirname, arrays, budget=64 << 20):
    """Writes each array as DIR/<name>.npy in float32 (complex values as (re, im) pairs), column-major order flattened.
    An array larger than its share of `budget` bytes is replaced by a fixed sample: the elements at sorted indices
    drawn without replacement by RandomState(0), written as <name>_sample.npy next to <name>_sample_index.npy
    (float64), so that two builds run with the same arguments can be compared element for element."""
    os.makedirs(dirname, exist_ok=True)
    share = budget // len(arrays) - 1024                  # room for the .npy headers
    written = {}
    for name, a in sorted(arrays.items()):
        flat = np.asarray(a).ravel(order="F")
        per = 8 if np.iscomplexobj(flat) else 4
        idx = None
        if flat.size * per > share:
            keep = share // (per + 8)
            idx = np.sort(np.random.RandomState(0).choice(flat.size, keep, replace=False))
            flat, name = flat[idx], name + "_sample"
        if np.iscomplexobj(flat):
            out = np.ascontiguousarray(flat.astype(np.complex64)).view(np.float32).reshape(-1, 2)
        else:
            out = flat.astype(np.float32)
        np.save(os.path.join(dirname, name + ".npy"), out)
        written[name] = list(out.shape)
        if idx is not None:
            np.save(os.path.join(dirname, name + "_index.npy"), idx.astype(np.float64))
            written[name + "_index"] = [int(idx.size)]
    return {"dir": dirname, "arrays": written}


def power_norm(B, AHA, team, nvox, rs, iters=6):
    """||A^H A||_2 by a few power iterations on the device (lamda of cfg4 is 1e-2 of it, SURVEY.md 8d)."""
    from indigo_b200 import synth
    v = B.copy_array(synth.rand64c(rs, nvox, 1)); w = B.zero_array((nvox, 1), C64)
    nrm = 1.0
    for _ in range(iters):
        AHA.eval(w, v)
        if team is not None:
            team.allreduce_array(w)
        nrm = float(np.sqrt(B.norm2(w)))
        B.axpby(0, v, 1.0 / max(nrm, 1e-30), w)
    return nrm


def e2e_region(B, torch, dist, team, world, rank, AHA, apply, x_h, y_h, x_d, y_d, nvox, steps, sync_all, apply_on=None):
    """The same metric through the public call with HOST buffers: every step moves the image from pinned host memory
    to the device and the result back.  N = 1: explicit copies vs evaluation on device-mapped views (faster is
    reported).  N > 1: each rank uploads its 1/N slab of the image and the slabs are all-gathered over NVLink (one
    PCIe crossing of the image per step in total instead of N), the partial images are reduce-scattered and each rank
    downloads its slab of the result: the result lands in host memory distributed by slab, like the work."""
    out = {"alt": None}
    if world == 1:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sync_all()
        for a, b in ev:
            a.record()
            x_d.copy_from(x_h)                      # pinned -> device, async on the stream
            apply()
            y_d.copy_to(y_h)                        # device -> pinned, synchronises
            b.record()
        sync_all()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        out.update(ms=ms, h2d=int(x_h.nbytes), d2h=int(y_h.nbytes),
                   path="pinned host -> cudaMemcpyAsync -> AHA.eval -> cudaMemcpyAsync -> pinned host")
        try:
            x_m, y_m = B.mapped_array(x_h), B.mapped_array(y_h)
            y_ref = np.array(y_h)
            AHA.eval(y_m, x_m); sync_all()
            err = float(np.linalg.norm(np.asarray(y_h) - y_ref) / max(np.linalg.norm(y_ref), 1e-30))
            if err > 1e-6:
                raise RuntimeError("mapped path deviates from the copy path: %.3e" % err)
            m_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            sync_all()
            for a, b in m_ev:
                a.record(); AHA.eval(y_m, x_m); b.record()
                b.synchronize()                                 # the result is in host memory before the next step starts
            sync_all()
            m_ms = sum(a.elapsed_time(b) for a, b in m_ev)
            out["alt"] = {"copy_path_ms_per_step": ms / steps, "mapped_path_ms_per_step": m_ms / steps}
            if m_ms < ms:
                out["ms"] = m_ms
                out["path"] = ("AHA.eval on device-mapped views of the pinned host buffers (B.mapped_array): H2D inside the "
                               "first pass' load, D2H inside the last pass' store")
        except Exception as exc:                                # keep the copy path's number
            out["alt"] = {"mapped_path_error": str(exc)[:200]}
        # pipelined path (a user reconstructing a series of images): two device buffers per direction and three
        # streams -- the upload of image k+1 and the download of result k-1 run under apply k.  Every step still moves
        # its image in and its result out inside the timed region; the region ends when the last result is in host memory.
        try:
            if apply_on is None:
                raise RuntimeError("not applicable (captured graph or solver step)")
            from indigo_b200.team import as_torch
            cs = torch.cuda.current_stream()
            up, down = torch.cuda.Stream(), torch.cuda.Stream()
            xb = [x_d, B.empty_array(x_d.shape, x_d.dtype)]
            yb = [y_d, B.empty_array(y_d.shape, y_d.dtype)]
            xt, yt = [as_torch(a) for a in xb], [as_torch(a) for a in yb]
            xh_t = torch.from_numpy(np.asarray(x_h).view(np.float32).reshape(-1))
            yh_t = torch.from_numpy(np.asarray(y_h).view(np.float32).reshape(-1))
            y_ref = np.array(y_h)
            e_up = [torch.cuda.Event() for _ in range(steps)]
            e_done = [torch.cuda.Event() for _ in range(steps)]
            e_down = [torch.cuda.Event() for _ in range(steps)]
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sync_all()
            t0.record(cs)
            up.wait_event(t0); down.wait_event(t0)
            for k in range(steps):
                i = k & 1
                if k >= 2:
                    up.wait_event(e_done[k - 2])                 # apply k-2 has read this input buffer
                with torch.cuda.stream(up):
                    xt[i].copy_(xh_t, non_blocking=True)
                    e_up[k].record(up)
                cs.wait_event(e_up[k])
                if k >= 2:
                    cs.wait_event(e_down[k - 2])                 # result k-2 has left this output buffer
                apply_on(yb[i], xb[i])
                e_done[k].record(cs)
                down.wait_event(e_done[k])
                with torch.cuda.stream(down):
                    yh_t.copy_(yt[i], non_blocking=True)
                    e_down[k].record(down)
            cs.wait_event(e_down[steps - 1])
            t1.record(cs)
            sync_all()
            p_ms = t0.elapsed_time(t1)
            err = float(np.linalg.norm(np.asarray(y_h) - y_ref) / max(np.linalg.norm(y_ref), 1e-30))
            if err > 1e-6:
                raise RuntimeError("pipelined path deviates from the copy path: %.3e" % err)
            out["alt"] = dict(out["alt"] or {}, pipelined_path_ms_per_step=p_ms / steps)
            if p_ms < out["ms"]:
                out["ms"] = p_ms
                out["path"] = ("series of images, double-buffered: pinned host -> device copy of image k+1 and device -> pinned "
                               "host copy of result k-1 on their own streams under AHA.eval of image k; region = first upload to "
                               "last result in host memory")
            del xb, yb, xt, yt
        except Exception as exc:
            out["alt"] = dict(out["alt"] or {}, pipelined_path_error=str(exc)[:200])
        return out
    # ---- N > 1 -------------------------------------------------------------------------------------------------
    from indigo_b200.team import as_torch
    slab = -(-nvox // world)
    pad = slab * world
    xt = torch.zeros(2 * pad, dtype=torch.float32, device="cuda")              # gathered image (padded to equal slabs)
    yt = torch.zeros(2 * pad, dtype=torch.float32, device="cuda")
    ys = torch.zeros(2 * slab, dtype=torch.float32, device="cuda")
    lo, hi = rank * slab, min(nvox, (rank + 1) * slab)
    xh_t = torch.from_numpy(np.asarray(x_h).view(np.float32).reshape(-1))      # views of the pinned host buffers
    yh_t = torch.from_numpy(np.asarray(y_h).view(np.float32).reshape(-1))
    x_flat, y_flat = as_torch(x_d), as_torch(y_d)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    sync_all()
    for a, b in ev:
        a.record()
        xt[2 * lo:2 * hi].copy_(xh_t[2 * lo:2 * hi], non_blocking=True)        # this rank's slab: pinned -> device
        dist.all_gather_into_tensor(xt, xt[2 * rank * slab:2 * (rank + 1) * slab].clone())
        x_flat.copy_(xt[:2 * nvox])
        AHA.eval(y_d, x_d)                                                    # partial image of this rank's coils
        yt[:2 * nvox].copy_(y_flat)
        dist.reduce_scatter_tensor(ys, yt, op=dist.ReduceOp.SUM)
        yh_t[2 * lo:2 * hi].copy_(ys[:2 * (hi - lo)], non_blocking=True)       # this rank's slab of the result -> pinned
        b.record()
        b.synchronize()
    sync_all()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    out.update(ms=ms, h2d=int(8 * nvox), d2h=int(8 * nvox),
               path="per rank: 1/%d slab of the image pinned host -> device, NCCL all-gather, AHA.eval on the rank's coils, NCCL "
                    "reduce-scatter, slab of the result -> pinned host (bytes are whole-job totals)" % world)
    return out


def run_checks(B, A, AHA, team, world, rank, x_h, y_h, y_d, args):
    """Correctness at the benchmarked size, outside every timed region (no oracle involved; the float64 single-output
    checks are tests/test_gpu_fullsize.py): adjointness of the operator that was timed, fused recipe against the
    six-call recipe, and -- for N > 1 -- the all-reduced image against the digest of the N = 1 run."""
    import hashlib
    from indigo_b200 import synth
    out = {}
    rs = np.random.RandomState(99)
    x = np.asarray(x_h).copy()
    nvox = x.shape[0]
    y = synth.rand64c(rs, A.shape[0], 1)
    Ax, AHy = A * x, A.H * y
    lhs = np.vdot(Ax.astype(np.complex128), y.astype(np.complex128))
    rhs = np.vdot(x.astype(np.complex128), AHy.astype(np.complex128))
    out["adjointness_rel"] = float(abs(lhs - rhs) / abs(lhs))
    AHA.eval(y_d, B.copy_array(x))
    if team is not None:
        team.allreduce_array(y_d)
    img = y_d.to_host()
    # digest: coarse fingerprint that survives the 1e-7 differences between coil partitions
    sub = img.ravel(order='F')[::997].astype(np.complex128)
    out["image_norm"] = float(np.linalg.norm(img.astype(np.complex128)))
    digest_path = os.path.join(REPO, "profiles", "digest_%s.npz" % args.workload)
    if world == 1 and not args.coils:
        if args.write_digest:
            np.savez(digest_path, sub=sub.astype(np.complex64), norm=out["image_norm"])
            out["digest"] = "written"
        if args.tree == "fused" and args.check_tree:
            from indigo_b200.sense import sense_operator_device, normal_operator
            # six-call recipe on device-built CSR operands of the same problem
            wl = WORKLOADS[args.workload]
            maps = synth.unit_rss_maps(np.random.RandomState(2024), wl["N"], wl["C"])
            Au = sense_operator_device(B, wl["N"], make_traj(wl["traj"]), maps, wl["oversamp"])
            ref = normal_operator(Au) * x
            out["fused_vs_six_call_rel"] = float(np.linalg.norm(img - ref) / np.linalg.norm(ref))
    if os.path.exists(digest_path) and not args.coils:
        d = np.load(digest_path)
        out["vs_n1_digest_rel"] = float(np.linalg.norm(sub - d["sub"]) / np.linalg.norm(d["sub"]))
        out["vs_n1_norm_rel"] = float(abs(out["image_norm"] - float(d["norm"])) / float(d["norm"]))
    bad = [k for k, v in out.items() if k.endswith("_rel") and v > 1e-5]
    out["passed"] = not bad
    if bad and rank == 0:
        print("CHECK FAILED: %s" % {k: out[k] for k in bad}, file=sys.stderr)
    return out


# --------------------------------------------------------------------------- CPU baseline / reference arm
def cpu_baseline(workload, steps=1, warmup=0):
    """The reference's CPU path on a bounded sample of the workload.

    Sample: CS coils on the full oversampled grid (FFT + IFFT + P expand/combine) and the gridding SpMM pair on every
    `frac`-th spoke with the same CS coils as right-hand sides.  One apply = (C/CS) x [FFT part] + (C/CS) x frac x
    [gridding part]: every term is linear in the coil count and in the number of samples.  Two sets of numbers:
      * multi-threaded: SpMM through the reference's own OpenMP kernel (_customcpu.c:14-114, compiled unchanged into
        oracle/_ref) with OMP_NUM_THREADS = os.cpu_count(), FFTs through scipy.fft with workers = os.cpu_count()
        (pocketfft, the library numpy calls, threaded over the batch) -- the headline `value`;
      * single-threaded numpy/scipy exactly as indigo/backends/np.py issues them (`single_thread`)."""
    from indigo_b200 import synth
    from oracle import np_oracle as K
    from oracle import sense as osense
    import scipy.fft as sfft

    wl = WORKLOADS[workload]
    N, C = wl["N"], wl["C"]
    threads = os.cpu_count() or 1
    frac = 64 if workload == "cfg3" else 1
    CS = 4 if C >= 4 else C
    coord = make_traj(wl["traj"])[:, :, ::frac]            # every frac-th spoke: same angular coverage
    rs = np.random.RandomState(2024)
    maps = synth.unit_rss_maps(rs, N, CS)
    op = osense.SenseOperator(N, coord, maps, wl["oversamp"])
    ref = K.load_ref_customcpu()
    nvox, on = int(np.prod(N)), int(np.prod(op.oN))
    x = synth.rand64c(rs, nvox, 1)
    os.environ["OMP_NUM_THREADS"] = str(threads)

    def spmm(y, A, xin, adjoint, multi):
        if multi and ref is not None and xin.shape[1] > 1:
            ref.csrmm(adjoint, A.shape[0], xin.shape[1], A.shape[1], 1.0 + 0j, A.data, A.indices, A.indptr,
                      xin, xin.shape[0], 0j, y, y.shape[0], False)
        else:
            K.ccsrmm(y, A.shape, A.indices, A.indptr, A.data, xin, 1, 0, adjoint=adjoint)

    def one(multi):
        t = {}
        g = np.zeros((on * CS, 1), dtype=C64, order="F")
        t0 = time.perf_counter(); spmm(g, op.PH, x, True, False); t["P"] = time.perf_counter() - t0
        G4 = g.reshape(op.oN + (CS,), order="F"); F4 = np.zeros_like(G4, order="F")
        t0 = time.perf_counter()
        if multi:
            F4[...] = sfft.fftn(G4, axes=(0, 1, 2), workers=threads)
        else:
            K.fftn(F4, G4)
        t["fft"] = time.perf_counter() - t0
        f = F4.reshape((on, CS), order="F")
        k = np.zeros((op.M, CS), dtype=C64, order="F")
        t0 = time.perf_counter(); spmm(k, op.G, f, False, multi); t["G"] = time.perf_counter() - t0
        t0 = time.perf_counter(); spmm(f, op.G, k, True, multi); t["GH"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        if multi:
            G4[...] = sfft.ifftn(F4, axes=(0, 1, 2), workers=threads) * float(on)
        else:
            K.ifftn(G4, F4)
        t["ifft"] = time.perf_counter() - t0
        yv = np.zeros((nvox, 1), dtype=C64, order="F")
        t0 = time.perf_counter(); spmm(yv, op.PH, G4.reshape((on * CS, 1), order="F"), False, False); t["PH"] = time.perf_counter() - t0
        return t

    def full_apply_seconds(t):
        return (C / CS) * (t["P"] + t["fft"] + t["ifft"] + t["PH"]) + (C / CS) * frac * (t["G"] + t["GH"])

    for _ in range(warmup):
        one(True)
    tm = [one(True) for _ in range(max(1, steps))]
    tm = {k: float(np.median([d[k] for d in tm])) for k in tm[0]}
    ts = one(False)
    full_m, full_s = full_apply_seconds(tm), full_apply_seconds(ts)
    step_m = sum(tm.values())
    kind_ = "reference" if ref is not None else "port"
    return {"value": 1.0 / full_m, "unit": "applies/s", "cores": threads if ref is not None else 1, "kind": kind_,
            "threads_available": threads, "omp_num_threads": threads, "extrapolated": True,
            "units_per_step": step_m / full_m, "seconds_per_step": step_m,
            "sample": "%d of %d coils on the full %s grid (scipy.fft workers=%d: fft %.2fs, ifft %.2fs; P pair %.2fs) + "
                      "gridding pair with %d right-hand sides on 1/%d of the spokes through the reference's OpenMP "
                      "_customcpu.csrmm (%d threads: G %.3fs, G^H %.3fs); extrapolated linearly to %d coils x all samples "
                      "= %.1f s per apply" % (CS, C, "x".join(str(v) for v in op.oN), threads, tm["fft"], tm["ifft"],
                                              tm["P"] + tm["PH"], CS, frac, threads, tm["G"], tm["GH"], C, full_m),
            "seconds_per_apply": full_m, "parts": tm,
            "single_thread": {"value": 1.0 / full_s, "seconds_per_apply": full_s, "cores": 1, "parts": ts,
                              "what": "numpy pocketfft + scipy csr_matvecs as indigo/backends/np.py calls them"}}


def run_reference(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = "cfg3" if args.workload in ("cfg4", "cfg5") else args.workload
    wl = WORKLOADS[workload]
    t0 = time.time()
    nsteps = max(1, min(args.steps, 3))
    base = cpu_baseline(workload, steps=nsteps, warmup=min(args.warmup, 1))
    # a step of this arm is the bounded sample; value = applies per step / seconds per step
    line = {"impl": "reference", "metric": "SENSE-NUFFT A^H A applies/sec", "value": base["value"], "unit": "applies/s",
            "n_gpus": world, "steps": nsteps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * base["seconds_per_step"],
            "units_per_step": base["units_per_step"], "extrapolated": True,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "complex64",
            "data": "synthetic (same seeded generators as the B200 arm)",
            "config": {"workload": wl["desc"], "tree": "-O3", "parallelism": "host CPU, %d threads" % base["cores"]},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "applies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": round(time.time() - t0, 1)}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--coils", type=int, default=0,
                    help="development only: override the workload's coil count (e.g. 2 = the per-GPU shard of cfg3 at 8 GPUs)")
    ap.add_argument("--tree", default="fused", choices=["fused", "o3"],
                    help="fused: backend-specific fused recipe (default); o3: the reference's six Backend calls")
    ap.add_argument("--graph", action="store_true", help="replay the apply as one CUDA graph (launch-bound workloads)")
    ap.add_argument("--check", action="store_true", help="correctness checks at the benchmarked size, outside the timed regions")
    ap.add_argument("--check-tree", action="store_true", help="with --check at N=1: also compare with the six-call recipe")
    ap.add_argument("--write-digest", action="store_true", help="with --check at N=1: store the image digest N>1 runs compare with")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all; "
                         "larger outputs as a fixed seeded sample)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
