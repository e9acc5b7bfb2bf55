#!/usr/bin/env python3
"""bench.py -- headline benchmark: SPH particles/sec projected to map (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            this repository's CUDA path
  python bench.py --impl reference [...]                          the reference's own CPU path (oracle/_ref)
  python bench.py [...] --dump-outputs DIR                        also writes the last timed step's map to DIR (dump_map)

Workload (BASELINE.json configs[2], the one north_star quotes its target on): synthetic 512^3 = 134 217 728 gas
particles (recipe S1 of SURVEY.md 8(d): jittered lattice in a unit periodic box, seed 12345) projected onto a
4096 x 4096 mass map, M4 cubic spline (the reference kernel), smoothing lengths h = d_48 from the periodic k-NN
(io/SWIFT/_SnapshotSWIFT.py:62-83 convention; a particle then covers ~4000 pixels, so the accumulation is
FP32-issue-bound, not HBM-bound -- SURVEY 7.2 H1; the `regimes` key shows the HBM-bound end of the same path).
A "step" is one full pass of the hot path over the particle set: bin -> scan -> emit -> sort -> pair records ->
tile accumulate (-> NCCL sum-reduce of the partial maps when N > 1).  N > 1 is STRONG scaling: the same 134 M
particles sharded by index over the ranks (the reference's per-rank particle split, io/EAGLE/_SnapshotEAGLE.py:120-130).

One JSON line is printed by rank 0: value = device-resident throughput, e2e = the same through the public host-buffer
API (H2D + D2H inside the timed region), parity = the GPU map against the CPU oracle on a window of the very map
that was timed, roofline = the dominant kernel against the measured HBM peak, cpu_baseline = the oracle's OpenMP
restatement on the host cores.  Sub-records (N = 1): c2 (configs[1]), c4 (configs[3], 3-D gridding), c5 (configs[4],
k-NN; also at N > 1, queries sharded over the ranks).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "SPH particles/sec projected to map"
UNIT = "particles/s"
WIN0 = 0.5            # parity / CPU windows start at map coordinate 0.5 on both axes (box interior: no periodic wrap)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline measurement (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the map the last one computed to DIR/mass_map.npy (see dump_map)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=512, help="lattice size (particles = n^3, all ranks together)")
    ap.add_argument("--npix", type=int, default=4096)
    ap.add_argument("--k", type=int, default=48)
    ap.add_argument("--h-scale", type=float, default=1.0, help="multiplies h = d_k (footprint sweep)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="full footprint sweep (h scale 1/64 .. 1) instead of the three default regimes")
    ap.add_argument("--no-regimes", action="store_true", help="skip the footprint regimes")
    ap.add_argument("--no-sub", action="store_true", help="skip the c2 / c4 / c5 sub-records")
    ap.add_argument("--sub", default="c5,c2,c4", help="which sub-records to run")
    ap.add_argument("--cpu-target-s", type=float, default=12.0)
    ap.add_argument("--c5-full-n", type=int, default=1024, help="lattice size of the full-size config-5 record (8 GPUs, or --sub c5full)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the map of this repository's CUDA path; it does not apply to --impl reference")
    return args


DUMP_BYTES = 32 << 20     # a larger map is dumped as a fixed sample of this many bytes of its pixels


def dump_map(dirname, img):
    """Write the float64 map `img` (device tensor) to DIR/mass_map.npy so that two builds run with the same arguments can be
    compared pixel for pixel: the whole (nx, ny) map when it fits DUMP_BYTES, else the pixels at DUMP_BYTES / 8 flat indices
    drawn without replacement by np.random.default_rng(0), in ascending order (the same pixels for the same map size)."""
    import torch
    flat = img.reshape(-1)
    if flat.numel() * 8 > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_BYTES // 8, replace=False))
        host = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    else:
        host = img.cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "mass_map.npy"), host.astype(np.float64, copy=False))


def hbm_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def workload_config(args, world):
    """identical in both arms (the reference arm prints the same dict)"""
    N = args.n ** 3
    return {"workload": f"S1 {args.n}^3 = {N} particles -> {args.npix}^2 projected mass map, cubic spline (reference kernel), axis Z, "
                        f"h = d_{args.k} (periodic k-NN, self included)",
            "h_scale": args.h_scale,
            "l2": f"inputs {N * 40 / 1e6:.0f} MB per step exceed the 126 MB L2, no explicit flush",
            "parallelism": (f"particles sharded by index over {world} GPU(s) (strong scaling), NCCL sum-reduce of the partial maps"
                            if world > 1 else "1 GPU")}


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """number of samples read so far (brackets the timed region)"""
        return len(self.lines)

    def stop(self, first=0, last=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        window = self.lines[first:(last if last is not None else len(self.lines)) + 1]
        if not window:
            window = self.lines[max(0, first - 4):first + 1]
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------- windows of the map
def window_bounds(npix, wp):
    """a wp x wp pixel window of the npix^2 map over [0,1]^2 whose lower corner is the pixel at WIN0; exact in float64"""
    p0 = int(round(WIN0 * npix))
    lo = p0 / npix
    return p0, lo, (p0 + wp) / npix


def select_column(pos, lo, hi, margin):
    """rows of pos whose in-plane (x, y) coordinates lie within `margin` of the window [lo, hi)^2"""
    return ((pos[:, 0] >= lo - margin) & (pos[:, 0] < hi + margin) & (pos[:, 1] >= lo - margin) & (pos[:, 1] < hi + margin))


def oracle_window(oracle, pos, h, props, npix, wp, kernel="cubic_spline_3d"):
    """float64 oracle map of the wp^2 window (all particles that can touch it must be in pos); returns (map(s), seconds)"""
    _, lo, hi = window_bounds(npix, wp)
    t0 = time.perf_counter()
    ref = oracle.project2d(pos, h, props, (wp, wp), 2, lo, hi, lo, hi, kernel=kernel, nthreads=0)
    return ref, time.perf_counter() - t0


def parity_of(gpu_crop, ref):
    num = float(np.linalg.norm(gpu_crop - ref)); den = float(np.linalg.norm(ref))
    return {"rel_l2": num / den if den > 0 else num, "total_rel": abs(float(gpu_crop.sum()) - float(ref.sum())) / abs(float(ref.sum())),
            "support_equal": bool(np.array_equal(gpu_crop != 0, ref != 0))}


# ---------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """--impl reference: the reference's own CPU implementation (oracle/_ref; serial by construction,
    tools/projections/_projector.py:111) on a bounded sample of the same config: one 32 x 32-pixel chunk of the 4096^2 map
    (the reference's own unit of work, chunk_size = 32) fed every particle of the 512^3 set that can touch it, with the same
    h rule as the CUDA arm (h = d_48 of the periodic k-NN, here from scipy on the column of particles around the window --
    bit-equal to the full-box search).  value = particles-equivalent per second: N * (window area / map area) / seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from astro_sph_tools_b200 import synthetic
    from scipy.spatial import cKDTree
    n, npix, k = args.n, args.npix, args.k
    N = n ** 3
    wp = 32
    _, lo, hi = window_bounds(npix, wp)
    h_cap = 1.25 * synthetic.s1_h_lattice_estimate(n, k)          # bound on d_k of the jittered lattice (checked below)
    reach = 2.0 * h_cap * max(args.h_scale, 1.0)                  # a particle further than this from the window cannot touch it
    col = []
    for _, _, blk in synthetic.s1_blocks(n, 1.0, 12345):
        col.append(blk[select_column(blk, lo, hi, reach + h_cap)])  # + h_cap: every neighbour of the particles kept below
    col = np.ascontiguousarray(np.concatenate(col))
    inner = select_column(col, lo, hi, reach)
    hk = cKDTree(col, boxsize=[0.0, 0.0, 1.0]).query(col[inner], k=k, workers=-1)[0][:, k - 1]
    assert hk.max() <= h_cap, "window superset too narrow for the k-NN h"
    p = np.ascontiguousarray(col[inner]); hh = hk * args.h_scale; a = np.full(len(hh), 1.0 / N)
    kind = "reference"
    try:
        mod, Axes = oracle.reference_module()
        def step():
            return mod.create_image(p, hh, a, (wp, wp), 32, Axes.Z, lo, hi, lo, hi)
        cores = 1
    except Exception:
        kind = "port"
        cores = oracle.max_threads()
        def step():
            return oracle.project2d(p, hh, a, (wp, wp), 2, lo, hi, lo, hi)
    for _ in range(args.warmup):
        step()
    t0 = time.time()
    for _ in range(args.steps):
        img = step()
    dt = (time.time() - t0) / max(args.steps, 1)
    equiv = N * (wp / npix) ** 2
    val = equiv / dt
    sample = (f"one {wp}x{wp}-pixel chunk of the {npix}^2 map at [{lo:g},{hi:g})^2 with all {len(hh)} particles of the {n}^3 set within "
              f"2 h_cap of it (halo included), h = d_{k} from scipy on that column (bit-equal to the full periodic search); "
              f"{dt:.2f} s per create_image call; value = N * (window area / map area) / seconds = {equiv:.0f} particles-equivalent per call; "
              f"sum(img)*A_pix = {float(img.sum()) / npix ** 2:.6e}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": workload_config(args, max(args.gpus, 1)),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------- helpers of the CUDA arm
class Ctx:
    pass


def timed_device(ctx, fn, steps, warm):
    """CUDA events around `steps` calls on the current stream, barrier + synchronize on both sides, max over ranks -> ms per step"""
    import torch
    import torch.distributed as dist
    for _ in range(warm):
        fn()
    ctx.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    ctx.sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps


def timed_wall(ctx, fn, steps, warm):
    """host wall clock around `steps` calls of a host-buffer API, barrier + synchronize on both sides, max over ranks -> ms"""
    import torch
    import torch.distributed as dist
    res = None
    for _ in range(warm):
        res = fn()
    ctx.sync_all()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = fn()
    ctx.sync_all()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    return float(dt.item()) / steps * 1e3, res


def pin(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def sub_c5(ctx, args, pos_all_d, peak):
    """configs[4]: smoothing-length k-NN, k = 48, periodic.  1 GPU: the workload's own 512^3 set (and 256^3);
    N GPUs: positions replicated, queries sharded by index.  CPU beside it: scipy cKDTree.query (the reference's arithmetic)."""
    import torch
    from astro_sph_tools_b200 import distributed as astd, synthetic
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    sol = SmoothingLengthSolver(device=ctx.dev)
    n, k = args.n, args.k
    N = n ** 3
    lo, hi = astd.shard_bounds(N, ctx.world, ctx.rank)
    q = dict(q_begin=lo, q_count=hi - lo) if ctx.world > 1 else {}
    ms = timed_device(ctx, lambda: sol.solve(pos_all_d, k, 1.0, **q), 2, 1)
    rec = {"config": f"k-NN k={k} periodic, S1 {n}^3 = {N} particles" +
                     (f", positions replicated, queries sharded over {ctx.world} GPUs" if ctx.world > 1 else ", 1 GPU"),
           "ms": ms, "queries_per_s": N / (ms * 1e-3), "n_gpus": ctx.world,
           "roofline": {"bound": "hbm", "achieved": N * 32 / (ms * 1e-3) / 1e9, "peak": peak * ctx.world, "unit": "GB/s",
                        "frac": N * 32 / (ms * 1e-3) / 1e9 / (peak * ctx.world), "algorithmic_bytes": N * 32,
                        "note": "N*(24+8) bytes; the selection kernel evaluates ~585 float32 candidate distances per query twice (histogram pass, band pass): FP32-issue / shared-memory bound, DRAM traffic ~= the input (profiles/r02_v13_ncu_knn_select.txt)"}}
    if ctx.world > 1:
        # the same search WITHOUT replicating the positions: slabs of equal count along x + ghost zones, one all-to-all of
        # positions and one of results (distributed.smoothing_lengths_slabs); must give the very same bits
        import torch.distributed as dist
        pos_loc = pos_all_d[lo:hi].contiguous()
        f = lambda: astd.smoothing_lengths_slabs(pos_loc, k, 1.0, solver=sol, return_stats=True)
        ms_s = timed_device(ctx, f, 2, 1)
        h_s, st = f()
        h_r = sol.solve(pos_all_d, k, 1.0, **q)
        bad = (h_s != h_r).sum().to(torch.int64).reshape(1)
        dist.all_reduce(bad, op=dist.ReduceOp.SUM)
        rec["slabs_with_ghost_zones"] = {"ms": ms_s, "queries_per_s": N / (ms_s * 1e-3), "iterations": st["iterations"],
                                         "ghost_fraction_rank0": st["ghost_fraction"], "local_set_rank0": st["local_set"],
                                         "mismatches_vs_replicated_search": int(bad.item()),
                                         "note": "includes the exchange of positions and results (NCCL all-to-all) and the slab plan"}
        del pos_loc, h_s, h_r
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline:
        from scipy.spatial import cKDTree
        ns = 128
        pos_s, _ = synthetic.s1_positions(ns)
        t0 = time.perf_counter(); tree = cKDTree(pos_s, boxsize=1.0); t_build = time.perf_counter() - t0
        rng = np.random.default_rng(5)
        q1 = rng.choice(len(pos_s), 60000, replace=False)
        t0 = time.perf_counter(); d1 = tree.query(pos_s[q1], k=k, workers=1)[0][:, k - 1]; t1 = time.perf_counter() - t0
        qa = rng.choice(len(pos_s), 400000, replace=False)
        t0 = time.perf_counter(); da = tree.query(pos_s[qa], k=k, workers=-1)[0][:, k - 1]; ta = time.perf_counter() - t0
        hs = sol.solve(torch.from_numpy(pos_s).to(ctx.dev), k, 1.0).cpu().numpy()
        rec["cpu_baseline"] = {"value": len(q1) / t1, "value_all_cores": len(qa) / ta, "unit": "queries/s", "cores": 1,
                               "cores_all": os.cpu_count(), "kind": "reference",
                               "sample": f"scipy.spatial.cKDTree(S1 {ns}^3, boxsize=1).query(k={k}): 60000 queries workers=1 in {t1:.2f} s, "
                                         f"400000 queries workers=-1 in {ta:.2f} s; tree build {t_build:.2f} s (not counted)"}
        rec["parity"] = {"bit_equal_to_scipy": bool(np.array_equal(hs[q1], d1) and np.array_equal(hs[qa], da)), "queries": int(len(q1) + len(qa))}
    sol._ws = None
    return rec


def sub_c5_full(ctx, args, peak, n=1024):
    """configs[4] as worded: k-NN (k = 48, periodic) on 1024^3 = 1.07e9 particles across the GPUs of the box.  Every rank
    generates ITS index range of the jittered lattice on the device (x-planes, counter-free torch CUDA generator seeded per rank:
    the set is reproducible per (n, world)), nothing is replicated: slabs + ghost zones, one all-to-all of positions, one of
    results (distributed.smoothing_lengths_slabs).  Parity: h of a cube inside rank 0's slab against scipy on that cube + margin."""
    import torch
    import torch.distributed as dist
    from astro_sph_tools_b200 import distributed as astd, synthetic
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    k = args.k
    N = n ** 3
    planes = n // ctx.world
    p0 = ctx.rank * planes
    g = torch.Generator(device=ctx.dev); g.manual_seed(777 + ctx.rank)
    ax = (torch.arange(n, dtype=torch.float64, device=ctx.dev) + 0.5) / n
    pos = torch.empty((planes * n * n, 3), dtype=torch.float64, device=ctx.dev)
    step = max(1, planes // 16)
    for i0 in range(0, planes, step):                           # slab by slab: no slab-sized temporaries
        i1 = min(planes, i0 + step)
        blk = torch.stack(torch.meshgrid(ax[p0 + i0:p0 + i1], ax, ax, indexing="ij"), dim=-1).reshape(-1, 3)
        blk = torch.remainder(blk + torch.randn(blk.shape, dtype=torch.float64, device=ctx.dev, generator=g) * (0.2 / n), 1.0)
        blk[blk >= 1.0] = 0.0
        pos[i0 * n * n:i1 * n * n] = blk
    del blk
    torch.cuda.empty_cache()
    sol = SmoothingLengthSolver(device=ctx.dev)
    f = lambda: astd.smoothing_lengths_slabs(pos, k, 1.0, solver=sol, return_stats=True)
    ms = timed_device(ctx, f, 1, 1)
    h, st = f()
    rec = {"config": f"k-NN k={k} periodic, jittered lattice {n}^3 = {N} particles generated per rank on the device, slabs + ghost zones "
                     f"over {ctx.world} GPUs (nothing replicated)",
           "ms": ms, "queries_per_s": N / (ms * 1e-3), "n_gpus": ctx.world, "iterations": st["iterations"],
           "ghost_fraction_rank0": st["ghost_fraction"], "local_set_rank0": st["local_set"],
           "roofline": {"bound": "hbm", "achieved": N * 32 / (ms * 1e-3) / 1e9, "peak": peak * ctx.world, "unit": "GB/s",
                        "frac": N * 32 / (ms * 1e-3) / 1e9 / (peak * ctx.world), "algorithmic_bytes": N * 32}}
    if ctx.rank == 0:
        from scipy.spatial import cKDTree
        h_cap = 1.25 * synthetic.s1_h_lattice_estimate(n, k)
        c = (0.5 + planes // 2) / n                               # a cube in the middle of rank 0's slab (x), box centre (y, z)
        half = 12.0 / n
        lo = torch.tensor([c - half, 0.5 - half, 0.5 - half], dtype=torch.float64, device=ctx.dev); hi = lo + 2 * half
        near = ((pos > lo - h_cap) & (pos < hi + h_cap)).all(dim=1)
        P = pos[near].cpu().numpy(); H = h[near].cpu().numpy()
        inner = np.all((P > lo.cpu().numpy()) & (P < hi.cpu().numpy()), axis=1)
        ref = cKDTree(P).query(P[inner], k=k, workers=-1)[0][:, k - 1]
        ok = bool(ref.max() <= h_cap and np.array_equal(H[inner], ref)) if c - half - h_cap > 0 and c + half + h_cap < planes / n else None
        rec["parity"] = {"bit_equal_to_scipy": ok, "queries": int(inner.sum()), "note": "cube of 24^3 lattice cells inside rank 0's slab + margin"}
    sol._ws = None
    del pos, h
    torch.cuda.empty_cache()
    return rec


def sub_c2(ctx, args, peak):
    """configs[1]: S1 256^3 -> 2048^2 mass + temperature-weighted maps in one pass (round 1's headline workload)"""
    import torch
    import oracle
    from astro_sph_tools_b200 import CoordinateAxes, synthetic
    from astro_sph_tools_b200.tools.projections import Projector2D, create_images, quartic_spline_kernel
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    n, npix, k = 256, 2048, args.k
    pos, rng = synthetic.s1_positions(n)
    N = len(pos)
    m = np.full(N, 1.0 / N); mT = m * 10.0 ** rng.uniform(4.0, 7.0, N)
    pos_d = torch.from_numpy(pos).to(ctx.dev)
    sol = SmoothingLengthSolver(device=ctx.dev)
    h_d = sol.solve(pos_d, k, 1.0)
    sol._ws = None
    props_d = [torch.from_numpy(m).to(ctx.dev), torch.from_numpy(mT).to(ctx.dev)]
    eng = Projector2D(device=ctx.dev)
    out = torch.empty((2, npix, npix), dtype=torch.float64, device=ctx.dev)
    size, bounds = (npix, npix), (0.0, 1.0, 0.0, 1.0)
    f = lambda: eng.project(pos_d, h_d, props_d, size, CoordinateAxes.Z, bounds, "cubic_spline_3d", out=out)
    ms = timed_device(ctx, f, 5, 3)
    eng.project(pos_d, h_d, props_d, size, CoordinateAxes.Z, bounds, "cubic_spline_3d", out=out, timing=True)
    stage = [float(x) for x in eng.last_stats["stage_ms"]]
    alg = N * 48 + 2 * npix * npix * 8
    h = h_d.cpu().numpy()
    rec = {"config": f"S1 {n}^3 = {N} particles -> {npix}^2 mass + T-weighted maps (one pass), cubic spline, h = d_{k}, 1 GPU",
           "ms": ms, "particles_per_s": N / (ms * 1e-3), "stage_ms": stage, "pairs": eng.last_stats["n_pairs"],
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes": alg}}
    # SURVEY 8(d): the same particles in a fixed random order (the cost of an incoherent input order; presort="auto" looks at a
    # sample of the order and projects a tile-ordered copy, "never" runs on the order as given)
    perm = torch.randperm(N, device=ctx.dev, generator=torch.Generator(device=ctx.dev).manual_seed(1))
    pos_r, h_r, props_r = pos_d[perm].contiguous(), h_d[perm].contiguous(), [q[perm].contiguous() for q in props_d]
    out_r = torch.empty_like(out)
    ro = {}
    for mode in ("auto", "never"):
        fr = lambda: eng.project(pos_r, h_r, props_r, size, CoordinateAxes.Z, bounds, "cubic_spline_3d", out=out_r, presort=mode)
        ro[mode] = timed_device(ctx, fr, 3, 2)
        if mode == "auto":
            ro["reordered"] = bool(eng.last_stats["reordered"])
            ro["rel_l2_vs_lattice_order_map"] = float(((out_r - out).norm() / out.norm()).item())
    rec["random_order"] = {"ms_presort_auto": ro["auto"], "ms_presort_never": ro["never"], "reordered": ro["reordered"],
                           "rel_l2_vs_lattice_order_map": ro["rel_l2_vs_lattice_order_map"]}
    del pos_r, h_r, props_r, out_r, perm
    # parity on a window of the timed maps
    wp = 128
    p0, lo, hi = window_bounds(npix, wp)
    sel = select_column(pos, lo, hi, 2.0 * float(h.max()))
    ref, _ = oracle_window(oracle, pos[sel], h[sel], np.stack([m[sel], mT[sel]]), npix, wp)
    crop = out[:, p0:p0 + wp, p0:p0 + wp].cpu().numpy()
    rec["parity"] = {"window": f"{wp}^2 pixels at [{lo:g},{hi:g})^2, {int(sel.sum())} particles", "mass": parity_of(crop[0], ref[0]),
                     "mass_T": parity_of(crop[1], ref[1])}
    if not args.no_e2e:
        pp, hp, mp, tp = pin(pos), pin(h), pin(m), pin(mT)
        ms_e, _ = timed_wall(ctx, lambda: create_images(pp, hp, [mp, tp], size, 32, CoordinateAxes.Z, *bounds, kernel_func=quartic_spline_kernel), 3, 2)
        rec["e2e"] = {"ms": ms_e, "particles_per_s": N / (ms_e * 1e-3), "h2d_bytes_per_step": N * 48, "d2h_bytes_per_step": 2 * npix * npix * 8}
    return rec


def nfw_positions_device(torch, dev, N, n_haloes=512, seed=12345, background=0.3):
    """recipe S2 of SURVEY 8(d) on the device (haloes with NFW profiles, c = 5..10, + 30 % uniform background, unit box)"""
    g = torch.Generator(device=dev); g.manual_seed(seed)
    U = lambda *s: torch.rand(*s, dtype=torch.float64, device=dev, generator=g)
    n_bg = int(N * background); n_h = N - n_bg
    centres = U(n_haloes, 3); conc = 5.0 + 5.0 * U(n_haloes); rvir = 0.04 * (0.5 + U(n_haloes))
    which = torch.randint(0, n_haloes, (n_h,), device=dev, generator=g)
    c = conc[which]
    mfun = lambda x: torch.log1p(x) - x / (1.0 + x)
    target = U(n_h) * mfun(c)
    lo = torch.zeros_like(c); hi = c.clone()
    for _ in range(50):                                   # inverse CDF of the NFW enclosed mass by bisection
        mid = 0.5 * (lo + hi)
        big = mfun(mid) > target
        hi = torch.where(big, mid, hi); lo = torch.where(big, lo, mid)
    r = 0.5 * (lo + hi) / c * rvir[which]
    v = torch.randn(n_h, 3, dtype=torch.float64, device=dev, generator=g)
    v = v / v.norm(dim=1, keepdim=True)
    pos = torch.cat([centres[which] + r[:, None] * v, U(n_bg, 3)])
    pos = torch.remainder(pos, 1.0)
    pos[pos >= 1.0] = 0.0
    return pos[torch.randperm(N, device=dev, generator=g)].contiguous()


def sub_c4(ctx, args, peak):
    """configs[3]: 3-D voxel gridding of 256^3 NFW-clustered particles onto a 512^3 grid (periodic), h = d_48"""
    import torch
    import oracle
    from astro_sph_tools_b200.tools.projections import Gridder3D
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    n, k = 256, args.k
    N = n ** 3
    ng = 2 * n
    pos_d = nfw_positions_device(torch, ctx.dev, N)
    sol = SmoothingLengthSolver(device=ctx.dev)
    h_d = sol.solve(pos_d, k, 1.0)
    sol._ws = None
    m_d = torch.full((N,), 1.0 / N, dtype=torch.float64, device=ctx.dev)
    g = Gridder3D(device=ctx.dev)
    out = torch.empty((ng,) * 3, dtype=torch.float64, device=ctx.dev)
    f = lambda: g.grid(pos_d, h_d, m_d, (ng,) * 3, (0, 0, 0), (1, 1, 1), periodic=True, box=1.0, out=out)
    ms = timed_device(ctx, f, 3, 2)
    g.grid(pos_d, h_d, m_d, (ng,) * 3, (0, 0, 0), (1, 1, 1), periodic=True, box=1.0, out=out, timing=True)
    alg = N * 40 + ng ** 3 * 8
    rec = {"config": f"S2 NFW-clustered {n}^3 = {N} particles (512 haloes + 30 % background) -> {ng}^3 voxels, periodic, cubic spline, h = d_{k}, 1 GPU",
           "ms": ms, "particles_per_s": N / (ms * 1e-3), "stage_ms": [float(x) for x in g.last_stats["stage_ms"]],
           "pairs": g.last_stats["n_pairs"], "n_huge": g.last_stats["n_huge"], "mass_sum": float(out.sum().item()) / ng ** 3,
           "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes": alg}}
    # parity + CPU baseline: the oracle on a window of the grid around the densest halo voxel ... (interior, so no wrap)
    pos = pos_d.cpu().numpy(); h = h_d.cpu().numpy()
    wv = 48
    v0 = ng // 2 - wv // 2
    lo, hi = v0 / ng, (v0 + wv) / ng
    r2 = 2.0 * h
    sel = np.all((pos + r2[:, None] > lo) & (pos - r2[:, None] < hi), axis=1)
    assert lo - 2 * h[sel].max() > 0.0 and hi + 2 * h[sel].max() < 1.0
    mm = np.full(int(sel.sum()), 1.0 / N)
    t0 = time.perf_counter()
    ref = oracle.grid3d(pos[sel], h[sel], mm, (wv,) * 3, (lo,) * 3, (hi,) * 3, nthreads=0)
    t_cpu = time.perf_counter() - t0
    crop = out[v0:v0 + wv, v0:v0 + wv, v0:v0 + wv].cpu().numpy()
    rec["parity"] = dict(parity_of(crop, ref), window=f"{wv}^3 voxels at [{lo:g},{hi:g})^3, {int(sel.sum())} particles")
    if not args.no_cpu_baseline:
        rec["cpu_baseline"] = {"value": N * (wv / ng) ** 3 / t_cpu, "unit": UNIT, "cores": oracle.max_threads(), "kind": "port",
                               "sample": f"oracle/sph_oracle.c OpenMP float64 scatter on the {wv}^3-voxel window with its {int(sel.sum())} "
                                         f"contributing particles in {t_cpu:.2f} s; value = N * (window volume / grid volume) / seconds"}
    return rec


# ---------------------------------------------------------------------------------------------- the CUDA arm
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from astro_sph_tools_b200 import CoordinateAxes, distributed as astd, synthetic
    from astro_sph_tools_b200.tools.projections import Projector2D, quartic_spline_kernel
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver

    ctx = Ctx()
    ctx.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.rank = rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    ctx.dev = dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    ctx.sync_all = sync_all
    peak, peak_src = hbm_peak()
    t_setup = time.time()

    # ---- inputs: every rank draws the whole S1 set block by block (identical on all ranks), keeps its own index range on
    # the host, uploads everything once for the k-NN (positions replicated); rank 0 also keeps the column around the window
    n, npix, k = args.n, args.npix, args.k
    N = n ** 3
    lo_i, hi_i = astd.shard_bounds(N, world, rank)
    n_loc = hi_i - lo_i
    wp_max = max(32, min(1024, npix // 4))
    _, wlo, whi_max = window_bounds(npix, wp_max)
    h_cap = 1.25 * synthetic.s1_h_lattice_estimate(n, k)
    pos_all_d = torch.empty((N, 3), dtype=torch.float64, device=dev)
    pos_loc = torch.empty((n_loc, 3), dtype=torch.float64, pin_memory=True).numpy()
    col = []
    for i0, i1, blk in synthetic.s1_blocks(n, 1.0, 12345):
        pos_all_d[i0:i1].copy_(torch.from_numpy(blk))
        a, b = max(i0, lo_i), min(i1, hi_i)
        if a < b:
            pos_loc[a - lo_i:b - lo_i] = blk[a - i0:b - i0]
        if rank == 0:
            col.append(blk[select_column(blk, wlo, whi_max, 2.0 * h_cap * max(args.h_scale, 1.0))])
    sol = SmoothingLengthSolver(device=dev)
    if rank == 0:
        col = np.ascontiguousarray(np.concatenate(col))
        col_h = sol.query(pos_all_d, torch.from_numpy(col).to(dev), k, 1.0)[0][:, k - 1].contiguous().cpu().numpy()
        assert col_h.max() <= h_cap, "window superset too narrow for the k-NN h"
        col_h = col_h * args.h_scale
    h_loc_d = sol.solve(pos_all_d, k, 1.0, **(dict(q_begin=lo_i, q_count=n_loc) if world > 1 else {})) * args.h_scale
    h_note = f"d_{k} from the CUDA k-NN (periodic)"
    subs = {}
    want = [] if args.no_sub else [s for s in args.sub.split(",") if s]
    if "c5" in want:
        if world == 1:
            try:
                subs["c5"] = sub_c5(ctx, args, pos_all_d, peak)
            except Exception as e:                                # a sub-record must not lose the headline line
                subs["c5"] = {"error": f"{type(e).__name__}: {e}"}
        else:                                                     # (collectives inside: every rank fails or none)
            subs["c5"] = sub_c5(ctx, args, pos_all_d, peak)
    run_c5_full = ("c5full" in want) or ("c5" in want and world == 8)
    sol._ws = None
    pos_d = pos_all_d[lo_i:hi_i].clone() if world > 1 else pos_all_d
    del pos_all_d
    torch.cuda.empty_cache()
    m_loc = torch.full((n_loc,), 1.0 / N, dtype=torch.float64, pin_memory=True).numpy()
    m_d = torch.from_numpy(m_loc).to(dev)
    size = (npix, npix)
    bounds = (0.0, 1.0, 0.0, 1.0)
    eng = Projector2D(device=dev)
    out = torch.empty((1,) + size, dtype=torch.float64, device=dev)
    t_setup = time.time() - t_setup

    def step():
        astd.project_sharded(eng, pos_d, h_loc_d, [m_d], size, CoordinateAxes.Z, bounds, "cubic_spline_3d", out=out)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    sync_all()
    launches_per_step = eng.last_stats["n_launches"]
    if rank == 0:                     # nvidia-smi needs a few hundred ms to deliver its first sample
        t_wait = time.time()
        while sampler.proc is not None and sampler.mark() == 0 and time.time() - t_wait < 3.0:
            if world == 1:
                step()
                torch.cuda.synchronize()
            else:                     # step() holds a collective: rank 0 must not run it alone
                time.sleep(0.02)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    m0 = sampler.mark()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    sync_all()
    m1 = sampler.mark()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop(m0, m1) if rank == 0 else None
    ms_per_step = float(ms.item()) / args.steps
    value = N / (ms_per_step * 1e-3)
    if rank == 0 and args.dump_outputs:          # before the calls below overwrite `out` (rank 0 holds the reduced map)
        dump_map(args.dump_outputs, out[0])

    # ---- parity of the map that was just timed (rank 0 holds the reduced map) against the CPU oracle, on a window
    parity = cpu = timed_crop = None
    if rank == 0:
        import oracle
        pc0 = window_bounds(npix, 64)[0]
        timed_crop = out[0, pc0:pc0 + 64, pc0:pc0 + 64].cpu().numpy()          # of the reduced map (later calls overwrite `out`)
        m_col = np.full(len(col), 1.0 / N)
        wp = 128 if world > 1 else 64
        def run_window(wp):
            p0, lo, hi = window_bounds(npix, wp)
            sel = select_column(col, lo, hi, 2.0 * h_cap * max(args.h_scale, 1.0))
            ref, t = oracle_window(oracle, col[sel], col_h[sel], m_col[sel], npix, wp)
            crop = out[0, p0:p0 + wp, p0:p0 + wp].cpu().numpy()
            return dict(parity_of(crop, ref), window=f"{wp}^2 pixels of the timed map at [{lo:g},{hi:g})^2 vs oracle/sph_oracle.c fed the "
                                                    f"{int(sel.sum())} particles within 2 h_max of it"), t, int(sel.sum())
        parity, t_w, n_w = run_window(wp)
        if not (parity["rel_l2"] <= 1e-5 and parity["total_rel"] <= 1e-6):
            raise SystemExit(f"PARITY FAILURE: the timed map does not match the oracle: {parity}")      # no number without parity
        if world == 1 and not args.no_cpu_baseline:
            # bounded CPU sample: grow the window until the oracle runs for about cpu_target_s seconds
            rate = wp * wp / max(t_w, 1e-3)
            wp2 = int(min(wp_max, max(wp, np.sqrt(rate * args.cpu_target_s) // 32 * 32)))
            if wp2 > wp:
                parity, t_w, n_w = run_window(wp2)
                wp = wp2
            cpu = {"value": N * (wp / npix) ** 2 / t_w, "unit": UNIT, "cores": oracle.max_threads(), "kind": "port",
                   "sample": f"oracle/sph_oracle.c OpenMP float64 scatter on a {wp}^2-pixel window of the workload's map with the {n_w} particles "
                             f"that can touch it, {t_w:.2f} s; value = N * (window area / map area) / seconds"}

    # ---- per-stage device times (CUDA events recorded inside the library on the launching stream)
    stage_names = ["bin+direct", "scan", "emit", "sort", "pair_records", "tile_accumulate", "memset", "total"]
    acc = np.zeros(8)
    reps = 2
    for _ in range(reps):
        eng.project(pos_d, h_loc_d, [m_d], size, CoordinateAxes.Z, bounds, "cubic_spline_3d", out=out, timing=True)
        acc += np.array(eng.last_stats["stage_ms"])
    stage_ms = acc / reps
    stats = eng.last_stats
    dom = int(np.argmax(stage_ms[:6]))
    alg_bytes = N * 40 + size[0] * size[1] * 8                      # SURVEY 8(d): N*(24+8+8) + nx*ny*8
    alg_rank = n_loc * 40 + size[0] * size[1] * 8                   # what this rank's launch processes
    traffic = traffic_src = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = tj.get(stage_names[dom]); traffic_src = tj.get("source")
    except Exception:
        pass
    achieved = alg_rank / (stage_ms[dom] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": stage_names[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes": alg_rank,
                "kernel_ms": float(stage_ms[dom]), "whole_step_frac": alg_bytes / (ms_per_step * 1e-3) / 1e9 / (peak * world),
                "note": "h = d_48 footprints (~4000 pixel updates per particle) make this stage FP32-issue/MUFU-bound (see fp32); "
                        "regimes[0] is the HBM-bound end of the same path"}
    h_mean = float(h_loc_d.mean().item())
    px_per_particle = float(np.pi * (2.0 * h_mean * npix) ** 2)
    sm_hz = 148 * 1.965e9
    fp32 = {"pixel_updates_per_particle": px_per_particle,
            "updates_per_s": n_loc * px_per_particle / (stage_ms[5] * 1e-3) if stage_ms[5] > 0 else None,
            "lane_instr_per_evaluated_pixel_sass": {"full": 9.6, "outer_annulus": 6.6},
            "issue_peak_lane_instr_per_s": sm_hz * 4 * 32, "mufu_peak_sqrt_per_s": sm_hz * 16}
    if fp32["updates_per_s"]:
        fp32["useful_issue_frac_at_max_clock"] = fp32["updates_per_s"] * 9.6 / fp32["issue_peak_lane_instr_per_s"]
        fp32["useful_mufu_frac_at_max_clock"] = fp32["updates_per_s"] / fp32["mufu_peak_sqrt_per_s"]
    fp32["ncu"] = {"source": "profiles/r02_v13_ncu_accum.txt (rowcol_accum_kernel<cubic,1>, config 3, one launch, final build of round 2)", "issue_active": 0.826,
                   "xu_pipe": 0.713, "fma_pipe": 0.551, "thread_instr_per_useful_update": 13.2, "evaluated_pixels_inside_support": 0.69}

    # ---- end to end through the public host-buffer API (pinned host arrays in, numpy map out on rank 0)
    e2e = None
    if not args.no_e2e:
        h_host = torch.empty(n_loc, dtype=torch.float64, pin_memory=True)
        h_host.copy_(h_loc_d)
        h_host = h_host.numpy()

        def e2e_step():
            return astd.create_images_sharded(pos_loc, h_host, [m_loc], size, 32, CoordinateAxes.Z, *bounds,
                                              kernel_func=quartic_spline_kernel)
        ms_e, res = timed_wall(ctx, e2e_step, args.steps, 2)
        e2e = {"value": N / (ms_e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(N * 40), "d2h_bytes_per_step": int(size[0] * size[1] * 8),
               "ms_per_step": ms_e}
        if rank == 0 and timed_crop is not None:
            p0 = window_bounds(npix, 64)[0]
            e2e["rel_l2_vs_device_resident_map_window"] = float(np.linalg.norm(res[0, p0:p0 + 64, p0:p0 + 64] - timed_crop) /
                                                                np.linalg.norm(timed_crop))
        del res

    # ---- footprint regimes: the same particle set with h scaled down; shows where the path is HBM-bound (sub-pixel supports,
    # every particle deposited by the binning kernel) and where it is FP32-issue-bound (SPH-realistic supports)
    sweep = None
    if not args.no_regimes and world == 1:
        sweep = []
        for sc in ((1 / 64, 1 / 32, 1 / 16, 1 / 8, 1 / 4, 1 / 2) if args.sweep else (1 / 64, 1 / 8)):
            hs = h_loc_d * sc
            f = lambda: eng.project(pos_d, hs, [m_d], size, CoordinateAxes.Z, bounds, out=out)
            t = timed_device(ctx, f, 3, 2)
            eng.project(pos_d, hs, [m_d], size, CoordinateAxes.Z, bounds, out=out, timing=True)
            sweep.append({"h_scale": sc, "support_radius_px": float(2 * hs.mean().item() * npix), "ms": t,
                          "particles_per_s": N / (t * 1e-3), "hbm_frac": alg_bytes / (t * 1e-3) / 1e9 / peak,
                          "stage_ms": [round(x, 4) for x in eng.last_stats["stage_ms"]], "pairs": eng.last_stats["n_pairs"]})

    # ---- sub-records of the other BASELINE configs (1 GPU; c5 ran above while the positions were still replicated)
    del out, pos_d, m_d, h_loc_d
    eng._ws = None
    torch.cuda.empty_cache()
    if run_c5_full:                                               # configs[4] at its full size, on the 8 GPUs of the box
        try:
            subs["c5_1024cubed"] = sub_c5_full(ctx, args, peak, args.c5_full_n)
        except Exception as e:                                    # (every rank fails or none: the collectives inside stay matched)
            subs["c5_1024cubed"] = {"error": f"{type(e).__name__}: {e}"}
        torch.cuda.empty_cache()
    if world == 1:
        for name, fn in (("c2", sub_c2), ("c4", sub_c4)):
            if name in want:
                try:
                    subs[name] = fn(ctx, args, peak)
                except Exception as e:                                 # a sub-record must not lose the headline line
                    subs[name] = {"error": f"{type(e).__name__}: {e}"}
                torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 kernel shape and weights, f64 index work and accumulation", "data": "synthetic",
            "config": workload_config(args, world),
            "details": {"h": h_note, "particles_per_rank": n_loc, "pairs_per_step_rank0": stats["n_pairs"], "rounds": stats["n_rounds"],
                        "setup_s": round(t_setup, 1)},
            "clocks": clocks, "e2e": e2e, "parity": parity, "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roofline, "fp32": fp32, "stages_ms": dict(zip(stage_names, [float(x) for x in stage_ms])),
            "cpu_baseline": cpu,
        }
        if sweep:
            line["regimes"] = sweep
        line.update(subs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
