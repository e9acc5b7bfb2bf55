#!/usr/bin/env python3
"""Multi-GPU configurations of BASELINE.json (launch with torchrun, one rank per GPU):
  --which c3   config 3: S1 512^3 = 134 M particles -> 4096^2 projection, particles sharded by index over the ranks
               (STRONG scaling: total work fixed), NCCL sum-reduce of the partial maps
  --which c5   config 5 slice: k-NN k=48 periodic on n^3 particles; positions replicated on every rank (generated on the
               device from a fixed seed), rank g answers queries [g*N/G, (g+1)*N/G)
  --which c4   config 4: 256^3 NFW-clustered particles -> 512^3 voxels, periodic, through distributed.grid_sharded: particles
               sharded by index, each rank owns one x-slab of the grid (1/G of it); parity on a 48^3 window of the assembled
               grid against the float64 oracle, as in bench.py's c4 sub-record
Rank 0 prints one JSON object per configuration.  Timing: CUDA events, barrier + synchronize on both sides, max over ranks."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--which", default="c3,c5")
    ap.add_argument("--lattice", dest="n", type=int, default=512)
    ap.add_argument("--npix", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from astro_sph_tools_b200 import CoordinateAxes, distributed as astd, synthetic
    from astro_sph_tools_b200.tools.projections import Projector2D
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()

    def timed(fn, reps):
        fn(); sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); sync()
        t = torch.tensor([e0.elapsed_time(e1) / reps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n = args.n
    N = n ** 3
    # S1-like jittered lattice generated on the device, identical on every rank (fixed seed)
    g = torch.Generator(device=dev); g.manual_seed(12345)
    ax = (torch.arange(n, dtype=torch.float64, device=dev) + 0.5) / n
    pos = torch.empty((N, 3), dtype=torch.float64, device=dev)
    slab = max(1, n // 32)                                      # generated slab by slab: no N-sized temporaries
    for i0 in range(0, n, slab):
        i1 = min(n, i0 + slab)
        blk = torch.stack(torch.meshgrid(ax[i0:i1], ax, ax, indexing="ij"), dim=-1).reshape(-1, 3)
        blk = torch.remainder(blk + torch.randn(blk.shape, dtype=torch.float64, device=dev, generator=g) * (0.2 / n), 1.0)
        blk[blk >= 1.0] = 0.0
        pos[i0 * n * n:i1 * n * n] = blk
    del blk
    torch.cuda.empty_cache()
    lo, hi = astd.shard_bounds(N, world, rank)
    sol = SmoothingLengthSolver(device=dev)
    out = {}
    if "c5" in args.which:
        ms = timed(lambda: sol.solve(pos, 48, 1.0, q_begin=lo, q_count=hi - lo), 2)
        if rank == 0:
            print(json.dumps({"config": f"C5 slice: k-NN k=48 periodic, {n}^3 = {N} particles replicated, queries sharded over {world} GPU(s)",
                              "ms": ms, "queries_per_s": N / (ms * 1e-3), "n_gpus": world}))
    if "c3" in args.which:
        h_loc = sol.solve(pos, 48, 1.0, q_begin=lo, q_count=hi - lo)
        sol._ws = None                                          # release the k-NN workspace before the projection
        torch.cuda.empty_cache()
        pos_loc = pos[lo:hi].contiguous()
        m_loc = torch.full((hi - lo,), 1.0 / N, dtype=torch.float64, device=dev)
        eng = Projector2D(device=dev)
        size = (args.npix, args.npix)
        buf = torch.empty((1,) + size, dtype=torch.float64, device=dev)
        step = lambda: astd.project_sharded(eng, pos_loc, h_loc, m_loc, size, CoordinateAxes.Z, (0.0, 1.0, 0.0, 1.0), out=buf)
        ms = timed(step, args.steps)
        total = float(buf.sum().item()) / args.npix ** 2 if rank == 0 else 0.0
        if rank == 0:
            alg = N * 40 + args.npix ** 2 * 8
            peak = 6554.2
            try:
                peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            except Exception:
                pass
            print(json.dumps({"config": f"C3: S1 {n}^3 = {N} particles -> {args.npix}^2, h = d_48, cubic spline, sharded over {world} GPU(s), "
                                        f"NCCL reduce", "ms": ms, "particles_per_s": N / (ms * 1e-3), "n_gpus": world, "scaling": "strong",
                              "hbm_frac_vs_one_gpu_roofline": alg / (ms * 1e-3) / 1e9 / peak, "sum_img_times_pixel_area": total,
                              "pairs_rank0": eng.last_stats["n_pairs"]}))
    if "c4" in args.which:
        c4(torch, dist, astd, dev, world, rank, timed, sync)
    if world > 1:
        dist.destroy_process_group()


def c4(torch, dist, astd, dev, world, rank, timed, sync):
    import oracle
    from bench import nfw_positions_device, parity_of
    from astro_sph_tools_b200.tools.projections import Gridder3D
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    n, ng = 256, 512
    N = n ** 3
    size, lo, hi = (ng,) * 3, (0.0, 0.0, 0.0), (1.0, 1.0, 1.0)
    pos = nfw_positions_device(torch, dev, N)                  # the same set on every rank (fixed seed)
    sol = SmoothingLengthSolver(device=dev)
    h = sol.solve(pos, 48, 1.0)
    sol._ws = None
    torch.cuda.empty_cache()
    a, b = astd.shard_bounds(N, world, rank)
    pos_l, h_l = pos[a:b].contiguous(), h[a:b].contiguous()
    m_l = torch.full((b - a,), 1.0 / N, dtype=torch.float64, device=dev)
    g = Gridder3D(device=dev)
    router = astd.default_grid_router(dev)
    edges = astd.grid_slab_planes(ng, world)
    route_ms = timed(lambda: router.route(pos_l, h_l, m_l, edges, size, lo, hi, True, 1.0), 3)
    e8 = astd.grid_slab_planes(ng, 8)                          # routing (count + write) of this rank's particles into 8 slabs
    route8_ms = timed(lambda: router.route(pos_l, h_l, m_l, e8, size, lo, hi, True, 1.0), 3)
    out = {}
    step = lambda: out.__setitem__("r", astd.grid_sharded(g, pos_l, h_l, m_l, size, lo, hi, periodic=True, box=1.0, return_stats=True))
    ms = timed(step, 3)
    slab, x0, st = out["r"]
    loads = torch.tensor([[float(st["n_pairs"]), float(st["received"]), float(sum(st["sent"]))]], dtype=torch.float64, device=dev)
    parts = [torch.zeros_like(loads) for _ in range(world)]
    if world > 1:
        dist.all_gather(parts, loads)
    else:
        parts = [loads]
    loads = torch.cat(parts).cpu().numpy()
    rec = {"config": f"C4: S2 NFW {n}^3 = {N} particles -> {ng}^3 voxels, periodic, grid_sharded over {world} GPU(s), x-slabs of "
                     f"{ng // world if ng % world == 0 else 'about ' + str(ng // world)} planes",
           "ms": ms, "route_ms_rank0": route_ms, "route_into_8_slabs_ms_rank0": route8_ms, "n_gpus": world, "fan_out": float(loads[:, 2].sum() / N),
           "n_pairs_max": float(loads[:, 0].max()), "n_pairs_mean": float(loads[:, 0].mean()), "rows_received_max": float(loads[:, 1].max())}
    if world == 1:
        whole = torch.empty(size, dtype=torch.float64, device=dev)
        rec["gridder3d_ms"] = timed(lambda: g.grid(pos, h, m_l, size, lo, hi, periodic=True, box=1.0, out=whole), 3)
    whole = astd.collect_slabs(slab, ng, dst=0)
    if rank == 0:
        wv, v0 = 48, ng // 2 - 24
        wlo, whi = v0 / ng, (v0 + wv) / ng
        p, hh = pos.cpu().numpy(), h.cpu().numpy()
        sel = np.all((p + 2.0 * hh[:, None] > wlo) & (p - 2.0 * hh[:, None] < whi), axis=1)
        ref = oracle.grid3d(p[sel], hh[sel], np.full(int(sel.sum()), 1.0 / N), (wv,) * 3, (wlo,) * 3, (whi,) * 3)
        crop = whole[v0:v0 + wv, v0:v0 + wv, v0:v0 + wv].cpu().numpy()
        rec["parity"] = dict(parity_of(crop, ref), window=f"{wv}^3 voxels at [{wlo:g},{whi:g})^3")
        print(json.dumps(rec), flush=True)
    sync()


if __name__ == "__main__":
    main()
