#!/usr/bin/env python3
"""Config 4 (S2 NFW 256^3 -> 512^3 voxels, periodic, h = d_48) through distributed.grid_sharded on G in-process ranks of ONE
GPU (the thread ranks of tests/inprocess_dist.py, real CUDA kernels): the load counts of a G-rank job -- rows sent, fan-out
(rows sent / particles), rows received and n_pairs per rank -- which do not depend on how many GPUs run the ranks.  The ranks
share the GPU, so this prints no timing; multi-GPU times come from `torchrun ... benchmarks/bench_multi.py --which c4`.
Prints one JSON line."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", type=int, default=8)
    args = ap.parse_args()
    import pytest
    import torch
    from bench import nfw_positions_device
    from inprocess_dist import InProcessRanks
    from astro_sph_tools_b200 import distributed as astd
    from astro_sph_tools_b200.tools.projections import Gridder3D
    from astro_sph_tools_b200.tools.smoothing import SmoothingLengthSolver
    dev = torch.device("cuda", 0)
    N, ng, world = 256 ** 3, 512, args.ranks
    pos = nfw_positions_device(torch, dev, N)
    sol = SmoothingLengthSolver(device=dev)
    h = sol.solve(pos, 48, 1.0)
    sol._ws = None
    torch.cuda.empty_cache()
    m = torch.full((N,), 1.0 / N, dtype=torch.float64, device=dev)

    def body(r):
        a, b = astd.shard_bounds(N, world, r)
        slab, _, st = astd.grid_sharded(Gridder3D(device=dev), pos[a:b].contiguous(), h[a:b].contiguous(), m[a:b].contiguous(),
                                        (ng,) * 3, (0, 0, 0), (1, 1, 1), periodic=True, box=1.0, return_stats=True)
        total = float(slab.sum().item())
        del slab
        return st, total

    mp = pytest.MonkeyPatch()
    ranks = InProcessRanks(timeout=600)
    ranks.install(mp)
    try:
        res = ranks.run(world, body)
    finally:
        mp.undo()
    pairs = [st["n_pairs"] for st, _ in res]
    print(json.dumps({"config": f"C4 through grid_sharded on {world} in-process ranks of one GPU (counts only)",
                      "fan_out": sum(sum(st["sent"]) for st, _ in res) / N, "n_pairs_per_rank": pairs, "n_pairs_max": max(pairs),
                      "n_pairs_mean": float(np.mean(pairs)), "rows_received_per_rank": [st["received"] for st, _ in res],
                      "mass_sum": sum(t for _, t in res) / ng ** 3}))


if __name__ == "__main__":
    main()
