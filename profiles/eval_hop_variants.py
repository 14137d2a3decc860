"""A/B of hop_bfs_kernel variants: the hop kernel's time on one full block (1 GB of distances + hop distances) of
each workload of profiles/eval_b200.py, and a digest of the block (equal for every variant).  Run once per library
(SYMPA_B200_LIB); prints one JSON line.  The variants were built from hop_kernels.cuh with -DSY_HOP_CTAS_PER_SM in
{1, 2, 4} and -DSY_HOP_SMEM_VISITED_BYTES=0 (visited set = the output row, atomicCAS in global memory) or the
default (visited bitmap in shared memory), sympa_b200.cu compiled with the flags of sympa_b200/build.py and linked
with the library's other objects; eval_hop_variants_b200.txt holds two alternating rounds on one B200 (1000 W),
"main" = the shipped 2 CTAs / SM with the shared-memory bitmap."""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from sympa_b200 import graphs, ops
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(0)
    ids, gd, n3 = graphs.product_cartesian_triplets(3, 3, 5, 3)
    work = [("config3", n3, ids[gd == 1], n3)]
    nt = (4 ** 9 - 1) // 3
    k = torch.arange(1, nt)
    work.append(("tree_4_8", nt, torch.stack((k, (k - 1) // 4), 1), (1 << 30) // (12 * nt)))
    rnd = 1 << 17
    k = torch.arange(1, rnd)
    parent = torch.from_numpy((rng.random(rnd - 1) * np.arange(1, rnd)).astype(np.int64))
    work.append(("random_tree_2_17", rnd, torch.stack((k, parent), 1), (1 << 30) // (12 * rnd)))
    out = {"lib": os.path.basename(os.path.dirname(os.environ.get("SYMPA_B200_LIB", "main/x")))}
    for name, n, edges, block in work:
        adj = graphs.adjacency_csr(edges, n)
        adj = (adj[0].to(dev), adj[1].to(dev))
        h = torch.empty(block, n, dtype=torch.int32, device=dev)
        ops.hop_distances(adj, 0, block, out=h)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(5):
            s.record()
            ops.hop_distances(adj, 0, block, out=h)
            e.record()
            torch.cuda.synchronize()
            times.append(s.elapsed_time(e) / 1e3)
        ops.check_status()
        out[name] = {"block": block, "sec_median": float(np.median(times)), "sec_min": min(times),
                     "digest": hashlib.sha256(h.cpu().numpy().tobytes()).hexdigest()[:16]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
