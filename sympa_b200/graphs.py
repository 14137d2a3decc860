"""Synthetic graphs of the BASELINE configs as (src, dst, distance) triplets, the format
preprocess.py:118-126 writes (all pairs i < j with their shortest-path distance).  Grid and balanced
tree distances are computed directly (no networkx / networkit needed)."""
import itertools

import torch


def grid_triplets(side, dims=2):
    """`side`^dims grid graph (preprocess.py: nx.grid_graph); distance = Manhattan distance."""
    coords = torch.tensor(list(itertools.product(range(side), repeat=dims)), dtype=torch.int64)
    n = coords.shape[0]
    i, j = torch.triu_indices(n, n, offset=1)
    dist = (coords[i] - coords[j]).abs().sum(-1)
    return torch.stack((i, j), 1).contiguous(), dist.double(), n


def balanced_tree_triplets(branching, height):
    """nx.balanced_tree(branching, height): node k has parent (k - 1) // branching."""
    n = (branching ** (height + 1) - 1) // (branching - 1)
    depth = torch.zeros(n, dtype=torch.int64)
    parent = torch.zeros(n, dtype=torch.int64)
    for k in range(1, n):
        parent[k] = (k - 1) // branching
        depth[k] = depth[parent[k]] + 1
    i, j = torch.triu_indices(n, n, offset=1)
    a, b = i.clone(), j.clone()
    d = torch.zeros_like(a)
    # climb the deeper node until both meet
    for _ in range(2 * height + 1):
        deeper_a = depth[a] > depth[b]
        deeper_b = depth[b] > depth[a]
        same = (~deeper_a) & (~deeper_b) & (a != b)
        d += deeper_a.long() + deeper_b.long() + 2 * same.long()
        a = torch.where(deeper_a | same, parent[a], a)
        b = torch.where(deeper_b | same, parent[b], b)
    return torch.stack((i, j), 1).contiguous(), d.double(), n


def product_cartesian_triplets(branching, height, side, dims):
    """Cartesian product of nx.balanced_tree(branching, height) and the `side`^dims grid (preprocess.py:53-60,
    BASELINE config 3).  Nodes are the pairs (tree node, grid node) in sorted order - id = tree_id * |grid| +
    grid_id, what nx.convert_node_labels_to_integers(ordering="sorted") gives the tuple labels (preprocess.py:151-152) -
    and the shortest-path distance of a Cartesian product is the sum of the factor distances.  The reference's CLI
    defaults (tree 3/3, nodes 125, grid_dims 3) give 40 x 125 = 5000 nodes and 12 497 500 pairs."""
    t_idx, t_dist, t_n = balanced_tree_triplets(branching, height)
    g_idx, g_dist, g_n = grid_triplets(side, dims)
    dt = torch.zeros(t_n, t_n, dtype=torch.int64)
    dt[t_idx[:, 0], t_idx[:, 1]] = t_dist.long()
    dt = dt + dt.t()
    dg = torch.zeros(g_n, g_n, dtype=torch.int64)
    dg[g_idx[:, 0], g_idx[:, 1]] = g_dist.long()
    dg = dg + dg.t()
    n = t_n * g_n
    i, j = torch.triu_indices(n, n, offset=1)
    dist = dt[i // g_n, j // g_n] + dg[i % g_n, j % g_n]
    return torch.stack((i, j), 1).contiguous(), dist.double(), n


def product_tree_grid_triplets(branching, height, side, dims):
    return product_cartesian_triplets(branching, height, side, dims)


def adjacency_csr(edges, num_nodes):
    """CSR adjacency (ptr, idx) of the undirected graph with the (E, 2) int64 node pairs `edges` over nodes
    [0, num_nodes): both directions, duplicates and self loops removed, every row sorted.  ptr has num_nodes + 1
    entries; the neighbours of u are idx[ptr[u]:ptr[u + 1]].  Returned on the device of `edges`.
    From triplets: adjacency_csr(ids[gd == 1], n); a tree's edges are (k, parent(k)), e.g. (k, (k - 1) // b)."""
    edges = torch.as_tensor(edges)
    if edges.dtype != torch.int64 or edges.dim() != 2 or edges.shape[1] != 2:
        raise ValueError("edges must be an (E, 2) int64 tensor")
    if edges.numel() and (int(edges.min()) < 0 or int(edges.max()) >= num_nodes):
        raise ValueError(f"edge endpoints must lie in [0, {num_nodes})")
    e = torch.cat((edges, edges.flip(1)))
    e = e[e[:, 0] != e[:, 1]]
    key = torch.unique(e[:, 0] * num_nodes + e[:, 1])        # sorted: by source, then by destination
    src, idx = key // num_nodes, key % num_nodes
    ptr = torch.zeros(num_nodes + 1, dtype=torch.int64, device=edges.device)
    ptr[1:] = torch.cumsum(torch.bincount(src, minlength=num_nodes), 0)
    return ptr, idx.contiguous()


def shortest_path_triplets(adj, block_bytes=1 << 30):
    """(src, dst, distance) triplets of every pair i < j joined by a path in the undirected graph adj = (ptr, idx)
    (adjacency_csr), distance = hop count: the format and order of the generators above, for any graph - what
    preprocess.py:114 gets from networkit's all-pairs shortest paths.  Hop distances come from breadth-first search
    on the GPU (ops.hop_distances) in blocks of max(1, block_bytes // (4 N)) source rows, on adj's device when it
    is a CUDA device and on the current one otherwise; the result is returned on adj's device.  Meant for graphs
    whose triplets fit in memory (24 bytes per pair)."""
    from . import ops

    ptr, idx = adj
    out_dev = torch.as_tensor(ptr).device
    dev = out_dev if out_dev.type == "cuda" else torch.device("cuda", torch.cuda.current_device())
    ptr = torch.as_tensor(ptr, dtype=torch.int64).to(dev).contiguous()
    idx = torch.as_tensor(idx, dtype=torch.int64).to(dev).contiguous()
    n = ptr.numel() - 1
    block = max(1, min(block_bytes // (4 * max(n, 1)), max(n, 1)))
    cols = torch.arange(n, device=dev)
    ids, dist = [], []
    for r0 in range(0, n, block):
        rc = min(block, n - r0)
        h = ops.hop_distances((ptr, idx), r0, rc)
        keep = (h > 0) & (cols[None, :] > torch.arange(r0, r0 + rc, device=dev)[:, None])
        rc_idx = keep.nonzero()
        rc_idx[:, 0] += r0
        ids.append(rc_idx.to(out_dev))
        dist.append(h[keep].double().to(out_dev))
    ops.check_status(dev)
    if not ids:
        return torch.zeros(0, 2, dtype=torch.int64, device=out_dev), torch.zeros(0, dtype=torch.float64, device=out_dev), n
    return torch.cat(ids).contiguous(), torch.cat(dist), n
