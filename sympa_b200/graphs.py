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
