"""Per-step neighbour lists of the score and confidence models, built on the ddb200_radius_* / ddb200_graph_fill kernels.

Two protocols.  Sync-free: count -> int32 scan -> fill into a capacity buffer (an upper bound that holds for any pose), with
the live edge count kept in device memory, so a step has static shapes and can be captured in a CUDA graph.  Host-sized:
``ops.radius`` reads the edge count back and returns exactly-sized lists.

An edge group is ``(tgt_int32, src_int32, edge_attr, edge_vec, edge_weight | None[, extras])``, CSR-sorted by target, as
``TensorProductConvLayer.forward_groups`` takes it."""
from __future__ import annotations

import torch

from . import ops
from .layers import edge_weight


def _i32(t):
    return t.to(torch.int32).contiguous()


def flat_weight(w):
    """A group's edge weight: the per-edge tensor flattened, or None for the constant weight 1."""
    return w.reshape(-1).contiguous() if torch.is_tensor(w) else None


def cross_cutoff(tr_sigma, dynamic_max_cross, cross_max_distance):
    """``(r, r_per_graph)`` of the ligand-receptor graph for ``ops.radius`` / ``ops.radius_count``: 3 tr_sigma + 20 per
    complex with dynamic_max_cross, else the fixed distance (models/cg_model.py:321-327)."""
    if dynamic_max_cross:
        return 1.0, (tr_sigma * 3 + 20).reshape(-1).float().contiguous()
    return float(cross_max_distance), None


# ------------------------------------------------------------------------------------------------------------- sync-free
def capacity_graph(x, y, x_ptr, y_batch32, capacity, r, r_per_graph=None, max_num_neighbors=32, exclude_self=False,
                   pre_cnt=None, **fill):
    """Neighbours of every y among the x of its complex in a buffer of ``capacity`` edges: ddb200_radius_count (+
    ``pre_cnt`` extra edges per y row, the bond CSR of ``fill``'s ``pre_ptr`` / ``pre_col``), int32 scan, ddb200_graph_fill.
    Returns ``ops.graph_fill``'s (row, col, vec, eid, perm) and the live edge count [1] on the device."""
    cnt = ops.radius_count(x, y, x_ptr, y_batch32, r=r, r_per_graph=r_per_graph, max_num_neighbors=max_num_neighbors,
                           exclude_self=exclude_self)
    if pre_cnt is not None:
        cnt = cnt + pre_cnt
    incl = torch.cumsum(cnt, 0, dtype=torch.int32)
    out = ops.graph_fill(x, y, x_ptr, y_batch32, (incl - cnt).contiguous(), capacity, r=r, r_per_graph=r_per_graph,
                         max_num_neighbors=max_num_neighbors, exclude_self=exclude_self, **fill)
    return out + (incl[-1:],)


def ligand_graph(pos, c, r, node_sigma_emb, expansion, edge_embedding, smooth):
    """ligand <- ligand group: bond edges + radius graph (models/cg_model.py:467-497), CSR by target.  ``c`` holds the
    per-batch bond CSR (``pre_ptr`` / ``pre_col`` / ``pre_cnt`` / ``pre_attr``, row -1 of ``pre_attr`` for radius edges),
    ``lig_ptr``, ``lig_batch32`` and the capacity ``cap_ll``.  radius_graph(max_num_neighbors=32) is radius with cap 33
    minus the self hit."""
    tgt, src, vec, eid, _, n = capacity_graph(pos, pos, c['lig_ptr'], c['lig_batch32'], c['cap_ll'], r,
                                              max_num_neighbors=33, exclude_self=True, pre_cnt=c['pre_cnt'],
                                              pre_ptr=c['pre_ptr'], pre_col=c['pre_col'], want_eid=True, fill_row=0)
    attr = torch.cat([c['pre_attr'][eid.long()], node_sigma_emb[tgt.long()], expansion(vec.norm(dim=-1))], 1)
    ea = edge_embedding(attr)
    return tgt, src, ea, vec, flat_weight(edge_weight(vec, r, smooth)), dict(n_edges_dev=n)


def cross_graph(pos, lig_ptr, lig_batch32, xpos, x_ptr, x_batch32, x_max, capacity, x_offset, r, r_per_graph, embed,
                vec_sign, fill_row):
    """ligand <- x group (x = residues or atoms, numbered from ``x_offset`` in the joint node list) and its reverse
    x <- ligand as a permutation of the same edges.  ``x_max``: most x of one complex.  ``embed(tgt, vec, n_dev)`` gives the
    forward edges' (edge_attr, edge_weight | None), which the reverse group reuses; its harmonics are evaluated at
    ``vec_sign`` * the forward vector.  ``fill_row``: value of the target rows beyond the live count, 0 when library ops
    gather over the whole buffer, None when only the kernels read it (they stop at the live count)."""
    slot = torch.empty((pos.shape[0], max(x_max, 1)), dtype=torch.int32, device=pos.device)
    f_tgt, f_src, f_vec, _, _, n = capacity_graph(xpos, pos, x_ptr, lig_batch32, capacity, r, r_per_graph,
                                                  max_num_neighbors=10000, slot_out=slot, slot_ld=slot.shape[1],
                                                  col_offset=x_offset, fill_row=fill_row)
    b_tgt, b_src, _, _, b_perm, _ = capacity_graph(pos, xpos, lig_ptr, x_batch32, capacity, r, r_per_graph,
                                                   max_num_neighbors=1 << 30, want_vec=False, slot_in=slot, y_ptr=x_ptr,
                                                   slot_ld=slot.shape[1], want_perm=True, row_offset=x_offset)
    ea, ew = embed(f_tgt, f_vec, n)
    return ((f_tgt, f_src, ea, f_vec, ew, dict(n_edges_dev=n)),
            (b_tgt, b_src, ea, f_vec, ew, dict(n_edges_dev=n, edge_perm=b_perm, vec_sign=vec_sign)))


# ----------------------------------------------------------------------------------------------------------- host-sized
def ligand_graph_host(pos, lig_ptr, lig_batch, ll, r, n_bond_features):
    """Bond edges, then the radius graph, unsorted as in the reference (models/cg_model.py:467-497): (target, gathered
    atom, bond attributes with zero rows for the radius edges)."""
    centre, nbr, _ = ops.radius(pos, pos, lig_ptr, lig_batch, r=r, max_num_neighbors=33, exclude_self=True)  # cap 32 (+ self)
    tgt = torch.cat([ll.edge_index[0].long(), nbr.long()])
    src = torch.cat([ll.edge_index[1].long(), centre.long()])
    bond_attr = torch.cat([ll.edge_attr.float(), pos.new_zeros(nbr.shape[0], n_bond_features)], 0)
    return tgt, src, bond_attr


def cross_graph_host(pos, xpos, x_ptr, lig_batch, r, r_per_graph=None):
    """ligand <- x edges within the cut-off, sorted by ligand atom: (ligand index, x index, x - ligand vector)."""
    li, xi, _ = ops.radius(xpos, pos, x_ptr, lig_batch, r=r, r_per_graph=r_per_graph, max_num_neighbors=10000)
    li, xi = li.long(), xi.long()
    return li, xi, xpos[xi] - pos[li]


def cross_groups_host(li, xi, x_offset, ea, vec, ew, vec_sign):
    """ligand <- x group of a host-sized cross graph and its reverse x <- ligand: the same pairs stably sorted by x, with
    the forward attributes and the harmonics of ``vec_sign`` * the forward vector."""
    x_tgt, rev = torch.sort(xi, stable=True)
    r_vec = vec[rev] if vec_sign > 0 else -vec[rev]
    return ((_i32(li), _i32(xi + x_offset), ea, vec.contiguous(), flat_weight(ew)),
            (_i32(x_tgt + x_offset), _i32(li[rev]), ea[rev], r_vec.contiguous(),
             flat_weight(ew[rev]) if torch.is_tensor(ew) else None))


def merge_groups(groups):
    """All groups as one (one radial MLP for every edge type, differentiate_convolutions=False)."""
    return [tuple(torch.cat([g[k] for g in groups]) if groups[0][k] is not None else None for k in range(5))]
