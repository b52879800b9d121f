"""Drop-in for the reference's coarse-grained score model ``models/cg_model.py:CGModel`` (score mode).

Same constructor keywords, ``forward(data) -> (tr_pred, rot_pred, tor_pred, sidechain_pred)`` contract, ``state_dict``
keys and side effects on ``data`` (SURVEY.md section 8(b)); ``utils/sampling.py:116`` can call it unchanged.  What runs
underneath is B200-native: neighbour search and the tensor-product convolutions (SH + Clebsch-Gordan contraction +
segmented reduction + BatchNorm/residual epilogue) are hand-written sm_100a kernels behind the C ABI
(include/diffdock_b200.h); every edge list is produced already CSR-sorted by its convolution target; the score-norm
tables are device buffers (no host round trips for so3/torus look-ups).

CUDA only, inference only.  No CPU fallback.
"""
from __future__ import annotations

import math
import os

import numpy as np
import torch
from torch import nn

from . import graphs, ops
from .irreps import irreps_str, sh_irreps
from .layers import AtomEncoder, GaussianSmearing, _mlp, edge_weight
from .synthetic import LIG_FEATURE_DIMS as lig_feature_dims, REC_RESIDUE_FEATURE_DIMS as rec_residue_feature_dims
from .tensor_layers import TensorProductConvLayer, get_irrep_seq
from .tp_table import full_tensor_product

_TABLES = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'tables', 'score_norm_tables.npz')
# utils/so3.py:6 and utils/torus.py:25-26
SO3_MIN_EPS, SO3_MAX_EPS, SO3_N_EPS = 0.0005, 4, 2000
TORUS_SIGMA_MIN, TORUS_SIGMA_MAX, TORUS_SIGMA_N = 3e-3, 2, 5000


def _sh_l2(vec):
    """Component-normalised l=2 real spherical harmonics of the normalised vectors (o3.spherical_harmonics("2e", ...),
    models/cg_model.py:411)."""
    v = torch.nn.functional.normalize(vec, dim=-1)
    x, y, z = v[:, 0], v[:, 1], v[:, 2]
    s5, s15 = math.sqrt(5.0), math.sqrt(15.0)
    return torch.stack([s15 * x * z, s15 * x * y, s5 * (y * y - 0.5 * (x * x + z * z)), s15 * y * z,
                        0.5 * s15 * (z * z - x * x)], dim=-1)


def _sh_full(vec, lmax):
    v = torch.nn.functional.normalize(vec, dim=-1)
    cols = [torch.ones_like(v[:, :1])]
    if lmax >= 1:
        cols.append(math.sqrt(3.0) * v)
    if lmax >= 2:
        cols.append(_sh_l2(vec))
    return torch.cat(cols, dim=-1)


class CGModel(nn.Module):
    def __init__(self, t_to_sigma, device, timestep_emb_func, in_lig_edge_features=4, sigma_embed_dim=32, sh_lmax=2,
                 ns=16, nv=4, num_conv_layers=2, lig_max_radius=5, rec_max_radius=30, cross_max_distance=250,
                 center_max_distance=30, distance_embed_dim=32, cross_distance_embed_dim=32, no_torsion=False,
                 scale_by_sigma=True, norm_by_sigma=True, use_second_order_repr=False, batch_norm=True,
                 dynamic_max_cross=False, dropout=0.0, smooth_edges=False, odd_parity=False,
                 separate_noise_schedule=False, lm_embedding_type=None, confidence_mode=False,
                 confidence_dropout=0, confidence_no_batchnorm=False,
                 asyncronous_noise_schedule=False, affinity_prediction=False, parallel=1,
                 parallel_aggregators="mean max min std", num_confidence_outputs=1, atom_num_confidence_outputs=1,
                 fixed_center_conv=False, no_aminoacid_identities=False, include_miscellaneous_atoms=False,
                 differentiate_convolutions=True, tp_weights_layers=2, num_prot_emb_layers=0, reduce_pseudoscalars=False,
                 embed_also_ligand=False, atom_confidence=False, sidechain_pred=False, depthwise_convolution=False):
        super().__init__()
        assert parallel == 1, "not implemented"
        unsupported = dict(confidence_mode=confidence_mode, separate_noise_schedule=separate_noise_schedule,
                           asyncronous_noise_schedule=asyncronous_noise_schedule,
                           include_miscellaneous_atoms=include_miscellaneous_atoms, sidechain_pred=sidechain_pred,
                           depthwise_convolution=depthwise_convolution, atom_confidence=atom_confidence)
        bad = [k for k, v in unsupported.items() if v]
        if bad:
            raise NotImplementedError(f"{bad}: outside the score-model hot path built so far (SURVEY.md section 8)")
        if lm_embedding_type not in (None, 'precomputed'):
            raise NotImplementedError("on-the-fly ESM embeddings are preprocessing (out of scope); use 'precomputed'")
        self.t_to_sigma, self.device, self.timestep_emb_func = t_to_sigma, device, timestep_emb_func
        self.in_lig_edge_features, self.sigma_embed_dim = in_lig_edge_features, sigma_embed_dim
        self.lig_max_radius, self.rec_max_radius = lig_max_radius, rec_max_radius
        self.cross_max_distance, self.dynamic_max_cross = cross_max_distance, dynamic_max_cross
        self.center_max_distance = center_max_distance
        self.distance_embed_dim, self.cross_distance_embed_dim = distance_embed_dim, cross_distance_embed_dim
        self.sh_lmax = sh_lmax
        self.sh_irreps = irreps_str(sh_irreps(sh_lmax))
        self.ns, self.nv = ns, nv
        self.scale_by_sigma, self.norm_by_sigma = scale_by_sigma, norm_by_sigma
        self.no_torsion, self.smooth_edges, self.odd_parity = no_torsion, smooth_edges, odd_parity
        self.confidence_mode = False
        self.num_conv_layers, self.num_prot_emb_layers = num_conv_layers, num_prot_emb_layers
        self.fixed_center_conv, self.no_aminoacid_identities = fixed_center_conv, no_aminoacid_identities
        self.differentiate_convolutions, self.reduce_pseudoscalars = differentiate_convolutions, reduce_pseudoscalars
        self.embed_also_ligand = embed_also_ligand
        self.lm_embedding_type = lm_embedding_type
        lm_dim = 1280 if lm_embedding_type == 'precomputed' else 0
        S, D, Dx = sigma_embed_dim, distance_embed_dim, cross_distance_embed_dim

        self.lig_node_embedding = AtomEncoder(emb_dim=ns, feature_dims=lig_feature_dims, sigma_embed_dim=S)
        self.lig_edge_embedding = _mlp(in_lig_edge_features + S + D, ns, ns, dropout)
        self.rec_node_embedding = AtomEncoder(emb_dim=ns, feature_dims=rec_residue_feature_dims, sigma_embed_dim=0,
                                              lm_embedding_dim=lm_dim)
        self.rec_edge_embedding = _mlp(D, ns, ns, dropout)
        self.rec_sigma_embedding = _mlp(S, ns, ns, dropout)
        self.cross_edge_embedding = _mlp(S + Dx, ns, ns, dropout)
        self.lig_distance_expansion = GaussianSmearing(0.0, lig_max_radius, D)
        self.rec_distance_expansion = GaussianSmearing(0.0, rec_max_radius, D)
        self.cross_distance_expansion = GaussianSmearing(0.0, cross_max_distance, Dx)

        seq = get_irrep_seq(ns, nv, use_second_order_repr, reduce_pseudoscalars)
        faster = sh_lmax == 1 and not use_second_order_repr

        def conv(i, groups):
            return TensorProductConvLayer(in_irreps=seq[min(i, len(seq) - 1)], sh_irreps=self.sh_irreps,
                                          out_irreps=seq[min(i + 1, len(seq) - 1)], n_edge_features=3 * ns,
                                          hidden_features=3 * ns, residual=True, batch_norm=batch_norm, dropout=dropout,
                                          faster=faster, tp_weights_layers=tp_weights_layers, edge_groups=groups)

        self.rec_emb_layers = nn.ModuleList([conv(i, 1) for i in range(num_prot_emb_layers)])
        if embed_also_ligand:
            self.lig_emb_layers = nn.ModuleList([conv(i, 1) for i in range(num_prot_emb_layers)])
        last = num_prot_emb_layers + num_conv_layers - 1
        self.conv_layers = nn.ModuleList([
            conv(i, 1 if not differentiate_convolutions else (2 if i == last else 4))
            for i in range(num_prot_emb_layers, num_prot_emb_layers + num_conv_layers)])

        # translation / rotation head
        self.center_distance_expansion = GaussianSmearing(0.0, center_max_distance, D)
        self.center_edge_embedding = _mlp(D + S, ns, ns, dropout)
        self.final_conv = TensorProductConvLayer(in_irreps=self.conv_layers[-1].out_irreps, sh_irreps=self.sh_irreps,
                                                 out_irreps='2x1o + 2x1e' if not odd_parity else '1x1o + 1x1e',
                                                 n_edge_features=2 * ns, residual=False, dropout=dropout,
                                                 batch_norm=batch_norm)
        self.tr_final_layer = nn.Sequential(nn.Linear(1 + S, ns), nn.Dropout(dropout), nn.ReLU(), nn.Linear(ns, 1))
        self.rot_final_layer = nn.Sequential(nn.Linear(1 + S, ns), nn.Dropout(dropout), nn.ReLU(), nn.Linear(ns, 1))
        if not no_torsion:
            self.final_edge_embedding = _mlp(D, ns, ns, dropout)
            T, tor_sh = full_tensor_product(self.sh_irreps, '1x2e')       # o3.FullTensorProduct(sh, "2e"), :240
            self.register_buffer('_tor_tp', torch.from_numpy(T).float(), persistent=False)
            self.tor_bond_conv = TensorProductConvLayer(in_irreps=self.conv_layers[-1].out_irreps,
                                                        sh_irreps=irreps_str(tor_sh),
                                                        out_irreps=f'{ns}x0o + {ns}x0e' if not odd_parity else f'{ns}x0o',
                                                        n_edge_features=3 * ns, residual=False, dropout=dropout,
                                                        batch_norm=batch_norm)
            self.tor_final_layer = nn.Sequential(nn.Linear(2 * ns if not odd_parity else ns, ns, bias=False), nn.Tanh(),
                                                 nn.Dropout(dropout), nn.Linear(ns, 1, bias=False))
        # score-norm tables (utils/so3.py:59, utils/torus.py:72-76) as device buffers; not part of the state_dict
        z = np.load(_TABLES)
        self.register_buffer('_so3_table', torch.from_numpy(z['so3_exp_score_norms']).float(), persistent=False)
        self.register_buffer('_torus_table', torch.from_numpy(z['torus_score_norm']).float(), persistent=False)
        self._sync_free = None

    # ---------------------------------------------------------------------------------------------------------
    def load_state_dict(self, state_dict, strict=True, **kw):
        """Accepts reference checkpoints: e3nn's TensorProduct modules register buffers (``*.tp.weight``,
        ``*.tp.output_mask``, ``final_tp_tor.*``, compiled ``_w3j_*`` constants) that have no counterpart here."""
        drop = [k for k in state_dict if '.tp.' in k or k.startswith('final_tp_tor.') or '_w3j' in k]
        if drop:
            state_dict = {k: v for k, v in state_dict.items() if k not in drop}
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def set_score_norm_tables(self, so3_exp_score_norms, torus_score_norm):
        """Install the tables of the caller's reference installation (torus.score_norm_ is a Monte-Carlo estimate that
        differs per machine, SURVEY.md section 5)."""
        self._so3_table.copy_(torch.as_tensor(so3_exp_score_norms, dtype=torch.float32))
        self._torus_table.copy_(torch.as_tensor(torus_score_norm, dtype=torch.float32))

    # ---------------------------------------------------------------------------------------------------------
    def _so3_score_norm(self, eps):
        """utils/so3.py:89-93 evaluated on the device (fp32 index arithmetic, round-half-even like np.around)."""
        lo, hi = math.log10(SO3_MIN_EPS), math.log10(SO3_MAX_EPS)
        idx = (torch.log10(eps.float()) - np.float32(lo)) / np.float32(hi - lo) * SO3_N_EPS
        idx = torch.round(idx).clamp(0, SO3_N_EPS - 1).long()
        return self._so3_table[idx]

    def _torus_score_norm(self, sigma):
        """utils/torus.py:79-83 on the device."""
        lo, hi = math.log(TORUS_SIGMA_MIN), math.log(TORUS_SIGMA_MAX)
        s = torch.log(sigma.float() / np.float32(np.pi))
        s = (s - np.float32(lo)) / np.float32(hi - lo) * TORUS_SIGMA_N
        s = torch.round(s.clamp(0, TORUS_SIGMA_N)).long()
        return self._torus_table[s]

    # ---------------------------------------------------------------------------------------------------------
    def _static(self, data):
        """Pose-independent quantities, cached on ``data`` like the reference does (models/cg_model.py:273,292-295)."""
        rec, rr, lig, ll = data['receptor'], data['receptor', 'receptor'], data['ligand'], data['ligand', 'ligand']
        if hasattr(rec, 'rec_node_attr') and hasattr(rr, '_b200'):
            return rr._b200
        B = data.num_graphs
        c = {}
        ei = rr.edge_index.long()
        uniq = getattr(rec, '_unique', None)       # (nodes, edges, copies): the batch holds `copies` identical receptors
        if uniq is not None and uniq[2] == B and uniq[0] * B == rec.pos.shape[0] and uniq[1] * B == ei.shape[1]:
            # N poses of one complex (inference.py:236-239): embed the receptor ONCE and tile the result; the reference
            # recomputes the identical 1280-wide embedding for every pose of the batch (models/cg_model.py:272-295)
            n1, e1 = uniq[0], uniq[1]
            ei1 = ei[:, :e1]
            vec1 = (rec.pos[ei1[1]] - rec.pos[ei1[0]]).float()
            ea1 = self.rec_edge_embedding(self.rec_distance_expansion(vec1.norm(dim=-1)))
            na1 = self.rec_node_embedding(rec.x[:n1])
            ew1 = edge_weight(vec1, self.rec_max_radius, self.smooth_edges)
            for layer in self.rec_emb_layers:
                ea_ = torch.cat([ea1, na1[ei1[0], :self.ns], na1[ei1[1], :self.ns]], -1)
                na1 = layer(na1, ei1, ea_, None, edge_weight=ew1, edge_vec=vec1)
            vec, rec_edge_attr, rec_node_attr = vec1.repeat(B, 1), ea1.repeat(B, 1), na1.repeat(B, 1)
            ew = ew1.repeat(B, 1) if torch.is_tensor(ew1) else ew1
        else:
            vec = (rec.pos[ei[1]] - rec.pos[ei[0]]).float()
            rec_edge_attr = self.rec_edge_embedding(self.rec_distance_expansion(vec.norm(dim=-1)))
            rec_node_attr = self.rec_node_embedding(rec.x)
            ew = edge_weight(vec, self.rec_max_radius, self.smooth_edges)
            for layer in self.rec_emb_layers:
                ea_ = torch.cat([rec_edge_attr, rec_node_attr[ei[0], :self.ns], rec_node_attr[ei[1], :self.ns]], -1)
                rec_node_attr = layer(rec_node_attr, ei, ea_, None, edge_weight=ew, edge_vec=vec)
        rec.rec_node_attr, rr.rec_edge_attr, rr.edge_weight = rec_node_attr, rec_edge_attr, ew
        rr.edge_sh = None   # evaluated inside the convolution kernel from the edge vectors; kept for attribute parity
        # CSR order of the static receptor graph (target = edge_index[0])
        tgt, order = torch.sort(ei[0], stable=True)
        c['rr_tgt'], c['rr_src'] = tgt, ei[1][order]
        c['rr_vec'] = vec[order].contiguous()
        c['rr_ea'] = rec_edge_attr[order].contiguous()
        c['rr_ew'] = ew[order].contiguous() if torch.is_tensor(ew) else None
        c['rr_tgt_batch'] = rec.batch[tgt]
        c['rec_ptr'] = ops.segment_ptr(rec.batch, B)
        c['lig_ptr'] = ops.segment_ptr(lig.batch, B)
        # rotatable bonds are static too
        mask = lig.edge_mask
        bonds = ll.edge_index[:, mask].long()
        c['bonds'], c['n_bonds'] = bonds, int(bonds.shape[1])
        c['bond_batch'] = lig.batch[bonds[0]] if bonds.shape[1] else None
        self._static_sync_free(data, c)
        rr._b200 = c
        return c

    def _static_sync_free(self, data, c):
        """Per-batch constants of the sync-free forward: node counts, the bond edges as a CSR by target atom, capacities of
        the per-step edge buffers (upper bounds that hold for ANY pose), int32 views.  One host read per batch."""
        rec, lig, ll = data['receptor'], data['ligand'], data['ligand', 'ligand']
        B, dev = data.num_graphs, lig.pos.device
        i32 = lambda t: t.to(torch.int32).contiguous()
        n_lig, n_rec = lig.batch.shape[0], rec.batch.shape[0]
        lig_cnt = (c['lig_ptr'][1:] - c['lig_ptr'][:-1])
        rec_cnt = (c['rec_ptr'][1:] - c['rec_ptr'][:-1])
        host = torch.stack([lig_cnt, rec_cnt]).cpu()                       # the one host read of the batch
        c['lig_cnt_f'] = lig_cnt.float().unsqueeze(1)
        c['rec_max'] = int(host[1].max()) if B else 0
        c['cap_cross'] = int((host[0].long() * host[1].long()).sum())      # every ligand atom x every residue of its complex
        c['lig_batch32'], c['rec_batch32'] = i32(lig.batch), i32(rec.batch)
        c['rr_gid32'] = i32(c['rr_tgt_batch'])
        # bond edges grouped by their convolution target (edge_index[0]), original order kept inside a group
        ei = ll.edge_index.long()
        order = torch.sort(ei[0], stable=True).indices
        c['pre_col'] = i32(ei[1][order])
        cnt = torch.bincount(ei[0], minlength=n_lig)[:n_lig] if ei.shape[1] else torch.zeros(n_lig, dtype=torch.long, device=dev)
        ptr = torch.zeros(n_lig + 1, dtype=torch.int32, device=dev)
        ptr[1:] = torch.cumsum(cnt, 0)
        c['pre_ptr'], c['pre_cnt'] = ptr, i32(cnt)
        attr = ll.edge_attr.float()[order] if ei.shape[1] else torch.zeros((0, self.in_lig_edge_features), device=dev)
        c['pre_attr'] = torch.cat([attr, torch.zeros((1, attr.shape[1]), device=dev)], 0)     # row -1: "not a bond"
        # radius_graph(max_num_neighbors=32) = radius with cap 33 minus the self hit: an atom whose own index is not among its
        # first 33 hits keeps 33 neighbours
        c['cap_ll'] = int(ei.shape[1]) + 33 * n_lig
        c['bond_lig_batch'] = lig.batch[c['bonds'][0]] if c['n_bonds'] else None
        c['cap_tor'] = 32 * c['n_bonds']
        c['bond_batch32'] = i32(c['bond_batch']) if c['n_bonds'] else None

    def _ligand_graph(self, data, c):
        """Bond edges + radius graph, sorted by convolution target (models/cg_model.py:467-497)."""
        lig = data['ligand']
        lig.node_sigma_emb = self.timestep_emb_func(lig.node_t['tr'])
        pos = lig.pos.float()
        row0, row1, bond_attr = graphs.ligand_graph_host(pos, c['lig_ptr'], lig.batch, data['ligand', 'ligand'],
                                                         self.lig_max_radius, self.in_lig_edge_features)
        tgt, order = torch.sort(row0, stable=True)
        src = row1[order]
        vec = pos[src] - pos[tgt]
        edge_attr = torch.cat([bond_attr[order], lig.node_sigma_emb[tgt], self.lig_distance_expansion(vec.norm(dim=-1))], 1)
        node_attr = torch.cat([lig.x.float(), lig.node_sigma_emb], 1)
        return node_attr, tgt, src, edge_attr, vec, edge_weight(vec, self.lig_max_radius, self.smooth_edges)

    # ---------------------------------------------------------------------------------------------------------
    def sync_free_capable(self):
        """The forward can run without any host synchronisation (and so inside a CUDA graph) when every convolution of the
        stack has a shape the fully fused kernel supports; otherwise the neighbour-list sizes go through the host."""
        if self._sync_free is None:
            ok = self.embed_also_ligand
            for layer in list(self.conv_layers) + list(getattr(self, 'lig_emb_layers', [])):
                ok = ok and layer.fused_capable(self.ns, self.ns)
            self._sync_free = bool(ok)
        return self._sync_free

    def _capacities_fit(self, c):
        """The 10000-neighbour cap of the cross graph (models/cg_model.py:546) is not binding, so the capacity buffers of the
        sync-free forward hold every edge."""
        return c['rec_max'] <= 10000

    @torch.no_grad()
    def forward(self, data):
        name = type(self).__name__
        if self.training:
            raise RuntimeError(f"diffdock_b200.{name} is inference-only: call .eval()")
        lig, rec = data['ligand'], data['receptor']
        if not lig.pos.is_cuda:
            raise RuntimeError(f"diffdock_b200.{name} runs on CUDA tensors only (no CPU fallback): data.to('cuda')")
        if self.no_aminoacid_identities:
            rec.x = rec.x * 0
        c = self._static(data)
        if self.sync_free_capable() and self._capacities_fit(c):
            return self._forward_sync_free(data, c)
        return self._forward_host_sized(data, c)

    # ---------------------------------------------------------------------------------------------------------
    def _forward_sync_free(self, data, c):
        """The whole forward without a device->host read: every per-step neighbour list is written into an upper-bound
        buffer by ddb200_graph_fill with its live length kept in device memory, the reverse direction of the cross graph is
        an index permutation of the forward one, the ligand-receptor edge embedding is one kernel, and the convolutions
        take (capacity, device count).  Shapes are static for a given batch, so a reverse-diffusion step can be captured in
        a CUDA graph (diffdock_b200/sampling.py)."""
        lig, rec = data['ligand'], data['receptor']
        ns = self.ns
        tr_sigma, rot_sigma, tor_sigma = self.t_to_sigma(*[data.complex_t[k] for k in ('tr', 'rot', 'tor')])
        n_lig = lig.batch.shape[0]
        pos, rpos = lig.pos.float().contiguous(), rec.pos.float().contiguous()

        # -- embeddings (models/cg_model.py:272-306) --------------------------------------------------------------
        sig = self.rec_sigma_embedding(self.timestep_emb_func(data.complex_t['tr'])).contiguous()      # [B, ns]
        rec_node = rec.rec_node_attr.clone()
        rec_node[:, :ns] += sig[rec.batch]
        lig.node_sigma_emb = self.timestep_emb_func(lig.node_t['tr'])

        # -- ligand graph: bonds + radius graph, CSR by target, built on the device (:467-497) -------------------------
        g_ll = graphs.ligand_graph(pos, c, self.lig_max_radius, lig.node_sigma_emb, self.lig_distance_expansion,
                                   self.lig_edge_embedding, self.smooth_edges)
        lig_node = self.lig_node_embedding(torch.cat([lig.x.float(), lig.node_sigma_emb], 1))
        for layer in self.lig_emb_layers:
            lig_node = layer.forward_groups(lig_node, [g_ll], gather_scalars=ns)

        # -- cross graph, both directions (:321-327, :539-562) ------------------------------------------------------------
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        lr = (self.cross_edge_embedding, self.cross_distance_expansion)
        g_lr, g_rl = graphs.cross_graph(pos, c['lig_ptr'], c['lig_batch32'], rpos, c['rec_ptr'], c['rec_batch32'], c['rec_max'],
                                        c['cap_cross'], n_lig, r, rpg, self._cross_embedder(lig, *lr, r, rpg), vec_sign=-1.0,
                                        fill_row=self._cross_fill_row(*lr))

        # -- joint graph: four edge groups (:329-338) ---------------------------------------------------------------
        node = torch.cat([lig_node, rec_node], 0)
        rr_tgt32 = c.setdefault('rr_tgt32', {}).get(n_lig)
        if rr_tgt32 is None:
            i32 = lambda t: t.to(torch.int32).contiguous()
            rr_tgt32 = c['rr_tgt32'][n_lig] = (i32(c['rr_tgt'] + n_lig), i32(c['rr_src'] + n_lig))
        groups = [
            g_ll,                                                                                         # lig <- lig
            g_lr,                                                                                         # lig <- rec
            (rr_tgt32[0], rr_tgt32[1], c['rr_ea'], c['rr_vec'], graphs.flat_weight(c['rr_ew']),
             dict(ea_add=sig, ea_add_idx=c['rr_gid32'])),                                                 # rec <- rec
            g_rl,                                                                                         # rec <- lig
        ]
        L = len(self.conv_layers)
        shared = self._shared_receptor_messages(data, c, rec, rec_node, sig, n_lig) if L > 1 else None
        for l, layer in enumerate(self.conv_layers):
            use = groups if l < L - 1 else groups[:2]       # last layer: only edges that end on ligand atoms (:347-349)
            if l == 0 and shared is not None:               # receptor <- receptor messages of layer 0: computed once per complex
                node = layer.forward_groups(node, [use[0], use[1], None, use[3]], gather_scalars=ns, init=shared)
            else:
                node = layer.forward_groups(node, use, gather_scalars=ns)
        lig_node = node[:n_lig]
        return self._heads(data, c, lig_node, tr_sigma, rot_sigma, tor_sigma, sync_free=True)

    def _shared_receptor_messages(self, data, c, rec, rec_node, sig, n_lig):
        """Layer-0 receptor<-receptor messages when the batch holds B poses of ONE complex at ONE diffusion time: the residue
        features entering the first interaction layer (static embedding + sigma embedding) and the contact graph are then the
        same in every copy, so the messages are computed for one copy (E/B edges) and added to all copies' accumulators.
        The reference recomputes them per pose (models/cg_model.py:342-349 over the B-fold receptor).  Needs the sampler's
        promise that all graphs of the batch share t (``data._uniform_t``; the model API allows per-graph times)."""
        uniq = getattr(rec, '_unique', None)
        if uniq is None or not getattr(data, '_uniform_t', False) or not self.differentiate_convolutions:
            return None
        n1, e1, B = uniq
        if B < 2 or n1 * B != rec_node.shape[0] or c['rr_tgt'].shape[0] != e1 * B:
            return None
        layer = self.conv_layers[0]
        if 'rr0' not in c:          # copy 0 of the CSR-sorted contact graph (targets of copy 0 sort first), local numbering
            i32 = lambda t: t.to(torch.int32).contiguous()
            c['rr0'] = (i32(c['rr_tgt'][:e1]), i32(c['rr_src'][:e1]), c['rr_ea'][:e1].contiguous(), c['rr_vec'][:e1].contiguous(),
                        c['rr_ew'][:e1].reshape(-1).contiguous() if c['rr_ew'] is not None else None)
        t0, s0, ea0, vec0, ew0 = c['rr0']
        zero_idx = c.setdefault('rr0_zero', torch.zeros(e1, dtype=torch.int32, device=ea0.device))
        g0 = (t0, s0, ea0, vec0, ew0, dict(ea_add=sig[:1].contiguous(), ea_add_idx=zero_idx))
        sum0, cnt0 = layer.accumulate_group(rec_node[:n1], g0, 2, n1, gather_scalars=self.ns)
        N = n_lig + rec_node.shape[0]
        sum_buf = torch.zeros((N, layer.out_size), dtype=torch.float32, device=sum0.device)
        cnt_buf = torch.zeros((N,), dtype=torch.float32, device=sum0.device)
        sum_buf[n_lig:].view(B, n1, layer.out_size).add_(sum0.unsqueeze(0))
        cnt_buf[n_lig:].view(B, n1).add_(cnt0.unsqueeze(0))
        return sum_buf, cnt_buf

    def _cross_edge_embedding(self, node_sigma_emb, vec, row, n_dev, mlp, gs):
        """``mlp``(cat[sigma_emb[lig], ``gs``(d)]) of ligand <- x edges, e.g. cross_edge_embedding with the cross distance
        expansion (models/cg_model.py:326,553-554): the sigma half of the first Linear is applied per ligand NODE, the rest
        per edge in one kernel (ddb200_edge_embed)."""
        l1, l2 = mlp[0], mlp[-1]
        S = node_sigma_emb.shape[1]
        if self._edge_embed_in_kernel(mlp, gs):
            u = torch.addmm(l1.bias, node_sigma_emb, l1.weight[:, :S].t()).contiguous()
            return ops.edge_embed(vec, row, u, l1.weight[:, S:].contiguous(), l2.weight.contiguous(), l2.bias.contiguous(),
                                  gs.offset.contiguous(), float(gs.coeff), n_dev)
        attr = torch.cat([node_sigma_emb[row.long()], gs(vec.norm(dim=-1))], 1)      # library path on the padded buffer
        return mlp(attr)

    def _cross_embedder(self, lig, mlp, gs, r=None, rpg=None):
        """``embed`` of graphs.cross_graph: edge attributes through ``mlp`` / ``gs`` and, with smooth_edges, the edge weight
        at the cut-off (``r``, or ``rpg`` per complex)."""
        def embed(tgt, vec, n_dev):
            ea = self._cross_edge_embedding(lig.node_sigma_emb, vec, tgt, n_dev, mlp, gs)
            if not self.smooth_edges:
                return ea, None
            return ea, graphs.flat_weight(edge_weight(vec, rpg[lig.batch[tgt.long()]] if rpg is not None else r, True))
        return embed

    def _edge_embed_in_kernel(self, mlp, gs):
        return (gs.offset.shape[0], self.ns) in ops.EDGE_EMBED_SHAPES and len(mlp) == 4

    def _cross_fill_row(self, mlp, gs):
        """``fill_row`` of a sync-free cross graph: rows beyond the live count must be valid (zero) when library ops gather
        over the whole buffer - the smooth edge weight, or the embedding MLP when its shape is outside the edge-embedding
        kernel's templates."""
        return 0 if self.smooth_edges or not self._edge_embed_in_kernel(mlp, gs) else None

    # ---------------------------------------------------------------------------------------------------------
    def _forward_host_sized(self, data, c):
        """Forward with exactly-sized neighbour lists (one host read of each edge count): convolution shapes outside the
        fused kernel's templates, or more than 10000 residues per complex."""
        lig, rec = data['ligand'], data['receptor']
        ns = self.ns
        tr_sigma, rot_sigma, tor_sigma = self.t_to_sigma(*[data.complex_t[k] for k in ('tr', 'rot', 'tor')])

        # -- embeddings (models/cg_model.py:272-306) --------------------------------------------------------------
        sig = self.rec_sigma_embedding(self.timestep_emb_func(data.complex_t['tr']))
        rec_node = rec.rec_node_attr.clone()
        rec_node[:, :ns] += sig[rec.batch]
        rr_ea = c['rr_ea'] + sig[c['rr_tgt_batch']]
        lig_x, ll_tgt, ll_src, ll_ea, ll_vec, ll_ew = self._ligand_graph(data, c)
        lig_node = self.lig_node_embedding(lig_x)
        ll_ea = self.lig_edge_embedding(ll_ea)
        assert self.embed_also_ligand, "otherwise reimplement padding"
        ll_ei = torch.stack([ll_tgt, ll_src])
        for layer in self.lig_emb_layers:
            ea_ = torch.cat([ll_ea, lig_node[ll_tgt, :ns], lig_node[ll_src, :ns]], -1)
            lig_node = layer(lig_node, ll_ei, ea_, None, edge_weight=ll_ew, edge_vec=ll_vec, assume_sorted=True)

        # -- cross graph (:321-327) ---------------------------------------------------------------------------------
        lp = lig.pos.float()
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        li, ri, lr_vec = graphs.cross_graph_host(lp, rec.pos.float(), c['rec_ptr'], lig.batch, r, rpg)
        lr_ea = torch.cat([lig.node_sigma_emb[li], self.cross_distance_expansion(lr_vec.norm(dim=-1))], 1)
        cutoff_d = rpg[lig.batch[li]] if rpg is not None else r
        lr_ew = edge_weight(lr_vec, cutoff_d, self.smooth_edges)
        lr_ea = self.cross_edge_embedding(lr_ea)

        # -- joint graph: four edge groups, each CSR-sorted by target (:329-338) ------------------------------------
        n_lig = lig_node.shape[0]
        node = torch.cat([lig_node, rec_node], 0)
        i32 = lambda t: t.to(torch.int32).contiguous()
        rr_tgt32 = c.setdefault('rr_tgt32', {}).get(n_lig)
        if rr_tgt32 is None:      # static receptor graph: int32 indices in the joint numbering, once per batch
            rr_tgt32 = c['rr_tgt32'][n_lig] = (i32(c['rr_tgt'] + n_lig), i32(c['rr_src'] + n_lig))
        g_lr, g_rl = graphs.cross_groups_host(li, ri, n_lig, lr_ea, lr_vec, lr_ew, vec_sign=-1.0)
        groups = [   # (target, gathered node, edge attr, edge vector, edge weight): int32, CSR-sorted, built once per forward
            (i32(ll_tgt), i32(ll_src), ll_ea, ll_vec.contiguous(), graphs.flat_weight(ll_ew)),           # lig <- lig
            g_lr,                                                                                        # lig <- rec
            (rr_tgt32[0], rr_tgt32[1], rr_ea, c['rr_vec'], graphs.flat_weight(c['rr_ew'])),              # rec <- rec
            g_rl,                                                                                        # rec <- lig, SH(-v)
        ]
        L = len(self.conv_layers)
        for l, layer in enumerate(self.conv_layers):
            use = groups if l < L - 1 else groups[:2]       # last layer: only edges that end on ligand atoms (:347-349)
            if not self.differentiate_convolutions:         # one radial MLP for all edge types: a single merged group
                use = graphs.merge_groups(use)
            node = layer.forward_groups(node, use, gather_scalars=ns)
        lig_node = node[:n_lig]
        return self._heads(data, c, lig_node, tr_sigma, rot_sigma, tor_sigma, sync_free=False)

    def _heads(self, data, c, lig_node, tr_sigma, rot_sigma, tor_sigma, sync_free):
        lig = data['ligand']
        ns, B = self.ns, data.num_graphs
        n_lig = lig_node.shape[0]
        # -- translation / rotation head (:368-395) -----------------------------------------------------------------
        pos = lig.pos.float()
        arange = torch.arange(n_lig, device=pos.device)
        center = torch.zeros((B, 3), device=pos.device).index_add_(0, lig.batch, pos)
        center = center / c['lig_cnt_f']
        c_vec = pos - center[lig.batch]
        c_ea = torch.cat([self.center_distance_expansion(c_vec.norm(dim=-1)), lig.node_sigma_emb], 1)
        c_ea = self.center_edge_embedding(c_ea)
        idx = arange if self.fixed_center_conv else lig.batch            # hazard C.6: graph id indexes lig_node
        c_ea = torch.cat([c_ea, lig_node[idx, :ns]], -1)
        glob = self.final_conv(lig_node, torch.stack([lig.batch, arange]), c_ea, None, out_nodes=B, edge_vec=c_vec,
                               assume_sorted=True)
        tr_pred = glob[:, :3] + (glob[:, 6:9] if not self.odd_parity else 0)
        rot_pred = glob[:, 3:6] + (glob[:, 9:] if not self.odd_parity else 0)
        data.graph_sigma_emb = self.timestep_emb_func(data.complex_t['tr'])
        tr_norm = torch.linalg.vector_norm(tr_pred, dim=1).unsqueeze(1)
        tr_pred = tr_pred / tr_norm * self.tr_final_layer(torch.cat([tr_norm, data.graph_sigma_emb], dim=1))
        rot_norm = torch.linalg.vector_norm(rot_pred, dim=1).unsqueeze(1)
        rot_pred = rot_pred / rot_norm * self.rot_final_layer(torch.cat([rot_norm, data.graph_sigma_emb], dim=1))
        if self.scale_by_sigma:
            tr_pred = tr_pred / tr_sigma.unsqueeze(1)
            rot_pred = rot_pred * self._so3_score_norm(rot_sigma).unsqueeze(1)

        if self.no_torsion or c['n_bonds'] == 0:
            return tr_pred, rot_pred, torch.empty(0, device=self.device), None

        # -- torsion head (:406-423) --------------------------------------------------------------------------------
        bonds = c['bonds']
        n_bonds = c['n_bonds']
        bond_pos = ((pos[bonds[0]] + pos[bonds[1]]) / 2).contiguous()
        if sync_free:
            # upper-bound buffer (32 atoms per bond, models/cg_model.py:630); slots beyond the live count point at an extra
            # dummy bond row (index n_bonds) that is dropped after the convolution
            bi32, ai32, t_vec, _, _, _ = graphs.capacity_graph(pos.contiguous(), bond_pos, c['lig_ptr'], c['bond_batch32'],
                                                               c['cap_tor'], self.lig_max_radius, max_num_neighbors=32,
                                                               fill_row=n_bonds)
            bi, ai = bi32.long(), ai32.long()
            bi_g = bi.clamp_max(n_bonds - 1)            # gathers of per-bond quantities for the dummy slots: any valid row
            n_out = n_bonds + 1
        else:
            bi, ai, _ = ops.radius(pos, bond_pos, c['lig_ptr'], c['bond_batch'], r=self.lig_max_radius, max_num_neighbors=32)
            bi, ai = bi.long(), ai.long()
            t_vec = pos[ai] - bond_pos[bi]
            bi_g, n_out = bi, n_bonds
        t_ea = self.final_edge_embedding(self.lig_distance_expansion(t_vec.norm(dim=-1)))
        bond_vec = pos[bonds[1]] - pos[bonds[0]]
        bond_attr = lig_node[bonds[0]] + lig_node[bonds[1]]
        t_sh = torch.einsum('ea,eb,abc->ec', _sh_full(t_vec, self.sh_lmax), _sh_l2(bond_vec)[bi_g], self._tor_tp)
        t_ea = torch.cat([t_ea, lig_node[ai, :ns], bond_attr[bi_g, :ns]], -1)
        tor_pred = self.tor_bond_conv(lig_node, torch.stack([bi, ai]), t_ea, t_sh, out_nodes=n_out, reduce='mean',
                                      edge_weight=edge_weight(t_vec, self.lig_max_radius, self.smooth_edges), assume_sorted=True)
        tor_pred = self.tor_final_layer(tor_pred[:n_bonds]).squeeze(1)
        edge_sigma = tor_sigma[c['bond_lig_batch']]
        if self.scale_by_sigma:
            tor_pred = tor_pred * torch.sqrt(self._torus_score_norm(edge_sigma))
        return tr_pred, rot_pred, tor_pred, None
