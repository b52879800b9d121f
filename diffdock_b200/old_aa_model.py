"""Drop-in for the reference's ALL-ATOM confidence model ``models/old_aa_model.py:AAOldModel`` in confidence mode - what
``inference.py:192,209`` builds when the confidence model's parameters say ``all_atoms`` (the released DiffDock-L ranking
model) and ``utils/sampling.py:208-227`` calls once per batch of final poses (SURVEY.md section 8, rows f2 / f3).

Same constructor keywords, ``forward(data) -> confidence [B]`` (``[B, 2]`` with affinity_prediction) and ``state_dict`` keys
as the reference class for: confidence_mode=True, use_old_atom_encoder=True (the only encoder the reference class can be
built with - its new AtomEncoder rejects the ``lm_embedding_type`` keyword, models/old_aa_model.py:71), one noise schedule,
parallel=1.  Three node types and nine convolutions per interaction layer (:105-121, :229-266), all on the same sm_100a
kernels as the score model: neighbour lists from ddb200_radius_*, spherical harmonics evaluated in-kernel from the edge
vectors, OldTensorProductConvLayer on the fully fused tcgen05 kernel when its shapes allow.  The reversed directions
(atom<-ligand, residue<-ligand, residue<-atom) reuse the forward edge attributes AND the forward vector's harmonics, as the
reference does (:246-266).

CUDA only, inference only.  No CPU fallback.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch import nn

from . import graphs, ops
from .irreps import irreps_str, sh_irreps
from .layers import GaussianSmearing, OldAtomEncoder, _mlp, edge_weight
from .old_cg_model import ConfidenceModel
from .synthetic import (LIG_FEATURE_DIMS as lig_feature_dims, REC_ATOM_FEATURE_DIMS as rec_atom_feature_dims,
                        REC_RESIDUE_FEATURE_DIMS as rec_residue_feature_dims)
from .tensor_layers import OldTensorProductConvLayer


class AAOldModel(ConfidenceModel):
    def __init__(self, t_to_sigma, device, timestep_emb_func, in_lig_edge_features=4, sigma_embed_dim=32, sh_lmax=2,
                 ns=16, nv=4, num_conv_layers=2, lig_max_radius=5, rec_max_radius=30, cross_max_distance=250,
                 center_max_distance=30, distance_embed_dim=32, cross_distance_embed_dim=32, no_torsion=False,
                 scale_by_sigma=True, norm_by_sigma=True, use_second_order_repr=False, batch_norm=True,
                 dynamic_max_cross=False, dropout=0.0, smooth_edges=False, odd_parity=False,
                 separate_noise_schedule=False, lm_embedding_type=False, confidence_mode=False, confidence_dropout=0,
                 confidence_no_batchnorm=False, asyncronous_noise_schedule=False, affinity_prediction=False, parallel=1,
                 parallel_aggregators="mean max min std", num_confidence_outputs=1, fixed_center_conv=False,
                 no_aminoacid_identities=False, include_miscellaneous_atoms=False, use_old_atom_encoder=False,
                 lm_embedding_dim=1280):
        super().__init__()
        lm_embedding_type = lm_embedding_type or None
        assert (not no_aminoacid_identities) or (lm_embedding_type is None), "no language model emb without identities"
        if parallel != 1:
            raise NotImplementedError("parallel > 1 (affinity aggregation over several poses) is outside the hot-path scope")
        if not confidence_mode:
            raise NotImplementedError("diffdock_b200.AAOldModel is built in confidence mode only (SURVEY.md rows f2/f3); "
                                      "the score model is diffdock_b200.cg_model.CGModel")
        if not use_old_atom_encoder:
            raise NotImplementedError("models/old_aa_model.py can only be constructed with use_old_atom_encoder=True")
        if include_miscellaneous_atoms or separate_noise_schedule or asyncronous_noise_schedule or use_second_order_repr:
            raise NotImplementedError("misc atoms / separate or asynchronous noise schedules / second-order irreps are "
                                      "outside the hot-path scope (SURVEY.md section 8)")
        self.t_to_sigma, self.device, self.timestep_emb_func = t_to_sigma, device, timestep_emb_func
        self.in_lig_edge_features, self.sigma_embed_dim = in_lig_edge_features, sigma_embed_dim
        self.lig_max_radius, self.rec_max_radius = lig_max_radius, rec_max_radius
        self.cross_max_distance, self.dynamic_max_cross = cross_max_distance, dynamic_max_cross
        self.sh_lmax, self.sh_irreps = sh_lmax, irreps_str(sh_irreps(sh_lmax))
        self.ns, self.nv, self.smooth_edges = ns, nv, smooth_edges
        self.confidence_mode, self.num_conv_layers = confidence_mode, num_conv_layers
        self.affinity_prediction, self.no_aminoacid_identities = affinity_prediction, no_aminoacid_identities
        S, D, Dx = sigma_embed_dim, distance_embed_dim, cross_distance_embed_dim
        kw = dict(lm_embedding_dim=lm_embedding_dim) if lm_embedding_type is not None else {}
        self.lig_node_embedding = OldAtomEncoder(ns, lig_feature_dims, S)
        self.lig_edge_embedding = _mlp(in_lig_edge_features + S + D, ns, ns, dropout)
        self.rec_node_embedding = OldAtomEncoder(ns, rec_residue_feature_dims, S, lm_embedding_type=lm_embedding_type, **kw)
        self.rec_edge_embedding = _mlp(S + D, ns, ns, dropout)
        self.atom_node_embedding = OldAtomEncoder(ns, rec_atom_feature_dims, S)
        self.atom_edge_embedding = _mlp(S + D, ns, ns, dropout)
        self.lr_edge_embedding = _mlp(S + Dx, ns, ns, dropout)
        self.ar_edge_embedding = _mlp(S + D, ns, ns, dropout)
        self.la_edge_embedding = _mlp(S + Dx, ns, ns, dropout)
        self.lig_distance_expansion = GaussianSmearing(0.0, lig_max_radius, D)
        self.rec_distance_expansion = GaussianSmearing(0.0, rec_max_radius, D)
        self.cross_distance_expansion = GaussianSmearing(0.0, cross_max_distance, Dx)
        seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e',
               f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']
        convs = []
        for i in range(num_conv_layers):
            p = dict(in_irreps=seq[min(i, 3)], sh_irreps=self.sh_irreps, out_irreps=seq[min(i + 1, 3)],
                     n_edge_features=3 * ns, residual=False, batch_norm=batch_norm, dropout=dropout)
            convs += [OldTensorProductConvLayer(**p) for _ in range(9)]       # 3 intra & 6 inter per layer (:119-120)
        self.conv_layers = nn.ModuleList(convs)
        bn = (lambda: nn.Identity()) if confidence_no_batchnorm else (lambda: nn.BatchNorm1d(ns))
        out_dim = (num_confidence_outputs + 1) if affinity_prediction else num_confidence_outputs
        self.confidence_predictor = nn.Sequential(
            nn.Linear(2 * ns if num_conv_layers >= 3 else ns, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout),
            nn.Linear(ns, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout), nn.Linear(ns, out_dim))

    def _static_graph(self, data, nt, pos, edge_embedding, node_embedding, expansion, max_r):
        """Receptor-residue / receptor-atom graph on precomputed edges (:400-445); row 0 = target, row 1 = gathered node."""
        st = data[nt]
        st.node_sigma_emb = self.timestep_emb_func(st.node_t['tr'])
        ei = data[nt, nt].edge_index.long()
        vec = pos[ei[1]] - pos[ei[0]]
        ea = edge_embedding(torch.cat([st.node_sigma_emb[ei[0]], expansion(vec.norm(dim=-1))], 1))
        node = node_embedding(torch.cat([st.x.float(), st.node_sigma_emb], 1))
        return node, ei, ea, vec, edge_weight(vec, max_r, self.smooth_edges)

    @torch.no_grad()
    def forward(self, data):                                            # models/old_aa_model.py:202-286
        if self.training:
            raise RuntimeError("diffdock_b200.AAOldModel is inference-only: call .eval()")
        lig_s, rec_s, atom_s = data['ligand'], data['receptor'], data['atom']
        if not lig_s.pos.is_cuda:
            raise RuntimeError("diffdock_b200.AAOldModel runs on CUDA tensors only (no CPU fallback): data.to('cuda')")
        if self.no_aminoacid_identities:
            rec_s.x = rec_s.x * 0
        B, ns, L, C = data.num_graphs, self.ns, self.num_conv_layers, self.conv_layers
        tr_sigma = data.complex_t['tr']                                 # confidence mode: times are used as they are (:209)
        lp, rp, ap = lig_s.pos.float(), rec_s.pos.float(), atom_s.pos.float()
        lig_ptr = ops.segment_ptr(lig_s.batch, B)
        rec_ptr, atom_ptr = ops.segment_ptr(rec_s.batch, B), ops.segment_ptr(atom_s.batch, B)

        # ligand graph (:358-398): bonds + radius graph
        lig_s.node_sigma_emb = self.timestep_emb_func(lig_s.node_t['tr'])
        row0, row1, bond_attr = graphs.ligand_graph_host(lp, lig_ptr, lig_s.batch, data['ligand', 'ligand'],
                                                         self.lig_max_radius, self.in_lig_edge_features)
        lig_ei = torch.stack([row0, row1])
        lig_vec = lp[lig_ei[1]] - lp[lig_ei[0]]
        lig_ea = torch.cat([bond_attr, lig_s.node_sigma_emb[lig_ei[0]], self.lig_distance_expansion(lig_vec.norm(dim=-1))], 1)
        lig_w = edge_weight(lig_vec, self.lig_max_radius, self.smooth_edges)
        lig = self.lig_node_embedding(torch.cat([lig_s.x.float(), lig_s.node_sigma_emb], 1))
        lig_ea = self.lig_edge_embedding(lig_ea)

        rec, rec_ei, rec_ea, rec_vec, rec_w = self._static_graph(data, 'receptor', rp, self.rec_edge_embedding,
                                                                 self.rec_node_embedding, self.rec_distance_expansion,
                                                                 self.rec_max_radius)
        atom, at_ei, at_ea, at_vec, at_w = self._static_graph(data, 'atom', ap, self.atom_edge_embedding,
                                                              self.atom_node_embedding, self.lig_distance_expansion,
                                                              self.lig_max_radius)

        # cross graphs (:447-491): ligand-residue (cut-off per complex), ligand-atom (lig_max_radius), atom-residue (given)
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        li, ri, lr_vec = graphs.cross_graph_host(lp, rp, rec_ptr, lig_s.batch, r, rpg)
        lr = torch.stack([li, ri])
        lr_ea = self.lr_edge_embedding(torch.cat([lig_s.node_sigma_emb[lr[0]],
                                                  self.cross_distance_expansion(lr_vec.norm(dim=-1))], 1))
        lr_w = edge_weight(lr_vec, rpg[lig_s.batch[lr[0]]] if rpg is not None else r, self.smooth_edges)
        la_l, la_a, la_vec = graphs.cross_graph_host(lp, ap, atom_ptr, lig_s.batch, float(self.lig_max_radius))
        la = torch.stack([la_l, la_a])
        la_ea = self.la_edge_embedding(torch.cat([lig_s.node_sigma_emb[la[0]],
                                                  self.cross_distance_expansion(la_vec.norm(dim=-1))], 1))
        la_w = edge_weight(la_vec, self.lig_max_radius, self.smooth_edges)
        ar = data['atom', 'receptor'].edge_index.long()
        ar_vec = rp[ar[1]] - ap[ar[0]]
        ar_ea = self.ar_edge_embedding(torch.cat([atom_s.node_sigma_emb[ar[0]],
                                                  self.rec_distance_expansion(ar_vec.norm(dim=-1))], 1))

        cat = lambda e, a, b: torch.cat([e, a[:, :ns], b[:, :ns]], -1)
        flip = lambda ei: torch.flip(ei, dims=[0])
        for l in range(L):
            k = 9 * l
            lig_up = C[k](lig, lig_ei, cat(lig_ea, lig[lig_ei[0]], lig[lig_ei[1]]), None, edge_weight=lig_w, edge_vec=lig_vec)
            lr_up = C[k + 1](rec, lr, cat(lr_ea, lig[lr[0]], rec[lr[1]]), None, out_nodes=lig.shape[0], edge_weight=lr_w,
                             edge_vec=lr_vec, assume_sorted=True)
            la_up = C[k + 2](atom, la, cat(la_ea, lig[la[0]], atom[la[1]]), None, out_nodes=lig.shape[0], edge_weight=la_w,
                             edge_vec=la_vec, assume_sorted=True)
            if l != L - 1:
                at_up = C[k + 3](atom, at_ei, cat(at_ea, atom[at_ei[0]], atom[at_ei[1]]), None, edge_weight=at_w, edge_vec=at_vec)
                al_up = C[k + 4](lig, flip(la), cat(la_ea, atom[la[1]], lig[la[0]]), None, out_nodes=atom.shape[0],
                                 edge_weight=la_w, edge_vec=la_vec)
                ar_up = C[k + 5](rec, ar, cat(ar_ea, atom[ar[0]], rec[ar[1]]), None, out_nodes=atom.shape[0], edge_weight=1.0,
                                 edge_vec=ar_vec)
                rec_up = C[k + 6](rec, rec_ei, cat(rec_ea, rec[rec_ei[0]], rec[rec_ei[1]]), None, edge_weight=rec_w,
                                  edge_vec=rec_vec)
                rl_up = C[k + 7](lig, flip(lr), cat(lr_ea, rec[lr[1]], lig[lr[0]]), None, out_nodes=rec.shape[0],
                                 edge_weight=lr_w, edge_vec=lr_vec)
                ra_up = C[k + 8](atom, flip(ar), cat(ar_ea, rec[ar[1]], atom[ar[0]]), None, out_nodes=rec.shape[0],
                                 edge_weight=1.0, edge_vec=ar_vec)
            lig = F.pad(lig, (0, lig_up.shape[-1] - lig.shape[-1])) + lig_up + la_up + lr_up
            if l != L - 1:
                atom = F.pad(atom, (0, at_up.shape[-1] - atom.shape[-1])) + at_up + al_up + ar_up
                rec = F.pad(rec, (0, rec_up.shape[-1] - rec.shape[-1])) + rec_up + ra_up + rl_up
        return self._confidence(lig, lig_s.batch, B)
