"""Drop-in for the reference's confidence model ``models/old_cg_model.py:CGOldModel`` in confidence mode - the ranking
model ``utils/sampling.py:208-227`` calls once per batch of final poses (SURVEY.md section 8, row f2).

Same constructor keywords, ``forward(data) -> confidence [B]`` (``[B, 2]`` with affinity_prediction) and ``state_dict``
keys as the reference class for: confidence_mode=True, use_old_atom_encoder=True (the only encoder the reference class
can be built with - its new AtomEncoder rejects the ``lm_embedding_type`` keyword, models/old_cg_model.py:63-66), no
miscellaneous atoms, one noise schedule.  The convolutions are the same sm_100a kernels as the score model's: every
OldTensorProductConvLayer call goes through the fully fused tcgen05 kernel (csrc/fused_conv.cu) when its shapes allow,
neighbour lists come from ddb200_radius_*, spherical harmonics are evaluated in-kernel from the edge vectors.

CUDA only, inference only.  No CPU fallback.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch import nn

from . import graphs, ops
from .irreps import irreps_str, sh_irreps
from .layers import GaussianSmearing, OldAtomEncoder, _mlp, edge_weight
from .synthetic import LIG_FEATURE_DIMS as lig_feature_dims, REC_RESIDUE_FEATURE_DIMS as rec_residue_feature_dims
from .tensor_layers import OldTensorProductConvLayer


class ConfidenceModel(nn.Module):
    """What the coarse-grained and the all-atom confidence models share: loading reference checkpoints, and the head that
    pools the ligand's scalar features per complex."""

    def load_state_dict(self, state_dict, strict=True, **kw):
        """Reference checkpoints carry e3nn's tensor-product buffers (``*.tp.*``): dropped, the kernels have their own tables."""
        sd = {k: v for k, v in state_dict.items() if '.tp.' not in k}
        return super().load_state_dict(sd, strict=strict, **kw)

    def _confidence(self, lig_node, lig_batch, B):
        """confidence_predictor of the per-complex mean of the ligand scalars: the 0e channels, and the 0o channels too with
        three or more layers (models/old_cg_model.py:285-301)."""
        ns = self.ns
        scal = torch.cat([lig_node[:, :ns], lig_node[:, -ns:]], 1) if self.num_conv_layers >= 3 else lig_node[:, :ns]
        pooled = torch.zeros((B, scal.shape[1]), device=scal.device, dtype=scal.dtype).index_add_(0, lig_batch, scal)
        pooled = pooled / torch.bincount(lig_batch, minlength=B).clamp(min=1).unsqueeze(1)
        return self.confidence_predictor(pooled).squeeze(dim=-1)


class CGOldModel(ConfidenceModel):
    def __init__(self, t_to_sigma, device, timestep_emb_func, in_lig_edge_features=4, sigma_embed_dim=32, sh_lmax=2,
                 ns=16, nv=4, num_conv_layers=2, lig_max_radius=5, rec_max_radius=30, cross_max_distance=250,
                 center_max_distance=30, distance_embed_dim=32, cross_distance_embed_dim=32, no_torsion=False,
                 scale_by_sigma=True, norm_by_sigma=True, use_second_order_repr=False, batch_norm=True,
                 dynamic_max_cross=False, dropout=0.0, smooth_edges=False, odd_parity=False,
                 separate_noise_schedule=False, lm_embedding_type=None, confidence_mode=False, confidence_dropout=0,
                 confidence_no_batchnorm=False, asyncronous_noise_schedule=False, affinity_prediction=False, parallel=1,
                 parallel_aggregators="mean max min std", num_confidence_outputs=1, fixed_center_conv=False,
                 no_aminoacid_identities=False, include_miscellaneous_atoms=False, use_old_atom_encoder=False,
                 lm_embedding_dim=1280):
        super().__init__()
        assert parallel == 1, "not implemented"
        assert (not no_aminoacid_identities) or (lm_embedding_type is None), "no language model emb without identities"
        if not confidence_mode:
            raise NotImplementedError("diffdock_b200.CGOldModel is built in confidence mode only (SURVEY.md row f2); "
                                      "the score model is diffdock_b200.cg_model.CGModel")
        if not use_old_atom_encoder:
            raise NotImplementedError("models/old_cg_model.py can only be constructed with use_old_atom_encoder=True")
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
        kw = dict(lm_embedding_dim=lm_embedding_dim) if lm_embedding_type is not None else {}
        self.lig_node_embedding = OldAtomEncoder(ns, lig_feature_dims, sigma_embed_dim)
        self.lig_edge_embedding = _mlp(in_lig_edge_features + sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.rec_node_embedding = OldAtomEncoder(ns, rec_residue_feature_dims, sigma_embed_dim,
                                                 lm_embedding_type=lm_embedding_type, **kw)
        self.rec_edge_embedding = _mlp(sigma_embed_dim + distance_embed_dim, ns, ns, dropout)
        self.cross_edge_embedding = _mlp(sigma_embed_dim + cross_distance_embed_dim, ns, ns, dropout)
        self.lig_distance_expansion = GaussianSmearing(0.0, lig_max_radius, distance_embed_dim)
        self.rec_distance_expansion = GaussianSmearing(0.0, rec_max_radius, distance_embed_dim)
        self.cross_distance_expansion = GaussianSmearing(0.0, cross_max_distance, cross_distance_embed_dim)
        seq = [f'{ns}x0e', f'{ns}x0e + {nv}x1o', f'{ns}x0e + {nv}x1o + {nv}x1e',
               f'{ns}x0e + {nv}x1o + {nv}x1e + {ns}x0o']
        lig, rec, l2r, r2l = [], [], [], []
        for i in range(num_conv_layers):
            p = dict(in_irreps=seq[min(i, 3)], sh_irreps=self.sh_irreps, out_irreps=seq[min(i + 1, 3)],
                     n_edge_features=3 * ns, hidden_features=3 * ns, residual=False, batch_norm=batch_norm,
                     dropout=dropout)
            lig.append(OldTensorProductConvLayer(**p))           # creation order of the reference (:118-125)
            rec.append(OldTensorProductConvLayer(**p))
            l2r.append(OldTensorProductConvLayer(**p))
            r2l.append(OldTensorProductConvLayer(**p))
        self.lig_conv_layers, self.rec_conv_layers = nn.ModuleList(lig), nn.ModuleList(rec)
        self.lig_to_rec_conv_layers, self.rec_to_lig_conv_layers = nn.ModuleList(l2r), nn.ModuleList(r2l)
        bn = (lambda: nn.Identity()) if confidence_no_batchnorm else (lambda: nn.BatchNorm1d(ns))
        self.confidence_predictor = nn.Sequential(
            nn.Linear(2 * ns if num_conv_layers >= 3 else ns, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout),
            nn.Linear(ns, ns), bn(), nn.ReLU(), nn.Dropout(confidence_dropout),
            nn.Linear(ns, 2 if affinity_prediction else 1))

    @torch.no_grad()
    def forward(self, data):                                            # models/old_cg_model.py:203-301
        if self.training:
            raise RuntimeError("diffdock_b200.CGOldModel is inference-only: call .eval()")
        lig, rec = data['ligand'], data['receptor']
        if not lig.pos.is_cuda:
            raise RuntimeError("diffdock_b200.CGOldModel runs on CUDA tensors only (no CPU fallback): data.to('cuda')")
        if self.no_aminoacid_identities:
            rec.x = rec.x * 0
        B, ns = data.num_graphs, self.ns
        tr_sigma = data.complex_t['tr']                                 # confidence mode: times are used as they are
        lp, rp = lig.pos.float(), rec.pos.float()
        lig_ptr, rec_ptr = ops.segment_ptr(lig.batch, B), ops.segment_ptr(rec.batch, B)

        # ligand graph (:361-391): bonds + radius graph; row 0 = convolution target, row 1 = gathered node
        lig.node_sigma_emb = self.timestep_emb_func(lig.node_t['tr'])
        row0, row1, bond_attr = graphs.ligand_graph_host(lp, lig_ptr, lig.batch, data['ligand', 'ligand'], self.lig_max_radius,
                                                         self.in_lig_edge_features)
        lig_ei = torch.stack([row0, row1])
        lig_vec = lp[lig_ei[1]] - lp[lig_ei[0]]
        lig_ea = torch.cat([bond_attr, lig.node_sigma_emb[lig_ei[0]], self.lig_distance_expansion(lig_vec.norm(dim=-1))], 1)
        lig_ew = edge_weight(lig_vec, self.lig_max_radius, self.smooth_edges)
        lig_node = self.lig_node_embedding(torch.cat([lig.x.float(), lig.node_sigma_emb], 1))
        lig_ea = self.lig_edge_embedding(lig_ea)

        # receptor graph (:393-414)
        rec.node_sigma_emb = self.timestep_emb_func(rec.node_t['tr'])
        rec_ei = data['receptor', 'receptor'].edge_index.long()
        rec_vec = rp[rec_ei[1]] - rp[rec_ei[0]]
        rec_ea = self.rec_edge_embedding(torch.cat([rec.node_sigma_emb[rec_ei[0]],
                                                    self.rec_distance_expansion(rec_vec.norm(dim=-1))], 1))
        rec_ew = edge_weight(rec_vec, self.rec_max_radius, self.smooth_edges)
        rec_node = self.rec_node_embedding(torch.cat([rec.x.float(), rec.node_sigma_emb], 1))

        # cross graph (:439-461): row 0 = ligand atom, row 1 = receptor residue, vector receptor - ligand
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        li, ri, lr_vec = graphs.cross_graph_host(lp, rp, rec_ptr, lig.batch, r, rpg)
        lr_ei, rl_ei = torch.stack([li, ri]), torch.stack([ri, li])
        lr_ea = self.cross_edge_embedding(torch.cat([lig.node_sigma_emb[li],
                                                     self.cross_distance_expansion(lr_vec.norm(dim=-1))], 1))
        lr_ew = edge_weight(lr_vec, rpg[lig.batch[li]] if rpg is not None else r, self.smooth_edges)

        L = len(self.lig_conv_layers)
        for l in range(L):
            ea_ = torch.cat([lig_ea, lig_node[lig_ei[0], :ns], lig_node[lig_ei[1], :ns]], -1)
            lig_intra = self.lig_conv_layers[l](lig_node, lig_ei, ea_, None, edge_weight=lig_ew, edge_vec=lig_vec)
            cross_ea_ = torch.cat([lr_ea, lig_node[li, :ns], rec_node[ri, :ns]], -1)
            lig_inter = self.rec_to_lig_conv_layers[l](rec_node, lr_ei, cross_ea_, None, out_nodes=lig_node.shape[0],
                                                       edge_weight=lr_ew, edge_vec=lr_vec, assume_sorted=True)
            if l != L - 1:
                ea_ = torch.cat([rec_ea, rec_node[rec_ei[0], :ns], rec_node[rec_ei[1], :ns]], -1)
                rec_intra = self.rec_conv_layers[l](rec_node, rec_ei, ea_, None, edge_weight=rec_ew, edge_vec=rec_vec)
                # ligand -> receptor messages reuse the ligand-centred attributes AND harmonics Y(receptor - ligand),
                # i.e. of the vector target - gathered (:275-276)
                rec_inter = self.lig_to_rec_conv_layers[l](lig_node, rl_ei, cross_ea_, None, out_nodes=rec_node.shape[0],
                                                           edge_weight=lr_ew, edge_vec=lr_vec)
            lig_node = F.pad(lig_node, (0, lig_intra.shape[-1] - lig_node.shape[-1])) + lig_intra + lig_inter
            if l != L - 1:
                rec_node = F.pad(rec_node, (0, rec_intra.shape[-1] - rec_node.shape[-1])) + rec_intra + rec_inter
        return self._confidence(lig_node, lig.batch, B)
