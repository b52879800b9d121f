"""Drop-in for the reference's all-atom score model ``models/aa_model.py:AAModel`` (score mode) - SURVEY.md section 8, row f3.

Same constructor keywords, ``forward(data) -> (tr_pred, rot_pred, tor_pred, None)`` contract, ``state_dict`` keys and side
effects on ``data`` (the cached receptor / atom embeddings of models/aa_model.py:319-333) as the reference class.  It is the
coarse-grained model (diffdock_b200/cg_model.py) with a third node type - receptor atoms - and nine edge groups per
interaction layer instead of four (three in the last layer, models/aa_model.py:401-430); every group runs on the same
sm_100a convolution kernels through ``TensorProductConvLayer.forward_groups`` (fully fused tcgen05 kernel when the shape
allows), neighbour lists come from ddb200_radius_*, spherical harmonics are evaluated in-kernel.

Two reference behaviours are reproduced on purpose: the reversed groups (residue<-ligand, residue<-atom, atom<-ligand) reuse
the FORWARD direction's spherical harmonics (:405-406; the coarse-grained model evaluates Y(-v) instead, cg_model.py:556-557),
and ligand-atom distances go through the ligand distance expansion (:613) into an MLP sized for the cross expansion (:108).

CUDA only, inference only, score mode only.  No CPU fallback.  Like the coarse-grained model the forward has a sync-free
form (``_forward_sync_free``: every per-step neighbour list in a capacity buffer with its live count on the device, the three
reversed groups as permutations of the forward lists, sigma terms of the four static groups added inside the kernel), so the
sampler captures the all-atom step in a CUDA graph too; ``_forward_host_sized`` reads the neighbour-list sizes back and is
used for shapes outside the fused kernel or more than 10000 residues / atoms per complex."""
from __future__ import annotations

import torch
from torch import nn

from . import graphs, ops
from .cg_model import CGModel
from .layers import AtomEncoder, _mlp
from .synthetic import REC_ATOM_FEATURE_DIMS as rec_atom_feature_dims
from .tensor_layers import TensorProductConvLayer, get_irrep_seq


class AAModel(CGModel):
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
                 embed_also_ligand=False, atom_confidence=False, sidechain_pred=False, depthwise_convolution=False,
                 crop_beyond=None):
        if crop_beyond is not None:
            raise NotImplementedError("models/aa_model.py:366-368 raises for crop_beyond too")
        if smooth_edges:
            raise NotImplementedError("the reference AAModel cannot run with smooth_edges (it concatenates the integer "
                                      "atom-residue edge weight with tensors, models/aa_model.py:413-416)")
        super().__init__(t_to_sigma, device, timestep_emb_func, in_lig_edge_features=in_lig_edge_features,
                         sigma_embed_dim=sigma_embed_dim, sh_lmax=sh_lmax, ns=ns, nv=nv, num_conv_layers=num_conv_layers,
                         lig_max_radius=lig_max_radius, rec_max_radius=rec_max_radius,
                         cross_max_distance=cross_max_distance, center_max_distance=center_max_distance,
                         distance_embed_dim=distance_embed_dim, cross_distance_embed_dim=cross_distance_embed_dim,
                         no_torsion=no_torsion, scale_by_sigma=scale_by_sigma, norm_by_sigma=norm_by_sigma,
                         use_second_order_repr=use_second_order_repr, batch_norm=batch_norm,
                         dynamic_max_cross=dynamic_max_cross, dropout=dropout, smooth_edges=False, odd_parity=odd_parity,
                         separate_noise_schedule=separate_noise_schedule, lm_embedding_type=lm_embedding_type,
                         confidence_mode=confidence_mode, asyncronous_noise_schedule=asyncronous_noise_schedule,
                         affinity_prediction=affinity_prediction, parallel=parallel, fixed_center_conv=fixed_center_conv,
                         no_aminoacid_identities=no_aminoacid_identities,
                         include_miscellaneous_atoms=include_miscellaneous_atoms,
                         differentiate_convolutions=differentiate_convolutions, tp_weights_layers=tp_weights_layers,
                         num_prot_emb_layers=num_prot_emb_layers, reduce_pseudoscalars=reduce_pseudoscalars,
                         embed_also_ligand=embed_also_ligand, atom_confidence=atom_confidence, sidechain_pred=sidechain_pred,
                         depthwise_convolution=depthwise_convolution)
        S, D, Dx = sigma_embed_dim, distance_embed_dim, cross_distance_embed_dim
        del self.cross_edge_embedding
        self.atom_node_embedding = AtomEncoder(emb_dim=ns, feature_dims=rec_atom_feature_dims, sigma_embed_dim=0)
        self.atom_edge_embedding = _mlp(D, ns, ns, dropout)
        self.lr_edge_embedding = _mlp(S + Dx, ns, ns, dropout)
        self.ar_edge_embedding = _mlp(D, ns, ns, dropout)
        self.la_edge_embedding = _mlp(S + Dx, ns, ns, dropout)
        seq = get_irrep_seq(ns, nv, use_second_order_repr, reduce_pseudoscalars)
        faster = sh_lmax == 1 and not use_second_order_repr

        def conv(i, groups):
            return TensorProductConvLayer(in_irreps=seq[min(i, len(seq) - 1)], sh_irreps=self.sh_irreps,
                                          out_irreps=seq[min(i + 1, len(seq) - 1)], n_edge_features=3 * ns,
                                          hidden_features=3 * ns, residual=True, batch_norm=batch_norm, dropout=dropout,
                                          faster=faster, tp_weights_layers=tp_weights_layers, edge_groups=groups)

        d = differentiate_convolutions
        self.rec_emb_layers = nn.ModuleList([conv(i, 4 if d else 1) for i in range(num_prot_emb_layers)])
        last = num_prot_emb_layers + num_conv_layers - 1
        self.conv_layers = nn.ModuleList([conv(i, 1 if not d else (3 if i == last else 9))
                                          for i in range(num_prot_emb_layers, num_prot_emb_layers + num_conv_layers)])

    def sync_free_capable(self):
        """As CGModel.sync_free_capable; additionally every edge type must have its own radial MLP (the merged single-group
        form concatenates edge lists, which needs their sizes on the host)."""
        return self.differentiate_convolutions and super().sync_free_capable()

    def _capacities_fit(self, c):
        return super()._capacities_fit(c) and c['atom_max'] <= 10000         # the 10000 caps (:595,:610) not binding

    # ---------------------------------------------------------------------------------------------------------
    @staticmethod
    def _csr(tgt, src, n_rows, *payload):
        """(tgt32, src32, payload...) sorted stably by target."""
        t32, order, _ = ops.csr_sort_by_target(tgt.to(torch.int32).contiguous(), n_rows)
        return (t32, src[order].to(torch.int32).contiguous()) + tuple(p[order].contiguous() for p in payload)

    def _static(self, data):
        """Pose-independent part, cached on ``data`` like models/aa_model.py:276-333: residue / atom node embeddings, the
        edge embeddings of the three static graphs (residue-residue, atom-atom, atom-residue), the optional protein
        embedding layers over their four groups, and the CSR-sorted static edge groups of the joint graph."""
        rec, atom, lig = data['receptor'], data['atom'], data['ligand']
        rr, aa, ar, ll = data['receptor', 'receptor'], data['atom', 'atom'], data['atom', 'receptor'], data['ligand', 'ligand']
        if hasattr(rec, 'rec_node_attr') and hasattr(rr, '_b200aa'):
            return rr._b200aa
        ns, B = self.ns, data.num_graphs
        rp, ap = rec.pos.float(), atom.pos.float()
        n_rec, n_atom, n_lig = rp.shape[0], ap.shape[0], lig.pos.shape[0]
        rr_ei, aa_ei, ar_ei = rr.edge_index.long(), aa.edge_index.long(), ar.edge_index.long()
        rr_vec, aa_vec = rp[rr_ei[1]] - rp[rr_ei[0]], ap[aa_ei[1]] - ap[aa_ei[0]]
        ar_vec = rp[ar_ei[1]] - ap[ar_ei[0]]
        rr_ea = self.rec_edge_embedding(self.rec_distance_expansion(rr_vec.norm(dim=-1)))
        aa_ea = self.atom_edge_embedding(self.lig_distance_expansion(aa_vec.norm(dim=-1)))
        ar_ea = self.ar_edge_embedding(self.rec_distance_expansion(ar_vec.norm(dim=-1)))
        r_node, a_node = self.rec_node_embedding(rec.x), self.atom_node_embedding(atom.x)
        if len(self.rec_emb_layers):
            # joint numbering [residues | atoms] (:301-311): residue<-residue, atom<-residue, atom<-atom, residue<-atom
            node = torch.cat([r_node, a_node], 0)
            n = n_rec + n_atom
            groups = [self._csr(rr_ei[0], rr_ei[1], n, rr_ea, rr_vec) + (None,),
                      self._csr(ar_ei[0] + n_rec, ar_ei[1], n, ar_ea, ar_vec) + (None,),
                      self._csr(aa_ei[0] + n_rec, aa_ei[1] + n_rec, n, aa_ea, aa_vec) + (None,),
                      self._csr(ar_ei[1], ar_ei[0] + n_rec, n, ar_ea, ar_vec) + (None,)]      # reversed: forward harmonics
            for layer in self.rec_emb_layers:
                node = layer.forward_groups(node, groups, gather_scalars=ns)
            r_node, a_node = node[:n_rec], node[n_rec:]
        rec.rec_node_attr, rr.rec_edge_attr, rr.edge_sh, rr.edge_weight = r_node, rr_ea, None, 1.0
        atom.atom_node_attr, aa.atom_edge_attr, aa.edge_sh, aa.edge_weight = a_node, aa_ea, None, 1.0
        ar.edge_attr, ar.edge_sh, ar.edge_weight = ar_ea, None, 1
        c = {}
        N = n_lig + n_rec + n_atom
        o_r, o_a = n_lig, n_lig + n_rec
        # static groups of the joint graph [ligand | residues | atoms], CSR by target, with the graph id of the sigma term
        gid = lambda b: b.to(torch.int64)
        c['rr'] = self._csr(rr_ei[0] + o_r, rr_ei[1] + o_r, N, rr_ea, rr_vec, gid(rec.batch[rr_ei[0]]))
        c['ra'] = self._csr(ar_ei[1] + o_r, ar_ei[0] + o_a, N, ar_ea, ar_vec, gid(atom.batch[ar_ei[0]]))    # residue <- atom
        c['aa'] = self._csr(aa_ei[0] + o_a, aa_ei[1] + o_a, N, aa_ea, aa_vec, gid(atom.batch[aa_ei[0]]))
        c['ar'] = self._csr(ar_ei[0] + o_a, ar_ei[1] + o_r, N, ar_ea, ar_vec, gid(atom.batch[ar_ei[0]]))    # atom <- residue
        c['rec_ptr'], c['atom_ptr'] = ops.segment_ptr(rec.batch, B), ops.segment_ptr(atom.batch, B)
        c['lig_ptr'] = ops.segment_ptr(lig.batch, B)
        c['lig_cnt_f'] = (c['lig_ptr'][1:] - c['lig_ptr'][:-1]).float().unsqueeze(1)
        bonds = ll.edge_index[:, lig.edge_mask].long()
        c['bonds'], c['n_bonds'] = bonds, int(bonds.shape[1])
        c['bond_batch'] = lig.batch[bonds[0]] if bonds.shape[1] else None
        c['bond_lig_batch'] = c['bond_batch']
        # constants of the sync-free forward: CGModel's (ligand / residue counts, bond CSR, capacities) + the atom side
        c['rr_tgt_batch'] = rec.batch[rr_ei[0]]
        self._static_sync_free(data, c)
        i32 = lambda t: t.to(torch.int32).contiguous()
        atom_cnt = c['atom_ptr'][1:] - c['atom_ptr'][:-1]
        lig_cnt = c['lig_ptr'][1:] - c['lig_ptr'][:-1]
        c['atom_max'] = int(atom_cnt.max()) if B else 0
        c['cap_la'] = int((lig_cnt.long() * atom_cnt.long()).sum())      # every ligand atom x every atom of its complex
        c['atom_batch32'] = i32(atom.batch)
        c['gid32'] = {k: i32(c[k][4]) for k in ('rr', 'ra', 'aa', 'ar')}
        rr._b200aa = c
        return c

    def _forward_sync_free(self, data, c):
        """The forward without a device->host read (see CGModel._forward_sync_free): ligand graph, ligand-residue and
        ligand-atom graphs written into upper-bound buffers with device-side counts; the reversed groups (residue<-ligand,
        atom<-ligand) are permutations of the forward lists and - as in the reference, models/aa_model.py:405-406 - keep the
        FORWARD direction's edge vector (vec_sign = +1); the four static groups get their sigma term inside the kernel."""
        lig, rec, atom = data['ligand'], data['receptor'], data['atom']
        ns = self.ns
        tr_sigma, rot_sigma, tor_sigma = self.t_to_sigma(*[data.complex_t[k] for k in ('tr', 'rot', 'tor')])
        n_lig, n_rec = lig.batch.shape[0], rec.batch.shape[0]
        o_r, o_a = n_lig, n_lig + n_rec
        pos, rpos, apos = lig.pos.float().contiguous(), rec.pos.float().contiguous(), atom.pos.float().contiguous()

        sig = self.rec_sigma_embedding(self.timestep_emb_func(data.complex_t['tr'])).contiguous()
        rec_node, atom_node = rec.rec_node_attr.clone(), atom.atom_node_attr.clone()
        rec_node[:, :ns] += sig[rec.batch]
        atom_node[:, :ns] += sig[atom.batch]
        lig.node_sigma_emb = self.timestep_emb_func(lig.node_t['tr'])

        # -- ligand graph: bonds + radius graph (models/aa_model.py:538-568 = cg_model.py:467-497) ---------------------------
        g_ll = graphs.ligand_graph(pos, c, self.lig_max_radius, lig.node_sigma_emb, self.lig_distance_expansion,
                                   self.lig_edge_embedding, self.smooth_edges)
        lig_node = self.lig_node_embedding(torch.cat([lig.x.float(), lig.node_sigma_emb], 1))
        for layer in self.lig_emb_layers:
            lig_node = layer.forward_groups(lig_node, [g_ll], gather_scalars=ns)

        # -- ligand cross graphs (:588-623): residues within the (per-complex) cut-off, atoms within lig_max_radius ---------
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        lr, la = (self.lr_edge_embedding, self.cross_distance_expansion), (self.la_edge_embedding, self.lig_distance_expansion)
        g_lr, g_rl = graphs.cross_graph(pos, c['lig_ptr'], c['lig_batch32'], rpos, c['rec_ptr'], c['rec_batch32'], c['rec_max'],
                                        c['cap_cross'], o_r, r, rpg, self._cross_embedder(lig, *lr), vec_sign=1.0,
                                        fill_row=self._cross_fill_row(*lr))
        g_la, g_al = graphs.cross_graph(pos, c['lig_ptr'], c['lig_batch32'], apos, c['atom_ptr'], c['atom_batch32'], c['atom_max'],
                                        c['cap_la'], o_a, float(self.lig_max_radius), None, self._cross_embedder(lig, *la),
                                        vec_sign=1.0, fill_row=self._cross_fill_row(*la))

        # -- joint graph [ligand | residues | atoms]: nine groups in the reference's order (:401-417) --------------------
        node = torch.cat([lig_node, rec_node, atom_node], 0)
        stat = lambda k: (c[k][0], c[k][1], c[k][2], c[k][3], None, dict(ea_add=sig, ea_add_idx=c['gid32'][k]))
        groups = [g_ll, g_lr, g_la, stat('rr'), g_rl, stat('ra'), stat('aa'), g_al, stat('ar')]
        L = len(self.conv_layers)
        for l, layer in enumerate(self.conv_layers):
            node = layer.forward_groups(node, groups if l < L - 1 else groups[:3], gather_scalars=ns)
        return self._heads(data, c, node[:n_lig], tr_sigma, rot_sigma, tor_sigma, sync_free=True)

    def _forward_host_sized(self, data, c):
        """Forward with exactly-sized neighbour lists (the sizes are read back to the host)."""
        lig, rec, atom = data['ligand'], data['receptor'], data['atom']
        ns = self.ns
        tr_sigma, rot_sigma, tor_sigma = self.t_to_sigma(*[data.complex_t[k] for k in ('tr', 'rot', 'tor')])
        n_lig, n_rec = lig.pos.shape[0], rec.pos.shape[0]
        o_r, o_a = n_lig, n_lig + n_rec

        # -- embeddings (:335-362): sigma term on residue / atom scalars and on the three static edge-attribute sets ----
        sig = self.rec_sigma_embedding(self.timestep_emb_func(data.complex_t['tr']))
        rec_node, atom_node = rec.rec_node_attr.clone(), atom.atom_node_attr.clone()
        rec_node[:, :ns] += sig[rec.batch]
        atom_node[:, :ns] += sig[atom.batch]
        lig_x, ll_tgt, ll_src, ll_ea, ll_vec, _ = self._ligand_graph(data, c)
        lig_node = self.lig_node_embedding(lig_x)
        ll_ea = self.lig_edge_embedding(ll_ea)
        assert self.embed_also_ligand, "otherwise reimplement padding"
        i32 = lambda t: t.to(torch.int32).contiguous()
        g_ll = (i32(ll_tgt), i32(ll_src), ll_ea, ll_vec.contiguous(), None)
        for layer in self.lig_emb_layers:
            lig_node = layer.forward_groups(lig_node, [g_ll], gather_scalars=ns)

        # -- ligand cross graphs (:588-623): residues within the (per-complex) cut-off, atoms within lig_max_radius ---------
        lp = lig.pos.float()
        r, rpg = graphs.cross_cutoff(tr_sigma, self.dynamic_max_cross, self.cross_max_distance)
        li, ri, lr_vec = graphs.cross_graph_host(lp, rec.pos.float(), c['rec_ptr'], lig.batch, r, rpg)
        lr_ea = self.lr_edge_embedding(torch.cat([lig.node_sigma_emb[li], self.cross_distance_expansion(lr_vec.norm(dim=-1))], 1))
        la_l, la_a, la_vec = graphs.cross_graph_host(lp, atom.pos.float(), c['atom_ptr'], lig.batch, float(self.lig_max_radius))
        la_ea = self.la_edge_embedding(torch.cat([lig.node_sigma_emb[la_l], self.lig_distance_expansion(la_vec.norm(dim=-1))], 1))

        # -- joint graph [ligand | residues | atoms]: nine groups in the reference's order (:401-417) --------------------
        node = torch.cat([lig_node, rec_node, atom_node], 0)
        g_lr, g_rl = graphs.cross_groups_host(li, ri, o_r, lr_ea, lr_vec, None, vec_sign=1.0)
        g_la, g_al = graphs.cross_groups_host(la_l, la_a, o_a, la_ea, la_vec, None, vec_sign=1.0)
        stat = lambda k: (c[k][0], c[k][1], c[k][2] + sig[c[k][4]], c[k][3], None)
        # reversed groups (residue <- ligand, residue <- atom, atom <- ligand) with the forward harmonics
        groups = [g_ll, g_lr, g_la, stat('rr'), g_rl, stat('ra'), stat('aa'), g_al, stat('ar')]
        L = len(self.conv_layers)
        for l, layer in enumerate(self.conv_layers):
            use = groups if l < L - 1 else groups[:3]           # last layer: only the groups that end on ligand atoms (:429-430)
            if not self.differentiate_convolutions:             # one radial MLP for all edge types: a single merged group
                use = graphs.merge_groups(use)
            node = layer.forward_groups(node, use, gather_scalars=ns)
        return self._heads(data, c, node[:n_lig], tr_sigma, rot_sigma, tor_sigma, sync_free=False)
