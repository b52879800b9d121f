"""Embedding layers with the reference's parameter names (models/layers.py) - plain PyTorch modules on the device
(small dense ops; the hot convolution lives in csrc/)."""
import numpy as np
import torch
from torch import nn

from .tensor_layers import FCBlock  # noqa: F401  (re-export: the reference keeps FCBlock in models/layers.py)


def _mlp(n_in, n_hidden, n_out, dropout):
    """Linear - ReLU - Dropout - Linear: the edge / sigma embeddings of the models."""
    return nn.Sequential(nn.Linear(n_in, n_hidden), nn.ReLU(), nn.Dropout(dropout), nn.Linear(n_hidden, n_out))


def edge_weight(edge_vec, max_norm, smooth):
    """Edge weight of smooth_edges, 0.5 (cos(pi |v| / max_norm) + 1) clipped at |v| = max_norm, else the constant 1
    (models/cg_model.py:459-465).  ``max_norm`` is a number or a per-edge tensor."""
    if smooth:
        nrm = torch.clip(edge_vec.norm(dim=-1) * np.pi / max_norm, max=np.pi)
        return 0.5 * (torch.cos(nrm) + 1.0).unsqueeze(-1)
    return 1.0


class GaussianSmearing(nn.Module):
    """Radial basis expansion exp(coeff * (d - mu_k)^2), mu = linspace(start, stop, K)  (models/layers.py:20-30)."""

    def __init__(self, start=0.0, stop=5.0, num_gaussians=50):
        super().__init__()
        mu = torch.linspace(start, stop, num_gaussians)
        self.coeff = -0.5 / (mu[1] - mu[0]).item() ** 2
        self.register_buffer('offset', mu)

    def forward(self, dist):
        diff = dist.reshape(-1, 1) - self.offset.reshape(1, -1)
        return torch.exp(self.coeff * diff * diff)


class AtomEncoder(nn.Module):
    """Sum of one embedding table per categorical column, then a Linear over [embedding | remaining float columns]
    (models/layers.py:33-67)."""

    def __init__(self, emb_dim, feature_dims, sigma_embed_dim, lm_embedding_dim=0):
        super().__init__()
        cat_dims, n_scalar = feature_dims
        self.num_categorical_features = len(cat_dims)
        self.additional_features_dim = n_scalar + sigma_embed_dim + lm_embedding_dim
        self.atom_embedding_list = nn.ModuleList()
        for d in cat_dims:
            table = nn.Embedding(d, emb_dim)
            nn.init.xavier_uniform_(table.weight.data)
            self.atom_embedding_list.append(table)
        if self.additional_features_dim > 0:
            self.additional_features_embedder = nn.Linear(self.additional_features_dim + emb_dim, emb_dim)

    def forward(self, x):
        nc = self.num_categorical_features
        assert x.shape[1] == nc + self.additional_features_dim
        idx = x[:, :nc].long()
        h = self.atom_embedding_list[0](idx[:, 0])
        for i in range(1, nc):
            h = h + self.atom_embedding_list[i](idx[:, i])
        if self.additional_features_dim > 0:
            h = self.additional_features_embedder(torch.cat([h, x[:, nc:].to(h.dtype)], dim=1))
        return h


class OldAtomEncoder(nn.Module):
    """models/layers.py:70-117: categorical embeddings + Linear(scalar features incl. sigma embedding), then an optional
    Linear([emb | LM columns]) - the encoder of the confidence model.  ``lm_embedding_dim`` (1280 in the reference,
    hard-wired for 'esm') is a keyword here so that small fixtures can be loaded."""

    def __init__(self, emb_dim, feature_dims, sigma_embed_dim, lm_embedding_type=None, lm_embedding_dim=1280):
        super().__init__()
        self.atom_embedding_list = nn.ModuleList()
        self.num_categorical_features = len(feature_dims[0])
        self.num_scalar_features = feature_dims[1] + sigma_embed_dim
        self.lm_embedding_type = lm_embedding_type
        for dim in feature_dims[0]:
            emb = nn.Embedding(dim, emb_dim)
            nn.init.xavier_uniform_(emb.weight.data)
            self.atom_embedding_list.append(emb)
        if self.num_scalar_features > 0:
            self.linear = nn.Linear(self.num_scalar_features, emb_dim)
        if lm_embedding_type is not None:
            if lm_embedding_type != 'esm':
                raise ValueError('LM Embedding type was not correctly determined. LM embedding type: ', lm_embedding_type)
            self.lm_embedding_dim = lm_embedding_dim
            self.lm_embedding_layer = nn.Linear(self.lm_embedding_dim + emb_dim, emb_dim)

    def forward(self, x):
        nc, nsf = self.num_categorical_features, self.num_scalar_features
        assert x.shape[1] == nc + nsf + (self.lm_embedding_dim if self.lm_embedding_type is not None else 0)
        out = 0
        for i in range(nc):
            out = out + self.atom_embedding_list[i](x[:, i].long())
        if nsf > 0:
            out = out + self.linear(x[:, nc:nc + nsf].float())
        if self.lm_embedding_type is not None:
            out = self.lm_embedding_layer(torch.cat([out, x[:, -self.lm_embedding_dim:].float()], 1))
        return out
