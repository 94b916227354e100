"""GIN graph classifier on the B200 aggregation kernels.

Drop-in for ``graph_classification/graph_neural_networks/models/gconv.py::GIN`` (:154-215) and for the PyG
2.0.2 pieces it calls (``GINConv``, ``global_add_pool``, ``global_mean_pool`` -- gconv.py:161,197,210-213):
same ``args`` fields, same sub-module names (``first_h, nns, convs[i].nn`` aliasing ``nns[i]``, ``convs[i].eps``,
``linears``), same quirks (layer-0 dropout is applied without ``training=`` :210; ``train_eps`` defaults to
``args.epochs`` :179; pooling includes the dummy node).

Hot ops: ``GINConv`` = one K1 launch with the ``(1 + eps) * x`` self term fused (torch_scatter's
index_select + atomic scatter_add in the reference), pooling = K3 segment readout.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import ops
from ..data import structure_of


class GINConv(nn.Module):
    """``out = nn((1 + eps) * x + sum_{j -> i} x_j)``.  ``forward`` takes the reference's ``(x, edge_index)``;
    pass ``structure=`` to reuse a compiled CSR (otherwise it is compiled per distinct edge_index and cached)."""

    def __init__(self, nn, eps=0.0, train_eps=False, **kw):
        super().__init__()
        self.nn = nn
        self.initial_eps = eps
        if train_eps:
            self.eps = torch.nn.Parameter(torch.Tensor([eps]))
        else:
            self.register_buffer("eps", torch.Tensor([eps]))
        self._cache = {}

    def _structure(self, x, edge_index):
        from ...graph import cached_for_tensor
        from ..data import GraphStructure
        return cached_for_tensor(self._cache, "structure", edge_index, x.size(0), lambda: GraphStructure(edge_index, x.size(0)))

    def forward(self, x, edge_index, structure=None):
        s = structure if structure is not None else self._structure(x, edge_index)
        if x.is_cuda and ops.gin_mlp_fusable(self.nn):
            # aggregation + Linear/BN/ReLU stages as one autograd node (tensor-core stages, eps read on the device)
            return ops.gin_conv(self.nn, x, self.eps, s.csr_in, s.csr_out)
        if isinstance(self.eps, nn.Parameter) and self.eps.requires_grad:
            # trainable eps: keep d/d eps on the autograd tape (agg + (1 + eps) * x); the self term is one
            # elementwise op instead of being fused, the gather-sum is still K1.
            out = ops.spmm_sum(x, s.csr_in, s.csr_out, 0.0) + (1 + self.eps) * x
        else:
            out = ops.spmm_sum(x, s.csr_in, s.csr_out, 1.0 + float(self.eps))
        return ops.apply_gin_mlp(self.nn, out)


def _ptr_of(batch, size=None):
    nb = (int(batch[-1].item()) + 1 if batch.numel() else 0) if size is None else size
    ptr = torch.zeros(nb + 1, dtype=torch.int32, device=batch.device)
    ptr[1:] = torch.cumsum(torch.bincount(batch, minlength=nb), 0).to(torch.int32)
    return ptr


def global_add_pool(x, batch, size=None, node_ptr=None):
    return ops.segment_sum(x, node_ptr if node_ptr is not None else _ptr_of(batch, size), None, mean=False)


def global_mean_pool(x, batch, size=None, node_ptr=None):
    return ops.segment_sum(x, node_ptr if node_ptr is not None else _ptr_of(batch, size), None, mean=True)


def _gin_mlp(din, dout):
    return nn.Sequential(ops.Linear(din, dout), nn.BatchNorm1d(dout), nn.ReLU(),
                         ops.Linear(dout, dout), nn.BatchNorm1d(dout), nn.ReLU())


class GIN(torch.nn.Module):
    def __init__(self, args):
        super().__init__()
        self.args = args
        self.num_features, self.hidden_dim, self.num_classes = args.num_features, args.hidden_dim, args.num_classes
        self.dropout = args.dropout_ratio
        config = args.additional if args.additional else {"train_eps": False, "num_layers": 2, "aggregation": "sum"}
        agg = config.get("aggregation", "sum")
        if agg == "sum":
            self.pooling = global_add_pool
        elif agg == "mean":
            self.pooling = global_mean_pool
        train_eps = config.get("train_eps", args.epochs)   # gconv.py:179
        self.embeddings_dim = [self.hidden_dim for _ in range(config.get("num_layers", 2))]
        self.no_layers = len(self.embeddings_dim)
        nns, convs, linears = [], [], []
        for layer, out_dim in enumerate(self.embeddings_dim):
            if layer == 0:
                self.first_h = _gin_mlp(self.num_features, out_dim)
            else:
                nns.append(_gin_mlp(self.embeddings_dim[layer - 1], out_dim))
                convs.append(GINConv(nns[-1], train_eps=train_eps))
            linears.append(ops.Linear(out_dim, self.num_classes))
        self.nns = nn.ModuleList(nns)
        self.convs = nn.ModuleList(convs)
        self.linears = nn.ModuleList(linears)

    def _fused(self):
        """the tensor-core GIN layers apply when every MLP is the reference's Linear/BN/ReLU stack in training mode."""
        return ops.gin_mlp_fusable(self.first_h) and all(ops.gin_mlp_fusable(m) for m in self.nns)

    def _forward_fused(self, data, s):
        """each layer is one autograd node producing (h, pooled h); the class scores are Linear(pooled) -- for layer 0
        pool(Linear(h)) = Linear(pool(h)) with the bias counted once per pooled row (gconv.py:210), so that GEMM runs on
        B rows instead of N."""
        mean = self.pooling is global_mean_pool
        x, out = data.x, 0
        if self.dropout == 0:
            # jumping-knowledge head as ONE GEMM: sum_l Linear_l(pooled_l) = [pooled_0 | ... | pooled_L] @ [W_0 | ... | W_L]^T
            # + biases (dropout with p = 0 is the identity).  Five (B x D) @ (D x C) GEMMs with their bias / dropout / add
            # kernels and their backward were ~40 launches of 2-3 us in a train step that is bound by launch count.
            pooled_all = []
            for layer in range(self.no_layers):
                if layer == 0:
                    x, pooled = ops.gin_layer(self.first_h, x, seg_ptr=s.node_ptr, row2seg=s.row2seg, mean=mean)
                else:
                    conv = self.convs[layer - 1]
                    x, pooled = ops.gin_layer(conv.nn, x, conv.eps, s.csr_in, s.csr_out, s.node_ptr, s.row2seg, mean)
                pooled_all.append(pooled)
            if ops.jk_head_supported(self.no_layers, self.hidden_dim, self.num_classes):
                # ... and with its log_softmax as one kernel each way (csrc/agg.cu jk_head_*): the concatenations, the GEMM,
                # the bias arithmetic and -- backward -- the slice copies of the concatenation gradient were ~25 launches
                return ops.jk_head(pooled_all, [lin.weight for lin in self.linears], [lin.bias for lin in self.linears],
                                   None if mean else s.node_ptr)
            w_all = torch.cat([lin.weight for lin in self.linears], dim=1)
            score = ops.linear(torch.cat(pooled_all, dim=1), w_all, None)
            bias_rest = torch.stack([lin.bias for lin in self.linears[1:]]).sum(0) if self.no_layers > 1 else 0
            if mean:
                score = score + (self.linears[0].bias + bias_rest)
            else:   # layer 0 pools Linear(h): its bias is counted once per pooled row (gconv.py:210)
                cnt = (s.node_ptr[1:] - s.node_ptr[:-1]).to(score.dtype).unsqueeze(1)
                score = score + (cnt * self.linears[0].bias + bias_rest)
            return F.log_softmax(score, dim=-1)
        for layer in range(self.no_layers):
            if layer == 0:
                x, pooled = ops.gin_layer(self.first_h, x, seg_ptr=s.node_ptr, row2seg=s.row2seg, mean=mean)
                lin = self.linears[0]
                if mean:
                    score = lin(pooled)
                else:
                    cnt = (s.node_ptr[1:] - s.node_ptr[:-1]).to(pooled.dtype).unsqueeze(1)
                    score = ops.linear(pooled, lin.weight, None) + cnt * lin.bias
                out = out + F.dropout(score, p=self.dropout)                                   # gconv.py:210 (no training=)
            else:
                conv = self.convs[layer - 1]
                x, pooled = ops.gin_layer(conv.nn, x, conv.eps, s.csr_in, s.csr_out, s.node_ptr, s.row2seg, mean)
                out = out + F.dropout(self.linears[layer](pooled), p=self.dropout, training=self.training)
        return F.log_softmax(out, dim=-1)

    def forward(self, data):
        x = data.x
        s = structure_of(data)
        if x.is_cuda and s.node_ptr is not None and self._fused():
            return self._forward_fused(data, s)
        out = 0
        for layer in range(self.no_layers):
            if layer == 0:
                x = ops.apply_gin_mlp(self.first_h, x)
                out += F.dropout(self.pooling(self.linears[layer](x), data.batch, node_ptr=s.node_ptr), p=self.dropout)
            else:
                # GINConv reads edge_index only without a compiled structure; a batch from the closed-form CONJ_ builder
                # would materialise it with a device->host read of the edge count
                x = self.convs[layer - 1](x, None, structure=s)
                out += F.dropout(self.linears[layer](self.pooling(x, data.batch, node_ptr=s.node_ptr)),
                                 p=self.dropout, training=self.training)
        return F.log_softmax(out, dim=-1)
