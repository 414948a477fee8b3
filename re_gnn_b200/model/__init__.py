"""The callers of the hot path, mirrored so that epoch time can be measured (and golden
parity checked) where the reference checkout is absent.  Same constructor arguments, sub-module /
parameter names and forward conventions as model/REGCN.py:6-46, model/REGAT.py:6-66,
model/REMixHop.py:19-101 and model/REGIN.py:35-84; the reference's own files also run unmodified on
``re_gnn_b200.layer`` (tests/test_layers_host.py, run with REGNN_REFERENCE set to a reference checkout)."""
import torch
from torch import nn

from ..layer import REGraphConv, RESAGEConv, REGATConv, REGATv2Conv, REMixHopConv, REGINConv


class _TypedInput(nn.Module):
    """Per-node-type input projection ``fc_list`` followed by concatenation in type order
    (model/REGCN.py:22-24,36-39; identical in the other two models)."""

    def _make_fc_list(self, feats_dim_list, width):
        self.fc_list = nn.ModuleList([nn.Linear(d, width, bias=True) for d in feats_dim_list])
        for fc in self.fc_list:
            nn.init.xavier_normal_(fc.weight, gain=1.414)

    def _project(self, features_list):
        # Type-contiguous rows and input widths up to 4231 (DBLP papers): one library GEMM per type is the right tool here
        # (measured: the grouped launch of functional.grouped_linear is slower on these shapes); the grouped kernel pays
        # off where rows of all types are interleaved and gathered, mag.REGNN.group_input.
        return torch.cat([fc(x) for fc, x in zip(self.fc_list, features_list)], 0)


class REGCN(_TypedInput):
    def __init__(self, g, num_etypes, R, in_feats, n_hidden, n_classes, n_layers, activation, dropout,
                 feats_dim_list, use_sage=False):
        super().__init__()
        self.g, self.num_layers = g, n_layers
        self._make_fc_list(feats_dim_list, in_feats)
        conv = RESAGEConv if use_sage else REGraphConv
        self.layers = nn.ModuleList()
        self.layers.append(conv(num_etypes, R, in_feats, n_hidden, bias=False, activation=None, dropout=dropout,
                                weight=False))
        for _ in range(1, n_layers - 1):
            self.layers.append(conv(num_etypes, R, n_hidden, n_hidden, activation=activation, dropout=dropout))
        self.layers.append(conv(num_etypes, R, n_hidden, n_classes, bias=False, dropout=dropout, weight=False))
        self.out_lin = nn.Linear(n_hidden, n_classes, bias=True)
        self.dropout = nn.Dropout(p=dropout)

    def forward(self, features_list, e_feat):
        h = self.layers[0](self.g, self._project(features_list), e_feat)
        for l in range(1, self.num_layers):
            h = self.layers[l](self.g, self.dropout(h), e_feat)
        return self.out_lin(h), h


class REGAT(_TypedInput):
    def __init__(self, g, num_etypes, R, num_layers, in_dim, num_hidden, num_classes, heads, activation,
                 feat_drop, attn_drop, negative_slope, residual, feats_dim_list, use_gatv2=False):
        super().__init__()
        self.g, self.num_etypes, self.num_layers = g, num_etypes, num_layers
        self.gat_layers, self.bns = nn.ModuleList(), nn.ModuleList()
        self.feats_dim_list, self.activation = feats_dim_list, activation
        self._make_fc_list(feats_dim_list, num_hidden)
        conv = REGATv2Conv if use_gatv2 else REGATConv
        self.gat_layers.append(conv(num_etypes, R, in_dim, num_hidden, heads[0], feat_drop, attn_drop,
                                    negative_slope, False, activation))
        for l in range(1, num_layers - 1):
            self.gat_layers.append(conv(num_etypes, R, num_hidden * heads[l - 1], num_hidden, heads[l], feat_drop,
                                        attn_drop, negative_slope, residual, activation))
        self.gat_layers.append(conv(num_etypes, R, num_hidden * heads[-2], num_hidden, heads[-2], feat_drop,
                                    attn_drop, negative_slope, residual, None, use_weight=False))
        self.out_lin = nn.Linear(num_hidden * heads[-2], num_classes)

    def forward(self, features_list, e_feat):
        h = self._project(features_list)
        for l in range(self.num_layers):          # includes the weight-less last layer ...
            h = self.gat_layers[l](self.g, h, e_feat).flatten(1)
        emb = self.gat_layers[-1](self.g, h, e_feat)   # ... which the reference applies a second time (Q3)
        return self.out_lin(emb.flatten(1)), emb.mean(1)


class REMixHop(_TypedInput):
    def __init__(self, g, num_etypes, R, in_dim, hid_dim, out_dim, num_layers, feats_dim_list, p=[0, 1, 2],
                 input_dropout=0.0, layer_dropout=0.0, activation=None, batchnorm=False):
        super().__init__()
        self.g, self.in_dim, self.hid_dim, self.out_dim = g, in_dim, hid_dim, out_dim
        self.num_layers, self.p = num_layers, p
        self.input_dropout, self.layer_dropout = input_dropout, layer_dropout
        self.activation, self.batchnorm = activation, batchnorm
        self.layers = nn.ModuleList()
        self.dropout = nn.Dropout(input_dropout)
        self._make_fc_list(feats_dim_list, in_dim)
        self.layers.append(REMixHopConv(num_etypes, R, in_dim, hid_dim, p=p, dropout=input_dropout,
                                        activation=activation, batchnorm=batchnorm))
        for _ in range(num_layers - 1):
            self.layers.append(REMixHopConv(num_etypes, R, hid_dim * len(p), hid_dim, p=p, dropout=layer_dropout,
                                            activation=activation, batchnorm=batchnorm))
        self.fc_layers = nn.Linear(hid_dim * len(p), out_dim, bias=False)

    def forward(self, features_list, e_feat):
        h = self.layers[0](self.g, self._project(features_list), e_feat)
        for l in range(1, self.num_layers):
            h = self.layers[l](self.g, self.dropout(h), e_feat)
        return self.fc_layers(h), h


class _GinMLP(nn.Module):
    """model/REGIN.py:9-32: declared as a two-layer MLP, but only dropout + ``linears[1]`` (input_dim -> output_dim) run;
    ``linears[0]`` exists for state_dict compatibility."""

    def __init__(self, input_dim, hidden_dim, output_dim, activation, dropout=0.):
        super().__init__()
        self.linears = nn.ModuleList([nn.Linear(input_dim, hidden_dim, bias=False),
                                      nn.Linear(input_dim, output_dim, bias=False)])
        self.dropout = nn.Dropout(dropout)
        self.activation = activation

    def reset_parameters(self):
        for lin in self.linears:
            lin.reset_parameters()

    def forward(self, x):
        return self.linears[1](self.dropout(x))


class REGIN(_TypedInput):
    def __init__(self, g, num_etypes, R, input_dim, hidden_dim, output_dim, n_layers, activation, dropout,
                 feats_dim_list):
        super().__init__()
        self.g, self.num_layers = g, n_layers
        self._make_fc_list(feats_dim_list, input_dim)
        self.layers = nn.ModuleList()
        for layer in range(n_layers):
            in_c = input_dim if layer == 0 else hidden_dim
            out_c = output_dim if layer == n_layers - 1 else hidden_dim
            if layer != n_layers - 1:
                self.layers.append(REGINConv(num_etypes, R, _GinMLP(in_c, hidden_dim, out_c, activation, dropout),
                                             activation=activation))
            else:   # the last layer aggregates only; the classifier is out_mlp
                self.layers.append(REGINConv(num_etypes, R, None, activation=None))
        self.out_mlp = _GinMLP(hidden_dim, hidden_dim, output_dim, activation, dropout)

    def forward(self, features_list, e_feat):
        h = self.layers[0](self.g, self._project(features_list), e_feat)
        for l in range(1, self.num_layers):
            h = self.layers[l](self.g, h, e_feat)
        return self.out_mlp(h), h
