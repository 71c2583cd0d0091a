"""Decoders of the hot path on B200 kernels.

NeRFDecoder             <- reference src/decoders.py:29-87
InstantNeRFDecoder      <- reference src/decoders.py:90-162   (tinycudann FullyFusedMLP x2 replaced)
DeformationNetwork      <- reference src/decoders.py:165-195
HashDeformationDecoder  <- reference src/decoders.py:264-318  (tinycudann FullyFusedMLP replaced)
TimeModulationNetwork   <- reference src/decoders.py:321-371

Parameter names/shapes equal the reference's state_dict (nn.Linear weight/bias; flat
``params`` for the fused MLPs) so checkpoints and run.py's optimizer groups keep working.
StandardMLP (Part 1 image fitting) and the dead DirectTimeDecoder are outside the
ray-marching hot path and are not provided.
"""
import math

import torch
from torch import nn

import b2n
from .abstract import BaseDecoder


def _pad16(n):
    return (n + 15) // 16 * 16


class _Dense(nn.Linear):
    """nn.Linear parameters (same init, same state_dict keys) evaluated by b2n_linear_*."""

    def forward(self, x, act="none"):
        return b2n.linear(x, self.weight, self.bias, act)


class FusedMLP(nn.Module):
    """Stand-in for ``tcnn.Network(..., {"otype": "FullyFusedMLP"})``: bias-free ReLU MLP whose
    matrices live in one flat ``params`` vector; in/out widths padded to multiples of 16
    (padding inputs are zeros, padded outputs are dropped -- SURVEY.md 8a/A4)."""

    def __init__(self, n_input_dims, n_output_dims, network_config, seed=1337):
        super().__init__()
        c = network_config
        if c.get("otype", "FullyFusedMLP") != "FullyFusedMLP" or c.get("activation", "ReLU") != "ReLU":
            raise ValueError("only ReLU FullyFusedMLP networks are on the hot path")
        self.n_input_dims, self.n_output_dims = n_input_dims, n_output_dims
        self.n_neurons, self.n_hidden = c["n_neurons"], c["n_hidden_layers"]
        self.output_activation = c.get("output_activation", "None")
        if self.output_activation not in ("None", "Sigmoid"):
            raise ValueError(self.output_activation)
        self.shapes = [(self.n_neurons, _pad16(n_input_dims))]
        self.shapes += [(self.n_neurons, self.n_neurons)] * (self.n_hidden - 1)
        self.shapes.append((_pad16(n_output_dims), self.n_neurons))
        gen = torch.Generator().manual_seed(seed)
        chunks = []
        for r, c_ in self.shapes:                       # Xavier uniform per matrix
            lim = math.sqrt(6.0 / (r + c_))
            chunks.append(((torch.rand(r, c_, generator=gen) * 2 - 1) * lim).reshape(-1))
        self.params = nn.Parameter(torch.cat(chunks))
        # content of the padded input columns: 0 here and in the oracle; b2n.checkpoint sets 1.0 when it loads weights
        # trained with an upstream tiny-cuda-nn whose Network pads its inputs with ones (those columns are then a bias)
        self.input_pad_value = 0.0

    def _pad_bias(self, W0, d_in):
        """the padded input columns' contribution as a first-layer bias: pad * sum_j W0[:, j >= d_in] (differentiable,
        so the gradient reaches the padded weight columns); None when there is nothing to add"""
        if self.input_pad_value == 0.0 or W0.shape[1] <= d_in:
            return None
        return W0[:, d_in:].sum(dim=1) * self.input_pad_value

    def matrices(self):
        out, off = [], 0
        for r, c in self.shapes:
            out.append(self.params[off:off + r * c].view(r, c))
            off += r * c
        return out

    def can_fuse(self, d_in=None):
        return (b2n.mlp_precision() == "bf16"
                and b2n.ops.fused_mlp_supported(self.n_input_dims if d_in is None else d_in, self.n_neurons, self.n_hidden,
                                                self.n_output_dims))

    def forward_fused(self, x0, x1=None):
        """whole network as one tensor-core kernel each way (b2n_fmlp_*); input = [x0 | x1]"""
        mats = self.matrices()
        act = "sigmoid" if self.output_activation == "Sigmoid" else "none"
        d_in = x0.shape[-1] + (x1.shape[-1] if x1 is not None else 0)
        biases = [self._pad_bias(mats[0], d_in)] + [None] * (len(mats) - 1)
        return b2n.ops.fused_mlp(x0, x1, mats[:-1] + [mats[-1][: self.n_output_dims]], biases, act)

    def forward(self, x):
        if x.is_cuda and self.can_fuse(x.shape[-1]):
            return self.forward_fused(x)
        mats = self.matrices()
        h = x
        for i, W in enumerate(mats[:-1]):
            h = b2n.linear(h, W, self._pad_bias(W, x.shape[-1]) if i == 0 else None, "relu")
        act = "sigmoid" if self.output_activation == "Sigmoid" else "none"
        return b2n.linear(h, mats[-1][: self.n_output_dims], None, act)


class NeRFDecoder(BaseDecoder):
    """x -> 8x256 ReLU trunk (skip concat [h, x] before layer ``skip_layer``) -> sigma (ReLU),
    feature (linear); cat[feature, d] -> view layer (ReLU) -> rgb (sigmoid)."""

    def __init__(self, pos_dim, dir_dim, hidden_dim=256, num_layers=8, skip_layer=4, view_dim=128):
        super().__init__()
        self.skip_layer = skip_layer
        layers = []
        for i in range(num_layers):
            in_dim = pos_dim if i == 0 else hidden_dim
            if i == skip_layer:
                in_dim += pos_dim
            layers.append(_Dense(in_dim, hidden_dim))
        self.pts_layers = nn.ModuleList(layers)
        self.sigma_layer = _Dense(hidden_dim, 1)
        self.feature_layer = _Dense(hidden_dim, hidden_dim)
        self.view_layer = _Dense(hidden_dim + dir_dim, view_dim)
        self.rgb_layer = _Dense(view_dim, 3)

    def forward(self, x, d):
        if (b2n.mlp_precision() == "bf16" and x.is_cuda and not d.requires_grad
                and b2n.ops.nerf_mlp_supported(self, x.shape[-1], d.shape[-1])):
            return b2n.ops.nerf_mlp(self, x, d)          # tcgen05 tensor-core path (fwd + bwd)
        h = x
        for i, layer in enumerate(self.pts_layers):
            if i == self.skip_layer:
                h = torch.cat([h, x], dim=-1)
            h = layer(h, "relu")
        sigma = self.sigma_layer(h, "relu")
        feat = self.feature_layer(h)
        hv = self.view_layer(torch.cat([feat, d], dim=-1), "relu")
        return self.rgb_layer(hv, "sigmoid"), sigma


class InstantNeRFDecoder(BaseDecoder):
    """sigma_net: pos -> 64 -> 16; sigma = softplus(h0 - 5); color_net: cat[h16, dir] -> 64 -> 64 -> 3 sigmoid."""

    def __init__(self, pos_dim, dir_dim, hidden_dim=64):
        super().__init__()
        self.sigma_net = FusedMLP(pos_dim, 16, {"otype": "FullyFusedMLP", "activation": "ReLU",
                                                "output_activation": "None", "n_neurons": hidden_dim,
                                                "n_hidden_layers": 1})
        self.color_net = FusedMLP(16 + dir_dim, 3, {"otype": "FullyFusedMLP", "activation": "ReLU",
                                                    "output_activation": "Sigmoid", "n_neurons": hidden_dim,
                                                    "n_hidden_layers": 2})

    def forward(self, x_enc, d_enc):
        """Module-API path on pre-encoded directions (layer-by-layer fp32 kernels)."""
        h = self.sigma_net(x_enc)
        sigma = b2n.sigma_head(h)
        rgb = self.color_net(torch.cat([h, d_enc], dim=-1))
        return rgb, sigma

    def density(self, x_enc, x_enc2=None):
        """sigma only, input = [x_enc | x_enc2]: the density branch without the colour network (occupancy sweeps,
        SURVEY 8f-3).  Same kernels and arithmetic as ``forward`` in fp32 mode; in bf16 mode the sigma network runs as
        one fused tensor-core kernel on the two sources (no concat, no direction features, no colour layers)."""
        net = self.sigma_net
        if x_enc.is_cuda and x_enc2 is not None and net.can_fuse(x_enc.shape[-1] + x_enc2.shape[-1]):
            return b2n.sigma_head(net.forward_fused(x_enc, x_enc2))
        if x_enc2 is not None:
            x_enc = torch.cat([x_enc, x_enc2], dim=-1)
        return b2n.sigma_head(net(x_enc))

    def can_fuse(self, dir_encoder):
        return (b2n.mlp_precision() == "bf16" and self.sigma_net.n_neurons == 64 and self.color_net.n_neurons == 64
                and self.sigma_net.n_input_dims <= 64 and dir_encoder.input_dim == 3 and dir_encoder.use_encoding
                and 0 <= dir_encoder.L <= 4 and self.color_net.n_input_dims == 16 + dir_encoder.out_dim)

    def forward_fused(self, x_enc, dirs, dir_encoder):
        """Whole decoder (+ direction Fourier features) as ONE tensor-core kernel each way
        (b2n_instant_mlp_fwd_tc / _bwd_tc); NeuralField.forward takes this path in bf16 mode."""
        if self.sigma_net.input_pad_value != self.color_net.input_pad_value:
            raise ValueError("sigma_net and color_net must share one input_pad_value")
        return b2n.instant_mlp(x_enc, dirs, dir_encoder.freq_bands, self.sigma_net.params, self.color_net.params,
                               self.sigma_net.input_pad_value)


class DeformationNetwork(BaseDecoder):
    """cat[gamma(x'), gamma(t')] -> (Linear, ReLU) x (num_layers - 1) -> Linear -> delta_x.
    ``net`` keeps nn.Sequential indexing (Linear at even indices) for checkpoint parity;
    the output layer starts at U(+-1e-4) weights / zero bias like the reference."""

    def __init__(self, pos_dim, time_dim, hidden_dim=128, num_layers=4):
        super().__init__()
        self.num_layers = num_layers
        mods = [_Dense(pos_dim + time_dim, hidden_dim), nn.ReLU()]
        for _ in range(num_layers - 2):
            mods += [_Dense(hidden_dim, hidden_dim), nn.ReLU()]
        last = _Dense(hidden_dim, 3)
        nn.init.uniform_(last.weight, -1e-4, 1e-4)
        nn.init.zeros_(last.bias)
        mods.append(last)
        self.net = nn.Sequential(*mods)

    def forward(self, x_feat, t_feat):
        dense = [m for m in self.net if isinstance(m, _Dense)]
        if (b2n.mlp_precision() == "bf16" and x_feat.is_cuda
                and b2n.ops.fused_mlp_supported(x_feat.shape[-1] + t_feat.shape[-1], dense[0].out_features,
                                                len(dense) - 1, 3)
                and all(m.out_features == dense[0].out_features for m in dense[:-1])):
            return b2n.ops.fused_mlp(x_feat, t_feat, [m.weight for m in dense], [m.bias for m in dense], "none")
        h = torch.cat([x_feat, t_feat], dim=-1)
        for m in dense[:-1]:
            h = m(h, "relu")
        return dense[-1](h)


class HashDeformationDecoder(BaseDecoder):
    """cat[hash_feat, time_mod] -> fused 64-wide MLP -> 3, times the learnable ``displacement_scale``."""

    def __init__(self, hash_dim, time_mod_dim, hidden_dim=64):
        super().__init__()
        self.deform_net = FusedMLP(hash_dim + time_mod_dim, 3, {"otype": "FullyFusedMLP", "activation": "ReLU",
                                                                "output_activation": "None",
                                                                "n_neurons": hidden_dim, "n_hidden_layers": 2})
        self.displacement_scale = nn.Parameter(torch.tensor(0.1))

    def forward(self, hash_feat, time_mod):
        if hash_feat.is_cuda and self.deform_net.can_fuse(hash_feat.shape[-1] + time_mod.shape[-1]):
            return self.deform_net.forward_fused(hash_feat, time_mod) * self.displacement_scale
        return self.deform_net(torch.cat([hash_feat, time_mod], dim=-1)) * self.displacement_scale


class TimeModulationNetwork(BaseDecoder):
    """gamma(t) -> Linear/ReLU stack -> sigmoid gate; last bias starts at -1 (reference :358-359)."""

    def __init__(self, time_dim, output_dim=64, hidden_dim=64, num_layers=2):
        super().__init__()
        self.output_dim = output_dim
        mods, in_dim = [], time_dim
        for i in range(num_layers):
            last = i == num_layers - 1
            mods.append(_Dense(in_dim, output_dim if last else hidden_dim))
            if not last:
                mods.append(nn.ReLU())
            in_dim = output_dim if last else hidden_dim
        self.net = nn.Sequential(*mods)
        nn.init.xavier_uniform_(mods[-1].weight)
        nn.init.constant_(mods[-1].bias, -1.0)

    def forward(self, time_feat):
        dense = [m for m in self.net if isinstance(m, _Dense)]
        if (b2n.mlp_precision() == "bf16" and time_feat.is_cuda and len(dense) >= 2
                and b2n.ops.fused_mlp_supported(time_feat.shape[-1], dense[0].out_features, len(dense) - 1,
                                                dense[-1].out_features)
                and all(m.out_features == dense[0].out_features for m in dense[:-1])):
            return b2n.ops.fused_mlp(time_feat, None, [m.weight for m in dense], [m.bias for m in dense], "sigmoid")
        h = time_feat
        for m in dense[:-1]:
            h = m(h, "relu")
        return dense[-1](h, "sigmoid")
