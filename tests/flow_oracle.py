"""float64 restatement of BigVGANFlowVAE's flow for the tests: the VITS ResidualCouplingBlock the reference copies
into backup/flows.py:613-792 (mean_only coupling layers, an unconditioned WN, a Flip after every coupling layer), over
a state dict with the reference's key names.  TEST INFRASTRUCTURE ONLY.

    layer:  x0, x1 = split(x);  h = pre(x0) mask;  h = WN(h, mask);  m = post(h) mask
            x1' = m + x1 mask (forward)  or  (x1 - m) mask (reverse);  cat(x0, x1')
    WN:     skip = 0; per layer i: a = in_layers[i](x) (dilation rate^i, padding (K d - d) / 2),
            acts = tanh(a[:, :H]) sigmoid(a[:, H:]), rs = res_skip_layers[i](acts);
            i < n - 1: x = (x + rs[:, :H]) mask, skip += rs[:, H:];  last: skip += rs;  return skip mask
    block:  forward: (layer, flip) in list order;  reverse: (flip, inverse layer) in reversed order"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _fold(sd, key):
    if key + ".weight_g" in sd:
        v, g = sd[key + ".weight_v"], sd[key + ".weight_g"]
        return v * (g / v.flatten(1).norm(dim=1).view(-1, 1, 1))
    return sd[key + ".weight"]


def _conv(sd, key, x, k=1, dilation=1):
    return F.conv1d(x, _fold(sd, key), sd[key + ".bias"], padding=int((k * dilation - dilation) / 2),
                    dilation=dilation)


def coupling_layer(sd, key, x, mask, reverse, hidden, n_layers=4, kernel_size=5, dilation_rate=1):
    half = x.shape[1] // 2
    x0, x1 = x[:, :half], x[:, half:]
    h = _conv(sd, key + ".pre", x0) * mask
    skip = 0
    for i in range(n_layers):
        d = dilation_rate ** i
        a = _conv(sd, f"{key}.enc.in_layers.{i}", h, kernel_size, d)
        acts = torch.tanh(a[:, :hidden]) * torch.sigmoid(a[:, hidden:])
        rs = _conv(sd, f"{key}.enc.res_skip_layers.{i}", acts)
        if i < n_layers - 1:
            h = (h + rs[:, :hidden]) * mask
            skip = skip + rs[:, hidden:]
        else:
            skip = skip + rs
    m = _conv(sd, key + ".post", skip * mask) * mask
    x1 = (x1 - m) * mask if reverse else m + x1 * mask
    return torch.cat([x0, x1], 1)


def flow(sd, h, x, mask, reverse=False, prefix="flow", n_flows=4, n_layers=4, kernel_size=5, dilation_rate=1):
    """ResidualCouplingBlock(latent_dim, flow_hidden_channels, kernel_size, dilation_rate, n_layers, n_flows) on x
    [B, C, T] with x_mask [B, 1, T], in the dtype of its inputs (float64 in the tests)."""
    layers = [f"{prefix}.flows.{2 * i}" for i in range(n_flows)]
    hidden = h["flow_hidden_channels"]
    if not reverse:
        for key in layers:
            x = coupling_layer(sd, key, x, mask, False, hidden, n_layers, kernel_size, dilation_rate)
            x = torch.flip(x, [1])
    else:
        for key in reversed(layers):
            x = torch.flip(x, [1])
            x = coupling_layer(sd, key, x, mask, True, hidden, n_layers, kernel_size, dilation_rate)
    return x
