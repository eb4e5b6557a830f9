"""Drop path (stochastic depth) for the CPU oracle, with the keep draw of the CUDA kernels.

The kernels draw one keep per record and residual branch from the dropout counter hash: branch j (0 attention,
1 feed-forward) of block l of a depth-D encoder uses site 4*D + 2 + 2*l + j and element index b (the record), at rate
drop_path_rate * l / (D - 1).  `inject_drop_path` scales the output of every PreNorm of an oracle encoder by that
per-record factor with forward hooks, so the oracle's modules and state_dict keys stay untouched."""
import torch

import ecg_b200


def path_site(depth, l, j):
    return 4 * depth + 2 + 2 * l + j


def path_keep(seed, site, rate, B):
    """fp32 [B]: 0 (dropped) or 1 / (1 - rate) (kept) per record"""
    return ecg_b200._lib.dropout_keep_mask(seed, site, rate, torch.arange(B))


def inject_drop_path(transformer, seed, rate):
    """hooks on the PreNorm modules of an oracle `Transformer`: returns their handles (call .remove() on each)"""
    layers = transformer.layers
    D = len(layers)
    rates = [float(v) for v in torch.linspace(0, rate, D)]
    handles = []
    for l, blk in enumerate(layers):
        for j, pre in enumerate(blk):
            def hook(_module, _inp, out, site=path_site(D, l, j), r=rates[l]):
                s = path_keep(seed, site, r, out.shape[0]).to(out.dtype)
                return out * s.view(-1, *([1] * (out.dim() - 1)))
            handles.append(pre.register_forward_hook(hook))
    return handles


def keeps(seed, depth, rate, B):
    """[(s_att, s_ff)] per block: the factors a forward with this seed used"""
    rates = [float(v) for v in torch.linspace(0, rate, depth)]
    return [(path_keep(seed, path_site(depth, l, 0), rates[l], B), path_keep(seed, path_site(depth, l, 1), rates[l], B))
            for l in range(depth)]
