"""
ORACLE (test infrastructure, NOT product code) -- CPU restatement of MAE-style pre-training
(`ecg_b200.EcgVitForMaskedAutoencoding`) on the modules of the restated `vit_pytorch.ViT` (`oracle/vit_restated.py`).

    a      = patchify(x)                                        [B, n, K]
    vis    = the visible positions of every record, ascending    [B, n_vis]
    x0     = [cls + pos[0] | a[vis] We^T + be + pos[1 + vis]] ; emb-dropout
    z      = encoder transformer(x0)                             [B, n_vis + 1, d]
    t      = decoder.embed(decoder.norm(z))                      [B, n_vis + 1, d_dec]
    u0     = [t[:, 0] | t[:, 1 + slot] where visible, else mask_token] + decoder.pos
    pred   = recon_head(decoder transformer(u0)[:, 1:])          [B, n, K]
    loss   = sum_{masked (b, w), k} (pred - a)^2 / (n_masked * K)

The mask is an INPUT (bool [B, n], the same count in every record), so the tests can inject the one the GPU drew.
`OracleMaskedPatchTrainer` (oracle/mpm_oracle.py) runs its training steps.

Only tests/ may import this.
"""
import torch
from torch import nn

from oracle.ecg_vit_oracle import OracleConfig
from oracle.vit_restated import ViT, Transformer


class OracleMaeDecoder(nn.Module):
    def __init__(self, dim, n_patch, dec_dim, depth, heads, mlp_dim):
        super().__init__()
        self.norm = nn.LayerNorm(dim)
        self.embed = nn.Linear(dim, dec_dim)
        self.mask_token = nn.Parameter(torch.zeros(1, 1, dec_dim))
        self.pos_embedding = nn.Parameter(torch.randn(1, n_patch + 1, dec_dim))
        self.transformer = Transformer(dec_dim, depth, heads, dec_dim // heads, mlp_dim, 0.0)


def visible_positions(bool_masked_pos):
    """int64 [B, n_vis]: the ascending positions of every record's visible patches"""
    B, n = bool_masked_pos.shape
    order = torch.argsort(bool_masked_pos.to(torch.int8), dim=1, stable=True)   # visible (0) first, in position order
    n_vis = n - int(bool_masked_pos[0].sum())
    return order[:, :n_vis]


def gather_visible(t, vis):
    """t [B, n, F] -> [B, n_vis, F], rows vis[b] of record b"""
    return torch.gather(t, 1, vis[..., None].expand(-1, -1, t.shape[-1]))


def unshuffle(t, bool_masked_pos, mask_token):
    """[B, n_vis + 1, F] (CLS first) -> [B, n + 1, F]: the visible rows back at their positions, the mask token at the
    masked ones"""
    B, n = bool_masked_pos.shape
    vis = visible_positions(bool_masked_pos)
    body = mask_token.expand(B, n, -1).clone()
    body = body.scatter(1, vis[..., None].expand(-1, -1, t.shape[-1]), t[:, 1:])
    return torch.cat((t[:, :1], body), dim=1)


class OracleMaskedAutoencoder(nn.Module):
    """state_dict keys: `vit.*` of `OracleEcgVit` without `vit.mlp_head.*`, then `decoder.*`, then `recon_head.{0,1}.*`"""

    def __init__(self, config=None, decoder_hidden_size=256, decoder_num_hidden_layers=4, decoder_num_attention_heads=4,
                 decoder_intermediate_size=1024):
        super().__init__()
        config = config if config is not None else OracleConfig()
        d, h = config.hidden_size, config.num_attention_heads
        self.config = config
        self.per_lead = bool(getattr(config, 'per_lead_tokens', False))
        self.vit = ViT(image_size=(config.num_channels if self.per_lead else 1, config.max_signal_length),
                       patch_size=(1, config.patch_size), num_classes=1, dim=d, depth=config.num_hidden_layers,
                       heads=h, mlp_dim=config.intermediate_size, pool='cls',
                       channels=1 if self.per_lead else config.num_channels, dim_head=d // h,
                       dropout=config.hidden_dropout_prob, emb_dropout=config.attention_probs_dropout_prob)
        del self.vit.mlp_head
        n = self.vit.pos_embedding.shape[1] - 1
        self.decoder = OracleMaeDecoder(d, n, decoder_hidden_size, decoder_num_hidden_layers,
                                        decoder_num_attention_heads, decoder_intermediate_size)
        patch_dim = config.patch_size * (1 if self.per_lead else config.num_channels)
        self.recon_head = nn.Sequential(nn.LayerNorm(decoder_hidden_size), nn.Linear(decoder_hidden_size, patch_dim))

    def patches(self, sample_values):
        img = sample_values.unsqueeze(1) if self.per_lead else sample_values.unsqueeze(-2)
        return self.vit.to_patch_embedding[0](img)   # [B, n, K]

    def encode(self, sample_values, bool_masked_pos):
        """(patch matrix a [B, n, K], encoder output z [B, n_vis + 1, d])"""
        vit = self.vit
        a = self.patches(sample_values)
        vis = visible_positions(bool_masked_pos)
        e = vit.to_patch_embedding[1](gather_visible(a, vis))
        b = e.shape[0]
        pos = vit.pos_embedding[0]
        x = torch.cat((vit.cls_token.expand(b, -1, -1) + pos[0], e + pos[1 + vis]), dim=1)
        return a, vit.transformer(vit.dropout(x))

    def forward(self, sample_values, bool_masked_pos):
        """(loss, reconstruction [B, n, K])"""
        a, z = self.encode(sample_values, bool_masked_pos)
        dec = self.decoder
        t = dec.embed(dec.norm(z))
        u = unshuffle(t, bool_masked_pos, dec.mask_token) + dec.pos_embedding
        pred = self.recon_head(dec.transformer(u)[:, 1:])
        m = bool_masked_pos[..., None].to(pred.dtype)
        loss = ((pred - a) ** 2 * m).sum() / (m.sum() * a.shape[-1])
        return loss, pred
