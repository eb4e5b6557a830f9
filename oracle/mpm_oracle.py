"""
ORACLE (test infrastructure, NOT product code) -- CPU restatement of masked-patch pre-training
(`ecg_b200.EcgVitForMaskedPatchModeling`) on the modules of the restated `vit_pytorch.ViT` (`oracle/vit_restated.py`).

SimMIM-style: masked patches keep their place in the sequence and enter it as a learned mask token; a LayerNorm +
Linear head predicts every patch from its encoder output and the loss is the MSE over the masked patches:

    a     = patchify(x)                                   (the Rearrange of to_patch_embedding[0])
    tok   = [cls | where(mask, mask_token, a We^T + be)] + pos ; emb-dropout
    z     = transformer(tok)
    pred  = recon_head(z[:, 1:])
    loss  = sum_{masked (b, w), k} (pred - a)^2 / (n_masked * K)

The mask is an INPUT (bool [B, n]), so the tests can inject the one the GPU drew.  The reference project has no
self-supervised objective; this restatement is the specification of the feature.

Only tests/ may import this.
"""
import torch
from torch import nn

from oracle.ecg_vit_oracle import OracleConfig, lr_lambda
from oracle.vit_restated import ViT


class OracleMaskedPatchModel(nn.Module):
    """state_dict keys: `vit.*` of `OracleEcgVit` without `vit.mlp_head.*`, plus `vit.mask_token` (after
    `vit.cls_token`), then `recon_head.{0,1}.*`"""

    def __init__(self, config=None):
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
        self.vit.mask_token = nn.Parameter(torch.zeros(1, 1, d))
        patch_dim = config.patch_size * (1 if self.per_lead else config.num_channels)
        self.recon_head = nn.Sequential(nn.LayerNorm(d), nn.Linear(d, patch_dim))

    def patches(self, sample_values):
        img = sample_values.unsqueeze(1) if self.per_lead else sample_values.unsqueeze(-2)
        return self.vit.to_patch_embedding[0](img)   # [B, n, K]

    def encode(self, sample_values, bool_masked_pos):
        """(patch matrix a [B, n, K], encoder output z [B, n + 1, d])"""
        vit = self.vit
        a = self.patches(sample_values)
        e = vit.to_patch_embedding[1](a)
        b, n, _ = e.shape
        e = torch.where(bool_masked_pos[..., None], vit.mask_token.expand(b, n, -1), e)
        x = torch.cat((vit.cls_token.expand(b, -1, -1), e), dim=1) + vit.pos_embedding[:, :n + 1]
        return a, vit.transformer(vit.dropout(x))

    def forward(self, sample_values, bool_masked_pos):
        """(loss, reconstruction [B, n, K])"""
        a, z = self.encode(sample_values, bool_masked_pos)
        pred = self.recon_head(z[:, 1:])
        m = bool_masked_pos[..., None].to(pred.dtype)
        loss = ((pred - a) ** 2 * m).sum() / (m.sum() * a.shape[-1])
        return loss, pred


class OracleMaskedPatchTrainer:
    """`OracleTrainer`'s step (zero_grad -> forward -> backward -> clip_grad_norm_ -> AdamW -> LambdaLR) on the
    masked-patch objective, with the mask as an input"""

    def __init__(self, model, learning_rate=3e-4, weight_decay=1e-2, schedule='constant', n_warmup=0, n_step=1000,
                 max_grad_norm=1.0):
        self.model = model
        self.optimizer = torch.optim.AdamW(model.parameters(), lr=learning_rate, weight_decay=weight_decay)
        self.scheduler = torch.optim.lr_scheduler.LambdaLR(
            self.optimizer, lambda s: lr_lambda(schedule, s, n_warmup, n_step))
        self.max_grad_norm = max_grad_norm

    def step(self, sample_values, bool_masked_pos):
        self.optimizer.zero_grad()
        loss, pred = self.model(sample_values, bool_masked_pos)
        loss.backward()
        total_norm = nn.utils.clip_grad_norm_(self.model.parameters(), max_norm=self.max_grad_norm,
                                              error_if_nonfinite=True)
        self.optimizer.step()
        self.scheduler.step()
        return loss.detach(), pred.detach(), total_norm.detach()
