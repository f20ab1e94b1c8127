"""A stand-in for the reference's denoiser (`Text2ImageTransformer`, transformer_utils.py) for the fused self-attention
tests, which must run where the reference source is absent.

`FullAttention` is restated from its known form (transformer_utils.py:24-62): key / query / value / proj = Linear(C, C);
q, k and v split into n_head heads; att = softmax(q kᵀ / √(C / n_head)); the return value is
(resid_drop(proj(att @ v with the heads merged)), att.mean(1)); `mask` is accepted and not used.  The class name is the
reference's, which is what `fuse_self_attention` matches.  `StandInDenoiser` has the surface `FusedDiffusionTransformer`
walks: `content_emb` (with `num_embed` = K + 1), `blocks` called as block(x, cond_emb, t) -> (x, att), `to_logits`
= LayerNorm + Linear(C, K), and `forward(x_t, cond_emb, t)` -> a `[B, K, N]` view of `[B, N, K]` logits."""
import math

import torch
from torch import nn
from torch.nn import functional as F


class FullAttention(nn.Module):
    def __init__(self, n_embd, n_head, attn_pdrop=0.0, resid_pdrop=0.0):
        super().__init__()
        self.key = nn.Linear(n_embd, n_embd)
        self.query = nn.Linear(n_embd, n_embd)
        self.value = nn.Linear(n_embd, n_embd)
        self.attn_drop = nn.Dropout(attn_pdrop)
        self.resid_drop = nn.Dropout(resid_pdrop)
        self.proj = nn.Linear(n_embd, n_embd)
        self.n_head = n_head

    def forward(self, x, encoder_output, mask=None):
        B, T, C = x.size()
        k = self.key(x).view(B, T, self.n_head, C // self.n_head).transpose(1, 2)
        q = self.query(x).view(B, T, self.n_head, C // self.n_head).transpose(1, 2)
        v = self.value(x).view(B, T, self.n_head, C // self.n_head).transpose(1, 2)
        att = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(k.size(-1)))
        att = F.softmax(att, dim=-1)
        att = self.attn_drop(att)
        y = att @ v
        y = y.transpose(1, 2).contiguous().view(B, T, C)
        att = att.mean(dim=1, keepdim=False)
        y = self.resid_drop(self.proj(y))
        return y, att


class CrossStandIn(nn.Module):
    """The block's cross-attention over the condition, reduced to a Linear of its mean (not what the tests exercise)."""

    def __init__(self, n_embd, cond_dim):
        super().__init__()
        self.proj = nn.Linear(cond_dim, n_embd)

    def forward(self, x, cond):
        return x + self.proj(cond.mean(1)).unsqueeze(1), None


class Block(nn.Module):
    def __init__(self, n_embd, n_head, cond_dim, T):
        super().__init__()
        self.t_emb = nn.Embedding(T, n_embd)
        self.ln1, self.ln2, self.ln3 = nn.LayerNorm(n_embd), nn.LayerNorm(n_embd), nn.LayerNorm(n_embd)
        self.attn1 = FullAttention(n_embd, n_head)
        self.attn2 = CrossStandIn(n_embd, cond_dim)
        self.mlp = nn.Sequential(nn.Linear(n_embd, 4 * n_embd), nn.GELU(), nn.Linear(4 * n_embd, n_embd))

    def forward(self, x, cond_emb, t, mask=None):
        a, att = self.attn1(self.ln1(x) + self.t_emb(t).unsqueeze(1), cond_emb, mask=mask)
        x = x + a
        a, att = self.attn2(self.ln2(x), cond_emb)
        x = a
        return x + self.mlp(self.ln3(x)), att


class ContentEmb(nn.Module):
    def __init__(self, num_embed, N, n_embd):
        super().__init__()
        self.num_embed = num_embed
        self.emb = nn.Embedding(num_embed, n_embd)
        self.pos = nn.Parameter(torch.randn(1, N, n_embd))

    def forward(self, x):
        return self.emb(x) + self.pos[:, : x.shape[1]]


class StandInDenoiser(nn.Module):
    def __init__(self, K, N, *, n_embd=64, n_head=16, n_layer=3, cond_dim=512, T=100, logit_gain=1.0):
        super().__init__()
        self.content_emb = ContentEmb(K + 1, N, n_embd)
        self.blocks = nn.ModuleList([Block(n_embd, n_head, cond_dim, T) for _ in range(n_layer)])
        self.to_logits = nn.Sequential(nn.LayerNorm(n_embd), nn.Linear(n_embd, K))
        with torch.no_grad():
            self.to_logits[1].weight.mul_(logit_gain)

    def forward(self, x_t, cond_emb, t):
        emb = self.content_emb(x_t)
        for block in self.blocks:
            emb, _ = block(emb, cond_emb, t)
        return self.to_logits(emb).permute(0, 2, 1)
