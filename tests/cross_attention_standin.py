"""A self-plus-cross stand-in for the reference's denoiser (`Text2ImageTransformer`, transformer_utils.py), for the fused
cross-attention tests, which must run where the reference source is absent.

`CrossAttention` is restated from its known form (the math `tools/attention_bench.py`'s `cross_arm` times): key / value =
Linear(condition_embd, n_embd), query / proj = Linear(n_embd, n_embd); q from the tokens, k and v from the condition rows,
split into n_head heads; att = softmax(q kᵀ / √(C / n_head)) over the condition tokens with no mask applied; the return
value is (resid_drop(proj(att @ v with the heads merged)), att.mean(1)).  Like the reference's causal variant it registers a
`mask` buffer that its forward never reads.  The class name is the reference's, which is what `fuse_cross_attention`
matches.  `CrossStandInDenoiser` has the surface of `tests/attention_standin.StandInDenoiser`, with blocks that run a
`FullAttention` and then this `CrossAttention`, each as a residual; a block returns the cross-attention's map."""
import math

import torch
from torch import nn
from torch.nn import functional as F

from tests.attention_standin import ContentEmb, FullAttention


class CrossAttention(nn.Module):
    def __init__(self, condition_seq_len, n_embd, condition_embd, n_head, seq_len=None, attn_pdrop=0.0, resid_pdrop=0.0,
                 causal=True):
        super().__init__()
        self.key = nn.Linear(condition_embd, n_embd)
        self.query = nn.Linear(n_embd, n_embd)
        self.value = nn.Linear(condition_embd, n_embd)
        self.attn_drop = nn.Dropout(attn_pdrop)
        self.resid_drop = nn.Dropout(resid_pdrop)
        self.proj = nn.Linear(n_embd, n_embd)
        self.n_head = n_head
        self.causal = causal
        if self.causal:
            self.register_buffer("mask", torch.tril(torch.ones(seq_len, seq_len)).view(1, 1, seq_len, seq_len))

    def forward(self, x, encoder_output, mask=None):
        B, T, C = x.size()
        B, T_E, _ = encoder_output.size()
        k = self.key(encoder_output).view(B, T_E, self.n_head, C // self.n_head).transpose(1, 2)
        q = self.query(x).view(B, T, self.n_head, C // self.n_head).transpose(1, 2)
        v = self.value(encoder_output).view(B, T_E, self.n_head, C // self.n_head).transpose(1, 2)
        att = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(k.size(-1)))
        att = F.softmax(att, dim=-1)
        att = self.attn_drop(att)
        y = att @ v
        y = y.transpose(1, 2).contiguous().view(B, T, C)
        att = att.mean(dim=1, keepdim=False)
        y = self.resid_drop(self.proj(y))
        return y, att


class CrossBlock(nn.Module):
    def __init__(self, n_embd, n_head, cond_dim, T, N):
        super().__init__()
        self.t_emb = nn.Embedding(T, n_embd)
        self.ln1, self.ln2, self.ln3 = nn.LayerNorm(n_embd), nn.LayerNorm(n_embd), nn.LayerNorm(n_embd)
        self.attn1 = FullAttention(n_embd, n_head)
        self.attn2 = CrossAttention(77, n_embd, cond_dim, n_head, seq_len=N)
        self.mlp = nn.Sequential(nn.Linear(n_embd, 4 * n_embd), nn.GELU(), nn.Linear(4 * n_embd, n_embd))

    def forward(self, x, cond_emb, t, mask=None):
        a, att = self.attn1(self.ln1(x) + self.t_emb(t).unsqueeze(1), cond_emb, mask=mask)
        x = x + a
        a, att = self.attn2(self.ln2(x), cond_emb, mask=mask)
        x = x + a
        return x + self.mlp(self.ln3(x)), att


class CrossStandInDenoiser(nn.Module):
    def __init__(self, K, N, *, n_embd=64, n_head=16, n_layer=3, cond_dim=512, T=100, logit_gain=1.0):
        super().__init__()
        self.content_emb = ContentEmb(K + 1, N, n_embd)
        self.blocks = nn.ModuleList([CrossBlock(n_embd, n_head, cond_dim, T, N) for _ in range(n_layer)])
        self.to_logits = nn.Sequential(nn.LayerNorm(n_embd), nn.Linear(n_embd, K))
        with torch.no_grad():
            self.to_logits[1].weight.mul_(logit_gain)

    def forward(self, x_t, cond_emb, t):
        emb = self.content_emb(x_t)
        for block in self.blocks:
            emb, _ = block(emb, cond_emb, t)
        return self.to_logits(emb).permute(0, 2, 1)
