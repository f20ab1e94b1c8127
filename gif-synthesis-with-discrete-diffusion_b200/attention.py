"""Fused self-attention for the denoiser's blocks (SURVEY §8 f3): `d3pm_self_attention` behind the reference's
`FullAttention` (transformer_utils.py:24-62).

The reference materialises `softmax(q kᵀ / √d)` as a `[B, heads, N, N]` fp32 tensor in every block (17 GB per layer at
B = 16, N = 4096); the kernel keeps the scores in registers.  Scope: inference - forward only, fp32, no autograd graph.
`FusedSelfAttention` hands every other call (training, dropout, autocast, a mask) to the original module unchanged.

    fuse_self_attention(denoiser)          # swap every FullAttention; state_dict keys and tensors are unchanged
    fuse_self_attention(denoiser, False)   # put the originals back
"""
from __future__ import annotations

import ctypes
import math

import torch
from torch import nn

from d3pm_b200 import _lib
from d3pm_b200._lib import D3PMError
from d3pm_b200.ops import _need_cuda, _stream

HEAD_DIM = 4  # the only head width the kernel implements (n_embd 64 / 16 heads, the shipped model)


def self_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, n_head: int, scale: float) -> torch.Tensor:
    """`softmax(scale · q kᵀ) v` per head on `[B, N, C]` fp32 tensors whose heads are the column groups of `C / n_head`
    (the outputs of FullAttention's `query` / `key` / `value` Linears, read in place) -> `[B, N, C]`, the reference's
    `y.transpose(1, 2).contiguous().view(B, T, C)`."""
    dev = _need_cuda(q, k, v)
    if q.dim() != 3 or q.shape != k.shape or q.shape != v.shape:
        raise D3PMError(f"q, k and v must be [B, N, C] of one shape, got {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    if any(x.dtype != torch.float32 for x in (q, k, v)):
        raise D3PMError("self_attention takes float32 tensors")
    B, N, C = q.shape
    if n_head <= 0 or C % n_head != 0:
        raise D3PMError(f"C = {C} is not a multiple of n_head = {n_head}")
    # read in place when the three share one row pitch (unit column stride, rows of a video consecutive); else copy
    pitch = q.stride(1) if N > 1 else (q.stride(0) if B > 1 else C)
    if (q.stride(2) != 1 or k.stride() != q.stride() or v.stride() != q.stride() or (B > 1 and q.stride(0) != N * pitch)
            or pitch < C or pitch % 4 != 0):
        q, k, v, pitch = q.contiguous(), k.contiguous(), v.contiguous(), C
    y = torch.empty(B, N, C, device=dev, dtype=torch.float32)
    d = _lib.AttnDesc(q=q.data_ptr(), k=k.data_ptr(), v=v.data_ptr(), y=y.data_ptr(), B=B, N=N, heads=n_head,
                      head_dim=C // n_head, pitch_qkv=pitch, pitch_y=C, scale=float(scale), stream=_stream(dev))
    _lib.check(_lib.load_library().d3pm_self_attention(ctypes.byref(d)), "d3pm_self_attention")
    return y


def _dropout_active(module: nn.Module) -> bool:
    return module.training and any(isinstance(m, nn.Dropout) and m.p > 0 for m in module.modules())


class FusedSelfAttention(nn.Module):
    """Stands in for one reference `FullAttention`.  Its children and buffers are the original's, registered under their
    own names, so `state_dict()` keys and tensors are unchanged; the original module is kept (unregistered) for
    delegation and for `fuse_self_attention(..., enable=False)`.

    `forward(x, encoder_output, mask=None)` runs the module's own `query` / `key` / `value` Linears, `d3pm_self_attention`
    and `proj`, and returns `(y, None)`: the head-averaged attention map (the reference's second output) is not formed -
    the blocks drop it (the self-attention map is overwritten by the cross-attention's before the block returns it).
    The original module runs instead, unchanged, when grad is enabled and `x` or a parameter requires grad, when a
    dropout is active (training mode with p > 0), under autocast or for non-fp32 `x`, and when a `mask` is given."""

    def __init__(self, original: nn.Module):
        super().__init__()
        object.__setattr__(self, "original", original)
        for name, child in original.named_children():
            setattr(self, name, child)
        for name, buf in original.named_buffers(recurse=False):
            self.register_buffer(name, buf, persistent=name not in original._non_persistent_buffers_set)
        self.n_head = int(original.n_head)
        self.train(original.training)

    def sync_original(self) -> nn.Module:
        """The original module with this module's training flag and buffers (which `.to()` may have replaced)."""
        self.original.training = self.training
        for name, buf in self.named_buffers(recurse=False):
            setattr(self.original, name, buf)
        return self.original

    def _delegate(self, x: torch.Tensor, mask) -> bool:
        if mask is not None or x.dtype != torch.float32 or torch.is_autocast_enabled(x.device.type) or _dropout_active(self):
            return True
        return torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))

    def forward(self, x, encoder_output, mask=None):
        if self._delegate(x, mask):
            return self.sync_original()(x, encoder_output, mask=mask)
        C = x.shape[-1]
        y = self_attention(self.query(x), self.key(x), self.value(x), self.n_head, 1.0 / math.sqrt(C // self.n_head))
        y = self.proj(y)
        drop = getattr(self, "resid_drop", None)
        return (drop(y) if drop is not None else y), None


def _qualifies(m: nn.Module) -> bool:
    """A reference FullAttention of the shape the kernel covers: key / query / value / proj = Linear(C, C), C / n_head = 4."""
    lin = [getattr(m, n, None) for n in ("key", "query", "value", "proj")]
    if not all(isinstance(x, nn.Linear) for x in lin):
        return False
    C = lin[0].in_features
    n_head = getattr(m, "n_head", None)
    return (all(x.in_features == C and x.out_features == C for x in lin) and isinstance(n_head, int) and n_head > 0
            and C % n_head == 0 and C // n_head == HEAD_DIM)


def fuse_self_attention(transformer: nn.Module, enable: bool = True) -> int:
    """Swap every submodule of `transformer` whose class is the reference's `FullAttention` (matched by class name: the
    reference is loaded by path) and whose shape the kernel covers for a `FusedSelfAttention`; `enable=False` puts the
    original modules back.  Idempotent: modules fused by an earlier call stay as they are.  Returns the number of fused
    modules after an enabling call, of restored ones after a disabling call.  Raises `D3PMError` when enabling leaves the
    model with none."""
    swaps, already = [], 0
    for parent in transformer.modules():
        for name, child in parent.named_children():
            if isinstance(child, FusedSelfAttention):
                if enable:
                    already += 1
                else:
                    swaps.append((parent, name, child.sync_original()))
            elif enable and type(child).__name__ == "FullAttention" and _qualifies(child):
                swaps.append((parent, name, FusedSelfAttention(child)))
    if enable and not swaps and not already:
        raise D3PMError("fuse_self_attention: no FullAttention with key / query / value / proj = Linear(C, C) and "
                        f"C / n_head = {HEAD_DIM} in this model")
    for parent, name, module in swaps:
        setattr(parent, name, module)
    return len(swaps) + already
