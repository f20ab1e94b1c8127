"""Training-side operators (SURVEY.md §8 f1): forward-process `q_pred`, and the variational-bound loss of
`_train_loss` (diffusion_transformer.py:391-457) with its gradient w.r.t. the denoiser logits, as one CUDA
kernel per pass (`d3pm_train_rows`).  CUDA only; nothing here falls back to PyTorch math.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from d3pm_b200 import _lib, ops
from d3pm_b200._lib import D3PMError


def q_pred_rows(rows: torch.Tensor, pitch: int, t: torch.Tensor, sched8: torch.Tensor, K: int, cumulative: bool) -> torch.Tensor:
    """q_pred (:201-218) / q_pred_one_timestep (:185-199) on token-major rows `[B, N, >=K+1]` -> rows `[B, N, pitch]`."""
    dev = ops._need_cuda(rows, t, sched8)
    B, N = rows.shape[:2]
    T = sched8.shape[1] - 1
    out = ops.alloc_rows(B, N, K + 1, dev)
    lib = _lib.load_library()
    _lib.check(lib.d3pm_q_pred(rows.data_ptr(), pitch, t.contiguous().data_ptr(), sched8.data_ptr(), 1 if cumulative else 0,
                               out.data_ptr(), out.shape[2], B, N, K, T, ops._stream(dev)), "d3pm_q_pred")
    return out


def q_sample_tokens(x0: torch.Tensor, t: torch.Tensor, sched8: torch.Tensor, K: int, *, seed: int, offset: int,
                    row_offset: int = 0, status=None) -> torch.Tensor:
    """`d3pm_q_sample_tokens`: x_t ~ q(x_t | x_0) on int64 tokens `[B, N]` with the library's Philox noise (:361-366)."""
    dev = ops._need_cuda(x0, t, sched8, status)
    B, N = x0.shape
    out = torch.empty_like(x0)
    lib = _lib.load_library()
    _lib.check(lib.d3pm_q_sample_tokens(x0.contiguous().data_ptr(), t.contiguous().data_ptr(), sched8.data_ptr(), B, N, K,
                                        sched8.shape[1] - 1, seed, offset, row_offset, out.data_ptr(), ops._ptr(status),
                                        ops._stream(dev)), "d3pm_q_sample_tokens")
    return out


def _logit_rows(logits_bkn: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """Denoiser output, logically `[B, K, N]` -> token-major `[B, N, K]` rows (zero-copy for the reference's layout).
    float32, float16 or bfloat16; the rows keep the element type."""
    got = ops.rows_of(logits_bkn)
    if got is not None and got[1] % (16 // logits_bkn.element_size()) == 0 and logits_bkn.data_ptr() % 16 == 0:
        return got
    rows = logits_bkn.permute(0, 2, 1).contiguous()
    return rows, rows.shape[2]


def stream_takes_16bit(rows: torch.Tensor, pitch: int) -> bool:
    """Whether `d3pm_train_rows` reads these float16 / bfloat16 rows (`[B, N, K]`, `pitch` elements apart) in place, with
    both arg-max outputs or neither: the persistent stream kernel's shapes.  Mirrors the library's predicate, so that a
    caller casts beforehand instead of meeting D3PM_ERR_UNSUPPORTED."""
    B, N, K = rows.shape
    return K in ops.STREAM_CODEBOOKS and B * N >= 2048 and pitch % 8 == 0 and rows.data_ptr() % 16 == 0


def _train_rows(rows, pitch, x0, x_t, t, coef_table, mask_weight, *, backward, w_main=None, w_aux=None,
                want_recon=False, status=None):
    """`d3pm_train_rows`: backward False / 0 = losses, True / 1 = gradient, 2 = both in one pass over the logits.
    float16 / bfloat16 rows (stream kernel shapes only, see `stream_takes_16bit`) give a gradient of the same type."""
    backward = int(backward)
    dev = ops._need_cuda(rows, x0, x_t, t, coef_table, w_main, w_aux, status)
    B, N, K = rows.shape
    d = _lib.TrainDesc()
    d.logits, d.x0, d.x_t, d.t, d.coef_table = rows.data_ptr(), x0.data_ptr(), x_t.data_ptr(), t.data_ptr(), coef_table.data_ptr()
    d.B, d.N, d.K, d.T = B, N, K, coef_table.shape[0]
    d.pitch = pitch
    d.logits_dtype = ops.LOGITS_DTYPES[rows.dtype]
    d.mask_weight_masked, d.mask_weight_unmasked = float(mask_weight[0]), float(mask_weight[1])
    d.status = ops._ptr(status)
    d.stream = ops._stream(dev)
    out = {}
    d.backward = backward
    if backward:
        out["grad"] = torch.empty(B, N, K, dtype=rows.dtype, device=dev)
        d.grad, d.pitch_grad = out["grad"].data_ptr(), K
        d.w_main, d.w_aux = w_main.data_ptr(), w_aux.data_ptr()
    if backward != 1:
        out["tok_main"] = torch.empty(B, N, dtype=torch.float32, device=dev)
        out["tok_aux"] = torch.empty(B, N, dtype=torch.float32, device=dev)
        d.tok_main, d.tok_aux = out["tok_main"].data_ptr(), out["tok_aux"].data_ptr()
        if want_recon:
            out["x0_recon"] = torch.empty(B, N, dtype=torch.int64, device=dev)
            out["xtm1_recon"] = torch.empty(B, N, dtype=torch.int64, device=dev)
            d.x0_recon, d.xtm1_recon = out["x0_recon"].data_ptr(), out["xtm1_recon"].data_ptr()
    lib = _lib.load_library()
    _lib.check(lib.d3pm_train_rows(ctypes.byref(d)), "d3pm_train_rows")
    return out


def scale_rows(rows: torch.Tensor, factor: torch.Tensor) -> torch.Tensor:
    """rows[b, n, :] *= factor[b] in place (d3pm_scale_rows); videos whose factor is exactly 1 cost nothing."""
    dev = ops._need_cuda(rows, factor)
    B, N, K = rows.shape
    lib = _lib.load_library()
    _lib.check(lib.d3pm_scale_rows(rows.data_ptr(), rows.stride(1), factor.contiguous().data_ptr(), B, N, K, ops._stream(dev)),
               "d3pm_scale_rows")
    return rows


class VBLoss(torch.autograd.Function):
    """vb_loss[b] = kl_loss[b] / pt[b] + aux_w[b] * aux[b] / pt[b]   (:431-455), differentiable in the logits.

    When the logits require grad, forward makes ONE pass over them that yields the losses AND the gradient rows for the
    upstream gradient the caller announces (`grad_scale`: d(final loss)/d(vb_loss[b]), e.g. 1 / (B N) for the reference's
    `loss.sum() / (B N)`, :546); backward then only rescales the videos whose true upstream gradient differs from it
    (none in the reference's training loop).  No `[B, K+1, N]` intermediate is ever stored.  A gradient flowing into the
    second output (kl_loss) takes the explicit recomputation path.

    float16 / bfloat16 logits (a denoiser run under autocast) are read in place, and the gradient is returned in their
    type.  Forward then computes the losses only, and backward recomputes the rows with the true upstream weights
    (one more 16-bit read of the logits).  A gradient written in forward at the announced scale 1 / (B N) would be of
    order 1e-6 per class at the shipped shape: float16 subnormals, most of which round to zero before a loss scaler
    could rescale them.  Shapes the 16-bit kernel does not take are cast to float32, run as above, and the gradient is
    cast back.
    """

    @staticmethod
    def forward(ctx, logits_bkn, x0, x_t, t, pt, aux_w, coef_table, mask_weight, status, grad_scale=1.0):
        if logits_bkn.dim() != 3 or logits_bkn.dtype not in ops.LOGITS_DTYPES:
            raise D3PMError("logits must be float32, float16 or bfloat16 [B, K, N]")
        rows, pitch = _logit_rows(logits_bkn.detach())
        if rows.dtype != torch.float32 and not stream_takes_16bit(rows, pitch):
            rows, pitch = _logit_rows(logits_bkn.detach().float())
        ctx.grad_dtype = logits_bkn.dtype
        x0, x_t, t = x0.contiguous(), x_t.contiguous(), t.contiguous()
        fused = bool(ctx.needs_input_grad[0]) and rows.dtype == torch.float32
        ctx.set_materialize_grads(False)  # an unused output (kl_loss is only read detached) arrives as None in backward
        ctx.grad_scale, ctx.grad = float(grad_scale), None
        if fused:
            w_main = (ctx.grad_scale / pt).float().contiguous()
            w_aux = (ctx.grad_scale * aux_w / pt).float().contiguous()
            out = _train_rows(rows, pitch, x0, x_t, t, coef_table, mask_weight, backward=2, w_main=w_main, w_aux=w_aux,
                              want_recon=True, status=status)
            ctx.grad = out["grad"]
        else:
            out = _train_rows(rows, pitch, x0, x_t, t, coef_table, mask_weight, backward=0, want_recon=True, status=status)
        kl_loss = out["tok_main"].sum(1)
        aux = out["tok_aux"].sum(1)
        vb = kl_loss / pt + aux_w * aux / pt
        ctx.save_for_backward(rows, x0, x_t, t, pt, aux_w, coef_table)
        ctx.pitch, ctx.mask_weight, ctx.status = pitch, tuple(mask_weight), status
        ctx.mark_non_differentiable(out["x0_recon"], out["xtm1_recon"])
        return vb, kl_loss, out["x0_recon"], out["xtm1_recon"]

    @staticmethod
    def backward(ctx, g_vb, g_kl, _g0, _g1):
        rows, x0, x_t, t, pt, aux_w, coef_table = ctx.saved_tensors
        g_vb = torch.zeros_like(pt) if g_vb is None else g_vb
        if ctx.grad is not None and g_kl is None:
            grad, ctx.grad = ctx.grad, None  # consumed: a second backward would need retain_graph semantics anyway
            scale_rows(grad, (g_vb / ctx.grad_scale).float())
            return grad.permute(0, 2, 1).to(ctx.grad_dtype), None, None, None, None, None, None, None, None, None
        w_main = (g_vb / pt + (0 if g_kl is None else g_kl)).float().contiguous()
        w_aux = (g_vb * aux_w / pt).float().contiguous()
        out = _train_rows(rows, ctx.pitch, x0, x_t, t, coef_table, ctx.mask_weight, backward=1, w_main=w_main,
                          w_aux=w_aux, status=ctx.status)
        return out["grad"].permute(0, 2, 1).to(ctx.grad_dtype), None, None, None, None, None, None, None, None, None
