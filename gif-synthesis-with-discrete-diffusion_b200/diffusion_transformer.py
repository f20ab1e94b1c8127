"""`FusedDiffusionTransformer`: host-side mirror of the reference's `DiffusionTransformer`.

Same constructor keywords, same registered buffer / parameter names (so reference checkpoints load)
and the same sampling-time method signatures as
`src/models/motionencoder/diffusion_transformer.py` (reference file:line cited per method), with
the per-step mathematics executed by `libd3pm_b200.so`.  Select it through the Hydra `_target_` of
`configs/model/motionencoder/diffusion_transformer.yaml:1` (see INTEGRATION.md).

Tensors returned where the reference returns `[B, K+1, N]` are `[B, K+1, N]`-shaped strided views of
token-major storage; integer tokens, not log-one-hots, are carried between reverse steps inside
`sample()` (the reference arg-maxes its log-one-hot immediately, :221, :255, :639).
"""
from __future__ import annotations

from typing import Callable, List, Optional

import numpy as np
import torch
from torch import nn

from d3pm_b200 import _lib, attention, head, ops, train
from d3pm_b200._lib import D3PMError

_SCHEDULE_BUFFERS = ("log_at", "log_bt", "log_ct", "log_1_min_ct",
                     "log_cumprod_at", "log_cumprod_bt", "log_cumprod_ct", "log_1_min_cumprod_ct")


def alpha_schedule(time_step, N=100, att_1=0.99999, att_T=0.000009, ctt_1=0.000009, ctt_T=0.99999):
    """Mask-and-replace schedule, same signature and return order as the reference (:56-69).

    Returns `(at, bt, ct, att, btt, ctt)`: per-step keep / replace / mask probabilities (length T) and
    their cumulative versions (length T+1, last slot = the identity "t = -1").  The arithmetic keeps
    the reference's operation order so the float64 values, and hence the float32 buffers, are
    bit-identical (checked in tests/test_host.py against the golden-pinned oracle).
    """
    frac = np.arange(0, time_step) / (time_step - 1)
    keep_cum = np.concatenate(([1], frac * (att_T - att_1) + att_1))
    mask_cum = np.concatenate(([0], frac * (ctt_T - ctt_1) + ctt_1))
    at = keep_cum[1:] / keep_cum[:-1]
    not_masked = 1 - mask_cum
    ct = 1 - not_masked[1:] / not_masked[:-1]
    bt = (1 - at - ct) / N
    att = np.concatenate((keep_cum[1:], [1]))
    ctt = np.concatenate((mask_cum[1:], [0]))
    btt = (1 - att - ctt) / N
    return at, bt, ct, att, btt, ctt


class FusedDiffusionTransformer(nn.Module):
    """Drop-in for `DiffusionTransformer` (:71-164) whose reverse step runs as one CUDA kernel."""

    def __init__(
        self,
        *,
        condition_emb_config=None,
        transformer=None,
        diffusion_step=100,
        alpha_init_type="cos",
        auxiliary_loss_weight=0,
        adaptive_auxiliary_loss=False,
        mask_weight=[1, 1],
        learnable_cf=False,
        guidance_scale=5,
        content_seq_len=1024,
    ):
        super().__init__()
        self.condition_emb = None  # the reference never instantiates one either (:92-98)
        self.transformer = transformer
        self.content_seq_len = content_seq_len
        self.amp = False
        self.num_classes = self.transformer.content_emb.num_embed  # K + 1 (:106)
        self.loss_type = "vb_stochastic"
        self.shape = content_seq_len
        self.num_timesteps = diffusion_step
        self.parametrization = "x0"
        self.auxiliary_loss_weight = auxiliary_loss_weight
        self.adaptive_auxiliary_loss = adaptive_auxiliary_loss
        self.mask_weight = mask_weight
        if alpha_init_type != "alpha1":  # the reference prints and then dies on an undefined name (:115-120)
            raise ValueError("alpha_init_type must be 'alpha1' (the only schedule the reference defines)")

        at, bt, ct, att, btt, ctt = alpha_schedule(self.num_timesteps, N=self.num_classes - 1)
        with np.errstate(divide="ignore"):
            as64 = lambda a: torch.tensor(np.asarray(a, dtype="float64"))  # noqa: E731
            log_at, log_bt, log_ct = torch.log(as64(at)), torch.log(as64(bt)), torch.log(as64(ct))
            log_cumprod_at, log_cumprod_bt = torch.log(as64(att)), torch.log(as64(btt))
            log_cumprod_ct = torch.log(as64(ctt))
        log_1_min_ct = torch.log(1 - log_ct.exp() + 1e-40)                  # log_1_min_a (:29-30)
        log_1_min_cumprod_ct = torch.log(1 - log_cumprod_ct.exp() + 1e-40)
        for lhs, rhs in ((log_ct, log_1_min_ct), (log_cumprod_ct, log_1_min_cumprod_ct)):  # (:136-137)
            top = torch.max(lhs, rhs)
            total = top + torch.log(torch.exp(lhs - top) + torch.exp(rhs - top))
            assert total.abs().sum().item() < 1.0e-5

        self.diffusion_acc_list = [0] * self.num_timesteps
        self.diffusion_keep_list = [0] * self.num_timesteps
        self.register_buffer("log_at", log_at.float())
        self.register_buffer("log_bt", log_bt.float())
        self.register_buffer("log_ct", log_ct.float())
        self.register_buffer("log_cumprod_at", log_cumprod_at.float())
        self.register_buffer("log_cumprod_bt", log_cumprod_bt.float())
        self.register_buffer("log_cumprod_ct", log_cumprod_ct.float())
        self.register_buffer("log_1_min_ct", log_1_min_ct.float())
        self.register_buffer("log_1_min_cumprod_ct", log_1_min_cumprod_ct.float())
        self.register_buffer("Lt_history", torch.zeros(self.num_timesteps))
        self.register_buffer("Lt_count", torch.zeros(self.num_timesteps))
        self.zero_vector = None
        self.empty_text_embed = nn.Parameter(torch.randn(size=(77, 512), requires_grad=True, dtype=torch.float64))

        self.prior_rule = 0     # only rule 0 (VQ-Diffusion v1 Gumbel sampling) is reachable in the reference (:157)
        self.prior_ps = 1024
        self.prior_weight = 0
        self.update_n_sample()
        self.learnable_cf = learnable_cf
        self.guidance_scale = guidance_scale

        # --- state of the CUDA path (not part of the reference surface) ---
        # Noise: a counter-based Philox stream keyed by (rng_seed, rng_offset, global row, class).  The key is taken
        # from torch.initial_seed() HERE and later torch.manual_seed() calls do not re-key it: `manual_seed()` below is
        # the re-keying path, `rng_state()` / `set_rng_state()` carry it across a checkpoint (it is deliberately NOT in
        # state_dict(), whose key set stays the reference's so that checkpoints load strictly in both directions).
        self.rng_seed = int(torch.initial_seed()) & (2**63 - 1)
        self.rng_offset = 0          # advanced by one per sampling call: every call draws fresh noise
        # global index of local row 0 when the batch is sharded across ranks.  None = derive it per call from the
        # process group (rank * local rows: equal shards, the layout of `distributed.shard_range`), 0 without one.
        self.row_offset = None
        self.inject_uniform: Optional[Callable[[tuple, torch.device], torch.Tensor]] = None
        # tests inject the Exp(1) noise torch.multinomial draws inside the purity-prior branch (:340): (B, N) -> tensor
        self.inject_exponential: Optional[Callable[[tuple, torch.device], torch.Tensor]] = None
        self._coef_cache = None
        self._status = None
        # one denoiser pass serves both guidance branches when the two conditionings are bitwise equal (see _same_conditioning)
        self.share_identical_conditioning = True
        self._same_cond_cache = None
        # SURVEY §8 f3: fold the denoiser's `to_logits` head into the update kernel (see enable_fused_head)
        self.fuse_head = False
        self._head_cache = None
        self._head_scratch = None

    # ------------------------------------------------------------------ bookkeeping
    def update_n_sample(self):
        """Tokens to reveal per step for the purity prior (:166-179); only its length matters for rule 0."""
        T = self.num_timesteps
        few = self.prior_ps <= 10
        table = {
            100: [1, 6 if few else 10] + [11, 10, 10] * 32 + [11, 15 if few else 11],
            50: [10] + [21, 20] * 24 + [30],
            25: [21] + [41] * 23 + [60],
            10: [69] + [102] * 8 + [139],
            200: [1, 3] + [6, 6, 4, 4] * 49 + [6, 9],
        }
        if T in table:
            self.n_sample = table[T]

    @property
    def device(self):
        return self.log_at.device

    def manual_seed(self, seed: int, offset: int = 0):
        """Re-key the in-kernel Philox stream."""
        self.rng_seed, self.rng_offset = int(seed) & (2**63 - 1), int(offset)
        return self

    def rng_state(self) -> dict:
        """The noise key as a picklable dict (store it next to the checkpoint; `set_rng_state` resumes the stream)."""
        return {"rng_seed": self.rng_seed, "rng_offset": self.rng_offset}

    def set_rng_state(self, state: dict):
        self.rng_seed, self.rng_offset = int(state["rng_seed"]) & (2**63 - 1), int(state["rng_offset"])
        return self

    def _next_offset(self) -> int:
        off = self.rng_offset
        self.rng_offset += 1
        return off

    def _row_offset(self, local_rows: int) -> int:
        """Global index of this rank's first token row: ranks of a data-parallel job must not noise different videos
        with the same stream (the reference's per-process torch generators differ by seed_everything + rank)."""
        if self.row_offset is not None:
            return int(self.row_offset)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank() * int(local_rows)
        return 0

    def coef_table(self) -> torch.Tensor:
        """Device coefficient table derived from the *registered buffers* (so a loaded checkpoint's
        schedule is honoured); rebuilt when a buffer is replaced, moved or modified in place."""
        bufs = [getattr(self, n) for n in _SCHEDULE_BUFFERS]
        key = tuple((b.data_ptr(), b._version, str(b.device)) for b in bufs)
        if self._coef_cache is None or self._coef_cache[0] != key:
            T1 = self.num_timesteps + 1
            sched = torch.zeros(8, T1, dtype=torch.float32, device=self.device)
            for i, b in enumerate(bufs):
                sched[i, : b.numel()] = b
            self._coef_cache = (key, ops.build_coef_table(sched, self.num_timesteps, self.num_classes - 1))
        return self._coef_cache[1]

    def _status_word(self) -> torch.Tensor:
        if self._status is None or self._status.device != self.device:
            self._status = ops.new_status(self.device)
        return self._status

    def check_status(self):
        """One host sync: raise if any kernel since the last check saw an out-of-range t or token
        (the reference asserts these eagerly with `.item()` syncs, :45-46, :253)."""
        if self._status is None:
            return
        word = int(self._status.item())
        self._status.zero_()
        if word & _lib.STATUS_BAD_T:
            raise AssertionError("t outside [0, num_timesteps)")
        if word & _lib.STATUS_BAD_TOKEN:
            raise AssertionError(f"token index >= num_classes ({self.num_classes})")

    # ------------------------------------------------------------------ fused denoiser head (SURVEY §8 f3)
    def enable_fused_head(self, enable: bool = True):
        """Let `p_sample_tokens` / `sample` run the denoiser's prediction head `to_logits = LayerNorm + Linear`
        (transformer_utils.py:352-356, :441) inside the update kernel (`d3pm_head_step`), so the `[B, N, K]` logits
        never exist in memory.  Needs `transformer.to_logits` to be exactly that Sequential with n_embd = 64 and K in
        (1024, 2048, 4096); `fused_head_active` tells whether the weights also satisfy the kernel's no-clamp bound (if
        not, the step keeps using the unfused CUDA path, which is exact for any weights)."""
        if enable:
            self._head_weights()  # raises D3PMError on an unsupported head
            tr = self.transformer
            if not (callable(getattr(tr, "hidden_states", None)) or (hasattr(tr, "blocks") and callable(getattr(tr, "content_emb", None)))):
                raise D3PMError("enable_fused_head: the denoiser must either be the reference's Text2ImageTransformer "
                                "(content_emb + blocks + to_logits, transformer_utils.py:429-444) or offer "
                                "hidden_states(x_t, cond_emb, t) -> [B, N, n_embd], the input of its to_logits head")
        self.fuse_head = bool(enable)
        return self

    def enable_fused_attention(self, enable: bool = True, cross: bool = False):
        """Run the self-attention of the denoiser's blocks (`FullAttention`, transformer_utils.py:24-62) on
        `d3pm_self_attention`, which never forms the `[B, heads, N, N]` score matrix: `attention.fuse_self_attention` on
        the denoiser (raises `D3PMError` if it has no FullAttention of head width 4).  With `cross=True` the blocks'
        cross-attention over the condition tokens (`CrossAttention`) runs on `d3pm_cross_attention` as well
        (`attention.fuse_cross_attention`; its head-averaged map, the block's second output, is then None - the
        denoiser drops it).  Inference only - training, autocast and masked calls still run the reference's modules;
        `state_dict()` is unchanged.  Composes with `enable_fused_head()` and the one-pass shared conditioning.  After
        the call the self-attention is fused iff `enable` and the cross-attention iff `enable and cross`: `enable=False`
        restores the original modules of both kinds."""
        attention.fuse_self_attention(self.transformer, enable)
        attention.fuse_cross_attention(self.transformer, enable and cross)
        return self

    def _head_weights(self) -> "head.HeadWeights":
        tl = self.transformer.to_logits
        params = [q for q in (tl[0].weight, tl[0].bias, tl[-1].weight, tl[-1].bias) if q is not None]
        key = tuple((q.data_ptr(), q._version, str(q.device)) for q in params)
        if self._head_cache is None or self._head_cache[0] != key:
            self._head_cache = (key, head.HeadWeights.from_module(tl))
        return self._head_cache[1]

    @property
    def fused_head_active(self) -> bool:
        return bool(self.fuse_head) and self._head_weights().valid

    def _hidden_rows(self, x_t, cond_emb, t) -> torch.Tensor:
        """The denoiser up to (not including) its head: `[B, N, D]` hidden states, contiguous.

        Nothing is swapped or hooked (re-entrant, CUDA-graph / DDP safe): a denoiser that offers
        `hidden_states(x_t, cond_emb, t)` is asked directly; the reference's `Text2ImageTransformer` is walked exactly as
        its own `forward` does (transformer_utils.py:433-440: `content_emb`, then every block with the timestep), stopping
        before `to_logits` (:441)."""
        tr = self.transformer

        def run():
            if callable(getattr(tr, "hidden_states", None)):
                return tr.hidden_states(x_t, cond_emb, t)
            emb = tr.content_emb(x_t)
            for block in tr.blocks:
                emb, _ = block(emb, cond_emb, t)
            return emb

        if self.amp:
            with torch.autocast("cuda"):
                out = run()
        else:
            out = run()
        assert out.dim() == 3 and out.size(0) == x_t.size(0) and out.size(1) == x_t.size(1)
        return out.float().contiguous()

    # ------------------------------------------------------------------ helpers
    def _denoise_rows(self, x_t: torch.Tensor, cond_emb, t: torch.Tensor, keep_16bit: bool = False) -> torch.Tensor:
        """Run the denoiser (:222-230) and hand its logits over as token-major rows `[B, N, K]`.
        The reference transformer returns a `[B, K, N]` permuted view of `[B, N, K]`
        (transformer_utils.py:442-443), so this is normally zero-copy.  Under autocast the denoiser returns float16 /
        bfloat16 logits; `keep_16bit` hands them on as they are (the production step reads them in place and widens in
        registers: the same numbers as the `.float()` the reference's `out.double()` implies, :231, without the cast pass)."""
        if self.amp:
            with torch.autocast("cuda"):
                out = self.transformer(x_t, cond_emb, t)
        else:
            out = self.transformer(x_t, cond_emb, t)
        assert out.size(0) == x_t.size(0)
        assert out.size(1) == self.num_classes - 1
        assert out.size()[2:] == x_t.size()[1:]
        if not (keep_16bit and out.dtype in (torch.float16, torch.bfloat16)):
            out = out.float()
        got = ops.rows_of(out)
        if got is not None and got[1] % (16 // out.element_size()) == 0 and out.data_ptr() % 16 == 0:
            return got[0]
        return out.permute(0, 2, 1).contiguous()

    def _tokens_of(self, log_x: torch.Tensor) -> torch.Tensor:
        """log_onehot_to_index (:53-54) on any layout."""
        if log_x.dtype == torch.int64 and log_x.dim() == 2:
            return log_x.contiguous()
        return ops.argmax_classes(log_x.float())

    def _noise_rows(self, B: int, N: int):
        """Uniform noise rows when a test injects the reference's `rand_like` tensor, else None (Philox)."""
        if self.inject_uniform is None:
            return None
        u = self.inject_uniform((B, self.num_classes, N), self.device)
        return ops.to_rows(u.to(self.device, torch.float32))

    def _same_conditioning(self, cond_emb, cf_cond_emb) -> bool:
        """True when the conditional and the unconditional pass of this step are the SAME computation: the two embeddings
        are bitwise equal and the denoiser is deterministic (eval mode).  The reference's shipped pipeline is exactly that
        case - its caller zeroes both text embeddings (networks/discrete_diffusion.py:25, :49) - and it runs the denoiser
        twice per step on identical inputs (diffusion_transformer.py:240-245).  The drop-in then runs it ONCE and hands the
        same logits to the kernel as both tensors: bit-identical to two passes (y = lu + s (lc - lu) with lc == lu), half the
        denoiser time, and the second read of every row comes from L2.  The comparison costs one host sync, so its result
        is cached per pair of tensor versions: `sample()` passes the same two tensors at every step."""
        if not self.share_identical_conditioning or cond_emb is None or cf_cond_emb is None or self.transformer.training:
            return False
        if cond_emb is cf_cond_emb:
            return True
        if cond_emb.shape != cf_cond_emb.shape or cond_emb.dtype != cf_cond_emb.dtype or cond_emb.device != cf_cond_emb.device:
            return False
        key = (cond_emb.data_ptr(), cond_emb._version, cf_cond_emb.data_ptr(), cf_cond_emb._version, tuple(cond_emb.shape))
        if self._same_cond_cache is None or self._same_cond_cache[0] != key:
            self._same_cond_cache = (key, bool(torch.equal(cond_emb, cf_cond_emb)))
        return self._same_cond_cache[1]

    def _guidance_off(self) -> bool:
        # the reference's own |s-1|<1e-3 branch raises AttributeError (:242-243); "off" here means the
        # result of predict_start alone, which is what that branch was written to return
        return abs(self.guidance_scale - 1) < 1e-3

    def _step(self, x_t, cond_emb, cf_cond_emb, t, *, sample_mode, want_post=False, want_recon=False,
              want_gap=False, guidance=True, x_prev_out=None, thin_factor=0.0, sample_from=_lib.FROM_POSTERIOR,
              want_score=False, sharpen=None, logits=None):
        if logits is not None:  # reuse the logits of an earlier call of the same step (purity prior, second pass)
            return self._step_on(logits[0], logits[1], x_t, t, sample_mode=sample_mode, want_post=want_post,
                                 want_recon=want_recon, want_gap=want_gap, x_prev_out=x_prev_out, thin_factor=thin_factor,
                                 sample_from=sample_from, want_score=want_score, sharpen=sharpen)
        # 16-bit logits (autocast) stay 16-bit when the step is the plain production one: the stream kernel reads them in place
        keep16 = (sample_mode in (_lib.SAMPLE_PHILOX, _lib.SAMPLE_PHILOX_EXACT) and self.inject_uniform is None
                  and not (want_post or want_recon or want_gap or want_score) and sharpen is None
                  and sample_from == _lib.FROM_POSTERIOR and (self.num_classes - 1) in ops.STREAM_CODEBOOKS)
        logits_c = self._denoise_rows(x_t, cond_emb, t, keep16)
        logits_u = None
        if guidance and not self._guidance_off() and self._same_conditioning(cond_emb, cf_cond_emb):
            logits_u = logits_c  # the unconditional pass would recompute these very logits
        elif guidance and not self._guidance_off():
            logits_u = self._denoise_rows(x_t, cf_cond_emb.type_as(cond_emb) if cond_emb is not None else cf_cond_emb, t, keep16)
            if logits_u.dtype != logits_c.dtype:
                logits_c, logits_u = logits_c.float(), logits_u.float()
            if logits_u.stride() != logits_c.stride():
                logits_u = logits_u.contiguous()
                logits_c = logits_c.contiguous()
        out = self._step_on(logits_c, logits_u, x_t, t, sample_mode=sample_mode, want_post=want_post,
                            want_recon=want_recon, want_gap=want_gap, x_prev_out=x_prev_out, thin_factor=thin_factor,
                            sample_from=sample_from, want_score=want_score, sharpen=sharpen)
        out["_logits"] = (logits_c, logits_u)
        return out

    def _step_on(self, logits_c, logits_u, x_t, t, *, sample_mode, want_post=False, want_recon=False, want_gap=False,
                 x_prev_out=None, thin_factor=0.0, sample_from=_lib.FROM_POSTERIOR, want_score=False, sharpen=None):
        B, N = x_t.shape
        gumbel = None
        uniform_given = False
        if sample_mode in (_lib.SAMPLE_PHILOX, _lib.SAMPLE_PHILOX_EXACT):
            noise = self._noise_rows(B, N)
            if noise is not None:
                gumbel, uniform_given, sample_mode = noise[0], True, _lib.SAMPLE_GUMBEL
        return ops.fused_step(
            logits_c, logits_u, x_t, t.contiguous(), self.coef_table(), guidance_scale=self.guidance_scale,
            sample_mode=sample_mode, gumbel=gumbel, gumbel_is_uniform=uniform_given, seed=self.rng_seed,
            offset=self._next_offset() if sample_mode != _lib.SAMPLE_NONE else 0, row_offset=self._row_offset(B * N),
            want_post=want_post, want_recon=want_recon, want_gap=want_gap, status=self._status_word(),
            x_prev_out=x_prev_out, thin_factor=thin_factor, sample_from=sample_from, want_score=want_score,
            sharpen=sharpen)

    # ------------------------------------------------------------------ reference method surface
    @torch.no_grad()
    def predict_start(self, log_x_t, cond_emb, t):
        """p(x0 | x_t): float64-accurate log-softmax of the denoiser logits, -70 [MASK] row, clamp (:220-238)."""
        x_t = self._tokens_of(log_x_t)
        out = self._step(x_t, cond_emb, None, t, sample_mode=_lib.SAMPLE_NONE, want_recon=True, guidance=False)
        self.check_status()
        return ops.as_logical(out["recon"], self.num_classes)

    @torch.no_grad()
    def cf_predict_start(self, log_x_t, cond_emb, cf_cond_emb, t):
        """Classifier-free guidance combine + renormalise + clamp (:240-249)."""
        x_t = self._tokens_of(log_x_t)
        out = self._step(x_t, cond_emb, cf_cond_emb, t, sample_mode=_lib.SAMPLE_NONE, want_recon=True)
        self.check_status()
        return ops.as_logical(out["recon"], self.num_classes)

    def q_posterior(self, log_x_start, log_x_t, t):
        """p_theta(x_{t-1} | x_t) from an arbitrary log p(x0) (:251-283), forward only.

        The differentiable use inside `_train_loss` (:405) does not go through this method: the training loss and
        its gradient with respect to the logits are one kernel (`d3pm_train_rows`, `train.VBLoss`).  A direct call on
        a tensor that requires grad is therefore refused rather than silently returning a result without a graph."""
        if torch.is_grad_enabled() and log_x_start.requires_grad:
            raise NotImplementedError("q_posterior is forward-only here; the differentiable route is _train_loss / "
                                      "train.VBLoss (d3pm_train_rows).  Call under torch.no_grad() or detach log_x_start")
        x_t = self._tokens_of(log_x_t)
        rows, pitch = ops.to_rows(log_x_start.detach().float())
        post = ops.q_posterior_rows(rows, pitch, x_t, t.contiguous(), self.coef_table(), self.num_classes - 1,
                                    self._status_word())
        self.check_status()  # the reference asserts the token range right here (:253)
        return ops.as_logical(post, self.num_classes)

    @torch.no_grad()
    def p_pred(self, log_x, cond_emb, cf_cond_emb, t):
        """(:285-296) -> (log_model_pred, log_x_recon), both `[B, K+1, N]`."""
        if self.parametrization != "x0":
            raise ValueError
        x_t = self._tokens_of(log_x)
        out = self._step(x_t, cond_emb, cf_cond_emb, t, sample_mode=_lib.SAMPLE_NONE, want_post=True, want_recon=True)
        self.check_status()
        return ops.as_logical(out["post"], self.num_classes), ops.as_logical(out["recon"], self.num_classes)

    @torch.no_grad()
    def p_sample(self, log_x, cond_emb, cf_cond_emb, t, sampled, to_sample):
        """One reverse step (:304-352): returns (log one-hot of x_{t-1} `[B, K+1, N]`, `sampled`).

        `prior_rule == 0` (the only value the reference's constructor sets, :157): Gumbel draw from the posterior for
        every token, `sampled = [1024] * B`.  `prior_rule` 1 / 2 with `t[0] > 0`: the purity-prior reveal of Improved
        VQ-Diffusion (:309-346), see `p_sample_tokens_purity`."""
        x_t = self._tokens_of(log_x)
        if self.prior_rule > 0 and int(t[0]) > 0:  # the reference reads t[0] on the host as well (:309)
            x_prev, sampled = self.p_sample_tokens_purity(x_t, cond_emb, cf_cond_emb, t, sampled, to_sample)
        else:
            x_prev, sampled = self.p_sample_tokens(x_t, cond_emb, cf_cond_emb, t), [1024] * log_x.shape[0]
        out = ops.tokens_to_log_onehot_rows(x_prev, self.num_classes, self._status_word())
        self.check_status()  # one host read per public call, where the reference syncs several times (:45-46, :253)
        return ops.as_logical(out, self.num_classes), sampled

    @torch.no_grad()
    def p_sample_tokens_purity(self, x_t, cond_emb, cf_cond_emb, t, sampled, to_sample):
        """The `prior_rule` 1 / 2 branch of `p_sample` (:309-346) on integer tokens -> (x_{t-1} `[B, N]`, sampled).

        One fused pass gives every token a candidate x0 ~ p(x0 | x_t) (Gumbel-max on `log_x_recon`, :327-329) and its
        purity max_k p(x0 = k | x_t) (:318); `d3pm_purity_select` then reveals, per video, `n_sample` of the [MASK]
        positions drawn without replacement with probability proportional to the normalised purity (:331-341).  With
        `prior_weight > 0` (:321-325) the candidates are drawn from softmax((1 + purity * r) * log_x_recon) instead, which
        needs the per-video purity maximum first: a second pass over the same logits.  `sampled` advances exactly like
        the reference's list (one device->host read of B integers)."""
        B, N = x_t.shape
        K = self.num_classes - 1
        sharpened = self.prior_rule != 1 and self.prior_weight > 0
        # the thinned Philox race draws the same candidate as exhaustive scoring (tests) at a fifth of the cost; with
        # injected noise `_step_on` switches to the Gumbel mode by itself
        first = self._step(x_t, cond_emb, cf_cond_emb, t, sample_mode=_lib.SAMPLE_NONE if sharpened else _lib.SAMPLE_PHILOX,
                           sample_from=_lib.FROM_RECON, want_score=True)
        score = first["score"]
        if sharpened:
            norm = score / (score.max(dim=1, keepdim=True).values + 1e-10)         # (:319)
            f = (1 + norm * self.prior_weight).float().contiguous()                 # (:323)
            cand = self._step(x_t, None, None, t, sample_mode=_lib.SAMPLE_PHILOX_EXACT, sample_from=_lib.FROM_RECON,
                              sharpen=f, logits=first["_logits"])["x_prev"]
        else:
            cand = first["x_prev"]
        n_reveal = []
        for i in range(B):                                                           # (:331-336)
            n = min(to_sample - sampled[i], self.prior_ps)
            if to_sample - sampled[i] - n == 1:
                n = to_sample - sampled[i]
            n_reveal.append(max(int(n), 0))
        expo = None
        if self.inject_exponential is not None:
            expo = self.inject_exponential((B, N), self.device).to(self.device, torch.float32).contiguous()
        x_out, revealed = ops.purity_select(
            x_t, cand, None if self.prior_rule == 1 else score, torch.tensor(n_reveal, dtype=torch.int32, device=self.device),
            K, expo=expo, seed=self.rng_seed, offset=self._next_offset(), row_offset=self._row_offset(B * N))
        sampled = [int(s) + int(r) for s, r in zip(sampled, revealed.tolist())]     # (:342-343)
        return x_out, sampled

    @torch.no_grad()
    def p_sample_tokens(self, x_t, cond_emb, cf_cond_emb, t, x_prev_out=None):
        """The same step on integer tokens: int64 `[B, N]` in, int64 `[B, N]` out (fast path of `sample`)."""
        if self.fuse_head and self.inject_uniform is None and self._head_weights().valid:
            hw = self._head_weights()
            hidden_c = self._hidden_rows(x_t, cond_emb, t)
            hidden_u = None
            if not self._guidance_off() and self._same_conditioning(cond_emb, cf_cond_emb):
                hidden_u = hidden_c
            elif not self._guidance_off():
                hidden_u = self._hidden_rows(x_t, cf_cond_emb.type_as(cond_emb) if cond_emb is not None else cf_cond_emb, t)
            B, N = x_t.shape
            if self._head_scratch is None or self._head_scratch[0].numel() != B * N or self._head_scratch[0].device != x_t.device:
                self._head_scratch = head.head_scratch(B, N, x_t.device)
            return head.head_step(hw, hidden_c, hidden_u, x_t, t.contiguous(), self.coef_table(),
                                  guidance_scale=self.guidance_scale, seed=self.rng_seed, offset=self._next_offset(),
                                  row_offset=self._row_offset(B * N), status=self._status_word(), x_prev_out=x_prev_out,
                                  scratch=self._head_scratch)
        out = self._step(x_t, cond_emb, cf_cond_emb, t, sample_mode=_lib.SAMPLE_PHILOX, x_prev_out=x_prev_out)
        return out["x_prev"]

    @torch.no_grad()
    def log_sample_categorical(self, logits):
        """Gumbel-max draw over dim 1 of `[B, C, N]` log-probs, returned as a log one-hot (:354-359)."""
        B, C, N = logits.shape
        rows, pitch = ops.to_rows(logits.float())
        noise = self._noise_rows(B, N) if C == self.num_classes else None
        if noise is not None:
            x = ops.gumbel_argmax_rows(rows, pitch, C, noise_rows=noise[0], pitch_noise=noise[1], noise_kind=1)
        else:
            x = ops.gumbel_argmax_rows(rows, pitch, C, noise_kind=2, seed=self.rng_seed, offset=self._next_offset(),
                                       row_offset=self._row_offset(B * N))
        return ops.as_logical(ops.tokens_to_log_onehot_rows(x, C, self._status_word()), C)

    @torch.no_grad()
    def sample(
        self,
        condition_token,
        condition_mask,
        condition_embed,
        cf_condition_embed,
        content_token=None,
        filter_ratio=0.5,
        temperature=1.0,
        return_att_weight=False,
        return_logits=False,
        content_logits=None,
        print_log=True,
        **kwargs,
    ):
        """Full reverse chain from the all-[MASK] state (:568-644) -> {'content_token': int64 [B, N]}.

        `filter_ratio > 0` (start from a noised `content_token`) calls `p_sample` with a stale
        signature in the reference and raises there (:628-636); it is refused here too."""
        if condition_token is not None:
            batch_size = len(condition_token)
        else:
            batch_size = kwargs["batch_size"]
        device = self.log_at.device
        start_step = int(self.num_timesteps * filter_ratio)
        if start_step != 0:
            raise NotImplementedError("sample(filter_ratio > 0) is unreachable in the reference (:628-636)")
        if condition_embed is None or cf_condition_embed is None:
            raise ValueError("condition_embed and cf_condition_embed are required (the reference leaves "
                             "cf_cond_emb undefined otherwise, :607-611)")
        cond_emb = condition_embed.float()
        cf_cond_emb = cf_condition_embed.float()

        N, K = self.shape, self.num_classes - 1
        self._status_word().zero_()  # a stale bit of an earlier, unchecked call must not fail this chain (no sync)
        x = torch.full((batch_size, N), K, dtype=torch.int64, device=device)  # all [MASK] (:615-618)
        x_next = torch.empty_like(x)
        for diffusion_index in range(self.num_timesteps - 1, -1, -1):
            t = torch.full((batch_size,), diffusion_index, device=device, dtype=torch.long)
            if self.prior_rule > 0 and diffusion_index > 0:
                # purity prior: reveal n_sample[t] tokens per video, repeating the step until every video got them (:623-626)
                sampled = [0] * batch_size
                while min(sampled) < self.n_sample[diffusion_index]:
                    x, sampled = self.p_sample_tokens_purity(x, cond_emb, cf_cond_emb, t, sampled,
                                                             self.n_sample[diffusion_index])
                continue
            # with prior_rule == 0 the reference's `while min(sampled) < n_sample[...]` body runs once (:624-626)
            self.p_sample_tokens(x, cond_emb, cf_cond_emb, t, x_prev_out=x_next)
            x, x_next = x_next, x
        self.check_status()
        output = {"content_token": x}
        if return_logits:
            log_z = ops.as_logical(ops.tokens_to_log_onehot_rows(x, self.num_classes), self.num_classes)
            output["logits"] = torch.exp(log_z)
        return output

    # ------------------------------------------------------------------ training side (SURVEY §8 f1)
    def _sched8(self) -> torch.Tensor:
        """The eight schedule buffers as one `[8, T+1]` device matrix (cached like the coefficient table)."""
        self.coef_table()
        key = self._coef_cache[0]
        if getattr(self, "_sched_cache", None) is None or self._sched_cache[0] != key:
            sched = torch.zeros(8, self.num_timesteps + 1, dtype=torch.float32, device=self.device)
            for i, n in enumerate(_SCHEDULE_BUFFERS):
                b = getattr(self, n)
                sched[i, : b.numel()] = b
            self._sched_cache = (key, sched)
        return self._sched_cache[1]

    @torch.no_grad()
    def q_pred(self, log_x_start, t):
        """q(x_t | x_0) in log space, t wrapped modulo T+1 (:201-218)."""
        rows, pitch = ops.to_rows(log_x_start.float())
        out = train.q_pred_rows(rows, pitch, t, self._sched8(), self.num_classes - 1, cumulative=True)
        return ops.as_logical(out, self.num_classes)

    @torch.no_grad()
    def q_pred_one_timestep(self, log_x_t, t):
        """q(x_t | x_{t-1}) in log space (:185-199)."""
        rows, pitch = ops.to_rows(log_x_t.float())
        out = train.q_pred_rows(rows, pitch, t, self._sched8(), self.num_classes - 1, cumulative=False)
        return ops.as_logical(out, self.num_classes)

    @torch.no_grad()
    def q_sample(self, log_x_start, t):
        """Forward noising draw x_t ~ q(x_t | x_0), returned as a log one-hot (:361-366)."""
        return self.log_sample_categorical(self.q_pred(log_x_start, t))

    @torch.no_grad()
    def q_sample_tokens(self, x_start, t):
        """The same on integer tokens: int64 `[B, N]` -> int64 `[B, N]`."""
        C = self.num_classes
        B, N = x_start.shape
        noise = self._noise_rows(B, N)
        if noise is None and (C - 1) % 4 == 0 and C - 1 <= 8192:
            # own noise: one kernel, none of the three [B, K+1, N] tensors (same tokens as the route below, tested)
            return train.q_sample_tokens(x_start, t, self._sched8(), C - 1, seed=self.rng_seed, offset=self._next_offset(),
                                         row_offset=self._row_offset(B * N), status=self._status_word())
        hot = ops.tokens_to_log_onehot_rows(x_start.contiguous(), C, self._status_word())
        qrows = train.q_pred_rows(hot, hot.shape[2], t, self._sched8(), C - 1, cumulative=True)
        if noise is not None:
            return ops.gumbel_argmax_rows(qrows, qrows.shape[2], C, noise_rows=noise[0], pitch_noise=noise[1], noise_kind=1)
        return ops.gumbel_argmax_rows(qrows, qrows.shape[2], C, noise_kind=2, seed=self.rng_seed,
                                      offset=self._next_offset(), row_offset=self._row_offset(B * N))

    def sample_time(self, b, device, method="uniform"):
        """Timestep sampler (:368-389): importance sampling on the running loss history once every step has
        been visited more than 10 times, uniform before that.  T-sized host-side logic, plain torch."""
        if method == "importance":
            if not (self.Lt_count > 10).all():
                return self.sample_time(b, device, method="uniform")
            Lt_sqrt = torch.sqrt(self.Lt_history + 1e-10) + 0.0001
            Lt_sqrt[0] = Lt_sqrt[1]  # overwrite the decoder term with L1
            pt_all = Lt_sqrt / Lt_sqrt.sum()
            t = torch.multinomial(pt_all, num_samples=b, replacement=True)
            return t, pt_all.gather(dim=0, index=t)
        if method == "uniform":
            t = torch.randint(0, self.num_timesteps, (b,), device=device).long()
            return t, torch.ones_like(t).float() / self.num_timesteps
        raise ValueError

    def _train_loss(self, x, cond_emb, is_train=True, need_log_model_prob=True):
        """The variational-bound loss (:391-457) -> (log_model_prob, vb_loss [B], x0_recon [B, N]).

        One denoiser forward, then `d3pm_train_rows` (forward) under autograd; its backward is the same kernel in
        gradient mode.  `log_model_prob` `[B, K+1, N]` is only materialised when asked for (the reference's
        `forward` exponentiates it for `out['logits']`)."""
        b, device = x.size(0), x.device
        assert self.loss_type == "vb_stochastic"
        x_start = x.contiguous()
        t, pt = self.sample_time(b, device, "importance")
        xt = self.q_sample_tokens(x_start, t)

        if self.amp:
            with torch.autocast("cuda"):
                out = self.transformer(xt, cond_emb, t)
        else:
            out = self.transformer(xt, cond_emb, t)
        assert out.size(0) == xt.size(0) and out.size(1) == self.num_classes - 1 and out.size()[2:] == xt.size()[1:]
        if out.dtype not in (torch.float16, torch.bfloat16):
            out = out.float()  # 16-bit logits (autocast) go to the loss kernel as they are; their gradient comes back 16-bit

        aux_on = self.auxiliary_loss_weight != 0 and is_train
        if aux_on:
            extra = (1 - t / self.num_timesteps) + 1.0 if self.adaptive_auxiliary_loss else torch.ones_like(pt)
            aux_w = (extra * self.auxiliary_loss_weight).float()
        else:
            aux_w = torch.zeros_like(pt)
        # d(final loss) / d(vb_loss[b]) as the caller will apply it (`forward` divides the sum by B N, :546): lets the
        # kernel write the final gradient in the same pass as the loss
        grad_scale, self._loss_grad_scale = getattr(self, "_loss_grad_scale", 1.0), 1.0
        vb_loss, kl_loss, x0_recon, xt_1_recon = train.VBLoss.apply(
            out, x_start, xt, t, pt.float(), aux_w, self.coef_table(), tuple(self.mask_weight), self._status_word(),
            grad_scale)

        # running accuracy lists (:407-417): one device->host copy instead of 2B `.item()` syncs
        with torch.no_grad():
            acc = (x0_recon == x_start).float().mean(1)
            keep = (xt_1_recon == xt).float().mean(1)
            self.check_status()  # out-of-range tokens / timesteps: the reference asserts (:45-46, :253); free next to .tolist()
            for this_t, a_, k_ in zip(t.tolist(), acc.tolist(), keep.tolist()):
                self.diffusion_acc_list[this_t] = a_ * 0.1 + self.diffusion_acc_list[this_t] * 0.9
                self.diffusion_keep_list[this_t] = k_ * 0.1 + self.diffusion_keep_list[this_t] * 0.9
            # loss history for the importance sampler (:434-438)
            Lt2 = kl_loss.detach().pow(2)
            Lt2_prev = self.Lt_history.gather(dim=0, index=t)
            self.Lt_history.scatter_(dim=0, index=t, src=(0.1 * Lt2 + 0.9 * Lt2_prev))
            self.Lt_count.scatter_add_(dim=0, index=t, src=torch.ones_like(Lt2))

        log_model_prob = None
        if need_log_model_prob:
            with torch.no_grad():
                rows, _ = train._logit_rows(out.detach().float())  # the row kernel that writes `post` reads fp32
                post = ops.fused_step(rows, None, xt, t.contiguous(), self.coef_table(), guidance_scale=1.0,
                                      sample_mode=_lib.SAMPLE_NONE, want_post=True, status=self._status_word())["post"]
                log_model_prob = ops.as_logical(post, self.num_classes)
        return log_model_prob, vb_loss, x0_recon

    def forward(self, input, return_loss=False, return_logits=True, return_att_weight=False, is_train=True, **kwargs):
        """Training entry point (:520-565): {'loss', 'logits', 'pred_data'} for a batch of clean tokens."""
        if kwargs.get("autocast") is True:
            self.amp = True
        sample_image = input["content_token"].type_as(input["content_token"])
        if input.get("condition_embed_token") is None:
            cond_emb = None
        else:
            cond_emb = input["condition_embed_token"].float()
        if not is_train:
            raise NotImplementedError("forward(is_train=False) leaves every output undefined in the reference (:552-565)")
        self._loss_grad_scale = 1.0 / (sample_image.size()[0] * sample_image.size()[1])
        log_model_prob, loss, sample_image_recon = self._train_loss(sample_image, cond_emb,
                                                                    need_log_model_prob=return_logits)
        loss = loss.sum() / (sample_image.size()[0] * sample_image.size()[1])
        out = {}
        if return_logits:
            out["logits"] = torch.exp(log_model_prob)
        if return_loss:
            out["loss"] = loss
        self.amp = False
        out["pred_data"] = sample_image_recon
        return out
