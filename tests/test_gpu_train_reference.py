"""The training loss kernels (`d3pm_train_rows`: the persistent stream kernel at >= 2048 rows and K in {1024, 2048, 4096},
the one-CTA-per-row kernel otherwise) against a float64 restatement of `oracle.train_loss`, row by row, on rows built to
reach each special case of the kernels; and both persistent kernels past the 256 timesteps whose coefficients they stage
in shared memory.  Needs a B200."""
import ctypes

import numpy as np
import pytest
import torch

import d3pm_b200
from d3pm_b200 import _lib, ops, train
from oracle import d3pm_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CHUNK = 1024  # rows per float64 reference pass

# Tolerances.  The fp32 comparisons of test_gpu_train.py (kernel against the fp32 oracle) allow 2e-5 relative on losses
# and 5e-5 relative on gradients.  Against float64 the kernels do much better; each bound below is about 4x the largest
# error observed over every case of this file (both kernels, every K) on a B200 at 1000 W.
TOK_REL = 1.5e-6   # per-token losses, relative part: observed 4.0e-7 (row kernel, K = 8), 3.3e-7 (stream, K = 4096)
TOK_ABS = 4e-6     # per-token losses, absolute part, for losses below 1: observed 9.6e-7 (row kernel, K = 8), 3.6e-7 (stream)
GRAD_REL = 1.5e-6  # gradient, relative to the row's own scale (_grad_row_error): observed 3.8e-7 (stream, K = 4096)
# x_{t-1} arg-max: rows whose two best float64 posterior log-probs are closer than this may swap in fp32.  The kernels'
# log-probs are within H.POST_TOL (1e-4) of the reference, so two classes closer than twice that are not ordered.
# Observed: at most 2 of 16384 rows that close, and no row differed.
NEAR_GAP = 2 * H.POST_TOL
NEAR_MAX_FRACTION = 1e-3


# --------------------------------------------------------------------------- float64 reference
def _log_onehot(x, num_classes, dtype):
    """`O.index_to_log_onehot` in `dtype` on x's device (the oracle casts to float32)."""
    hot = torch.nn.functional.one_hot(x, num_classes).to(dtype)
    return torch.log(hot.clamp(min=1e-30)).permute(0, 2, 1)


def _predict_start(logits, dtype):
    """`O.predict_start_from_logits` in `dtype` (the oracle rounds the log-softmax to float32)."""
    B, K, N = logits.shape
    lp = torch.log_softmax(logits.to(dtype), dim=1)
    floor_row = torch.full((B, 1, N), O.CLAMP_LO, dtype=dtype, device=logits.device)
    return torch.clamp(torch.cat((lp, floor_row), dim=1), O.CLAMP_LO, 0)


def _reference_chunk(sched, logits, x0, x_t, t, mask_weight, w_main, w_aux):
    """`oracle.train_loss` for R independent rows (each its own video of one token), float64 on the rows' device:
    -> tok_main, tok_aux, x0_recon, xtm1_recon, the top-2 gap of the posterior and d(w_main tok_main + w_aux tok_aux)/d logits."""
    R, K = logits.shape
    C = K + 1
    dt = torch.float64
    lg = logits.to(dt).unsqueeze(2).detach().requires_grad_(True)           # [R, K, 1]
    with torch.device(logits.device):  # the oracle's q_posterior allocates its constants on the default device
        log_x_start = _log_onehot(x0.unsqueeze(1), C, dt)
        log_xt = _log_onehot(x_t.unsqueeze(1), C, dt)
        log_x0_recon = _predict_start(lg, dt)
        log_model_prob = O.q_posterior(sched, log_x0_recon, log_xt, t)
        log_true_prob = O.q_posterior(sched, log_x_start, log_xt, t)
    kl = O.multinomial_kl(log_true_prob, log_model_prob)[:, 0]
    mask_region = (x_t == K).to(dt)
    w = mask_region * mask_weight[0] + (1.0 - mask_region) * mask_weight[1]
    decoder_nll = -(log_x_start.exp() * log_model_prob).sum(dim=1)[:, 0]
    kl_aux = O.multinomial_kl(log_x_start[:, :-1, :], log_x0_recon[:, :-1, :])[:, 0]
    at_zero = (t == 0).to(dt)
    tok_main = at_zero * decoder_nll + (1.0 - at_zero) * kl * w
    tok_aux = at_zero * decoder_nll + (1.0 - at_zero) * kl_aux * w
    (w_main.to(dt) * tok_main + w_aux.to(dt) * tok_aux).sum().backward()
    lmp = log_model_prob.detach()[:, :, 0]
    top2 = lmp.topk(2, dim=1).values
    return dict(tok_main=tok_main.detach(), tok_aux=tok_aux.detach(), x0_recon=log_x0_recon.detach()[:, :, 0].argmax(1),
                xtm1_recon=lmp.argmax(1), gap=top2[:, 0] - top2[:, 1], grad=lg.grad[:, :, 0])


def reference_rows(sched, logits, x0, x_t, t_row, mask_weight, w_row_main, w_row_aux):
    """The reference for token rows `logits [R, K]` (float32), `x0`, `x_t`, `t_row`, per-row weights `[R]`, in chunks of
    CHUNK rows on the logits' device.  `sched`: the float32 schedule the coefficient table is built from."""
    s64 = {k: v.to(device=logits.device, dtype=torch.float64) for k, v in sched.items()}
    parts = [_reference_chunk(s64, logits[a:a + CHUNK], x0[a:a + CHUNK], x_t[a:a + CHUNK], t_row[a:a + CHUNK], mask_weight,
                              w_row_main[a:a + CHUNK], w_row_aux[a:a + CHUNK]) for a in range(0, logits.shape[0], CHUNK)]
    return {k: torch.cat([p[k] for p in parts]) for k in parts[0]}


@pytest.mark.parametrize("K,aux,mask_weight,seed", [(64, 1e-3, (1, 1), 11), (4096, 5e-4, (0.3, 2.0), 12)])
def test_reference_matches_the_oracle(K, aux, mask_weight, seed):
    """The float64 restatement against `oracle.train_loss` (fp32, autograd) on the CPU, at the bounds of
    test_train_loss_and_gradient_against_oracle: the per-video loss and the gradient of the mean loss."""
    T, B, N = 100, 4, 6
    sched = O.make_schedule(T, K)
    rows = _make_rows(B, N, K, T, [0, 1, 37, 99], seed, "cpu")
    logits = rows["logits"].view(B, N, K)
    u = torch.rand(B, K + 1, N, generator=torch.Generator().manual_seed(seed))
    t = torch.tensor([0, 1, 37, 99])
    pt = torch.rand(B, generator=torch.Generator().manual_seed(seed + 1)) * 0.02 + 0.001
    ref_logits = logits.clone().requires_grad_(True)
    _, vb_o, x0r_o, xt_o, _ = O.train_loss(sched, ref_logits.permute(0, 2, 1), rows["x0"].view(B, N), t, pt, u,
                                          auxiliary_loss_weight=aux, adaptive_auxiliary_loss=True, mask_weight=mask_weight)
    (vb_o.sum() / (B * N)).backward()
    aux_w = ((1 - t / T) + 1.0) * aux
    w_main, w_aux = (1.0 / (B * N * pt)).double(), (aux_w / (B * N * pt)).double()
    rep = lambda v: v.repeat_interleave(N)  # noqa: E731  (per video -> per row)
    ref = reference_rows(sched, logits.reshape(-1, K), rows["x0"], xt_o.reshape(-1), rep(t), mask_weight, rep(w_main), rep(w_aux))
    vb = (ref["tok_main"].view(B, N).sum(1) + aux_w.double() * ref["tok_aux"].view(B, N).sum(1)) / pt.double()
    assert (vb - vb_o.double()).abs().max() <= 2e-5 * vb_o.abs().max()
    assert torch.equal(ref["x0_recon"].view(B, N), x0r_o)
    gw = ref_logits.grad.double().reshape(-1, K)
    assert (ref["grad"] - gw).abs().max() <= 5e-5 * gw.abs().max() + 1e-8


# --------------------------------------------------------------------------- rows that reach each branch
MASKED, KEPT, OTHER, RUNNER_FAST, RUNNER_GENERAL, WIDE, SPIKE, EDGE, TIE = range(9)
N_KINDS = 9


def _make_rows(B, N, K, T, tvals, seed, device, groups=None):
    """Token rows of every kind, interleaved.  `groups` = the stream kernel's group count G (one launch runs rows
    g, g + G, g + 2G, ... on group g, alternating its two ring slots): the kind of row r is then (r // G // 2 + r % G) mod
    N_KINDS, so every group sees every kind in both slots once it runs 2 N_KINDS rows.  Row kinds:
    MASKED       x_t = [MASK]
    KEPT         x_t = x0
    OTHER        x_t != x0, both codes
    RUNNER_FAST  x_t = the logits' arg-max with a margin >= 0.5, x0 elsewhere (runner-up search without clamps)
    RUNNER_GENERAL  the same with one class 90 below the rest (its recon clamp fires: general path, rescoring)
    WIDE         logits spread over 110 (> 70 - ln K: recon clamps fire for the lowest classes), masked and unmasked
    SPIKE        one class +200 (x0, x_t or another class): p_x0 and posterior clamps on both sides
    EDGE         x0 / x_t at classes 0, K - 1, 4 GT - 1, 4 GT (GT = K / 32: the first / last thread of a group, chunk ends)
    TIE          two or three exactly equal maxima away from x0 and x_t (lowest-index rule across threads, warps, CTAs)"""
    R = B * N
    rng = np.random.default_rng(seed)
    gen = torch.Generator(device=device).manual_seed(seed)
    logits = torch.randn(R, K, generator=gen, device=device)
    r = np.arange(R)
    kind = (r // groups // 2 + r % groups) % N_KINDS if groups else r % N_KINDS
    x0 = rng.integers(0, K, R)
    other = (x0 + 1 + rng.integers(0, K - 1, R)) % K     # a code != x0
    x_t = np.where(kind == MASKED, K, np.where(kind == KEPT, x0, other))
    gt = max(K // 32, 1)
    edges = np.array(sorted({c for c in (0, K - 1, 4 * gt - 1, 4 * gt) if 0 <= c < K}))

    sel = np.flatnonzero(kind == WIDE)
    x_t[sel] = np.where(sel % 2 == 0, K, x_t[sel])
    if len(sel):
        rows_ = logits[sel]
        lo, hi = rows_.min(1, keepdim=True).values, rows_.max(1, keepdim=True).values
        logits[sel] = (rows_ - lo) * (110.0 / (hi - lo)) - 55.0

    sel = np.flatnonzero(kind == EDGE)
    a = sel % len(edges)
    b = (sel // len(edges)) % (len(edges) + 1)
    x0[sel] = edges[a]
    x_t[sel] = np.where(b < len(edges), edges[np.minimum(b, len(edges) - 1)], K)

    sel = np.flatnonzero(kind == SPIKE)
    mode = sel % 4                                        # x_t = x0, [MASK], another code, another code
    x_t[sel] = np.where(mode == 0, x0[sel], np.where(mode == 1, K, other[sel]))
    target = (sel // 4) % 3                               # spike at x0, at x_t (x0 when masked), elsewhere
    spike = np.where(target == 0, x0[sel], np.where(target == 1, np.where(x_t[sel] == K, x0[sel], x_t[sel]),
                                                    rng.integers(0, K, len(sel))))
    idx = torch.as_tensor(sel, device=device)
    logits[idx, torch.as_tensor(spike, device=device)] += 200.0

    for kd in (RUNNER_FAST, RUNNER_GENERAL):
        sel = np.flatnonzero(kind == kd)
        if not len(sel):
            continue
        idx = torch.as_tensor(sel, device=device)
        j = torch.as_tensor(x_t[sel], device=device)      # OTHER-like: a code != x0
        top = logits[idx].max(1).values
        logits[idx, j] = top + 0.5 + torch.rand(len(sel), generator=gen, device=device)
        if kd == RUNNER_GENERAL:
            low = (x_t[sel] + 1 + rng.integers(0, K - 1, len(sel))) % K
            low = np.where(low == x0[sel], (low + 1) % K, low)
            low = np.where(low == x_t[sel], (low + 1) % K, low)
            logits[idx, torch.as_tensor(low, device=device)] = logits[idx].min(1).values - 90.0

    sel = np.flatnonzero(kind == TIE)
    x_t[sel] = np.where(sel % 3 == 0, K, x_t[sel])
    tops = (logits[torch.as_tensor(sel, device=device)].max(1).values + 1.0).tolist() if len(sel) else []
    for n, row in enumerate(sel):
        want = 2 + row % 2
        fixed = [4 * gt - 4, 4 * gt, K - 1][:want] if K >= 8 and (row // 2) % 3 == 0 else []
        avoid = {int(x0[row]), int(x_t[row])}
        cls = [c for c in fixed if 0 <= c < K and c not in avoid]
        while len(cls) < want:
            c = int(rng.integers(0, K))
            if c not in avoid and c not in cls:
                cls.append(c)
        logits[row, cls] = tops[n]                        # one fp32 value: an exact tie

    t_row = np.repeat(np.asarray(tvals), N)
    return dict(logits=logits, x0=torch.as_tensor(x0, device=device), x_t=torch.as_tensor(x_t, device=device),
                t=torch.as_tensor(np.asarray(tvals), device=device), t_row=torch.as_tensor(t_row, device=device),
                kind=torch.as_tensor(kind, device=device))


def _video_weights(B, seed):
    g = torch.Generator().manual_seed(seed)
    w_main = torch.rand(B, generator=g) * 2.0 + 0.05
    w_aux = torch.rand(B, generator=g) * 0.5
    w_main[B // 2] = 0.0  # a video whose gradient is its auxiliary term alone, and one without the auxiliary term
    w_aux[1] = 0.0
    return w_main.to(DEV), w_aux.to(DEV)


def _stream_groups(K):
    return torch.cuda.get_device_properties(DEV).multi_processor_count * (512 // (K // 32))


def _tvals(B, T):
    base = [0, 1, 2, 37, T - 2, T - 1]
    return (base * (B // len(base) + 1))[:B] if B >= len(base) else base[:B]


# --------------------------------------------------------------------------- comparisons
def _check(name, got, ref, rows, N, mask_weight, w_main, w_aux, stats):
    """Kernel outputs `got` (backward = 2 with both arg-maxes) against the reference `ref`, every row."""
    K = rows["logits"].shape[1]
    assert torch.equal(got["x0_recon"].reshape(-1), torch.argmax(rows["logits"], dim=1)), f"{name}: x0_recon"
    assert torch.equal(ref["x0_recon"], got["x0_recon"].reshape(-1)), f"{name}: x0_recon vs reference"
    near = (ref["gap"] > 0) & (ref["gap"] < NEAR_GAP)   # exact float64 ties are compared: lowest index
    diff = got["xtm1_recon"].reshape(-1) != ref["xtm1_recon"]
    runner = (rows["kind"] == RUNNER_FAST) | (rows["kind"] == RUNNER_GENERAL)
    n_near = int(near.sum())
    print(f"[{name}] x_t-1 arg-max: {n_near} of {near.numel()} rows excluded as near-ties (gap < {NEAR_GAP:g}), "
          f"{int((diff & near).sum())} of them differ")
    assert not (near & runner).any(), f"{name}: a built arg-max row is a near-tie"
    assert not (diff & ~near).any(), f"{name}: {int((diff & ~near).sum())} x_t-1 arg-maxes differ away from near-ties"
    assert n_near <= NEAR_MAX_FRACTION * near.numel(), f"{name}: {n_near} near-ties"
    for q in ("tok_main", "tok_aux"):
        g, w = got[q].reshape(-1).double(), ref[q]
        err = (g - w).abs()
        small = w.abs() < 1
        stats.setdefault((q, "abs", K), []).append(float(err[small].max()) if small.any() else 0.0)
        stats.setdefault((q, "rel", K), []).append(float((err[~small] / w[~small].abs()).max()) if (~small).any() else 0.0)
        assert (err <= TOK_REL * w.abs() + TOK_ABS).all(), f"{name}: {q} max err {float(err.max()):.3e}"
    weight = _row_weight(rows["x_t"], rows["t_row"], K, mask_weight, w_main.repeat_interleave(N), w_aux.repeat_interleave(N))
    rel = _grad_row_error(got["grad"].reshape(-1, K), ref["grad"], weight, name)
    stats.setdefault(("grad", "rel", K), []).append(float(rel.max()))
    worst = int(torch.argmax(rel))
    assert float(rel.max()) <= GRAD_REL, (f"{name}: gradient row error {float(rel.max()):.3e} of the row's scale "
                                          f"(row kind {int(rows['kind'][worst])}, t {int(rows['t_row'][worst])})")


def _row_weight(x_t, t_row, K, mask_weight, w_main, w_aux):
    """The weight of each row's loss terms in the gradient: (|w_main| + |w_aux|) times the mask weight, or without it at t = 0
    (the NLL is not mask-weighted).  A row's gradient is a softmax-weighted sum of its loss terms' derivatives with respect
    to its log-probabilities, which are at most of this size; where they nearly cancel (a confident row that is right, a
    row whose x0 class is clamped), the fp32 kernel keeps ~1e-7 of the terms, not of their sum."""
    wtok = torch.where(x_t == K, float(mask_weight[0]), float(mask_weight[1])).double()
    w = w_main.double().abs() + w_aux.double().abs()
    return torch.where(t_row == 0, w, w * wtok)


def _grad_row_error(got, want, weight, name):
    """max |got - want| of each row over that row's own scale: the larger of max |want| and its loss weight `weight`.
    Neither the other rows nor their weights enter, so rows at t = 0 and rows of small weight are held to their own size."""
    err = (got.double() - want).abs().amax(1)
    scale = torch.maximum(want.abs().amax(1), weight)
    live = scale > 0
    assert (err[~live] == 0).all(), f"{name}: gradient on rows of weight 0"
    return torch.where(live, err / scale.clamp_min(1e-300), torch.zeros_like(err))


def _launch(rows2d, pitch, rows, B, N, K, table, mask_weight, backward, w_main, w_aux, want_recon, grad_pitch=None, status=None):
    """`train._train_rows`, or with `grad_pitch` the same call through the C ABI with a pitched gradient."""
    x0, x_t, t = rows["x0"].view(B, N), rows["x_t"].view(B, N), rows["t"]
    logits = torch.as_strided(rows2d, (B, N, K), (N * pitch, pitch, 1))
    if grad_pitch is None:
        return train._train_rows(logits, pitch, x0, x_t, t, table, mask_weight, backward=backward, w_main=w_main, w_aux=w_aux,
                                 want_recon=want_recon, status=status)
    d = _lib.TrainDesc()
    d.logits, d.x0, d.x_t, d.t, d.coef_table = logits.data_ptr(), x0.data_ptr(), x_t.data_ptr(), t.data_ptr(), table.data_ptr()
    d.B, d.N, d.K, d.T, d.pitch, d.logits_dtype = B, N, K, table.shape[0], pitch, _lib.LOGITS_F32
    d.mask_weight_masked, d.mask_weight_unmasked = float(mask_weight[0]), float(mask_weight[1])
    d.stream, d.backward, d.status = ops._stream(torch.device(DEV)), backward, ops._ptr(status)
    grad = torch.full((B, N, grad_pitch), 7.0, device=DEV)  # the pad columns must stay untouched
    d.grad, d.pitch_grad, d.w_main, d.w_aux = grad.data_ptr(), grad_pitch, w_main.data_ptr(), w_aux.data_ptr()
    out = {name: torch.empty(B, N, dtype=dt, device=DEV) for name, dt in
           (("tok_main", torch.float32), ("tok_aux", torch.float32), ("x0_recon", torch.int64), ("xtm1_recon", torch.int64))}
    d.tok_main, d.tok_aux = out["tok_main"].data_ptr(), out["tok_aux"].data_ptr()
    d.x0_recon, d.xtm1_recon = out["x0_recon"].data_ptr(), out["xtm1_recon"].data_ptr()
    _lib.check(_lib.load_library().d3pm_train_rows(ctypes.byref(d)), "d3pm_train_rows")
    torch.cuda.synchronize()
    assert torch.equal(grad[:, :, K:], torch.full_like(grad[:, :, K:], 7.0)), "pitched gradient: pad columns written"
    out["grad"] = grad[:, :, :K]
    return out


def _run_case(name, B, N, K, T, seed, mask_weight, stats, *, stream, pitched=False):
    sched = O.make_schedule(T, K)
    table = ops.build_coef_table(O.pack_schedule(sched).to(DEV), T, K)
    rows = _make_rows(B, N, K, T, _tvals(B, T), seed, DEV, groups=_stream_groups(K) if stream else None)
    w_main, w_aux = _video_weights(B, seed)
    pitch = K + 64 if pitched else K
    rows2d = rows["logits"]
    if pitched:
        rows2d = torch.full((B * N, pitch), float("nan"), device=DEV)  # the pad columns must never be read
        rows2d[:, :K] = rows["logits"]
    status = ops.new_status(DEV)
    kw = dict(rows2d=rows2d, pitch=pitch, rows=rows, B=B, N=N, K=K, table=table, mask_weight=mask_weight, w_main=w_main,
              w_aux=w_aux)
    both = _launch(backward=2, want_recon=True, grad_pitch=pitch if pitched else None, status=status, **kw)
    fwd = _launch(backward=0, want_recon=True, **kw)
    fwd_plain = _launch(backward=0, want_recon=False, **kw)
    grad_only = _launch(backward=1, want_recon=False, **kw)
    both_plain = _launch(backward=2, want_recon=False, **kw)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    # the outputs the modes share are bit for bit the same
    for o in (fwd, fwd_plain, both_plain):
        assert torch.equal(o["tok_main"], both["tok_main"]) and torch.equal(o["tok_aux"], both["tok_aux"]), name
    assert torch.equal(fwd["x0_recon"], both["x0_recon"]) and torch.equal(fwd["xtm1_recon"], both["xtm1_recon"]), name
    for o in (grad_only, both_plain):
        assert torch.equal(o["grad"], both["grad"]), name
    ref = reference_rows(sched, rows["logits"], rows["x0"], rows["x_t"], rows["t_row"], mask_weight,
                         w_main.repeat_interleave(N), w_aux.repeat_interleave(N))
    _check(name, both, ref, rows, N, mask_weight, w_main, w_aux, stats)


def _report(stats):
    for key in sorted(stats):
        print(f"[observed max error] {key[0]} {key[1]} K={key[2]}: {max(stats[key]):.3e}")


STREAM_CASES = [  # B, N (2048 rows = the threshold, a ragged count, the benchmarked shape), mask weights
    (8, 256, (1, 1)),
    (6, 347, (0.3, 2.0)),
    (16, 1024, (1, 1)),
]


@pytest.mark.parametrize("K", [1024, 2048, 4096])
def test_stream_kernel_against_reference(K):
    """train_stream_kernel at every codebook and row count, every backward mode, against the float64 reference; the
    ragged shape at K = 2048 reads pitched logits and writes a pitched gradient, the 16 x 1024 one uses mask weights
    (0.3, 2.0) at K = 2048 instead."""
    T = 100
    stats = {}
    for B, N, mw in STREAM_CASES:
        if K == 2048 and B == 16:
            mw = (0.3, 2.0)
        _run_case(f"stream K={K} {B}x{N}", B, N, K, T, 1000 + K + B, mw, stats, stream=True, pitched=(K == 2048 and B == 6))
    _report(stats)


@pytest.mark.parametrize("K", [8, 1000, 2048, 8192])
def test_row_kernel_against_reference(K):
    """train_rows_kernel (fewer than 2048 rows) at V = 1, 1, 2 and 8 float4 chunks per thread."""
    stats = {}
    _run_case(f"rows K={K}", 6, 300, K, 100, 2000 + K, (0.3, 2.0) if K in (8, 2048) else (1, 1), stats, stream=False)
    _report(stats)


# --------------------------------------------------------------------------- past 256 timesteps
T_LONG = 400
T_LONG_VALUES = [0, 1, 255, 256, 257, 399]


@pytest.mark.parametrize("K", [2048, 4096])
def test_stream_kernel_past_256_timesteps(K):
    """T = 400: the training stream kernel reads the coefficient table from global memory."""
    stats = {}
    sched = O.make_schedule(T_LONG, K)
    assert sched["log_at"].numel() == T_LONG
    B, N = 6, 347
    table = ops.build_coef_table(O.pack_schedule(sched).to(DEV), T_LONG, K)
    rows = _make_rows(B, N, K, T_LONG, T_LONG_VALUES, 3000 + K, DEV, groups=_stream_groups(K))
    w_main, w_aux = _video_weights(B, 3000 + K)
    got = _launch(rows["logits"], K, rows, B, N, K, table, (0.3, 2.0), 2, w_main, w_aux, True)
    ref = reference_rows(sched, rows["logits"], rows["x0"], rows["x_t"], rows["t_row"], (0.3, 2.0),
                         w_main.repeat_interleave(N), w_aux.repeat_interleave(N))
    _check(f"stream T=400 K={K}", got, ref, rows, N, (0.3, 2.0), w_main, w_aux, stats)
    # t = T is out of range: the status word says so
    status = ops.new_status(DEV)
    bad = dict(rows, t=torch.tensor([0, 1, 255, T_LONG, 257, 399], device=DEV))
    _launch(rows["logits"], K, bad, B, N, K, table, (1, 1), 2, w_main, w_aux, True, status=status)
    torch.cuda.synchronize()
    assert int(status.item()) & _lib.STATUS_BAD_T
    _report(stats)


@pytest.mark.parametrize("K,s", [(4096, 2.0), (1024, None)])
def test_step_stream_kernel_past_256_timesteps(K, s):
    """T = 400: step_stream_kernel against the oracle on the uniforms it drew (as test_stream_kernel_parity) and against
    the rows kernel, which always reads the coefficient table from global memory."""
    B, N = 6, 400
    sched = O.make_schedule(T_LONG, K)
    table = ops.build_coef_table(O.pack_schedule(sched).to(DEV), T_LONG, K)
    g = torch.Generator(device=DEV).manual_seed(K + 400)
    lc = torch.randn(B, N, K, device=DEV, generator=g) * 2.0
    lu = None if s is None else torch.randn(B, N, K, device=DEV, generator=g) * 2.0
    t = torch.tensor(T_LONG_VALUES, device=DEV)
    x_t = torch.randint(0, K, (B, N), device=DEV, generator=g)
    x_t[:, ::3] = K
    kw = dict(guidance_scale=0.0 if s is None else s, sample_mode=_lib.SAMPLE_PHILOX, seed=41, offset=7, row_offset=999)
    status = ops.new_status(DEV)
    thin = ops.fused_step(lc, lu, x_t, t, table, kernel=_lib.KERNEL_STREAM, status=status, **kw)["x_prev"]
    torch.cuda.synchronize()
    assert int(status.item()) & (_lib.STATUS_BAD_T | _lib.STATUS_BAD_TOKEN) == 0
    rows = torch.arange(0, N, 8)
    u = ops.philox_uniform(B, N, K, seed=41, offset=7, row_offset=999, device=DEV)[:, rows, :K + 1].cpu().permute(0, 2, 1)
    out_o, post_o, _ = O.p_sample_step(sched, lc[:, rows].cpu().permute(0, 2, 1),
                                       None if lu is None else lu[:, rows].cpu().permute(0, 2, 1),
                                       O.index_to_log_onehot(x_t[:, rows].cpu(), K + 1), t.cpu(), kw["guidance_scale"], u)
    ties = O.near_ties(post_o, u).numpy()
    H.assert_tokens_match(thin[:, rows].cpu().numpy(), out_o.argmax(1).numpy(), ties, "stream T=400 vs oracle")
    for tf in (0.0, 1.0, 1e-3):  # batched survivor scoring, second thinned attempt, exhaustive
        o = ops.fused_step(lc, lu, x_t, t, table, kernel=_lib.KERNEL_STREAM, thin_factor=tf, want_winner_post=True, **kw)
        assert torch.equal(o["x_prev"], thin)
        want = post_o.gather(1, thin[:, rows].cpu().unsqueeze(1)).squeeze(1)
        assert (o["winner_post"][:, rows].cpu() - want).abs().max().item() <= H.POST_TOL, f"thin_factor {tf}"
    rowsk = ops.fused_step(lc, lu, x_t, t, table, kernel=_lib.KERNEL_ROWS, **kw)["x_prev"]
    H.assert_tokens_match(rowsk[:, rows].cpu().numpy(), out_o.argmax(1).numpy(), ties, "rows T=400 vs oracle")
    assert (rowsk != thin).float().mean() < 1e-3
    status.zero_()
    ops.fused_step(lc, lu, x_t, torch.tensor([0, 1, 255, T_LONG, 257, 399], device=DEV), table, kernel=_lib.KERNEL_STREAM,
                   status=status, **kw)
    torch.cuda.synchronize()
    assert int(status.item()) & _lib.STATUS_BAD_T


# --------------------------------------------------------------------------- the module, end to end
class _LeafDenoiser(torch.nn.Module):
    """Returns a leaf logits tensor as a [B, K, N] view of [B, N, K] (the reference transformer's layout) and keeps the
    x_t it was called with."""

    def __init__(self, K, logits_bnk):
        super().__init__()
        import types
        self.content_emb = types.SimpleNamespace(num_embed=K + 1)
        self.to_logits = torch.nn.Sequential(torch.nn.Identity(), torch.nn.Linear(1, 1))
        self.logits = logits_bnk
        self.x_t = None

    def forward(self, x_t, cond, t):
        self.x_t = x_t.clone()
        return self.logits.permute(0, 2, 1)


def test_module_loss_and_gradient_against_reference():
    """FusedDiffusionTransformer.forward(return_loss=True) + backward at 16 x 1024 tokens, K = 2048, adaptive auxiliary
    loss: the loss and logits.grad against the float64 reference summed the way VBLoss sums it."""
    T, K, B, N, aux = 100, 2048, 16, 1024, 5e-3
    rows = _make_rows(B, N, K, T, _tvals(B, T), 4242, DEV, groups=_stream_groups(K))  # only the logits and x0 are used
    logits = rows["logits"].view(B, N, K).clone().requires_grad_(True)
    x0 = rows["x0"].view(B, N)
    t = torch.tensor(_tvals(B, T), device=DEV)
    pt = (torch.rand(B, generator=torch.Generator().manual_seed(5)) * 0.02 + 0.001).to(DEV)
    u = torch.rand(B, K + 1, N, generator=torch.Generator().manual_seed(6))
    den = _LeafDenoiser(K, logits)
    m = d3pm_b200.FusedDiffusionTransformer(transformer=den, diffusion_step=T, alpha_init_type="alpha1", guidance_scale=2.0,
                                           content_seq_len=N, auxiliary_loss_weight=aux, adaptive_auxiliary_loss=True).to(DEV)
    m.sample_time = lambda b, device, method="uniform": (t, pt)
    m.inject_uniform = lambda shape, dev: u.to(dev)
    out = m({"content_token": x0, "condition_embed_token": torch.ones(B, 1, 512, device=DEV)}, return_loss=True,
            return_logits=False)
    out["loss"].backward()
    m.check_status()
    x_t = den.x_t
    # the forward noising drew what the oracle draws from the same uniforms (Gumbel near-ties aside)
    sched = {name: getattr(m, name).cpu() for name in O.SCHEDULE_NAMES}
    q = O.q_pred(sched, O.index_to_log_onehot(x0.cpu(), K + 1), t.cpu())
    want_xt = (O.gumbel_from_uniform(u) + q).argmax(1)
    H.assert_tokens_match(x_t.cpu().numpy(), want_xt.numpy(), O.near_ties(q, u).numpy(), "q_sample vs oracle")

    aux_w = ((1 - t / T) + 1.0) * aux
    w_main, w_aux = 1.0 / (B * N * pt), aux_w / (B * N * pt)
    ref = reference_rows(sched, rows["logits"], rows["x0"], x_t.reshape(-1), t.repeat_interleave(N), m.mask_weight,
                         w_main.repeat_interleave(N), w_aux.repeat_interleave(N))
    vb = (ref["tok_main"].view(B, N).sum(1) + aux_w.double() * ref["tok_aux"].view(B, N).sum(1)) / pt.double()
    want_loss = float(vb.sum() / (B * N))
    print(f"[module] loss {float(out['loss']):.9e} reference {want_loss:.9e} rel. err "
          f"{abs(float(out['loss']) - want_loss) / abs(want_loss):.3e}")
    assert abs(float(out["loss"]) - want_loss) <= TOK_REL * abs(want_loss)  # observed 6.9e-8 relative
    assert torch.equal(out["pred_data"].reshape(-1), ref["x0_recon"])
    weight = _row_weight(x_t.reshape(-1), t.repeat_interleave(N), K, m.mask_weight, w_main.repeat_interleave(N),
                         w_aux.repeat_interleave(N))
    rel = _grad_row_error(logits.grad.reshape(-1, K), ref["grad"], weight, "module")
    print(f"[module] gradient: max error {float(rel.max()):.3e} of the row's scale")
    assert float(rel.max()) <= GRAD_REL
