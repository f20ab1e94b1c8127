"""Training-side step (SURVEY §8 f1) at the reference's shipped training shape: batch 16, 4x16x16 = 1024 tokens,
4096 codes.  Times `d3pm_train_rows` forward and backward (CUDA events) and, with --cpu, the oracle port of the
reference's `_train_loss` + autograd backward on the host cores.

With --dtype float16 | bfloat16 it compares, at --videos and at 64 videos, the two ways to train on 16-bit logits:
(a) the losses (backward = 0) and then the gradient (backward = 1) straight on the 16-bit rows, and (b) the cast route:
`.float()`, the fp32 one-pass kernel (backward = 2), `grad.to(dtype)`, and the same with a `d3pm_scale_rows` factor
other than 1 (any run with a loss scaler).  The routes alternate in one process, CUDA events, median of the rounds.

    python tools/train_bench.py [--videos 16] [--tokens 1024] [--cpu] [--dtype float16|bfloat16]
"""
import argparse
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import d3pm_b200  # noqa: E402
from d3pm_b200 import train  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--videos", type=int, default=16)
ap.add_argument("--tokens", type=int, default=1024)
ap.add_argument("--codes", type=int, default=4096)
ap.add_argument("--cpu", action="store_true")
ap.add_argument("--dtype", choices=("float16", "bfloat16"), help="compare the 16-bit route with the cast route")
ap.add_argument("--rounds", type=int, default=7, help="alternated rounds of the --dtype comparison")
a = ap.parse_args()
B, N, K, T = a.videos, a.tokens, a.codes, 100
dev = torch.device("cuda", 0)


class _Stub(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.content_emb = type("E", (), {"num_embed": K + 1})()


m = d3pm_b200.FusedDiffusionTransformer(transformer=_Stub(), diffusion_step=T, alpha_init_type="alpha1", guidance_scale=2.0,
                                        content_seq_len=N, auxiliary_loss_weight=5e-4, adaptive_auxiliary_loss=True).to(dev)
g = torch.Generator(device=dev).manual_seed(0)
logits = torch.randn(B, N, K, device=dev, generator=g)
x0 = torch.randint(0, K, (B, N), device=dev, generator=g)
t = torch.randint(0, T, (B,), device=dev, generator=g)
pt = torch.full((B,), 1.0 / T, device=dev)
x_t = m.q_sample_tokens(x0, t)
w = torch.ones(B, device=dev)
table = m.coef_table()


def fwd():
    return train._train_rows(logits, K, x0, x_t, t, table, (1, 1), backward=False, want_recon=True)


def bwd():
    return train._train_rows(logits, K, x0, x_t, t, table, (1, 1), backward=True, w_main=w, w_aux=w)


def both():
    return train._train_rows(logits, K, x0, x_t, t, table, (1, 1), backward=2, w_main=w, w_aux=w, want_recon=True)




def compare_16bit(B, dtype, rounds, iters=10):
    """Times the 16-bit route against the cast route on the same [B, N, K] logits (inputs >> L2 at 64 videos)."""
    gen = torch.Generator(device=dev).manual_seed(1)
    l16 = torch.randn(B, N, K, device=dev, generator=gen).to(dtype)
    xs = torch.randint(0, K, (B, N), device=dev, generator=gen)
    ts = torch.randint(0, T, (B,), device=dev, generator=gen)
    xts = m.q_sample_tokens(xs, ts)
    ones, half = torch.ones(B, device=dev), torch.full((B,), 0.5, device=dev)

    def new():
        train._train_rows(l16, K, xs, xts, ts, table, (1, 1), backward=0, want_recon=True)
        return train._train_rows(l16, K, xs, xts, ts, table, (1, 1), backward=1, w_main=ones, w_aux=ones)["grad"]

    def cast(factor=None):
        out = train._train_rows(l16.float(), K, xs, xts, ts, table, (1, 1), backward=2, w_main=ones, w_aux=ones,
                                want_recon=True)
        if factor is not None:
            train.scale_rows(out["grad"], factor)
        return out["grad"].to(dtype)

    e = B * N * K  # bytes per route: the logits' and the gradient's reads and writes, 2 bytes per 16-bit, 4 per fp32 value
    routes = (("16-bit rows: losses, then gradient", new, e * (2 + 2 + 2)),
              ("cast route: .float(), one fp32 pass, .to(dtype)", cast, e * (2 + 4 + 4 + 4 + 4 + 2)),
              ("cast route with a loss-scale rescale", lambda: cast(half), e * (2 + 4 + 4 + 4 + 4 + 4 + 4 + 2)))
    for _, fn, _ in routes:
        fn()
    times = {name: [] for name, _, _ in routes}
    for _ in range(rounds):
        for name, fn, _ in routes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / iters)
    for name, _, nbytes in routes:
        ms = sorted(times[name])[len(times[name]) // 2]
        print(f"{dtype} {B}x{N} tokens x {K} codes, {name}: {ms:.3f} ms (median of {rounds}, spread "
              f"{min(times[name]):.3f}-{max(times[name]):.3f}), {nbytes / 1e9:.3f} GB algorithmic, {nbytes / ms / 1e6:.0f} GB/s")


if a.dtype:
    print(torch.cuda.get_device_name(dev))
    for videos in sorted({B, 64}):
        compare_16bit(videos, getattr(torch, a.dtype), a.rounds)
    sys.exit(0)

for name, fn, nbytes in (("forward (losses, arg-maxes)", fwd, B * N * K * 4), ("gradient only", bwd, 2 * B * N * K * 4),
                         ("forward + gradient, one pass", both, 2 * B * N * K * 4)):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print(f"d3pm_train_rows {name}: {ms:.3f} ms, {nbytes / ms / 1e6:.0f} GB/s algorithmic ({B}x{N} tokens x {K} codes)")

if a.cpu:
    from oracle import d3pm_oracle as O
    torch.set_num_threads(os.cpu_count())
    sched = O.make_schedule(T, K)
    lg = logits[:2].cpu().clone().requires_grad_(True)
    u = torch.rand(2, K + 1, N)
    t0 = time.perf_counter()
    _, vb, _, _, _ = O.train_loss(sched, lg.permute(0, 2, 1), x0[:2].cpu(), t[:2].cpu(), pt[:2].cpu(), u,
                                  auxiliary_loss_weight=5e-4, adaptive_auxiliary_loss=True)
    vb.sum().backward()
    dt = time.perf_counter() - t0
    print(f"oracle port of _train_loss fwd+bwd on {os.cpu_count()} host cores: {dt * 1e3:.0f} ms for 2 videos "
          f"-> {dt / 2 * B * 1e3:.0f} ms per {B}-video step")
