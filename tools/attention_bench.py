"""The denoiser's attentions at head dimension 4: the reference's math against `d3pm_self_attention` and
`d3pm_cross_attention`.

    python tools/attention_bench.py [--iters 20] [--shapes 16x4096,16x1024,1x1024] [--denoiser] [--standin] [--json out.json]

Per shape (B videos, N tokens, 16 heads of width 4; q, k, v ~ N(0, 1) from a fixed seed) three self-attention arms, each
warmed up and then timed over `--iters` launches with CUDA events (median reported):

  (a) `reference`: FullAttention's own math (transformer_utils.py:52-58): q kᵀ * scale, softmax, att @ v, att.mean(1);
  (b) `sdpa`: torch.nn.functional.scaled_dot_product_attention in fp32, whichever backend torch picks (comparison only);
  (c) `fused`: d3pm_self_attention.

Each arm's max error against a float64 restatement on 64 sampled query rows (of max|v|), ms, scores/s, and the fused
kernel against the exponential floor: B * heads * N² ex2 at 16 MUFU.EX2 per clock per SM.  Each arm's SM clock is the
median nvidia-smi reports while that arm runs back to back for about a second; the floor uses the fused arm's.  The card's
name and power limit are printed with them.  The blocks' cross-attention `attn2` over the 77 condition tokens is timed the
same way in two arms: `cross` is CrossAttention's math in PyTorch (it forms a [B, 16, N, 77] matrix and its head mean),
`cross_fused` is d3pm_cross_attention, with its scores/s and its fraction of the floor of B * heads * N * 77 ex2.

`--denoiser` (only where the reference is staged): two `Text2ImageTransformer` forwards and one `p_sample_tokens` step at
config 3 (B = 16, N = 4096, K = 4096) eager, with `enable_fused_attention()` and with `enable_fused_attention(cross=True)`.

`--standin`: one forward of a 19-block self-plus-cross stand-in denoiser (tests/cross_attention_standin.py: n_embd 64, 16
heads, condition 77 x 512, K = 4096) at config 3 (B = 16, N = 4096), eager, fused self and fused self + cross.  It is not
the reference's denoiser (no AdaLayerNorm, a plain GELU MLP): it measures what each attention costs in a pass of that shape
where the reference is not staged.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

HEADS, HD = 16, 4
EX2_PER_CLK_PER_SM = 16


def smi(fields: str) -> list:
    out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), f"--query-gpu={fields}",
                          "--format=csv,noheader,nounits"], capture_output=True, text=True).stdout.strip()
    return [f.strip() for f in out.split(",")]


def time_ms(fn, iters: int, warmup: int = 3) -> float:
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def sustained_clock_mhz(fn, seconds: float = 1.0) -> float:
    """Median SM clock nvidia-smi reports while `fn` runs back to back for about `seconds`."""
    samples, done = [], threading.Event()

    def poll():
        while not done.is_set():
            samples.append(float(smi("clocks.sm")[0]))
            done.wait(0.1)

    ms = time_ms(fn, 3, warmup=1)
    th = threading.Thread(target=poll)
    th.start()
    for _ in range(max(1, int(seconds * 1e3 / max(ms, 1e-3)))):
        fn()
    torch.cuda.synchronize()
    done.set()
    th.join()
    return statistics.median(samples)


def heads_of(x, B, N):
    return x.view(B, N, HEADS, HD).transpose(1, 2)


def reference_arm(q, k, v):
    B, N, C = q.shape
    qh, kh, vh = heads_of(q, B, N), heads_of(k, B, N), heads_of(v, B, N)
    att = (qh @ kh.transpose(-2, -1)) * (1.0 / math.sqrt(HD))
    att = F.softmax(att, dim=-1)
    y = (att @ vh).transpose(1, 2).contiguous().view(B, N, C)
    return y, att.mean(dim=1)


def sdpa_arm(q, k, v):
    B, N, C = q.shape
    y = F.scaled_dot_product_attention(heads_of(q, B, N), heads_of(k, B, N), heads_of(v, B, N))
    return y.transpose(1, 2).contiguous().view(B, N, C)


def cross_arm(q, kc, vc):
    """CrossAttention's math with 77 condition keys: softmax(q kcᵀ * scale) @ vc and the head mean of the map."""
    B, N, C = q.shape
    att = F.softmax((heads_of(q, B, N) @ heads_of(kc, B, 77).transpose(-2, -1)) * (1.0 / math.sqrt(HD)), dim=-1)
    return (att @ heads_of(vc, B, 77)).transpose(1, 2).contiguous().view(B, N, C), att.mean(dim=1)


def float64_rows(q, k, v, rows):
    B, N, C = q.shape
    M = k.shape[1]
    qs = q[:, rows].double().view(B, len(rows), HEADS, HD).transpose(1, 2)
    att = torch.softmax((qs @ heads_of(k.double(), B, M).transpose(-2, -1)) / math.sqrt(HD), dim=-1)
    return (att @ heads_of(v.double(), B, M)).transpose(1, 2).reshape(B, len(rows), C)


def ex2_floor_ms(pairs, mhz):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return pairs / (EX2_PER_CLK_PER_SM * sms * mhz * 1e6) * 1e3


def timed_arm(fn, rows, want, vmax, iters, pairs):
    """ms, scores/s, error against float64 (of max|v|) and SM clock of one arm."""
    with torch.no_grad():
        y = fn()
        err = float((y[:, rows].double() - want).abs().max()) / vmax
        del y
        ms = time_ms(fn, iters)
        mhz = sustained_clock_mhz(fn)
    torch.cuda.empty_cache()
    return {"ms": ms, "scores_per_s": pairs / (ms * 1e-3), "max_err_of_max_v": err, "sm_clock_mhz": mhz}


def bench_shape(B, N, iters):
    from d3pm_b200 import attention
    g = torch.Generator(device="cuda").manual_seed(1234)
    q, k, v = (torch.randn(B, N, HEADS * HD, device="cuda", generator=g) for _ in range(3))
    rows = torch.randperm(N, generator=torch.Generator().manual_seed(5))[:64].cuda()
    want = float64_rows(q, k, v, rows)
    vmax = float(v.abs().max())
    arms = {
        "reference": lambda: reference_arm(q, k, v)[0],
        "sdpa": lambda: sdpa_arm(q, k, v),
        "fused": lambda: attention.self_attention(q, k, v, HEADS, 1.0 / math.sqrt(HD)),
    }
    scores = B * HEADS * N * N
    out = {"B": B, "N": N, "heads": HEADS, "head_dim": HD, "scores": scores}
    for name, fn in arms.items():
        out[name] = timed_arm(fn, rows, want, vmax, iters, scores)
    floor_ms = ex2_floor_ms(scores, out["fused"]["sm_clock_mhz"])
    out["fused"].update({"ex2_floor_ms": floor_ms, "fraction_of_ex2_floor": floor_ms / out["fused"]["ms"]})
    kc, vc = (torch.randn(B, 77, HEADS * HD, device="cuda", generator=g) for _ in range(2))
    want_c = float64_rows(q, kc, vc, rows)
    vmax_c = float(vc.abs().max())
    cross_scores = B * HEADS * N * 77
    out["cross_scores"] = cross_scores
    out["cross"] = timed_arm(lambda: cross_arm(q, kc, vc)[0], rows, want_c, vmax_c, iters, cross_scores)
    out["cross_fused"] = timed_arm(lambda: attention.cross_attention(q, kc, vc, HEADS, 1.0 / math.sqrt(HD)), rows, want_c,
                                   vmax_c, iters, cross_scores)
    floor_ms = ex2_floor_ms(cross_scores, out["cross_fused"]["sm_clock_mhz"])
    out["cross_fused"].update({"ex2_floor_ms": floor_ms, "fraction_of_ex2_floor": floor_ms / out["cross_fused"]["ms"]})
    return out


def bench_denoiser(iters):
    from baseline import reference_loader as RL
    if not RL.reference_available():
        return {"ran": False, "why": "reference not staged (baseline/_ref absent): config-3 denoiser not measured"}
    from tools import config3
    B, N, K, T = 16, 4096, 4096, 100
    dev = torch.device("cuda", 0)
    _, ours = config3.build_models(B, N, K, T, [64, 64], dev)
    del _
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randint(0, K + 1, (B, N), device=dev, generator=g)
    cond = torch.randn(B, 77, 512, device=dev, generator=g)
    cf = torch.zeros(B, 77, 512, device=dev)
    t = torch.full((B,), 50, device=dev, dtype=torch.long)
    res = {"ran": True, "B": B, "N": N, "K": K}
    for arm, fused, cross in (("eager", False, False), ("fused", True, False), ("fused_self_cross", True, True)):
        ours.enable_fused_attention(fused, cross=cross)
        with torch.no_grad():
            two = time_ms(lambda: (ours.transformer(x, cond, t), ours.transformer(x, cf, t)), max(3, iters // 4), warmup=1)
            step = time_ms(lambda: ours.p_sample_tokens(x, cond, cf, t), max(3, iters // 4), warmup=1)
        res[arm] = {"two_forwards_ms": two, "p_sample_tokens_ms": step}
        torch.cuda.empty_cache()
    ours.enable_fused_attention(False)
    return res


def bench_standin(iters):
    """One forward of a 19-block self-plus-cross stand-in denoiser at config 3, eager / fused self / fused self + cross."""
    from d3pm_b200 import attention
    from tests.cross_attention_standin import CrossStandInDenoiser
    B, N, K = 16, 4096, 4096
    torch.manual_seed(0)
    model = CrossStandInDenoiser(K, N, n_layer=19).cuda().eval()
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randint(0, K + 1, (B, N), device="cuda", generator=g)
    cond = torch.randn(B, 77, 512, device="cuda", generator=g)
    t = torch.full((B,), 50, device="cuda", dtype=torch.long)
    res = {"what": "stand-in denoiser (tests/cross_attention_standin.py), not the reference's", "B": B, "N": N, "K": K,
           "n_layer": 19, "n_embd": 64, "heads": HEADS}
    n = max(3, iters // 4)
    with torch.no_grad():
        fwd = lambda: model(x, cond, t)  # noqa: E731
        res["eager"] = {"forward_ms": time_ms(fwd, n, warmup=1), "sm_clock_mhz": sustained_clock_mhz(fwd, 3.0)}
        torch.cuda.empty_cache()
        attention.fuse_self_attention(model)
        res["fused_self"] = {"forward_ms": time_ms(fwd, n), "sm_clock_mhz": sustained_clock_mhz(fwd)}
        attention.fuse_cross_attention(model)
        res["fused_self_cross"] = {"forward_ms": time_ms(fwd, n), "sm_clock_mhz": sustained_clock_mhz(fwd)}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--shapes", default="16x4096,16x1024,1x1024")
    ap.add_argument("--denoiser", action="store_true")
    ap.add_argument("--standin", action="store_true")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_bench needs a CUDA device")
    name, power = smi("name,power.limit")
    result = {"card": name, "power_limit_w": float(power), "shapes": []}
    print(f"card {name}, power limit {power} W")
    for s in args.shapes.split(","):
        B, N = (int(z) for z in s.split("x"))
        r = bench_shape(B, N, max(20, args.iters))
        result["shapes"].append(r)
        f = r["fused"]
        arm = lambda a: f"{r[a]['ms']:9.3f} ms at {r[a]['sm_clock_mhz']:.0f} MHz (err {r[a]['max_err_of_max_v']:.1e})"  # noqa: E731
        print(f"B={B:2d} N={N:5d}: reference {arm('reference')} | sdpa {arm('sdpa')} | fused {arm('fused')}, "
              f"{f['scores_per_s']:.3e} scores/s, ex2 floor {f['ex2_floor_ms']:.3f} ms = {100 * f['fraction_of_ex2_floor']:.0f} %; "
              f"cross (77 keys) {arm('cross')}")
        c = r["cross_fused"]
        print(f"            cross fused {arm('cross_fused')}, {c['scores_per_s']:.3e} scores/s, "
              f"ex2 floor {1e3 * c['ex2_floor_ms']:.1f} us = {100 * c['fraction_of_ex2_floor']:.0f} %")
    if args.denoiser:
        result["denoiser"] = bench_denoiser(args.iters)
        print("denoiser:", json.dumps(result["denoiser"]))
    if args.standin:
        result["standin"] = bench_standin(args.iters)
        print("stand-in:", json.dumps(result["standin"]))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
