"""The denoiser's self-attention at head dimension 4: the reference's math against `d3pm_self_attention`.

    python tools/attention_bench.py [--iters 20] [--shapes 16x4096,16x1024,1x1024] [--denoiser] [--json out.json]

Per shape (B videos, N tokens, 16 heads of width 4; q, k, v ~ N(0, 1) from a fixed seed) three arms, each warmed up and
then timed over `--iters` launches with CUDA events (median reported):

  (a) `reference`: FullAttention's own math (transformer_utils.py:52-58): q kᵀ * scale, softmax, att @ v, att.mean(1);
  (b) `sdpa`: torch.nn.functional.scaled_dot_product_attention in fp32, whichever backend torch picks (comparison only);
  (c) `fused`: d3pm_self_attention.

Each arm's max error against a float64 restatement on 64 sampled query rows (of max|v|), ms, scores/s, and the fused
kernel against the exponential floor: B * heads * N² ex2 at 16 MUFU.EX2 per clock per SM.  Each arm's SM clock is the
median nvidia-smi reports while that arm runs back to back for about a second; the floor uses the fused arm's.  The card's
name and power limit are printed with them.  For scale, `cross` times the math of the blocks' cross-attention `attn2` over the
77 condition tokens (left to PyTorch: it forms a [B, 16, N, 77] matrix) at the same B and N.

`--denoiser` (only where the reference is staged): two `Text2ImageTransformer` forwards and one `p_sample_tokens` step at
config 3 (B = 16, N = 4096, K = 4096) with and without `enable_fused_attention()`.
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
    qs = q[:, rows].double().view(B, len(rows), HEADS, HD).transpose(1, 2)
    att = torch.softmax((qs @ heads_of(k.double(), B, N).transpose(-2, -1)) / math.sqrt(HD), dim=-1)
    return (att @ heads_of(v.double(), B, N)).transpose(1, 2).reshape(B, len(rows), C)


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
        with torch.no_grad():
            y = fn()
            err = float((y[:, rows].double() - want).abs().max()) / vmax
            del y
            ms = time_ms(fn, iters)
            mhz = sustained_clock_mhz(fn)
        out[name] = {"ms": ms, "scores_per_s": scores / (ms * 1e-3), "max_err_of_max_v": err, "sm_clock_mhz": mhz}
        torch.cuda.empty_cache()
    kc, vc = (torch.randn(B, 77, HEADS * HD, device="cuda", generator=g) for _ in range(2))
    with torch.no_grad():
        cross = lambda: cross_arm(q, kc, vc)  # noqa: E731
        out["cross"] = {"ms": time_ms(cross, iters), "sm_clock_mhz": sustained_clock_mhz(cross)}
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    floor_ms = scores / (EX2_PER_CLK_PER_SM * sms * out["fused"]["sm_clock_mhz"] * 1e6) * 1e3
    out["fused"].update({"ex2_floor_ms": floor_ms, "fraction_of_ex2_floor": floor_ms / out["fused"]["ms"]})
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
    for fused in (False, True):
        ours.enable_fused_attention(fused)
        with torch.no_grad():
            two = time_ms(lambda: (ours.transformer(x, cond, t), ours.transformer(x, cf, t)), max(3, iters // 4), warmup=1)
            step = time_ms(lambda: ours.p_sample_tokens(x, cond, cf, t), max(3, iters // 4), warmup=1)
        res["fused" if fused else "eager"] = {"two_forwards_ms": two, "p_sample_tokens_ms": step}
        torch.cuda.empty_cache()
    ours.enable_fused_attention(False)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--shapes", default="16x4096,16x1024,1x1024")
    ap.add_argument("--denoiser", action="store_true")
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
              f"cross (77 keys) {r['cross']['ms']:.3f} ms at {r['cross']['sm_clock_mhz']:.0f} MHz")
    if args.denoiser:
        result["denoiser"] = bench_denoiser(args.iters)
        print("denoiser:", json.dumps(result["denoiser"]))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
