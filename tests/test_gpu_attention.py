"""The fused self-attention (`d3pm_self_attention`, `attention.FusedSelfAttention`) on the GPU.

* the kernel against a float64 restatement on sampled query rows, next to eager fp32's own error, over N from 1 to one
  too long to stage a head's keys in one pass, B in {1, 3, 16}, 16 heads, and inputs that stress the softmax (scores up to
  about ±300, all keys equal, one dominant key);
* delegation: with grad, under autocast and with a mask the original module runs, bit for bit;
* a whole stand-in denoiser (tests/attention_standin.py): fused logits within 4x eager fp32's error against float64;
* a teacher-forced chain at N = 1024, K = 4096 (as tests/test_gpu_config3.py): posterior within POST_TOL, tokens equal
  except at logged near-ties, with and without the fused head;
* CUDA-graph capture, a non-current device, and the real `Text2ImageTransformer` where the reference is staged.
"""
import contextlib
import copy
import math

import pytest
import torch

from baseline import reference_loader as RL
from d3pm_b200 import FusedDiffusionTransformer, attention, ops
from oracle import d3pm_oracle as O
from tests import helpers as H
from tests.attention_standin import FullAttention, StandInDenoiser

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
HEADS, HD = 16, 4
TOL = 2e-5  # of max|v|


def _inputs(kind, B, N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    shape = (B, N, HEADS * HD)
    q, k, v = (torch.randn(shape, device=DEV, generator=g) for _ in range(3))
    if kind == "large":        # scale 0.5: scores of std ~70, up to about ±300
        q, k = q * 8.5, k * 8.5
    elif kind == "equal_keys":  # uniform softmax: y = mean of v
        k = k[:, :1].expand(shape).contiguous()
    elif kind == "dominant":   # one key far above the rest for every query
        q = q.abs()
        k = k * 0.1
        k[:, N // 2] = 12.0
    return q.contiguous(), k, v


def _restated(q, k, v, rows, dtype):
    """softmax(scale q kᵀ) v per head for the query rows `rows`, in `dtype`."""
    B, N, C = q.shape
    qs = q[:, rows].to(dtype).view(B, len(rows), HEADS, HD).transpose(1, 2)
    kh = k.to(dtype).view(B, N, HEADS, HD).transpose(1, 2)
    vh = v.to(dtype).view(B, N, HEADS, HD).transpose(1, 2)
    att = torch.softmax((qs @ kh.transpose(-2, -1)) * (1.0 / math.sqrt(HD)), dim=-1)
    return (att @ vh).transpose(1, 2).reshape(B, len(rows), C)


SHAPES = [(1, 1), (3, 1), (3, 77), (16, 77), (1, 1000), (3, 1000), (1, 1024), (16, 1024), (3, 4096), (16, 4096),
          (1, 8200), (3, 8200)]


@pytest.mark.parametrize("kind", ["ln", "large", "equal_keys", "dominant"])
@pytest.mark.parametrize("B, N", SHAPES)
def test_kernel_matches_float64_on_sampled_rows(B, N, kind):
    q, k, v = _inputs(kind, B, N, seed=B * 100003 + N)
    y = attention.self_attention(q, k, v, HEADS, 1.0 / math.sqrt(HD))
    g = torch.Generator().manual_seed(N)
    rows = torch.unique(torch.cat((torch.tensor([0, N - 1]), torch.randint(0, N, (62,), generator=g)))).to(DEV)
    want = _restated(q, k, v, rows, torch.float64)
    eager = _restated(q, k, v, rows, torch.float32)
    scale = float(v.abs().max())
    err = float((y[:, rows].double() - want).abs().max()) / scale
    err_eager = float((eager.double() - want).abs().max()) / scale
    print(f"[attention B={B} N={N} {kind}] kernel {err:.2e}, eager fp32 {err_eager:.2e} of max|v|")
    assert torch.isfinite(y).all()
    assert err <= TOL


def test_more_videos_than_one_grid_holds():
    """B above the 65535 videos of one launch's grid: the batch runs as several launches, every video is computed."""
    B, N = 65537, 3
    q, k, v = _inputs("ln", B, N, seed=4)
    y = attention.self_attention(q, k, v, HEADS, 0.5)
    for b in (0, 65534, 65535, 65536):
        want = _restated(q[b:b + 1], k[b:b + 1], v[b:b + 1], torch.arange(N, device=DEV), torch.float64)
        assert float((y[b:b + 1].double() - want).abs().max()) <= TOL * float(v.abs().max()), b


def test_pitched_inputs_are_read_in_place():
    """q, k and v as column slices of one [B, N, 3C] tensor (pitch 3C) give the result of contiguous copies."""
    B, N, C = 2, 300, HEADS * HD
    qkv = torch.randn(B, N, 3 * C, device=DEV)
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    a = attention.self_attention(q, k, v, HEADS, 0.5)
    b = attention.self_attention(q.contiguous(), k.contiguous(), v.contiguous(), HEADS, 0.5)
    assert torch.equal(a, b)


def _pair(seed=0):
    torch.manual_seed(seed)
    ref = FullAttention(64, HEADS).to(DEV)
    return ref, attention.FusedSelfAttention(copy.deepcopy(ref))


def test_delegation_with_grad_is_bit_identical():
    ref, fused = _pair()
    x1 = torch.randn(2, 200, 64, device=DEV, requires_grad=True)
    x2 = x1.detach().clone().requires_grad_(True)
    y1, a1 = ref(x1, None)
    y2, a2 = fused(x2, None)
    assert torch.equal(y1, y2) and torch.equal(a1, a2)
    (y1.square().sum() + a1.sum()).backward()
    (y2.square().sum() + a2.sum()).backward()
    assert torch.equal(x1.grad, x2.grad)
    for p, q in zip(ref.parameters(), fused.parameters()):
        assert torch.equal(p.grad, q.grad)


def test_delegation_under_autocast_and_with_a_mask_is_bit_identical():
    ref, fused = _pair(1)
    x = torch.randn(2, 200, 64, device=DEV)
    with torch.no_grad():
        with torch.autocast("cuda"):
            y1, a1 = ref(x, None)
            y2, a2 = fused(x, None)
        assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
        mask = torch.ones(2, 200, 200, dtype=torch.bool, device=DEV)
        y1, a1 = ref(x, None, mask=mask)
        y2, a2 = fused(x, None, mask=mask)
        assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
        y3, a3 = fused(x, None)  # and the fused path itself: no map, the same output within the kernel's tolerance
        assert a3 is None and float((y3 - y1).abs().max()) <= 1e-4 * float(y1.abs().max())


@contextlib.contextmanager
def _fused_calls(model):
    """Counts the forwards of `model`'s FusedSelfAttention modules that ran the kernel (second output None) and those that
    delegated to the original module: a fused model that quietly delegated would have exactly eager's numbers."""
    calls = {"fused": 0, "delegated": 0}

    def hook(mod, args, out):
        calls["fused" if out[1] is None else "delegated"] += 1

    hooks = [m.register_forward_hook(hook) for m in model.modules() if isinstance(m, attention.FusedSelfAttention)]
    try:
        yield calls
    finally:
        for hk in hooks:
            hk.remove()


def _logit_errors(model, B, N, K, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randint(0, K + 1, (B, N), device=DEV, generator=g)
    cond = torch.randn(B, 77, 512, device=DEV, generator=g)
    t = torch.randint(0, 100, (B,), device=DEV, generator=g)
    with torch.no_grad():
        want = copy.deepcopy(model).double()(x, cond.double(), t)
        eager = model(x, cond, t)
        n = attention.fuse_self_attention(model)
        with _fused_calls(model) as calls:
            got = model(x, cond, t)
        attention.fuse_self_attention(model, False)
    assert calls == {"fused": n, "delegated": 0}
    return float((got.double() - want).abs().max()), float((eager.double() - want).abs().max())


def test_whole_standin_denoiser_logits():
    torch.manual_seed(0)
    K, N = 1024, 1024
    model = StandInDenoiser(K, N).to(DEV).eval()
    err, err_eager = _logit_errors(model, 2, N, K, 1)
    print(f"[stand-in denoiser B=2 N={N}] max |logit - float64|: fused {err:.2e}, eager fp32 {err_eager:.2e}")
    assert err <= 4 * err_eager


def _models(transformer, N):
    return FusedDiffusionTransformer(transformer=transformer, diffusion_step=100, alpha_init_type="alpha1",
                                     guidance_scale=2.0, content_seq_len=N).to(DEV)


def _teacher_forced(ours, B, N, K, steps, seed):
    """Each step twice from the same x_t: eager attention (the reference arm) and fused attention, on shared uniforms;
    then, with the fused head, the production token path of both arms on the same Philox key.  Both arms continue from
    the eager arm's x_{t-1}."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    cond = torch.randn(B, 77, 512, device=DEV, generator=g)
    cf = torch.randn(B, 77, 512, device=DEV, generator=g) * 0.1
    x_t = torch.full((B, N), K, dtype=torch.int64, device=DEV)
    worst, differ, near_total = 0.0, 0, 0
    with torch.no_grad():
        for ti in steps:
            t = torch.full((B,), ti, device=DEV, dtype=torch.long)
            u = torch.rand(B, K + 1, N, device=DEV, generator=g)
            log_z = ops.as_logical(ops.tokens_to_log_onehot_rows(x_t, K + 1), K + 1)
            arms = []
            for fused in (False, True):
                ours.enable_fused_attention(fused)
                with _fused_calls(ours) as calls:
                    post, recon = ours.p_pred(log_z, cond, cf, t)
                    ours.inject_uniform = lambda shape, dev: u
                    nxt, _ = ours.p_sample(log_z, cond, cf, t, [0] * B, ours.n_sample[ti])
                    ours.inject_uniform = None
                    ours.enable_fused_head()
                    assert ours.fused_head_active
                    tok_head = ours.manual_seed(11, 0).p_sample_tokens(x_t, cond, cf, t)
                    ours.enable_fused_head(False)
                assert calls["delegated"] == 0 and (calls["fused"] > 0) == fused
                arms.append((post, recon, nxt.argmax(1), tok_head))
            ours.enable_fused_attention(False)
            (post_r, recon_r, x_r, head_r), (post_f, recon_f, x_f, head_f) = arms
            worst = max(worst, float((post_f - post_r).abs().max()), float((recon_f - recon_r).abs().max()))
            near = O.near_ties(post_r.cpu(), u.cpu()).numpy()
            diff = (x_f != x_r).cpu().numpy()
            differ += int(diff.sum())
            near_total += int(near.sum())
            assert not (diff & ~near).any(), f"t={ti}: {int((diff & ~near).sum())} tokens differ away from near-ties"
            uh = ops.philox_uniform(B, N, K, seed=11, offset=0, device=DEV)[:, :, :K + 1].permute(0, 2, 1)
            near_h = O.near_ties(post_r.cpu(), uh.cpu()).numpy()
            diff_h = (head_f != head_r).cpu().numpy()
            differ += int(diff_h.sum())
            assert not (diff_h & ~near_h).any(), f"t={ti}: fused head, {int((diff_h & ~near_h).sum())} tokens differ"
            x_t = x_r
    return worst, differ, near_total


def test_teacher_forced_chain_n1024_k4096_standin():
    B, N, K = 2, 1024, 4096
    torch.manual_seed(0)
    ours = _models(StandInDenoiser(K, N, logit_gain=3.0), N).eval()
    worst, differ, near = _teacher_forced(ours, B, N, K, range(99, -1, -11), seed=5)
    print(f"[stand-in, N=1024 K=4096] teacher-forced: max |post/recon fused - eager| = {worst:.2e}; "
          f"{differ} tokens differ, all among {near} logged near-ties")
    assert worst <= H.POST_TOL


def test_cuda_graph_replays_to_the_eager_result():
    torch.manual_seed(0)
    model = StandInDenoiser(1024, 512).to(DEV).eval()
    attention.fuse_self_attention(model)
    x = torch.randint(0, 1025, (2, 512), device=DEV)
    cond = torch.randn(2, 77, 512, device=DEV)
    t = torch.tensor([3, 70], device=DEV)
    with torch.no_grad():
        with _fused_calls(model) as calls:
            eager = model(x, cond, t).clone()
        assert calls == {"fused": 3, "delegated": 0}
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            model(x, cond, t)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = model(x, cond, t)
        out.zero_()
        graph.replay()
        torch.cuda.synchronize()
    assert torch.equal(out, eager)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_tensors_on_a_non_current_device():
    q, k, v = _inputs("ln", 2, 700, seed=9)
    want = attention.self_attention(q, k, v, HEADS, 0.5)
    d1 = torch.device("cuda", 1)
    with torch.cuda.device(0):
        got = attention.self_attention(q.to(d1), k.to(d1), v.to(d1), HEADS, 0.5)
        torch.cuda.synchronize(d1)
    assert got.device == d1 and torch.equal(got.cpu(), want.cpu())


needs_reference = pytest.mark.skipif(not RL.reference_available(), reason="reference not staged (baseline/_ref absent)")


@needs_reference
def test_real_reference_denoiser_logits():
    """Fused against eager fp32 on the reference's own Text2ImageTransformer (19 layers); each fused layer's attention
    output is checked against a float64 restatement of its FullAttention on the same input."""
    torch.manual_seed(0)
    K, N, B = 1024, 1024, 2
    model = RL.build_denoiser(K, N, (32, 32)).to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randint(0, K + 1, (B, N), device=DEV, generator=g)
    cond = torch.randn(B, 77, 512, device=DEV, generator=g)
    t = torch.randint(0, 100, (B,), device=DEV, generator=g)
    errs = []

    def check(mod, args, out):
        assert out[1] is None  # the kernel ran, not the delegated original
        xin = args[0].double()
        with torch.no_grad():
            lin = lambda lay: torch.nn.functional.linear(xin, lay.weight.double(), lay.bias.double())  # noqa: E731
            Bx, T, C = xin.shape
            split = lambda z: z.view(Bx, T, mod.n_head, C // mod.n_head).transpose(1, 2)  # noqa: E731
            q, k, v = split(lin(mod.query)), split(lin(mod.key)), split(lin(mod.value))
            att = torch.softmax((q @ k.transpose(-2, -1)) / math.sqrt(C // mod.n_head), dim=-1)
            y = (att @ v).transpose(1, 2).reshape(Bx, T, C)
            want = torch.nn.functional.linear(y, mod.proj.weight.double(), mod.proj.bias.double())
            errs.append(float((out[0].double() - want).abs().max()) / float(want.abs().max()))

    with torch.no_grad():
        eager = model(x, cond, t)
        n = attention.fuse_self_attention(model)
        hooks = [m.register_forward_hook(check) for m in model.modules() if isinstance(m, attention.FusedSelfAttention)]
        got = model(x, cond, t)
        for hk in hooks:
            hk.remove()
        attention.fuse_self_attention(model, False)
    diff = float((got - eager).abs().max()) / float(eager.abs().max())
    print(f"[reference denoiser] {n} layers fused; logits vs eager fp32 {diff:.2e} of max|logit|; "
          f"worst layer vs float64 {max(errs):.2e}")
    assert n == 19 and len(errs) == 19
    assert max(errs) <= 1e-5 and diff <= 1e-4


@needs_reference
def test_real_reference_teacher_forced_chain():
    B, N, K = 2, 1024, 4096
    torch.manual_seed(0)
    tr = RL.build_denoiser(K, N, (32, 32))
    with torch.no_grad():
        tr.to_logits[-1].weight.mul_(3.0)
    ours = _models(tr, N).eval()
    worst, differ, near = _teacher_forced(ours, B, N, K, [99, 60, 20, 0], seed=6)
    print(f"[reference denoiser, N=1024 K=4096] teacher-forced: max |post/recon fused - eager| = {worst:.2e}; "
          f"{differ} tokens differ, all among {near} logged near-ties")
    assert worst <= H.POST_TOL
