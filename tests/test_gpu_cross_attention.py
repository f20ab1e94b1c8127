"""The fused cross-attention (`d3pm_cross_attention`, `attention.FusedCrossAttention`) on the GPU.

* the kernel against a float64 restatement on sampled query rows, next to eager fp32's own error, over M (condition rows)
  from 1 to past the kernel's 128-key staging tile, N from 1 to 8200, B in {1, 3, 16}, 16 heads, and inputs that stress the
  softmax (scores up to about ±300, all keys and values equal - the zeroed condition of the shipped pipeline -, one
  dominant key);
* a batch past one grid, pitched inputs, and delegation (grad, autocast, a mask), bit for bit;
* a self-plus-cross stand-in denoiser (tests/cross_attention_standin.py) with both attentions fused: logits within 4x eager
  fp32's error against float64, every fused module running its kernel;
* a teacher-forced chain at N = 1024, K = 4096 with `enable_fused_attention(cross=True)`, with and without the fused head;
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
from tests.cross_attention_standin import CrossAttention, CrossStandInDenoiser

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
HEADS, HD = 16, 4
TOL = 2e-5  # of max|v|


def _inputs(kind, B, N, M, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    q = torch.randn(B, N, HEADS * HD, device=DEV, generator=g)
    k, v = (torch.randn(B, M, HEADS * HD, device=DEV, generator=g) for _ in range(2))
    if kind == "large":         # scale 0.5: scores of std ~70, up to about ±300
        q, k = q * 8.5, k * 8.5
    elif kind == "equal_keys":  # key(0) and value(0): every row is the Linear's bias, y = that row of v
        k = k[:, :1].expand(B, M, HEADS * HD).contiguous()
        v = v[:, :1].expand(B, M, HEADS * HD).contiguous()
    elif kind == "dominant":    # one key far above the rest for every query
        q = q.abs()
        k = k * 0.1
        k[:, M // 2] = 12.0
    return q, k, v


def _restated(q, k, v, rows, dtype):
    """softmax(scale q kᵀ) v per head for the query rows `rows`, in `dtype`."""
    B, N, C = q.shape
    M = k.shape[1]
    qs = q[:, rows].to(dtype).view(B, len(rows), HEADS, HD).transpose(1, 2)
    kh = k.to(dtype).view(B, M, HEADS, HD).transpose(1, 2)
    vh = v.to(dtype).view(B, M, HEADS, HD).transpose(1, 2)
    att = torch.softmax((qs @ kh.transpose(-2, -1)) * (1.0 / math.sqrt(HD)), dim=-1)
    return (att @ vh).transpose(1, 2).reshape(B, len(rows), C)


# every M of {1, 31, 32, 33, 77, 300} and 129 / 1100 (past the 128-key staging tile), every N of {1, 77, 1000, 4096, 8200},
# every B of {1, 3, 16}
SHAPES = [(1, 1, 1), (3, 1, 77), (1, 77, 31), (3, 77, 32), (16, 77, 33), (16, 1000, 1), (1, 1000, 77), (3, 1000, 300),
          (1, 4096, 77), (3, 4096, 129), (16, 4096, 77), (16, 4096, 300), (1, 8200, 1100), (3, 8200, 77), (16, 8200, 33),
          (16, 8200, 129)]


@pytest.mark.parametrize("kind", ["ln", "large", "equal_keys", "dominant"])
@pytest.mark.parametrize("B, N, M", SHAPES)
def test_kernel_matches_float64_on_sampled_rows(B, N, M, kind):
    q, k, v = _inputs(kind, B, N, M, seed=B * 100003 + N * 101 + M)
    y = attention.cross_attention(q, k, v, HEADS, 1.0 / math.sqrt(HD))
    g = torch.Generator().manual_seed(N)
    rows = torch.unique(torch.cat((torch.tensor([0, N - 1]), torch.randint(0, N, (62,), generator=g)))).to(DEV)
    want = _restated(q, k, v, rows, torch.float64)
    eager = _restated(q, k, v, rows, torch.float32)
    scale = float(v.abs().max())
    err = float((y[:, rows].double() - want).abs().max()) / scale
    err_eager = float((eager.double() - want).abs().max()) / scale
    print(f"[cross-attention B={B} N={N} M={M} {kind}] kernel {err:.2e}, eager fp32 {err_eager:.2e} of max|v|")
    assert y.shape == q.shape and torch.isfinite(y).all()
    assert err <= TOL


def test_more_videos_than_one_grid_holds():
    """B above the 65535 videos of one launch's grid: the batch runs as several launches, each video against its own
    condition rows."""
    B, N, M = 65537, 3, 5
    q, k, v = _inputs("ln", B, N, M, seed=4)
    y = attention.cross_attention(q, k, v, HEADS, 0.5)
    for b in (0, 65534, 65535, 65536):
        want = _restated(q[b:b + 1], k[b:b + 1], v[b:b + 1], torch.arange(N, device=DEV), torch.float64)
        assert float((y[b:b + 1].double() - want).abs().max()) <= TOL * float(v.abs().max()), b


def test_pitched_inputs_are_read_in_place():
    """q a column slice of a [B, N, 2C] tensor, k and v column slices of one [B, M, 2C] tensor: the result of contiguous
    copies, bit for bit; and k, v of different strides (copied) too."""
    B, N, M, C = 3, 300, 77, HEADS * HD
    qx = torch.randn(B, N, 2 * C, device=DEV)
    kv = torch.randn(B, M, 2 * C, device=DEV)
    q, k, v = qx[..., C:], kv[..., :C], kv[..., C:]
    want = attention.cross_attention(q.contiguous(), k.contiguous(), v.contiguous(), HEADS, 0.5)
    assert torch.equal(attention.cross_attention(q, k, v, HEADS, 0.5), want)
    assert torch.equal(attention.cross_attention(q, k, v.contiguous(), HEADS, 0.5), want)


def _pair(seed=0, N=200):
    torch.manual_seed(seed)
    ref = CrossAttention(77, 64, 512, HEADS, seq_len=N).to(DEV)
    return ref, attention.FusedCrossAttention(copy.deepcopy(ref))


@pytest.mark.parametrize("grad_of", ["x", "encoder_output"])
def test_delegation_with_grad_is_bit_identical(grad_of):
    ref, fused = _pair()
    for m in (ref, fused):
        m.requires_grad_(False)
    x1 = torch.randn(2, 200, 64, device=DEV, requires_grad=grad_of == "x")
    c1 = torch.randn(2, 77, 512, device=DEV, requires_grad=grad_of == "encoder_output")
    x2 = x1.detach().clone().requires_grad_(x1.requires_grad)
    c2 = c1.detach().clone().requires_grad_(c1.requires_grad)
    y1, a1 = ref(x1, c1)
    y2, a2 = fused(x2, c2)
    assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
    (y1.square().sum() + a1.sum()).backward()
    (y2.square().sum() + a2.sum()).backward()
    t1, t2 = (x1, x2) if grad_of == "x" else (c1, c2)
    assert torch.equal(t1.grad, t2.grad)


def test_delegation_under_autocast_and_with_a_mask_is_bit_identical():
    ref, fused = _pair(1)
    x = torch.randn(2, 200, 64, device=DEV)
    c = torch.randn(2, 77, 512, device=DEV)
    with torch.no_grad():
        with torch.autocast("cuda"):
            y1, a1 = ref(x, c)
            y2, a2 = fused(x, c)
        assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
        mask = torch.ones(2, 200, 77, dtype=torch.bool, device=DEV)
        y1, a1 = ref(x, c, mask=mask)
        y2, a2 = fused(x, c, mask=mask)
        assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
        y3, a3 = fused(x, c)  # and the fused path itself: no map, the same output within the kernel's tolerance
        assert a3 is None and float((y3 - y1).abs().max()) <= 1e-4 * float(y1.abs().max())


@contextlib.contextmanager
def _fused_calls(model):
    """Counts, per kind, the forwards of `model`'s fused attention modules that ran the kernel (second output None) and
    those that delegated to the original module: a fused model that quietly delegated would have exactly eager's numbers."""
    calls = {"self": 0, "cross": 0, "delegated": 0}

    def hook(mod, args, out):
        kind = "cross" if isinstance(mod, attention.FusedCrossAttention) else "self"
        calls[kind if out[1] is None else "delegated"] += 1

    hooks = [m.register_forward_hook(hook) for m in model.modules()
             if isinstance(m, (attention.FusedSelfAttention, attention.FusedCrossAttention))]
    try:
        yield calls
    finally:
        for hk in hooks:
            hk.remove()


def test_whole_standin_denoiser_logits():
    torch.manual_seed(0)
    K, N, B = 1024, 1024, 2
    model = CrossStandInDenoiser(K, N).to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randint(0, K + 1, (B, N), device=DEV, generator=g)
    cond = torch.randn(B, 77, 512, device=DEV, generator=g)
    t = torch.randint(0, 100, (B,), device=DEV, generator=g)
    with torch.no_grad():
        want = copy.deepcopy(model).double()(x, cond.double(), t)
        eager = model(x, cond, t)
        n_self = attention.fuse_self_attention(model)
        n_cross = attention.fuse_cross_attention(model)
        with _fused_calls(model) as calls:
            got = model(x, cond, t)
        attention.fuse_self_attention(model, False)
        attention.fuse_cross_attention(model, False)
    assert n_self == n_cross == 3
    assert calls == {"self": 3, "cross": 3, "delegated": 0}
    err, err_eager = float((got.double() - want).abs().max()), float((eager.double() - want).abs().max())
    print(f"[self+cross stand-in denoiser B={B} N={N}] max |logit - float64|: fused {err:.2e}, eager fp32 {err_eager:.2e}")
    assert err <= 4 * err_eager


def _models(transformer, N):
    return FusedDiffusionTransformer(transformer=transformer, diffusion_step=100, alpha_init_type="alpha1",
                                     guidance_scale=2.0, content_seq_len=N).to(DEV)


def _teacher_forced(ours, B, N, K, steps, seed):
    """Each step twice from the same x_t: eager attention (the reference arm) and both attentions fused, on shared
    uniforms; then, with the fused head, the production token path of both arms on the same Philox key.  Both arms continue
    from the eager arm's x_{t-1}.  `cf` is the zeroed condition of the shipped pipeline."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    cond = torch.randn(B, 77, 512, device=DEV, generator=g)
    cf = torch.zeros(B, 77, 512, device=DEV)
    x_t = torch.full((B, N), K, dtype=torch.int64, device=DEV)
    worst, differ, near_total = 0.0, 0, 0
    with torch.no_grad():
        for ti in steps:
            t = torch.full((B,), ti, device=DEV, dtype=torch.long)
            u = torch.rand(B, K + 1, N, device=DEV, generator=g)
            log_z = ops.as_logical(ops.tokens_to_log_onehot_rows(x_t, K + 1), K + 1)
            arms = []
            for fused in (False, True):
                ours.enable_fused_attention(fused, cross=True)
                with _fused_calls(ours) as calls:
                    post, recon = ours.p_pred(log_z, cond, cf, t)
                    ours.inject_uniform = lambda shape, dev: u
                    nxt, _ = ours.p_sample(log_z, cond, cf, t, [0] * B, ours.n_sample[ti])
                    ours.inject_uniform = None
                    ours.enable_fused_head()
                    assert ours.fused_head_active
                    tok_head = ours.manual_seed(11, 0).p_sample_tokens(x_t, cond, cf, t)
                    ours.enable_fused_head(False)
                assert calls["delegated"] == 0
                assert (calls["self"] > 0) == fused and calls["cross"] == calls["self"]
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
    ours = _models(CrossStandInDenoiser(K, N, logit_gain=3.0), N).eval()
    worst, differ, near = _teacher_forced(ours, B, N, K, range(99, -1, -11), seed=5)
    print(f"[self+cross stand-in, N=1024 K=4096] teacher-forced: max |post/recon fused - eager| = {worst:.2e}; "
          f"{differ} tokens differ, all among {near} logged near-ties")
    assert worst <= H.POST_TOL


def test_cuda_graph_replays_to_the_eager_result():
    torch.manual_seed(0)
    model = CrossStandInDenoiser(1024, 512).to(DEV).eval()
    attention.fuse_self_attention(model)
    attention.fuse_cross_attention(model)
    x = torch.randint(0, 1025, (2, 512), device=DEV)
    cond = torch.randn(2, 77, 512, device=DEV)
    t = torch.tensor([3, 70], device=DEV)
    with torch.no_grad():
        with _fused_calls(model) as calls:
            eager = model(x, cond, t).clone()
        assert calls == {"self": 3, "cross": 3, "delegated": 0}
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
    q, k, v = _inputs("ln", 2, 700, 77, seed=9)
    want = attention.cross_attention(q, k, v, HEADS, 0.5)
    d1 = torch.device("cuda", 1)
    with torch.cuda.device(0):
        got = attention.cross_attention(q.to(d1), k.to(d1), v.to(d1), HEADS, 0.5)
        torch.cuda.synchronize(d1)
    assert got.device == d1 and torch.equal(got.cpu(), want.cpu())


needs_reference = pytest.mark.skipif(not RL.reference_available(), reason="reference not staged (baseline/_ref absent)")


@needs_reference
def test_real_reference_denoiser_logits():
    """Both attentions fused against eager fp32 on the reference's own Text2ImageTransformer (19 layers); each fused
    CrossAttention's output is checked against a float64 restatement of its own weights on the same input."""
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
        xin, cin = args[0].double(), args[1].double()
        with torch.no_grad():
            lin = lambda lay, z: torch.nn.functional.linear(z, lay.weight.double(), lay.bias.double())  # noqa: E731
            Bx, T, C = xin.shape
            split = lambda z: z.view(Bx, z.shape[1], mod.n_head, C // mod.n_head).transpose(1, 2)  # noqa: E731
            q, k, v = split(lin(mod.query, xin)), split(lin(mod.key, cin)), split(lin(mod.value, cin))
            att = torch.softmax((q @ k.transpose(-2, -1)) / math.sqrt(C // mod.n_head), dim=-1)
            y = (att @ v).transpose(1, 2).reshape(Bx, T, C)
            want = lin(mod.proj, y)
            errs.append(float((out[0].double() - want).abs().max()) / float(want.abs().max()))

    with torch.no_grad():
        eager = model(x, cond, t)
        attention.fuse_self_attention(model)
        n = attention.fuse_cross_attention(model)
        hooks = [m.register_forward_hook(check) for m in model.modules() if isinstance(m, attention.FusedCrossAttention)]
        got = model(x, cond, t)
        for hk in hooks:
            hk.remove()
        attention.fuse_self_attention(model, False)
        attention.fuse_cross_attention(model, False)
    diff = float((got - eager).abs().max()) / float(eager.abs().max())
    print(f"[reference denoiser] {n} cross-attention layers fused (and the self-attention); logits vs eager fp32 "
          f"{diff:.2e} of max|logit|; worst cross layer vs float64 {max(errs):.2e}")
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
    print(f"[reference denoiser, N=1024 K=4096, self+cross fused] teacher-forced: max |post/recon fused - eager| = "
          f"{worst:.2e}; {differ} tokens differ, all among {near} logged near-ties")
    assert worst <= H.POST_TOL
