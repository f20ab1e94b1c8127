"""The fused cross-attention without a GPU: argument validation of `d3pm_cross_attention` (before any launch), and the
module swap of `attention.fuse_cross_attention` on a CPU self-plus-cross stand-in of the denoiser (state dict with the
unread `mask` buffer, restore, delegation, `enable_fused_attention(cross=...)`)."""
import copy
import ctypes

import pytest
import torch

import d3pm_b200
from d3pm_b200 import FusedDiffusionTransformer, _lib, attention
from d3pm_b200._lib import D3PMError
from tests.cross_attention_standin import CrossAttention, CrossStandInDenoiser

ERR_INVALID, ERR_ALIGN, ERR_UNSUPPORTED = -1, -2, -3


def _desc(**kw):
    d = _lib.CrossAttnDesc(q=16, k=32, v=48, y=64, B=1, N=8, M=77, heads=16, head_dim=4, pitch_q=64, pitch_kv=64,
                           pitch_y=64, scale=0.5)
    for name, value in kw.items():
        setattr(d, name, value)
    return d


@pytest.mark.parametrize("kw, code, text", [
    ({"q": None}, ERR_INVALID, b"required"),
    ({"k": None}, ERR_INVALID, b"required"),
    ({"v": None}, ERR_INVALID, b"required"),
    ({"y": None}, ERR_INVALID, b"required"),
    ({"B": 0}, ERR_INVALID, b"positive"),
    ({"N": -1}, ERR_INVALID, b"positive"),
    ({"M": 0}, ERR_INVALID, b"positive"),
    ({"heads": 0}, ERR_INVALID, b"positive"),
    ({"head_dim": 8, "heads": 8}, ERR_UNSUPPORTED, b"head_dim"),
    ({"head_dim": 2}, ERR_UNSUPPORTED, b"head_dim"),
    ({"heads": 65536, "pitch_q": 262144, "pitch_kv": 262144, "pitch_y": 262144}, ERR_UNSUPPORTED, b"65535"),
    ({"pitch_q": 66}, ERR_ALIGN, b"multiples of 4"),
    ({"pitch_kv": 70}, ERR_ALIGN, b"multiples of 4"),
    ({"pitch_y": 62}, ERR_ALIGN, b"multiples of 4"),
    ({"pitch_q": 60}, ERR_INVALID, b"shorter"),
    ({"pitch_kv": 60}, ERR_INVALID, b"shorter"),
    ({"pitch_y": 32}, ERR_INVALID, b"shorter"),
    ({"q": 20}, ERR_ALIGN, b"aligned"),
    ({"k": 36}, ERR_ALIGN, b"aligned"),
    ({"v": 40}, ERR_ALIGN, b"aligned"),
    ({"y": 72}, ERR_ALIGN, b"aligned"),
    ({"scale": float("nan")}, ERR_INVALID, b"scale"),
    ({"scale": float("inf")}, ERR_INVALID, b"scale"),
])
def test_cross_attention_rejects_bad_arguments_before_any_launch(kw, code, text):
    lib = d3pm_b200.load_library()
    assert lib.d3pm_cross_attention(None) == ERR_INVALID
    assert b"null descriptor" in lib.d3pm_last_error()
    assert lib.d3pm_cross_attention(ctypes.byref(_desc(**kw))) == code
    assert text in lib.d3pm_last_error()


def test_thin_op_refuses_cpu_tensors():
    q, kv = torch.randn(1, 8, 64), torch.randn(1, 77, 64)
    with pytest.raises(D3PMError, match="CUDA"):
        attention.cross_attention(q, kv, kv, 16, 0.5)


def _model(seed=0):
    torch.manual_seed(seed)
    return CrossStandInDenoiser(K=64, N=32, n_layer=3).eval()


def test_fusing_keeps_the_state_dict_and_strict_loads_work_both_ways():
    model = _model()
    before = {k: v.clone() for k, v in model.state_dict().items()}
    assert "blocks.0.attn2.mask" in before  # the buffer CrossAttention registers and never reads
    originals = [b.attn2 for b in model.blocks]
    assert attention.fuse_cross_attention(model) == 3
    fused = [b.attn2 for b in model.blocks]
    assert all(isinstance(m, attention.FusedCrossAttention) for m in fused)
    assert all(isinstance(b.attn1, torch.nn.Module) and type(b.attn1).__name__ == "FullAttention" for b in model.blocks)
    assert attention.fuse_cross_attention(model) == 3     # a second call changes nothing
    assert all(b.attn2 is m for b, m in zip(model.blocks, fused))
    after = model.state_dict()
    assert list(after.keys()) == list(before.keys())
    for k, v in before.items():
        assert torch.equal(after[k], v), k
    plain = _model(seed=1)                                # different weights, unfused
    plain.load_state_dict(model.state_dict(), strict=True)
    for k, v in before.items():
        assert torch.equal(plain.state_dict()[k], v), k
    other = _model(seed=2)
    with torch.no_grad():
        for b in other.blocks:
            b.attn2.mask.mul_(2.0)                        # the buffer loads too
    model.load_state_dict(other.state_dict(), strict=True)  # an unfused checkpoint into the fused model
    for k, v in other.state_dict().items():
        assert torch.equal(model.state_dict()[k], v), k
    # the weights the fused module runs are the original module's own tensors
    assert all(b.attn2.key.weight is o.key.weight for b, o in zip(model.blocks, originals))
    # and the restored originals carry the loaded buffer
    attention.fuse_cross_attention(model, enable=False)
    assert all(torch.equal(b.attn2.mask, o.attn2.mask) for b, o in zip(model.blocks, other.blocks))


def test_disable_restores_the_original_module_objects():
    model = _model()
    originals = [b.attn2 for b in model.blocks]
    attention.fuse_cross_attention(model)
    assert attention.fuse_cross_attention(model, enable=False) == 3
    assert all(b.attn2 is o for b, o in zip(model.blocks, originals))
    assert attention.fuse_cross_attention(model, enable=False) == 0


def test_a_model_without_a_qualifying_cross_attention_raises():
    with pytest.raises(D3PMError, match="no CrossAttention"):
        attention.fuse_cross_attention(torch.nn.Sequential(torch.nn.Linear(64, 64)))
    wide = torch.nn.Sequential(CrossAttention(77, 64, 512, 8, seq_len=16))  # head width 8: not what the kernel covers
    with pytest.raises(D3PMError, match="no CrossAttention"):
        attention.fuse_cross_attention(wide)
    assert isinstance(wide[0], CrossAttention)
    # a FullAttention is not a CrossAttention (and the reverse)
    from tests.attention_standin import StandInDenoiser
    with pytest.raises(D3PMError, match="no CrossAttention"):
        attention.fuse_cross_attention(StandInDenoiser(K=64, N=32))


@pytest.mark.parametrize("grad_of", ["x", "encoder_output", "parameters"])
def test_grad_enabled_calls_delegate_to_the_original_module(grad_of):
    """Training-time calls run the reference's module itself: output and gradients are those of an unfused copy."""
    torch.manual_seed(3)
    ref = CrossAttention(77, 64, 512, 16, seq_len=16)
    fused = attention.FusedCrossAttention(copy.deepcopy(ref))
    if grad_of != "parameters":
        for m in (ref, fused):
            m.requires_grad_(False)
    x1 = torch.randn(2, 16, 64, requires_grad=grad_of == "x")
    c1 = torch.randn(2, 77, 512, requires_grad=grad_of == "encoder_output")
    x2 = x1.detach().clone().requires_grad_(x1.requires_grad)
    c2 = c1.detach().clone().requires_grad_(c1.requires_grad)
    y1, a1 = ref(x1, c1)
    y2, a2 = fused(x2, c2)
    assert a2 is not None and torch.equal(y1, y2) and torch.equal(a1, a2)
    (y1.square().sum() + a1.sum()).backward()
    (y2.square().sum() + a2.sum()).backward()
    for t1, t2 in ((x1, x2), (c1, c2)):
        assert (t1.grad is None) == (t2.grad is None)
        assert t1.grad is None or torch.equal(t1.grad, t2.grad)
    for (n, p), q in zip(ref.named_parameters(), fused.parameters()):
        assert (p.grad is None) == (q.grad is None), n
        assert p.grad is None or torch.equal(p.grad, q.grad), n


def test_fused_diffusion_transformer_enable_fused_attention_cross():
    ours = FusedDiffusionTransformer(transformer=_model(), diffusion_step=100, alpha_init_type="alpha1", guidance_scale=2.0,
                                     content_seq_len=32)
    keys = list(ours.state_dict().keys())
    crosses = [b.attn2 for b in ours.transformer.blocks]
    count = lambda cls: sum(isinstance(m, cls) for m in ours.modules())  # noqa: E731
    assert ours.enable_fused_attention() is ours                  # the default fuses the self-attention only
    assert count(attention.FusedSelfAttention) == 3 and count(attention.FusedCrossAttention) == 0
    assert all(b.attn2 is c for b, c in zip(ours.transformer.blocks, crosses))
    assert ours.enable_fused_attention(cross=True) is ours
    assert ours.enable_fused_attention(cross=True) is ours        # idempotent
    assert count(attention.FusedSelfAttention) == 3 and count(attention.FusedCrossAttention) == 3
    assert list(ours.state_dict().keys()) == keys
    ours.enable_fused_attention(False)
    assert count(attention.FusedSelfAttention) == 0 and count(attention.FusedCrossAttention) == 0
    assert all(b.attn2 is c for b, c in zip(ours.transformer.blocks, crosses))
