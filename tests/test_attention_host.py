"""The fused self-attention without a GPU: argument validation of `d3pm_self_attention` (before any launch), and the
module swap of `attention.fuse_self_attention` on a CPU stand-in of the denoiser (state dict, restore, delegation)."""
import copy
import ctypes

import pytest
import torch

import d3pm_b200
from d3pm_b200 import FusedDiffusionTransformer, _lib, attention
from d3pm_b200._lib import D3PMError
from tests.attention_standin import FullAttention, StandInDenoiser

ERR_INVALID, ERR_ALIGN, ERR_UNSUPPORTED = -1, -2, -3


def _desc(**kw):
    d = _lib.AttnDesc(q=16, k=32, v=48, y=64, B=1, N=8, heads=16, head_dim=4, pitch_qkv=64, pitch_y=64, scale=0.5)
    for name, value in kw.items():
        setattr(d, name, value)
    return d


@pytest.mark.parametrize("kw, code, text", [
    ({"q": None}, ERR_INVALID, b"required"),
    ({"v": None}, ERR_INVALID, b"required"),
    ({"y": None}, ERR_INVALID, b"required"),
    ({"B": 0}, ERR_INVALID, b"positive"),
    ({"N": -1}, ERR_INVALID, b"positive"),
    ({"heads": 0}, ERR_INVALID, b"positive"),
    ({"head_dim": 8, "heads": 8}, ERR_UNSUPPORTED, b"head_dim"),
    ({"head_dim": 2}, ERR_UNSUPPORTED, b"head_dim"),
    ({"pitch_qkv": 66}, ERR_ALIGN, b"multiples of 4"),
    ({"pitch_y": 70}, ERR_ALIGN, b"multiples of 4"),
    ({"pitch_qkv": 60}, ERR_INVALID, b"shorter"),
    ({"k": 36}, ERR_ALIGN, b"aligned"),
    ({"y": 72}, ERR_ALIGN, b"aligned"),
    ({"scale": float("nan")}, ERR_INVALID, b"scale"),
])
def test_self_attention_rejects_bad_arguments_before_any_launch(kw, code, text):
    lib = d3pm_b200.load_library()
    assert lib.d3pm_self_attention(None) == ERR_INVALID
    assert lib.d3pm_self_attention(ctypes.byref(_desc(**kw))) == code
    assert text in lib.d3pm_last_error()


def test_thin_op_refuses_cpu_tensors():
    q = torch.randn(1, 8, 64)
    with pytest.raises(D3PMError, match="CUDA"):
        attention.self_attention(q, q, q, 16, 0.5)


def _model(seed=0):
    torch.manual_seed(seed)
    return StandInDenoiser(K=64, N=32, n_layer=3).eval()


def test_fusing_keeps_the_state_dict_and_strict_loads_work_both_ways():
    model = _model()
    before = {k: v.clone() for k, v in model.state_dict().items()}
    originals = [b.attn1 for b in model.blocks]
    assert attention.fuse_self_attention(model) == 3
    fused = [b.attn1 for b in model.blocks]
    assert all(isinstance(m, attention.FusedSelfAttention) for m in fused)
    assert attention.fuse_self_attention(model) == 3     # a second call changes nothing
    assert all(b.attn1 is m for b, m in zip(model.blocks, fused))
    after = model.state_dict()
    assert list(after.keys()) == list(before.keys())
    for k, v in before.items():
        assert torch.equal(after[k], v), k
    plain = _model(seed=1)                               # different weights, unfused
    plain.load_state_dict(model.state_dict(), strict=True)
    for k, v in before.items():
        assert torch.equal(plain.state_dict()[k], v), k
    other = _model(seed=2)
    model.load_state_dict(other.state_dict(), strict=True)  # an unfused checkpoint into the fused model
    for k, v in other.state_dict().items():
        assert torch.equal(model.state_dict()[k], v), k
    # the weights the fused module runs are the original module's own tensors
    assert all(b.attn1.query.weight is o.query.weight for b, o in zip(model.blocks, originals))


def test_disable_restores_the_original_module_objects():
    model = _model()
    originals = [b.attn1 for b in model.blocks]
    attention.fuse_self_attention(model)
    assert attention.fuse_self_attention(model, enable=False) == 3
    assert all(b.attn1 is o for b, o in zip(model.blocks, originals))
    assert attention.fuse_self_attention(model, enable=False) == 0


def test_a_model_without_a_qualifying_full_attention_raises():
    with pytest.raises(D3PMError, match="no FullAttention"):
        attention.fuse_self_attention(torch.nn.Sequential(torch.nn.Linear(64, 64)))
    wide = torch.nn.Sequential(FullAttention(64, 8))  # head width 8: not what the kernel covers
    with pytest.raises(D3PMError, match="no FullAttention"):
        attention.fuse_self_attention(wide)
    assert isinstance(wide[0], FullAttention)


def test_grad_enabled_calls_delegate_to_the_original_module():
    """Training-time calls run the reference's module itself: output and gradients are those of an unfused copy."""
    torch.manual_seed(3)
    ref = FullAttention(64, 16)
    fused = attention.FusedSelfAttention(copy.deepcopy(ref))
    x1 = torch.randn(2, 16, 64, requires_grad=True)
    x2 = x1.detach().clone().requires_grad_(True)
    y1, a1 = ref(x1, None)
    y2, a2 = fused(x2, None)
    assert torch.equal(y1, y2) and torch.equal(a1, a2)
    (y1.square().sum() + a1.sum()).backward()
    (y2.square().sum() + a2.sum()).backward()
    assert torch.equal(x1.grad, x2.grad)
    for (n, p), q in zip(ref.named_parameters(), fused.parameters()):
        assert torch.equal(p.grad, q.grad), n


def test_fused_diffusion_transformer_enable_fused_attention():
    ours = FusedDiffusionTransformer(transformer=_model(), diffusion_step=100, alpha_init_type="alpha1", guidance_scale=2.0,
                                     content_seq_len=32)
    keys = list(ours.state_dict().keys())
    assert ours.enable_fused_attention() is ours
    assert ours.enable_fused_attention() is ours  # idempotent, like enable_fused_head()
    assert sum(isinstance(m, attention.FusedSelfAttention) for m in ours.modules()) == 3
    assert list(ours.state_dict().keys()) == keys
    ours.enable_fused_attention(False)
    assert not any(isinstance(m, attention.FusedSelfAttention) for m in ours.modules())
