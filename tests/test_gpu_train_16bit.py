"""float16 / bfloat16 denoiser logits on the training side: `d3pm_train_rows` reads them in place and writes their
gradient in the same type.  The reference for every comparison is the fp32 kernel on `logits.float()`, which
test_gpu_train.py pins to the reference's fixtures and the oracle.  Needs a B200."""
import ctypes
import types

import pytest
import torch

import d3pm_b200
from d3pm_b200 import _lib, ops, train

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = (torch.float16, torch.bfloat16)
MW = (1.0, 0.5)
ERR_ALIGN, ERR_UNSUPPORTED = -2, -3  # D3PM_ERR_ALIGN, D3PM_ERR_UNSUPPORTED


class LeafDenoiser(torch.nn.Module):
    """Returns a leaf logits tensor the way Text2ImageTransformer returns its output (a [B,K,N] view of [B,N,K])."""

    def __init__(self, K, logits_bnk):
        super().__init__()
        self.content_emb = types.SimpleNamespace(num_embed=K + 1)
        self.to_logits = torch.nn.Sequential(torch.nn.Identity(), torch.nn.Linear(1, 1))
        self.logits = logits_bnk

    def forward(self, x_t, cond, t):
        return self.logits.permute(0, 2, 1)


def _model(K, T, N, logits, aux=0.0):
    return d3pm_b200.FusedDiffusionTransformer(transformer=LeafDenoiser(K, logits), diffusion_step=T, alpha_init_type="alpha1",
                                               guidance_scale=2.0, content_seq_len=N, auxiliary_loss_weight=aux,
                                               adaptive_auxiliary_loss=True).to(DEV)


def _data(K, scale, B=3, N=1024, T=100):
    """The inputs of test_stream_kernel_equals_row_kernel: both clamps fire at scale 9, t = 0 is present, and some
    unmasked tokens kept their clean value."""
    g = torch.Generator().manual_seed(K + int(scale))
    logits = torch.randn(B, N, K, generator=g) * scale
    if scale > 5:
        logits[:, ::7, 5] += 200.0
    x0 = torch.randint(0, K, (B, N), generator=g).to(DEV)
    t = torch.tensor([0, 37, 99][:B]).to(DEV)
    m = _model(K, T, N, torch.zeros(1, 1, K, device=DEV))
    x_t = m.q_sample_tokens(x0, t)
    if B > 1:
        x_t[1, :50] = x0[1, :50]
    w_main = torch.tensor([0.7, 1.3, 0.01][:B], device=DEV)
    w_aux = torch.tensor([0.2, 0.0, 0.5][:B], device=DEV)
    return logits.to(DEV), x0, x_t, t, m.coef_table(), w_main, w_aux


def _runs(rows, pitch, x0, x_t, t, table, w_main, w_aux):
    return {bw: train._train_rows(rows, pitch, x0, x_t, t, table, MW, backward=bw, w_main=w_main, w_aux=w_aux,
                                  want_recon=bw != 1) for bw in (0, 1, 2)}


def _direct(rows, pitch, grad, pitch_grad, x0, x_t, t, table, w_main, w_aux, dtype):
    """d3pm_train_rows on caller-made rows, backward == 2 (0 when grad is None); returns (status code, tok_main)."""
    B, N, K = rows.shape
    tok = torch.empty(2, B, N, device=DEV)
    d = _lib.TrainDesc()
    d.logits, d.x0, d.x_t, d.t, d.coef_table = rows.data_ptr(), x0.data_ptr(), x_t.data_ptr(), t.data_ptr(), table.data_ptr()
    d.w_main, d.w_aux, d.tok_main, d.tok_aux = w_main.data_ptr(), w_aux.data_ptr(), tok[0].data_ptr(), tok[1].data_ptr()
    d.grad, d.pitch_grad = (0 if grad is None else grad.data_ptr()), pitch_grad
    d.B, d.N, d.K, d.T = B, N, K, table.shape[0]
    d.pitch, d.backward, d.logits_dtype = pitch, 2 if grad is not None else 0, ops.LOGITS_DTYPES[dtype]
    d.mask_weight_masked, d.mask_weight_unmasked = MW
    d.stream = ops._stream(torch.device(DEV))
    rc = d3pm_b200.load_library().d3pm_train_rows(ctypes.byref(d))
    return rc, tok[0]


@pytest.mark.parametrize("scale", [1.0, 9.0])
@pytest.mark.parametrize("dtype", DTYPES, ids=str)
@pytest.mark.parametrize("K", [1024, 2048, 4096])
def test_16bit_rows_equal_the_fp32_kernel_on_their_cast(K, dtype, scale):
    logits, x0, x_t, t, table, w_main, w_aux = _data(K, scale)
    l16 = logits.to(dtype)
    want = _runs(l16.float(), K, x0, x_t, t, table, w_main, w_aux)
    got = _runs(l16, K, x0, x_t, t, table, w_main, w_aux)
    for bw in (0, 2):
        for name in ("tok_main", "tok_aux", "x0_recon", "xtm1_recon"):
            assert torch.equal(got[bw][name], want[bw][name]), (bw, name)
    for bw in (1, 2):
        assert got[bw]["grad"].dtype == dtype
        assert torch.equal(got[bw]["grad"], want[bw]["grad"].to(dtype)), bw
    # one pass = the forward pass plus the gradient pass
    assert torch.equal(got[2]["grad"], got[1]["grad"])
    for name in ("tok_main", "tok_aux", "x0_recon", "xtm1_recon"):
        assert torch.equal(got[2][name], got[0][name]), name


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_16bit_pitches_and_refusals(dtype):
    K = 2048
    logits, x0, x_t, t, table, w_main, w_aux = _data(K, 9.0)
    l16 = logits.to(dtype)
    padded = torch.full((3, 1024, K + 8), 7.0, dtype=dtype, device=DEV)
    padded[..., :K] = l16
    grad_pad = torch.full((3, 1024, K + 8), 5.0, dtype=dtype, device=DEV)
    rc, tok = _direct(padded[..., :K], K + 8, grad_pad[..., :K], K + 8, x0, x_t, t, table, w_main, w_aux, dtype)
    assert rc == 0
    want = train._train_rows(l16.float(), K, x0, x_t, t, table, MW, backward=2, w_main=w_main, w_aux=w_aux)
    torch.cuda.synchronize()
    assert torch.equal(tok, want["tok_main"])
    assert torch.equal(grad_pad[..., :K], want["grad"].to(dtype))
    assert bool((grad_pad[..., K:] == 5.0).all())  # the padding is left alone
    # pitch K + 4: 16-bit rows would not start on 16-byte boundaries
    odd = torch.zeros(3, 1024, K + 4, dtype=dtype, device=DEV)
    assert _direct(odd[..., :K], K + 4, None, 0, x0, x_t, t, table, w_main, w_aux, dtype)[0] == ERR_ALIGN
    assert _direct(l16, K, odd[..., :K], K + 4, x0, x_t, t, table, w_main, w_aux, dtype)[0] == ERR_ALIGN
    # shapes the stream kernel does not take: the caller casts
    small = torch.zeros(3, 1024, 64, dtype=dtype, device=DEV)
    x0s = torch.zeros(3, 1024, dtype=torch.long, device=DEV)
    assert _direct(small, 64, None, 0, x0s, x0s, t, table, w_main, w_aux, dtype)[0] == ERR_UNSUPPORTED
    assert _direct(l16[:1], K, None, 0, x0[:1], x_t[:1], t[:1], table, w_main, w_aux, dtype)[0] == ERR_UNSUPPORTED


def _train_step(K, N, leaf, x0, tt, pt, *, return_logits=False, loss_factor=1.0, aux=1e-3):
    """One training step of a fresh module on the leaf logits, at fixed timesteps and noise."""
    m = _model(K, 100, N, leaf, aux=aux)
    m.sample_time = lambda b, device, method="uniform": (tt, pt)
    m.manual_seed(5)
    out = m({"content_token": x0}, return_loss=True, return_logits=return_logits)
    (out["loss"] * loss_factor).backward()
    return out


def _spy(monkeypatch):
    calls = []
    real = train._train_rows

    def spy(rows, pitch, x0, x_t, t, coef_table, mask_weight, **kw):
        calls.append(dict(rows=rows, pitch=pitch, x0=x0, x_t=x_t, t=t, table=coef_table, mw=mask_weight, **kw))
        return real(rows, pitch, x0, x_t, t, coef_table, mask_weight, **kw)
    monkeypatch.setattr(train, "_train_rows", spy)
    return calls


def _fp32_gradient(call, w_main, w_aux):
    """The fp32 kernel's gradient pass on the cast of the rows a 16-bit call saw, for the given weights."""
    return train._train_rows(call["rows"].float(), call["rows"].shape[2], call["x0"], call["x_t"], call["t"], call["table"],
                             call["mw"], backward=1, w_main=w_main, w_aux=w_aux)["grad"]


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_module_trains_on_16bit_logits_in_place(dtype, monkeypatch):
    K, B, N = 2048, 3, 1024
    g = torch.Generator().manual_seed(11)
    base = (torch.randn(B, N, K, generator=g) * 3).to(DEV).to(dtype)
    x0 = torch.randint(0, K, (B, N), generator=g).to(DEV)
    tt, pt = torch.tensor([0, 37, 99], device=DEV), torch.tensor([0.01, 0.02, 0.01], device=DEV)

    ref_leaf = base.float().requires_grad_(True)
    ref = _train_step(K, N, ref_leaf, x0, tt, pt, return_logits=True)
    leaf = base.clone().requires_grad_(True)
    calls = _spy(monkeypatch)
    out = _train_step(K, N, leaf, x0, tt, pt, return_logits=True)
    # forward: the losses only, on the 16-bit rows themselves (no fp32 copy); backward: the gradient pass
    assert [c["backward"] for c in calls] == [0, 1]
    for c in calls:
        assert c["rows"].dtype == dtype and c["rows"].data_ptr() == leaf.data_ptr()
    assert torch.equal(out["loss"], ref["loss"])
    assert torch.equal(out["pred_data"], ref["pred_data"])
    assert torch.equal(out["logits"], ref["logits"])
    assert leaf.grad.dtype == dtype
    want = _fp32_gradient(calls[1], calls[1]["w_main"], calls[1]["w_aux"]).to(dtype)
    assert torch.equal(leaf.grad, want)
    # the weights are the true upstream ones: the fp32 model's gradient, cast (up to one unit in the last place)
    assert (leaf.grad.float() - ref_leaf.grad.to(dtype).float()).abs().max() <= 8e-3 * ref_leaf.grad.abs().max()


@pytest.mark.parametrize("dtype", DTYPES, ids=str)
def test_module_casts_shapes_the_16bit_kernel_does_not_take(dtype, monkeypatch):
    K, B, N = 64, 1, 64
    g = torch.Generator().manual_seed(12)
    base = (torch.randn(B, N, K, generator=g) * 3).to(DEV).to(dtype)
    x0 = torch.randint(0, K, (B, N), generator=g).to(DEV)
    tt, pt = torch.tensor([37], device=DEV), torch.tensor([0.01], device=DEV)
    ref_leaf = base.float().requires_grad_(True)
    ref = _train_step(K, N, ref_leaf, x0, tt, pt)
    leaf = base.clone().requires_grad_(True)
    calls = _spy(monkeypatch)
    out = _train_step(K, N, leaf, x0, tt, pt)
    assert all(c["rows"].dtype == torch.float32 for c in calls)
    assert torch.equal(out["loss"], ref["loss"])
    assert leaf.grad.dtype == dtype and torch.equal(leaf.grad, ref_leaf.grad.to(dtype))


def _ulps(a, b):
    """|a - b| in float16 units in the last place (bit patterns mapped to ordered integers)."""
    def ordered(x):
        i = x.view(torch.int16).to(torch.int32)
        return torch.where(i < 0, -(i & 0x7FFF), i)
    return (ordered(a) - ordered(b)).abs()


def test_float16_gradient_under_a_loss_scaler(monkeypatch):
    K, B, N, S = 1024, 3, 1024, 65536.0
    g = torch.Generator().manual_seed(13)
    base = (torch.randn(B, N, K, generator=g) * 3).to(DEV).half()
    x0 = torch.randint(0, K, (B, N), generator=g).to(DEV)
    tt, pt = torch.tensor([0, 37, 99], device=DEV), torch.tensor([0.01, 0.02, 0.01], device=DEV)
    calls = _spy(monkeypatch)
    unscaled = base.clone().requires_grad_(True)
    _train_step(K, N, unscaled, x0, tt, pt)
    w_main, w_aux = calls[1]["w_main"], calls[1]["w_aux"]
    calls.clear()
    leaf = base.clone().requires_grad_(True)
    _train_step(K, N, leaf, x0, tt, pt, loss_factor=S)
    assert torch.equal(calls[1]["w_main"], w_main * S) and torch.equal(calls[1]["w_aux"], w_aux * S)
    assert torch.equal(leaf.grad, _fp32_gradient(calls[1], w_main * S, w_aux * S).half())
    monkeypatch.undo()
    # today's amp route: cast, one fp32 pass at the announced scale, rescale by the loss scale, cast back
    ref_leaf = base.float().requires_grad_(True)
    _train_step(K, N, ref_leaf, x0, tt, pt, loss_factor=S)
    assert int(_ulps(leaf.grad, ref_leaf.grad.half()).max()) <= 1
    # what the scaler is for: at the unscaled size many float16 entries underflow to zero, scaled they survive
    assert int((leaf.grad != 0).sum()) > int((unscaled.grad != 0).sum())
