"""Host logic of the native VQ-VAE decoder (SURVEY §8 f4), on the CPU: `decode.decoder_plan` turns the reference's `Decoder`
module into `LayerSpec`s (BatchNorm folding, tap tables of the parity classes of the transposed convolutions, weight
matrices).  Here the plan is executed by a plain-torch EMULATION of the contracts `include/d3pm_b200.h` states for
d3pm_dec_conv / d3pm_dec_axial_attention / d3pm_dec_col2im and compared with the oracle pinned to the reference's videos -
so what the GPU tests still have to prove is only that the kernels honour those contracts."""
import os

import numpy as np
import pytest
import torch

from d3pm_b200 import decode
from oracle import decoder_oracle as DO
from tests.helpers import vqvae_from_fixture

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def emulate_conv(spec, x, B, grid, residual=None):
    """The contract of d3pm_dec_conv (include/d3pm_b200.h) in float64 torch ops."""
    T, H, W = grid
    st, sh, sw = spec.stride
    a = x.double().view(B, T, H, W, spec.cin)
    if spec.in_affine is not None:
        a = torch.relu(a * spec.in_affine[0].double() + spec.in_affine[1].double())
    out = torch.zeros(B, T * st, H * sh, W * sw, spec.nout, dtype=torch.float64)
    for c, (offs, taps) in enumerate(zip(spec.classes, spec.taps)):
        acc = torch.zeros(B, T, H, W, spec.nout, dtype=torch.float64)
        wm = spec.wmat[c].double().view(spec.nout, len(taps), spec.cin)
        for i, (dt, dh, dw) in enumerate(taps):
            shifted = torch.zeros_like(a)   # a(pos + tap offset), zero outside the grid
            ts, hs, ws = (slice(max(0, -d), n - max(0, d)) for d, n in ((dt, T), (dh, H), (dw, W)))
            tsrc, hsrc, wsrc = (slice(max(0, d), n - max(0, -d)) for d, n in ((dt, T), (dh, H), (dw, W)))
            shifted[:, ts, hs, ws] = a[:, tsrc, hsrc, wsrc]
            acc += shifted @ wm[:, i].t()
        out[:, offs[0]::st, offs[1]::sh, offs[2]::sw] = acc
    out = out.view(-1, spec.nout)
    if spec.bias is not None:
        out = out + spec.bias.double()
    if residual is not None:
        out = out + residual.double()
    if spec.relu_out:
        out = torch.relu(out)
    return out.float()


def emulate_attention(qkv, B, grid, heads, C, scale=None):
    """d3pm_dec_axial_attention: qkv [M][3 axes (W, H, T)][q, k, v][heads][dh] -> att [M][3 axes][heads][dh]."""
    T, H, W = grid
    dh = C // heads
    scale = dh ** -0.5 if scale is None else scale
    z = qkv.double().view(B, T, H, W, 3, 3, heads, dh)
    outs = []
    for axis, dim in ((0, 3), (1, 2), (2, 1)):
        q, k, v = (z[..., axis, j, :, :].movedim(dim, -2) for j in range(3))   # [..., heads, L, dh]
        p = torch.softmax(q @ k.transpose(-1, -2) * scale, dim=-1)
        outs.append((p @ v).movedim(-2, dim))                                  # [B, T, H, W, heads, dh]
    return torch.stack(outs, 4).reshape(B * T * H * W, 3 * C).float()


def emulate_col2im(y, bias, B, grid, cout, stride):
    """d3pm_dec_col2im (on the untransposed contributions y [positions][64 * cout]): tap k of input i lands on
    y = (i + pf) * s + k - 3, pf = ceil((4 - s) / 2), per dimension."""
    T, H, W = grid
    To, Ho, Wo = (g * s for g, s in zip(grid, stride))
    yy = y.double().view(B, T, H, W, 4, 4, 4, cout)
    out = torch.zeros(B, cout, To, Ho, Wo, dtype=torch.float64)
    pf = [(4 - s + 1) // 2 for s in stride]
    for it in range(T):
        for kt in range(4):
            ot = (it + pf[0]) * stride[0] + kt - 3
            if not 0 <= ot < To:
                continue
            for ih in range(H):
                for kh in range(4):
                    oh = (ih + pf[1]) * stride[1] + kh - 3
                    if not 0 <= oh < Ho:
                        continue
                    for kw in range(4):
                        ow = (torch.arange(W) + pf[2]) * stride[2] + kw - 3
                        ok = (ow >= 0) & (ow < Wo)
                        out[:, :, ot, oh, ow[ok]] += yy[:, it, ih, ok, kt, kh, kw, :].permute(0, 2, 1)
    return (out + bias.double().view(1, -1, 1, 1, 1)).float()


def run_plan(plan, h):
    B, Cm, T, H, W = h.shape
    C = plan["C"]   # the width the kernels work on: the model's channels zero-padded
    x = torch.nn.functional.pad(h.permute(0, 2, 3, 4, 1).reshape(-1, Cm), (0, C - Cm)).contiguous()
    for L3, L1, Lq, Lf in plan["blocks"]:
        y = emulate_conv(L1, emulate_conv(L3, x, B, (T, H, W)), B, (T, H, W))
        att = emulate_attention(emulate_conv(Lq, y, B, (T, H, W)), B, (T, H, W), plan["heads"], C, plan["softmax_scale"])
        x = emulate_conv(Lf, att, B, (T, H, W), residual=x)
    grid = (T, H, W)
    for item in plan["convts"]:
        if item[0] == "conv":
            x = emulate_conv(item[1], x, B, grid)
            grid = tuple(g * s for g, s in zip(grid, item[2]))
        else:
            return emulate_col2im(emulate_conv(item[1], x, B, grid), item[3], B, grid, item[4], item[2])


@pytest.mark.parametrize("name", ["decode_h64", "decode_h128", "decode_small", "decode_k512"])   # the last two: n_hiddens 24, padded to 64
def test_plan_through_the_kernel_contracts_reproduces_the_reference_video(name):
    fx = np.load(os.path.join(GOLD, name + ".npz"))
    vq = vqvae_from_fixture(fx)
    plan = decode.decoder_plan(vq.decoder)
    got = run_plan(plan, torch.from_numpy(fx["h"]))
    want = torch.from_numpy(fx["video"])
    assert got.shape == want.shape
    assert (got - want).abs().max() <= 5e-6 * max(1.0, float(want.abs().max()))
    with pytest.raises(decode.D3PMError):
        decode.decoder_plan(vq.train().decoder)   # batch statistics are not something the folded plan can express


def test_transposed_convolution_classes_cover_every_tap_once():
    """Every (kt, kh, kw) of the 4x4x4 kernel belongs to exactly one parity class, with the offset the oracle's own
    conv_transpose3d implies (checked on a delta input)."""
    import torch.nn.functional as F
    for stride in ((1, 2, 2), (2, 2, 2), (1, 1, 2)):
        classes = decode._convt_taps(stride)
        seen = [k for _, taps in classes for k, _ in taps]
        assert sorted(seen) == sorted((a, b, c) for a in range(4) for b in range(4) for c in range(4))
        T = H = W = 5
        x = torch.zeros(1, 1, T, H, W)
        x[0, 0, 2, 2, 2] = 1.0
        w = torch.arange(64, dtype=torch.float32).view(1, 1, 4, 4, 4) + 1
        y = F.conv_transpose3d(F.pad(x, DO.same_pad((4, 4, 4), stride)), w, stride=stride, padding=(3, 3, 3))
        for (pt, ph, pw), taps in classes:
            for (kt, kh, kw), (dt, dh, dw) in taps:
                # output (m * s + parity) reads input m + d: the delta at 2 is seen from m = 2 - d
                ot, oh, ow = (2 - dt) * stride[0] + pt, (2 - dh) * stride[1] + ph, (2 - dw) * stride[2] + pw
                assert float(y[0, 0, ot, oh, ow]) == float(w[0, 0, kt, kh, kw])
