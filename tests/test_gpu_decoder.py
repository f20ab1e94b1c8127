"""Token -> video, second stage (SURVEY §8 f4): the native VQ-VAE decoder kernels against the contracts of
include/d3pm_b200.h (emulated in float64 torch ops, tests/test_decoder_plan.py), the fixtures generated from the imported
reference, the oracle, and the live reference `Decoder` module on the same GPU.  Needs a B200."""
import os

import numpy as np
import pytest
import torch

from baseline import reference_loader as RL
from d3pm_b200 import _lib, decode, ops
from d3pm_b200._lib import D3PMError
from oracle import decoder_oracle as DO
from tests.helpers import reference_vqvae_like, vqvae_from_fixture, vqvae_layout
from tests.test_decoder_plan import emulate_attention, emulate_col2im, emulate_conv

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# 3xTF32 products vs float64, relative to the largest output.  The products themselves are fp32-grade (2^-22); what shows at
# K = 27 x 256 = 6912 is the tensor core's accumulator, which does not round to nearest: ~3e-5 of the scale there, ~1e-6 at K <= 256
TOL_FP32 = 1e-4
TOL_TF32 = 5e-3   # single TF32 products (10-bit mantissas)


def _spec(g, *, nclass, nout, cin, taps, classes, stride=(1, 1, 1), bias=False, affine=False, relu=False):
    w = torch.randn(nclass, nout, len(taps[0]) * cin, generator=g) / (len(taps[0]) * cin) ** 0.5
    return decode.LayerSpec(w, cin=cin, taps=taps, classes=classes, stride=stride,
                            bias=torch.randn(nout, generator=g) if bias else None,
                            in_affine=(torch.rand(cin, generator=g) + 0.5, torch.randn(cin, generator=g) * 0.3) if affine else None,
                            relu_out=relu)


CONV3 = [(a - 1, b - 1, c - 1) for a in range(3) for b in range(3) for c in range(3)]
CONV_CASES = {
    # name: (B, grid, spec kwargs, residual, n_tile)
    "pointwise_k32": (2, (2, 4, 4), dict(nclass=1, nout=64, cin=32, taps=[[(0, 0, 0)]], classes=[(0, 0, 0)]), False, 128),
    "pointwise_bias_relu_res": (3, (3, 5, 5), dict(nclass=1, nout=256, cin=128, taps=[[(0, 0, 0)]], classes=[(0, 0, 0)], bias=True,
                                                   relu=True), True, 256),
    "qkv_2304": (1, (4, 8, 8), dict(nclass=1, nout=2304, cin=256, taps=[[(0, 0, 0)]], classes=[(0, 0, 0)]), False, 256),
    "conv3_affine": (2, (4, 6, 5), dict(nclass=1, nout=128, cin=256, taps=[CONV3], classes=[(0, 0, 0)], bias=True, affine=True,
                                        relu=True), False, 128),
    "conv3_ragged_two_tiles": (1, (3, 7, 9), dict(nclass=1, nout=32, cin=64, taps=[CONV3], classes=[(0, 0, 0)], affine=True), False, 128),
    "nout_192_padded": (2, (2, 6, 6), dict(nclass=1, nout=192, cin=64, taps=[[(0, 0, 0)]], classes=[(0, 0, 0)], affine=True), False, 256),
    "nout_192_tiles_of_128": (2, (2, 6, 6), dict(nclass=1, nout=192, cin=64, taps=[[(0, 0, 0)]], classes=[(0, 0, 0)]), False, 128),
}


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("terms", [3, 1])
@pytest.mark.parametrize("name", sorted(CONV_CASES))
def test_dec_conv_honours_its_contract(name, terms, pair):
    B, grid, kw, with_res, n_tile = CONV_CASES[name]
    g = torch.Generator().manual_seed(len(name))
    spec = _spec(g, **kw)
    M = B * grid[0] * grid[1] * grid[2]
    x = torch.randn(M, spec.cin, generator=g)
    res = torch.randn(M, spec.nout, generator=g) if with_res else None
    want = emulate_conv(spec, x, B, grid, residual=res)
    layer = decode._Layer(spec, torch.device(DEV), n_tile, cta_pair=pair)   # pair: cta_group::2, two CTAs per 256 positions
    got = layer(x.to(DEV), B, grid, terms=terms, residual=None if res is None else res.to(DEV)).cpu()
    assert got.shape == want.shape
    tol = (TOL_FP32 if terms == 3 else TOL_TF32) * float(want.abs().max())
    assert (got - want).abs().max().item() <= tol
    if not with_res:  # the transposed store of the epilogue (the layout col2im reads)
        got_t = layer(x.to(DEV), B, grid, terms=terms, transposed=True).cpu()   # planes [B * T, Nout, H * W]
        assert got_t.shape == (B * grid[0], spec.nout, grid[1] * grid[2])
        assert torch.equal(got_t.transpose(1, 2).reshape(M, spec.nout), got)


@pytest.mark.parametrize("stride", [(1, 2, 2), (2, 2, 2)])
def test_dec_conv_parity_classes_of_a_transposed_convolution(stride):
    """A whole SamePadConvTranspose3d (kernel 4) as parity classes, against torch's conv_transpose3d on the CPU."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(7)
    B, grid, cin, cout = 2, (3, 5, 6), 64, 96
    w = torch.randn(cin, cout, 4, 4, 4, generator=g) / (cin * 16) ** 0.5
    bias = torch.randn(cout, generator=g)
    x = torch.randn(B, cin, *grid, generator=g)
    want = F.conv_transpose3d(F.pad(x, DO.same_pad((4, 4, 4), stride)), w, bias, stride=stride, padding=(3, 3, 3))
    classes = decode._convt_taps(stride)
    mats = [torch.stack([w[:, :, kt, kh, kw].t() for (kt, kh, kw), _ in taps], 1).reshape(cout, -1) for _, taps in classes]
    spec = decode.LayerSpec(torch.stack(mats, 0), cin=cin, taps=[[d for _, d in taps] for _, taps in classes],
                            classes=[c for c, _ in classes], stride=stride, bias=bias)
    rows = x.permute(0, 2, 3, 4, 1).reshape(-1, cin).contiguous()
    for pair in (False, True):
        got = decode._Layer(spec, torch.device(DEV), cta_pair=pair)(rows.to(DEV), B, grid, terms=3).cpu()
        got = got.view(B, *(n * s for n, s in zip(grid, stride)), cout).permute(0, 4, 1, 2, 3)
        assert (got - want).abs().max().item() <= TOL_FP32 * float(want.abs().max()), pair


@pytest.mark.parametrize("B,grid,C", [(2, (4, 16, 16), 256), (1, (3, 5, 7), 128), (2, (2, 4, 4), 64), (1, (16, 16, 16), 256), (1, (1, 32, 2), 64)])
def test_axial_attention(B, grid, C):
    g = torch.Generator().manual_seed(C + grid[0])
    M = B * grid[0] * grid[1] * grid[2]
    qkv = torch.randn(M, 9 * C, generator=g)
    want = emulate_attention(qkv, B, grid, 2, C)
    att = torch.empty(M, 3 * C, device=DEV)
    lib = _lib.load_library()
    _lib.check(lib.d3pm_dec_axial_attention(qkv.to(DEV).data_ptr(), att.data_ptr(), B, *grid, 2, C // 2, 0.0, 0), "d3pm_dec_axial_attention")
    torch.cuda.synchronize()
    assert (att.cpu() - want).abs().max().item() <= 2e-5 * float(want.abs().max())


@pytest.mark.parametrize("stride", [(1, 2, 2), (2, 2, 2), (1, 1, 2)])
def test_col2im(stride):
    g = torch.Generator().manual_seed(3)
    B, grid, cout = 2, (3, 4, 5), 3
    y = torch.randn(B * grid[0] * grid[1] * grid[2], 64 * cout, generator=g)
    bias = torch.randn(cout, generator=g)
    want = emulate_col2im(y, bias, B, grid, cout, stride)
    out = torch.empty(*want.shape, device=DEV)
    lib = _lib.load_library()
    # the kernel reads the plane-transposed rows d3pm_dec_conv writes with out_transposed = 1: [B * T][64 * cout][H * W]
    y_t = y.view(B * grid[0], grid[1] * grid[2], 64 * cout).transpose(1, 2).contiguous().to(DEV)
    _lib.check(lib.d3pm_dec_col2im(y_t.data_ptr(), bias.to(DEV).data_ptr(), out.data_ptr(), B, *grid, cout, *stride, 0), "d3pm_dec_col2im")
    torch.cuda.synchronize()
    assert (out.cpu() - want).abs().max().item() <= 1e-5 * float(want.abs().max())


@pytest.mark.parametrize("name", ["decode_h64", "decode_h128", "decode_small", "decode_k512"])   # the last two: n_hiddens 24, padded to 64
def test_native_decoder_against_reference_fixture(name):
    """tokens -> video entirely on the library's kernels, against the video the imported reference's `VQVAE.decode` returned."""
    fx = np.load(os.path.join(GOLD, name + ".npz"))
    vq = vqvae_from_fixture(fx).to(DEV)
    tokens = torch.from_numpy(fx["tokens"]).to(DEV)
    want = torch.from_numpy(fx["video"])
    scale = float(want.abs().max())
    table = decode.DecodeTable.from_autoencoder(vq)
    status = ops.new_status(DEV)
    got = decode.decode(vq, tokens, table, decode.NativeDecoder(vq.decoder), status).cpu()
    assert got.shape == want.shape and int(status.item()) == 0
    assert (got - want).abs().max().item() <= 5e-5 * scale
    fast = decode.decode(vq, tokens, table, decode.NativeDecoder(vq.decoder, precision="tf32")).cpu()
    assert (fast - want).abs().max().item() <= 2e-2 * scale
    paired = decode.decode(vq, tokens, table, decode.NativeDecoder(vq.decoder, cta_pair=True)).cpu()
    assert (paired - want).abs().max().item() <= 5e-5 * scale
    if tokens.shape[0] > 1:  # a batch too large for the 32-bit element offsets is decoded in passes of whole videos
        small = decode.NativeDecoder(vq.decoder)
        small.max_elements = small.max_elements // (small.videos_per_pass(tokens.shape[1:])) + 1   # room for exactly one video
        assert small.videos_per_pass(tokens.shape[1:]) == 1
        assert torch.equal(decode.decode(vq, tokens, table, small).cpu(), got)
    # the reference's own entry: Decoder.forward on the channels-first tensor
    again = decode.NativeDecoder(vq.decoder)(torch.from_numpy(fx["h"]).to(DEV)).cpu()
    assert (again - want).abs().max().item() <= 5e-5 * scale
    with pytest.raises(D3PMError):
        decode.NativeDecoder(vq.decoder.train())


@pytest.mark.parametrize("B", [1, 3])
def test_native_decoder_at_the_shipped_shape_against_the_live_reference(B):
    """n_hiddens 256, 3 residual blocks, downsample [1, 8, 8], 4 x 128 x 128 video (ucf-ddiff-train.job:15): the native chain
    against the oracle (CPU, fp32; pinned to the reference's videos by tests/golden/decode_*.npz), and -
    where the reference is present - against the reference's own `VQVAE.decode` on this GPU in fp32 (TF32 off), same weights."""
    torch.manual_seed(21)
    vq = vqvae_layout(128, 4096, 256, 3, (1, 8, 8))
    with torch.no_grad():
        for m in vq.modules():
            if isinstance(m, torch.nn.BatchNorm3d):
                m.running_mean.normal_(0, 0.2)
                m.running_var.uniform_(0.5, 1.5)
    vq = vq.to(DEV)
    tokens = torch.randint(0, 4096, (B, 4, 16, 16), device=DEV)
    table = decode.DecodeTable.from_autoencoder(vq)
    got = decode.decode(vq, tokens, table, decode.NativeDecoder(vq.decoder)).cpu()
    assert got.shape == (B, 3, 4, 128, 128)
    sd = {k: v.detach().cpu() for k, v in vq.state_dict().items()}
    orc = DO.vqvae_decode(sd, tokens.cpu(), 3, (1, 8, 8))
    assert (got - orc).abs().max().item() <= 1e-4 * float(orc.abs().max())
    if RL.reference_available():
        ref = reference_vqvae_like(vq, embedding_dim=128, n_codes=4096, n_hiddens=256, n_res_layers=3, downsample=[1, 8, 8],
                                   sequence_length=4, resolution=128)
        tf32_conv, tf32_mm = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
        try:
            with torch.no_grad():
                want = ref.decode(tokens).cpu()
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32_conv, tf32_mm
        assert want.shape == got.shape
        assert (got - want).abs().max().item() <= 1e-4 * float(want.abs().max())


def test_sample_then_decode_like_the_reference_caller():
    """`DiscreteDiffusion.forward`'s inference branch (networks/discrete_diffusion.py:53-62): sample the tokens with the drop-in
    diffusion class, view them on the latent grid, decode natively - against the oracle's `VQVAE.decode` (CPU, fp32) and,
    where the reference is present, the reference's own `VQVAE.decode`."""
    import types
    import d3pm_b200
    K, B, grid = 256, 2, (2, 4, 4)
    N = grid[0] * grid[1] * grid[2]

    class Denoiser(torch.nn.Module):  # any module with the reference transformer's surface: logits [B, K, N] as a view of [B, N, K]
        def __init__(self):
            super().__init__()
            self.content_emb = types.SimpleNamespace(num_embed=K + 1)
            self.to_logits = torch.nn.Sequential(torch.nn.Identity(), torch.nn.Linear(1, 1))
            self.table = torch.nn.Parameter(torch.randn(K + 1, K, generator=torch.Generator().manual_seed(1)))

        def forward(self, x_t, cond, t):
            return self.table[x_t].permute(0, 2, 1)

    model = d3pm_b200.FusedDiffusionTransformer(transformer=Denoiser(), diffusion_step=20, alpha_init_type="alpha1", guidance_scale=2.0,
                                                content_seq_len=N).to(DEV)
    torch.manual_seed(5)
    vq = vqvae_layout(32, K, 64, 1, (1, 4, 4)).to(DEV)
    cond = torch.zeros(B, 1, 512, device=DEV)
    video = decode.sample_and_decode(model.manual_seed(3), vq, ["a"] * B, cond, cond, grid, decoder=decode.NativeDecoder(vq.decoder))
    tokens = model.manual_seed(3).sample(["a"] * B, None, cond, cond, content_token=None, filter_ratio=0)["content_token"]
    assert not (tokens == K).any()
    sd = {k: v.detach().cpu() for k, v in vq.state_dict().items()}
    orc = DO.vqvae_decode(sd, tokens.view(B, *grid).cpu(), 1, (1, 4, 4))
    assert video.shape == orc.shape == (B, 3, grid[0], 4 * grid[1], 4 * grid[2])
    assert (video.cpu() - orc).abs().max().item() <= 1e-4 * float(orc.abs().max())
    if RL.reference_available():
        ref = reference_vqvae_like(vq, embedding_dim=32, n_codes=K, n_hiddens=64, n_res_layers=1, downsample=[1, 4, 4],
                                   sequence_length=grid[0], resolution=4 * grid[1])
        with torch.no_grad():
            want = ref.decode(tokens.view(B, *grid))
        assert (video - want).abs().max().item() <= 2e-3 * float(want.abs().max())   # the reference arm runs cuDNN's default TF32 here


@pytest.mark.parametrize("pair", [False, True])
@pytest.mark.parametrize("name", ["conv3_ragged_two_tiles", "nout_192_padded", "pointwise_bias_relu_res"])
def test_dec_conv_writes_nothing_outside_its_rows_and_columns(name, pair):
    """Canaries around the output: rows past the last position and the columns between Nout and the row pitch stay untouched
    (ragged last tile, padded last N tile, the shared-memory-staged epilogue)."""
    B, grid, kw, with_res, n_tile = CONV_CASES[name]
    g = torch.Generator().manual_seed(11)
    spec = _spec(g, **kw)
    M = B * grid[0] * grid[1] * grid[2]
    x = torch.randn(M, spec.cin, generator=g).to(DEV)
    layer = decode._Layer(spec, torch.device(DEV), n_tile, cta_pair=pair)
    plain = layer(x, B, grid, terms=3)
    pitch, guard = spec.nout + 8, 5
    buf = torch.full((M + guard, pitch), 777.0, device=DEV)
    got = layer(x, B, grid, terms=3, out=buf[:M])
    assert got.data_ptr() == buf.data_ptr()
    assert torch.equal(buf[:M, :spec.nout], plain)
    assert bool((buf[M:] == 777.0).all()) and bool((buf[:M, spec.nout:] == 777.0).all())


@pytest.mark.parametrize("seed", range(16))
def test_dec_conv_random_shapes(seed):
    """Randomised shapes against the float64 emulation of the contract: odd grids, arbitrary tap sets, every stride / parity-class
    combination, padded N tiles, bias / affine / ReLU / residual in all mixes, both tile widths, single CTAs and pairs."""
    import random
    rnd = random.Random(1000 + seed)
    g = torch.Generator().manual_seed(seed)
    B, grid = rnd.randint(1, 3), tuple(rnd.randint(1, 7) for _ in range(3))
    cin, nout = rnd.choice([32, 64, 96]), 4 * rnd.randint(1, 75)
    stride = tuple(rnd.choice([1, 2]) for _ in range(3))
    classes = [(a, b, c) for a in range(stride[0]) for b in range(stride[1]) for c in range(stride[2])]
    ntaps = rnd.randint(1, 6)
    taps = [[tuple(rnd.randint(-2, 2) for _ in range(3)) for _ in range(ntaps)] for _ in classes]
    spec = _spec(g, nclass=len(classes), nout=nout, cin=cin, taps=taps, classes=classes, stride=stride, bias=rnd.random() < 0.5,
                 affine=rnd.random() < 0.5, relu=rnd.random() < 0.5)
    M = B * grid[0] * grid[1] * grid[2]
    x = torch.randn(M, cin, generator=g)
    res = torch.randn(M * stride[0] * stride[1] * stride[2], nout, generator=g) if rnd.random() < 0.5 else None
    want = emulate_conv(spec, x, B, grid, residual=res)
    layer = decode._Layer(spec, torch.device(DEV), rnd.choice([128, 256]), cta_pair=rnd.random() < 0.5)
    got = layer(x.to(DEV), B, grid, terms=3, residual=None if res is None else res.to(DEV)).cpu()
    assert (got - want).abs().max().item() <= TOL_FP32 * max(1.0, float(want.abs().max()))


def test_decoder_kernels_on_a_non_current_device():
    """The decoder entry points make the device that owns the tensors current for the call, like the rest of the C ABI (cluster
    launches and the SM count of the persistent grid included)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    other = torch.device("cuda", 1)
    torch.cuda.set_device(0)
    B, grid, kw, _, n_tile = CONV_CASES["conv3_affine"]
    g = torch.Generator().manual_seed(2)
    spec = _spec(g, **kw)
    x = torch.randn(B * grid[0] * grid[1] * grid[2], spec.cin, generator=g)
    want = decode._Layer(spec, torch.device(DEV), n_tile)(x.to(DEV), B, grid, terms=3).cpu()
    for pair in (False, True):
        got = decode._Layer(spec, other, n_tile, cta_pair=pair)(x.to(other), B, grid, terms=3)
        assert got.device == other and torch.cuda.current_device() == 0
        assert torch.equal(got.cpu(), want)
    qkv = torch.randn(2 * 4 * 4 * 4, 9 * 64, generator=g)
    outs = []
    for dev in (torch.device(DEV), other):
        att = torch.empty(qkv.shape[0], 3 * 64, device=dev)
        _lib.check(_lib.load_library().d3pm_dec_axial_attention(qkv.to(dev).data_ptr(), att.data_ptr(), 2, 4, 4, 4, 2, 32, 0.0,
                                                                torch.cuda.current_stream(dev).cuda_stream), "d3pm_dec_axial_attention")
        outs.append(att.cpu())
    assert torch.equal(outs[0], outs[1])


def test_native_decode_can_be_captured_in_a_cuda_graph():
    """Serving loops replay a captured graph: the whole native decode (gather, 3xTF32 GEMMs with cluster launches off and on,
    attention, col2im) records into a CUDA graph and replays to the eager result on new tokens."""
    fx = np.load(os.path.join(GOLD, "decode_h64.npz"))
    vq = vqvae_from_fixture(fx).to(DEV)
    table = decode.DecodeTable.from_autoencoder(vq)
    K = int(fx["hparams"][1])
    for pair in (False, True):
        dec = decode.NativeDecoder(vq.decoder, cta_pair=pair)
        static_tokens = torch.from_numpy(fx["tokens"]).to(DEV)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            decode.decode(vq, static_tokens, table, dec)   # warm-up outside the capture (lazy function attributes)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = decode.decode(vq, static_tokens, table, dec)
        new_tokens = torch.randint(0, K, static_tokens.shape, device=DEV)
        static_tokens.copy_(new_tokens)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_out, decode.decode(vq, new_tokens, table, dec))
