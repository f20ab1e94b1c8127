"""Shared helpers for the tests (the oracle is imported here as the CHECKER only)."""
import glob
import os

import numpy as np
import torch

from oracle import d3pm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
POST_TOL = 1e-4       # north_star: posterior log-probs within 1e-4 absolute in fp32
NEAR_TIE_GAP = 2e-4   # tokens must match except where the reference's own top-2 gap is below this


def step_fixtures():
    return sorted(glob.glob(os.path.join(GOLDEN, "step_k*.npz")))


def load(path):
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


def fixture_guidance(fx):
    s = float(fx["guidance_scale"])
    return None if s < 0 else s


def oracle_step_from_fixture(fx):
    """Run the op-faithful oracle on a fixture's inputs -> (tokens [B,N], post [B,N,K+1], recon [B,N,K+1])."""
    T, K = int(fx["T"]), int(fx["K"])
    sched = O.make_schedule(T, K)
    lc, lu = torch.from_numpy(fx["logits_c"]), torch.from_numpy(fx["logits_u"])
    x_t, t = torch.from_numpy(fx["x_t"]), torch.from_numpy(fx["t"])
    u = torch.from_numpy(fx["uniform"]).permute(0, 2, 1)
    s = fixture_guidance(fx)
    out, post, recon = O.p_sample_step(sched, lc.permute(0, 2, 1), None if s is None else lu.permute(0, 2, 1),
                                       O.index_to_log_onehot(x_t, K + 1), t, 0.0 if s is None else s, u)
    return out.argmax(1), post.permute(0, 2, 1), recon.permute(0, 2, 1)


def assert_tokens_match(got, want, near_tie, what=""):
    """Bit-exact except at (logged) near-ties."""
    got, want, near_tie = np.asarray(got), np.asarray(want), np.asarray(near_tie).astype(bool)
    diff = got != want
    if diff.any():
        print(f"[near-tie log] {what}: {int(diff.sum())} token(s) differ, {int((diff & near_tie).sum())} of them at near-ties; "
              f"{int(near_tie.sum())} near-tie position(s) in total")
    assert not (diff & ~near_tie).any(), f"{what}: {int((diff & ~near_tie).sum())} token mismatches away from near-ties"


class _Node(torch.nn.Module):
    """A container whose children are set as attributes (the reference's wrappers `SamePadConv3d.conv`,
    `SamePadConvTranspose3d.convt`, `AxialBlock.attn_w` ... are nothing more to the code under test)."""

    def __init__(self, **children):
        super().__init__()
        for name, child in children.items():
            setattr(self, name, child)


def _attention(C):
    return _Node(w_qs=torch.nn.Linear(C, C, bias=False), w_ks=torch.nn.Linear(C, C, bias=False),
                 w_vs=torch.nn.Linear(C, C, bias=False), fc=torch.nn.Linear(C, C), n_head=2, d_k=C // 2)


def vqvae_layout(E, K, C, R, downsample):
    """The parts of the reference's `VQVAE` (videogpt_vq_vae.py) that `decode.DecodeTable`, `decode.decoder_plan` and
    `decode.NativeDecoder` read - `codebook.embeddings`, `post_vq_conv.conv` and the `Decoder`'s `res_stack` / `convts` -
    under the reference's own parameter names, so that its state dict loads strictly into this and back.  Initialised by
    torch's default initialisers (seed the global generator for fixed weights), codebook N(0, 1); eval mode, on the CPU."""
    Ch = C // 2
    blocks = [_Node(block=torch.nn.Sequential(
        torch.nn.BatchNorm3d(C), torch.nn.ReLU(), _Node(conv=torch.nn.Conv3d(C, Ch, 3, bias=False)),
        torch.nn.BatchNorm3d(Ch), torch.nn.ReLU(), _Node(conv=torch.nn.Conv3d(Ch, C, 1, bias=False)),
        torch.nn.BatchNorm3d(C), torch.nn.ReLU(), _Node(attn_w=_attention(C), attn_h=_attention(C), attn_t=_attention(C))))
        for _ in range(R)]
    # the Decoder's upsampling (videogpt_vq_vae.py:265-275): log2(downsample) doublings per axis, one transposed convolution
    # per doubling of the most-upsampled axis, the last one to RGB
    todo = np.array([int(np.log2(d)) for d in downsample])
    convts, n_convts = [], int(todo.max())
    for i in range(n_convts):
        stride = tuple(2 if n > 0 else 1 for n in todo)
        cout = 3 if i == n_convts - 1 else C
        convts.append(_Node(convt=torch.nn.ConvTranspose3d(C, cout, 4, stride=stride, padding=3)))
        todo -= 1
    vq = _Node(codebook=_Node(embeddings=torch.nn.Parameter(torch.randn(K, E))),
               post_vq_conv=_Node(conv=torch.nn.Conv3d(E, C, 1)),
               decoder=_Node(res_stack=torch.nn.Sequential(*blocks, torch.nn.BatchNorm3d(C), torch.nn.ReLU()),
                             convts=torch.nn.ModuleList(convts)))
    return vq.eval()


def vqvae_from_fixture(fx):
    """`vqvae_layout` with the weights of a `tests/golden/decode_*.npz` fixture loaded strictly.  The fixture's `video` is
    what the reference's `VQVAE.decode` returned for these weights, so a test compares with the reference without importing
    it."""
    E, K, C, R, d0, d1, d2, _, _, _ = (int(v) for v in fx["hparams"])
    vq = vqvae_layout(E, K, C, R, (d0, d1, d2))
    state = {k[3:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("sd/")}
    vq.load_state_dict({k: v for k, v in state.items() if k.startswith(("decoder.", "post_vq_conv.", "codebook.embeddings"))},
                       strict=True)
    return vq


def reference_vqvae_like(vq, **hparams):
    """The reference's own `VQVAE` (imported; the reference must be present) holding the weights of `vq` (a `vqvae_layout`),
    on the same device, eval mode.  Only its encoder-side weights are its own."""
    from baseline import reference_loader as RL
    ref = RL.load_vqvae_module().VQVAE(checkpoint_path=None, **hparams)
    missing = ref.load_state_dict({k: v.detach().cpu() for k, v in vq.state_dict().items()}, strict=False).missing_keys
    assert all(k.startswith(("encoder.", "pre_vq_conv.", "codebook.")) and k != "codebook.embeddings" for k in missing), missing
    return ref.to(next(vq.parameters()).device).eval()
