"""The fused head + reverse step (d3pm_head_step) where the small tests of test_gpu_head.py never take it: at the benchmarked
shape and other shapes where every CTA of the persistent kernel runs two or more 128-row tiles, through its redo and
survivor-overflow paths, at the edge of the weights' validity bound (the guided mix clamped at -70), and on LayerNorm edge
rows.  Needs a B200 (tcgen05).

Three references, strongest first:
  * the oracle: float64 logits from the module's fp32 parameters, stepped by `d3pm_oracle.p_sample_step` with the very
    uniforms the kernel's Philox stream draws, on a row sample that covers later tiles, tile and video boundaries and the
    last, partial tile;
  * the CUDA-core exhaustive path (HEAD_REFERENCE) on every row;
  * the same call split at video boundaries that are also tile boundaries, each chunk with fewer tiles than SMs and its
    own `row_offset`: every row keeps its lane and tile-relative position, so only the tile loop differs and the tokens
    must be equal bit for bit.
"""
import copy
import math

import pytest
import torch

from d3pm_b200 import _lib, head, ops
from oracle import d3pm_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
D, T, TILE = 64, 100, 128
LOGIT_TOL = 5e-5  # HEAD_LOGITS against float64 where |logit| stays within a few tens (test_gpu_head.py's bound)
ROW_CHUNK = 8192  # rows per float64 reference block (256 MiB at K = 4096)


def _sms():
    return torch.cuda.get_device_properties(torch.device(DEV)).multi_processor_count


def _tiles(B, N):
    return -(-B * N // TILE)


def _multi_tile(B, N):
    """The kernel's grid is min(tiles, SMs): with at least twice as many tiles as SMs every CTA runs a second tile."""
    sms, tiles = _sms(), _tiles(B, N)
    assert tiles >= 2 * sms, f"{B} x {N} rows are {tiles} tiles on {sms} SMs: not every CTA would run a second tile"
    print(f"\n[tiles] {B} x {N} = {B * N} rows: {tiles} tiles on {sms} SMs, {tiles // sms}-{-(-tiles // sms)} tiles per CTA")
    return sms


def _head(K, seed, scale=3.0):
    """test_gpu_head.py's head: gamma ~ 1, small beta, |logit| ~ 10."""
    g = torch.Generator().manual_seed(seed)
    ln, lin = torch.nn.LayerNorm(D), torch.nn.Linear(D, K)
    with torch.no_grad():
        ln.weight.copy_(1 + 0.1 * torch.randn(D, generator=g))
        ln.bias.copy_(0.1 * torch.randn(D, generator=g))
        lin.weight.copy_(torch.randn(K, D, generator=g) * (scale / 8 / math.sqrt(3)))
        lin.bias.copy_(torch.randn(K, generator=g) * 0.5)
    return torch.nn.Sequential(ln, lin)


def _bench_head(K, seed):
    """bench.py's head: torch's default initialisation of LayerNorm(64) + Linear(64, K), here seeded."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        return torch.nn.Sequential(torch.nn.LayerNorm(D), torch.nn.Linear(D, K))


def _t_cycle(B):
    """Per-video timesteps cycling through 0, 99 and values between."""
    return torch.tensor([(0, 99, 50, 1, 98, 25, 75, 10)[b % 8] for b in range(B)])


def _x_t(B, N, K, t, g):
    """x_t masked with the schedule's probability at each video's t, random codes elsewhere."""
    p_mask = O.make_schedule(T, K)["log_cumprod_ct"][t].exp().view(B, 1)
    return torch.where(torch.rand(B, N, generator=g) < p_mask, torch.full((B, N), K), torch.randint(0, K, (B, N), generator=g))


def _table(K):
    return ops.build_coef_table(O.pack_schedule(O.make_schedule(T, K)).to(DEV), T, K)


def _logits64(tl64, h, r0, r1):
    with torch.no_grad():
        return tl64(h.reshape(-1, D)[r0:r1].double())


def _combined64(tl64, hc, hu, s, r0, r1):
    """s * Linear(LayerNorm(h_c)) + (1 - s) * Linear(LayerNorm(h_u)) in float64, rows r0 .. r1 of the flat batch."""
    lc = _logits64(tl64, hc, r0, r1)
    return lc if hu is None else s * lc + (1 - s) * _logits64(tl64, hu, r0, r1)


def _unfused_near_ties(tl64, hc, hu, x_t, t, table, s, K, **kw):
    """Near-tie positions of every row: d3pm_fused_step (exact Philox scoring) on the fp32-rounded float64 logits reports
    the reference's top-2 gap.  Also returns its tokens."""
    B, N, _ = hc.shape
    lc = torch.empty(B * N, K, device=DEV)
    lu = None if hu is None else torch.empty_like(lc)
    for r0 in range(0, B * N, ROW_CHUNK):
        lc[r0:r0 + ROW_CHUNK] = _logits64(tl64, hc, r0, r0 + ROW_CHUNK).float()
        if lu is not None:
            lu[r0:r0 + ROW_CHUNK] = _logits64(tl64, hu, r0, r0 + ROW_CHUNK).float()
    unf = ops.fused_step(lc.view(B, N, K), None if lu is None else lu.view(B, N, K), x_t, t, table, guidance_scale=s or 1.0,
                         sample_mode=_lib.SAMPLE_PHILOX_EXACT, want_gap=True, kernel=_lib.KERNEL_ROWS, **kw)
    return (unf["gap"] < H.NEAR_TIE_GAP).cpu().numpy(), unf["x_prev"].cpu().numpy()


def _sample_rows(B, N, sms, seed, n_random=1024):
    """~1-2 k flat rows: both sides of the boundaries of tiles around sms and 2 sms, one whole tile processed as some CTA's
    second or later tile, the last (partial) tile, both sides of every video boundary that falls inside a tile, and random
    rows, half of them from tiles >= sms."""
    rows, tiles = B * N, _tiles(B, N)
    pick = []
    for tile in (1, sms - 1, sms, sms + 1, 2 * sms - 1, 2 * sms, tiles - 1):
        if 0 < tile < tiles:
            pick.extend(range(tile * TILE - 2, min(tile * TILE + 2, rows)))
    pick.extend(range((tiles - 1) * TILE, rows))
    mid = (sms + tiles) // 2
    pick.extend(range(mid * TILE, (mid + 1) * TILE))
    for v in range(1, B):
        if (v * N) % TILE:
            pick.extend(range(v * N - 2, v * N + 2))
    g = torch.Generator().manual_seed(seed)
    pick.extend(torch.randint(sms * TILE, rows, (n_random // 2,), generator=g).tolist())
    pick.extend(torch.randint(0, rows, (n_random // 2,), generator=g).tolist())
    sel = torch.tensor(sorted(set(pick)))
    assert (sel // TILE >= 2 * sms).any() and (sel // TILE == tiles - 1).any()
    return sel


def _oracle_tokens(tl64, hc, hu, x_t, t, s, K, sel, *, seed, offset, row_offset):
    """(tokens, near-ties) of the oracle on the flat rows `sel` (each row a video of one token with its video's t)."""
    B, N, _ = hc.shape
    idx = sel.to(DEV)
    u = ops.philox_uniform(B, N, K, seed=seed, offset=offset, row_offset=row_offset, device=DEV)
    u = u.view(B * N, -1)[idx, :K + 1].cpu().unsqueeze(2)
    with torch.no_grad():
        lc = tl64(hc.reshape(-1, D)[idx].double()).cpu().unsqueeze(2)
        lu = None if hu is None else tl64(hu.reshape(-1, D)[idx].double()).cpu().unsqueeze(2)
    xs = x_t.reshape(-1)[idx].cpu().unsqueeze(1)
    out, post, _ = O.p_sample_step(O.make_schedule(T, K), lc, lu, O.index_to_log_onehot(xs, K + 1), t.cpu()[sel // N],
                                   0.0 if hu is None else s, u)
    return out.argmax(1)[:, 0].numpy(), O.near_ties(post, u)[:, 0].numpy()


def _check_case(tl, hc, hu, x_t, t, s, *, chunks, seed, offset, row_offset, what):
    """Every check of a multi-tile case; `hu is None` is guidance off, `chunks` are video indices (or None)."""
    B, N, _ = hc.shape
    K = tl[-1].out_features
    sms = _multi_tile(B, N)
    table = _table(K)
    hw = head.HeadWeights.from_module(tl)
    assert hw.valid
    gs = s if hu is not None else 1.0
    kw = dict(guidance_scale=gs, seed=seed, offset=offset, row_offset=row_offset)
    args = (hw, hc, hu, x_t, t, table)
    status = ops.new_status(DEV)
    fused = head.head_step(*args, status=status, **kw)
    assert int(status.item()) == 0, f"{what}: status {int(status.item())}"
    # the statistics pass in 3xTF32 instead of 1xTF32 only narrows the thinning thresholds: the very same tokens
    assert torch.equal(head.head_step(*args, stats_1xtf32=False, **kw), fused), f"{what}: 1xTF32 and 3xTF32 statistics differ"
    if chunks is not None:
        parts = []
        for v0, v1 in zip(chunks[:-1], chunks[1:]):
            assert (v0 * N) % TILE == 0 and _tiles(v1 - v0, N) < sms
            parts.append(head.head_step(hw, hc[v0:v1], None if hu is None else hu[v0:v1], x_t[v0:v1], t[v0:v1], table,
                                        guidance_scale=gs, seed=seed, offset=offset, row_offset=row_offset + v0 * N))
        joined = torch.cat(parts)
        assert torch.equal(joined, fused), \
            f"{what}: {int((joined != fused).sum())} tokens differ from the same rows stepped in single-tile-per-CTA chunks"
    ref = head.head_step(*args, mode=_lib.HEAD_REFERENCE, **kw)

    tl64 = copy.deepcopy(tl).double()
    near, unf = _unfused_near_ties(tl64, hc, hu, x_t, t, table, s, K, seed=seed, offset=offset, row_offset=row_offset)
    fused_np = fused.cpu().numpy()
    print(f"[near-ties] {what}: {int(near.sum())} of {B * N} rows")
    H.assert_tokens_match(fused_np, ref.cpu().numpy(), near, f"{what}: fused vs HEAD_REFERENCE")
    H.assert_tokens_match(fused_np, unf, near, f"{what}: fused vs unfused step on float64-made logits")

    sel = _sample_rows(B, N, sms, seed)
    want, ties = _oracle_tokens(tl64, hc, hu, x_t, t, s, K, sel, seed=seed, offset=offset, row_offset=row_offset)
    print(f"[oracle] {what}: {len(sel)} sampled rows, {int(ties.sum())} near-ties")
    H.assert_tokens_match(fused_np.reshape(-1)[sel.numpy()], want, ties, f"{what}: fused vs oracle")
    H.assert_tokens_match(ref.cpu().numpy().reshape(-1)[sel.numpy()], want, ties, f"{what}: HEAD_REFERENCE vs oracle")
    assert (fused != x_t).any()

    logits = head.head_step(hw, hc, hu, None, None, None, guidance_scale=gs, mode=_lib.HEAD_LOGITS)
    flat, err = logits.view(B * N, K), 0.0
    for r0 in range(0, B * N, ROW_CHUNK):
        err = max(err, (flat[r0:r0 + ROW_CHUNK].double() - _combined64(tl64, hc, hu, s, r0, r0 + ROW_CHUNK)).abs().max().item())
    print(f"[logits] {what}: max |HEAD_LOGITS - float64| = {err:.2e} (bound {LOGIT_TOL:.0e})")
    assert err <= LOGIT_TOL, f"{what}: combined logits differ from float64 torch by {err}"
    if chunks is not None:
        for v0, v1 in zip(chunks[:-1], chunks[1:]):
            part = head.head_step(hw, hc[v0:v1], None if hu is None else hu[v0:v1], None, None, None, guidance_scale=gs,
                                  mode=_lib.HEAD_LOGITS)
            assert torch.equal(part, logits[v0:v1]), f"{what}: HEAD_LOGITS of videos {v0}..{v1 - 1} differ from the whole-batch call"


# ---- A: the benchmarked shape and other multi-tile shapes -----------------------------------------------------------
# 53 x 1000: tiles straddle videos, the last tile holds 8 rows, videos 16 / 32 / 48 start on tile boundaries (37 x 1000 has
# the same layout but only 290 tiles, fewer than twice the 148 SMs of a B200).  44 x 2500: the last tile holds 48 rows; no
# video boundary below 32 videos is a tile boundary, so that case has no chunked run.
CASES = {
    "bench": dict(K=4096, B=16, N=4096, s=2.0, weights="bench", chunks=(0, 4, 8, 12, 16)),
    "bench_scale3": dict(K=4096, B=16, N=4096, s=2.0, weights="scale3", chunks=(0, 4, 8, 12, 16)),
    "straddle_k4096": dict(K=4096, B=53, N=1000, s=None, weights="scale3", chunks=(0, 16, 32, 48, 53)),
    "k2048_s3": dict(K=2048, B=44, N=2500, s=3.0, weights="scale3", chunks=None),
    "k1024": dict(K=1024, B=20, N=4096, s=None, weights="scale3", chunks=(0, 4, 8, 12, 16, 20)),
}


@pytest.mark.parametrize("name", list(CASES))
def test_multi_tile_shapes(name):
    c = CASES[name]
    K, B, N, s = c["K"], c["B"], c["N"], c["s"]
    g = torch.Generator().manual_seed(len(name))
    if c["weights"] == "bench":
        # bench.py (measure_next_rows): randn hidden states of a seeded device generator, every video at t = 50
        tl = _bench_head(K, 77).to(DEV)
        gen = torch.Generator(device=DEV).manual_seed(77)
        hc = torch.randn(B, N, D, device=DEV, generator=gen)
        hu = torch.randn(B, N, D, device=DEV, generator=gen)
        t = torch.full((B,), 50, dtype=torch.int64)
    else:
        tl = _head(K, 5).to(DEV)
        hc = (torch.randn(B, N, D, generator=g) * 2 + 0.3).to(DEV)
        hu = torch.randn(B, N, D, generator=g).to(DEV)
        t = _t_cycle(B)
    x_t = _x_t(B, N, K, t, g).to(DEV)
    _check_case(tl, hc, hu if s is not None else None, x_t, t.to(DEV), s, chunks=c["chunks"], seed=5, offset=3,
                row_offset=1000, what=name)


# ---- B: redo and survivor-overflow paths, bad inputs in late tiles ---------------------------------------------------
def test_redo_and_overflow_paths_at_scale():
    K, B, N, s = 4096, 16, 4096, 2.0
    sms = _multi_tile(B, N)
    tl = _bench_head(K, 78).to(DEV)
    g = torch.Generator().manual_seed(9)
    hc, hu = torch.randn(B, N, D, generator=g).to(DEV), torch.randn(B, N, D, generator=g).to(DEV)
    # mostly masked rows at t <= 1: their posterior is spread over the codes, ~thin_factor survivors per row
    t = torch.tensor([0, 1, 0, 1, 50, 0, 1, 0, 1, 0, 99, 1, 0, 1, 0, 1]).to(DEV)
    x_t = torch.where(torch.rand(B, N, generator=g) < 0.85, torch.full((B, N), K), torch.randint(0, K, (B, N), generator=g)).to(DEV)
    table = _table(K)
    hw = head.HeadWeights.from_module(tl)
    assert hw.valid
    kw = dict(guidance_scale=s, seed=12, offset=7, row_offset=0)
    args = (hw, hc, hu, x_t, t, table)

    def run(thin, x=x_t, tt=t, status=None):
        scratch = head.head_scratch(B, N, DEV)
        tok = head.head_step(hw, hc, hu, x, tt, table, thin_factor=thin, scratch=scratch, status=status, **kw)
        listed = scratch[0][:int(scratch[1].item())].long()
        assert listed.unique().numel() == listed.numel(), "a row was listed for the redo kernel twice"
        return tok, listed

    clean, listed0 = run(0.0)
    ref = head.head_step(*args, mode=_lib.HEAD_REFERENCE, **kw)
    near, _ = _unfused_near_ties(copy.deepcopy(tl).double(), hc, hu, x_t, t, table, s, K, seed=12, offset=7, row_offset=0)
    near = near.reshape(-1)
    H.assert_tokens_match(clean.view(-1).cpu().numpy(), ref.view(-1).cpu().numpy(), near, "default thinning vs HEAD_REFERENCE")
    print(f"[redo] default thinning: {listed0.numel()} of {B * N} rows redone; {int(near.sum())} near-ties")

    for thin, least in ((1e-3, 0.99), (64.0, 0.5)):
        tok, listed = run(thin)
        share = listed.numel() / (B * N)
        print(f"[redo] thin_factor={thin:g}: {listed.numel()} of {B * N} rows redone ({100 * share:.1f} %)")
        assert share >= least, f"thin_factor={thin}: only {100 * share:.1f} % of the rows reached the redo kernel"
        # a listed row is finished by head_redo_kernel, the arithmetic of HEAD_REFERENCE
        assert torch.equal(tok.view(-1)[listed], ref.view(-1)[listed]), f"thin_factor={thin}: redone rows differ from HEAD_REFERENCE"
        rest = torch.ones(B * N, dtype=torch.bool, device=DEV)
        rest[listed] = False
        rest = rest.cpu().numpy()
        H.assert_tokens_match(tok.view(-1).cpu().numpy()[rest], ref.view(-1).cpu().numpy()[rest], near[rest],
                              f"thin_factor={thin}: raced rows vs HEAD_REFERENCE")
        H.assert_tokens_match(tok.view(-1).cpu().numpy(), clean.view(-1).cpu().numpy(), near, f"thin_factor={thin} vs default")

    # one bad token and one bad t, each in a video all of whose tiles are some CTA's third or later tile
    v_late = -(-2 * sms * TILE // N)
    assert v_late + 2 < B
    vt, vT = v_late, v_late + 2
    row = vt * N + 777
    x_bad = x_t.clone()
    x_bad.view(-1)[row] = K + 7
    st = ops.new_status(DEV)
    tok, _ = run(0.0, x=x_bad, status=st)
    assert int(st.item()) == _lib.STATUS_BAD_TOKEN, f"status {int(st.item())} after an out-of-range token"
    keep = torch.ones(B * N, dtype=torch.bool, device=DEV)
    keep[row] = False
    assert torch.equal(tok.view(-1)[keep], clean.view(-1)[keep]), "an out-of-range token changed other rows"
    x_mask = x_t.clone()
    x_mask.view(-1)[row] = K
    assert torch.equal(tok, run(0.0, x=x_mask)[0]), "an out-of-range token is not stepped as [MASK]"

    t_bad = t.clone()
    t_bad[vT] = T + 5
    st = ops.new_status(DEV)
    tok, _ = run(0.0, tt=t_bad, status=st)
    assert int(st.item()) == _lib.STATUS_BAD_T, f"status {int(st.item())} after an out-of-range t"
    others = torch.ones(B, N, dtype=torch.bool, device=DEV)
    others[vT] = False
    assert torch.equal(tok[others], clean[others]), "an out-of-range t changed rows of other videos"
    t_last = t.clone()
    t_last[vT] = T - 1
    assert torch.equal(tok, run(0.0, tt=t_last)[0]), "an out-of-range t is not clamped to T - 1"


# ---- C: at the edge of the validity bound ---------------------------------------------------------------------------
def _edge_of_bound(K, seed):
    """A head whose validity bound is 99.9 % tight and hidden rows that point along one class of the conditional branch and
    against it (or along another class) in the unconditional one, swept from exactly along to pure noise."""
    g = torch.Generator().manual_seed(seed)
    L = 0.5 * (69.99 - math.log(K))
    W = torch.randn(K, D, generator=g, dtype=torch.float64)
    W -= W.mean(1, keepdim=True)  # LayerNorm outputs have mean 0: one can point along every row
    W[64:128] = -W[:64]           # classes 64 .. 127 are the antipodes of 0 .. 63
    Wn = W / W.norm(dim=1, keepdim=True)
    tl = torch.nn.Sequential(torch.nn.LayerNorm(D), torch.nn.Linear(D, K))
    with torch.no_grad():
        tl[1].weight.copy_(Wn * (0.999 * L / math.sqrt(D)))
        tl[1].bias.zero_()
    B, N = 4, 512
    i = torch.arange(N)
    theta = (math.pi / 2) * ((i // 4) % 64).double().view(1, N, 1) / 63

    def unit(x):
        x = x - x.mean(-1, keepdim=True)
        return x / x.norm(dim=-1, keepdim=True)

    k1 = torch.randint(0, 64, (B, N), generator=g)
    k3 = torch.randint(128, K, (B, N), generator=g)
    noise_c, noise_u = (unit(torch.randn(B, N, D, generator=g, dtype=torch.float64)) for _ in range(2))
    along_u = torch.where(((i // 256) % 2 == 0).view(1, N, 1), -Wn[k1], Wn[k3])
    # norm 8 = sqrt(D): unit variance, so eps hardly shortens the LayerNorm output
    hc = (8 * unit(theta.cos() * Wn[k1] + theta.sin() * noise_c)).float()
    hu = (8 * unit(theta.cos() * along_u + theta.sin() * noise_u)).float()
    return tl, hc, hu, torch.tensor([0, 1, 50, 99]), L, g


@pytest.mark.parametrize("K", [4096, 1024])
@pytest.mark.parametrize("s", [2.0, 5.0, None])
def test_at_the_edge_of_the_validity_bound(K, s):
    tl, hc, hu, t, L, g = _edge_of_bound(K, K + int(s or 0))
    B, N, _ = hc.shape
    tl64 = copy.deepcopy(tl).double()
    with torch.no_grad():
        lc64, lu64 = tl64(hc.double()), tl64(hu.double())
        ac, au = tl64[0](hc.double()), tl64[0](hu.double())
    lsc, lsu = torch.log_softmax(lc64, -1), torch.log_softmax(lu64, -1)
    # the premise of the fused kernel: neither branch reaches the -70 clamp
    assert lsc.min() > -70 and (s is None or lsu.min() > -70), (lsc.min().item(), lsu.min().item())
    if s is None:
        mix, hu = lsc, None
    else:
        mix = lsu + s * (lsc - lsu)
        mix = mix - torch.logsumexp(mix, -1, keepdim=True)
        fired = (mix < -70).any(-1).double().mean().item()
        print(f"\n[clamp] K={K} s={s:g}: the mix clamp fires on {100 * fired:.1f} % of the rows")
        assert fired >= 0.25, f"the mix clamp fires on only {100 * fired:.1f} % of the rows"
    kind = torch.arange(N).view(1, N) % 4  # x_t: masked, the dominant class, the most suppressed class, random
    x_t = torch.where(kind == 0, K, torch.where(kind == 1, mix.argmax(-1), torch.where(kind == 2, mix.argmin(-1),
                                                                                      torch.randint(0, K, (B, N), generator=g))))

    tl = tl.to(DEV)
    hw = head.HeadWeights.from_module(tl)
    assert hw.valid and hw.logit_bound >= 0.99 * L, (hw.logit_bound, L)
    table = _table(K)
    gs = s if s is not None else 1.0
    kw = dict(guidance_scale=gs, seed=21, offset=2, row_offset=5)
    args = (hw, hc.to(DEV), None if hu is None else hu.to(DEV), x_t.to(DEV), t.to(DEV), table)
    status = ops.new_status(DEV)
    fused = head.head_step(*args, status=status, **kw)
    assert int(status.item()) == 0
    assert torch.equal(head.head_step(*args, stats_1xtf32=False, **kw), fused), "1xTF32 and 3xTF32 statistics differ"
    ref = head.head_step(*args, mode=_lib.HEAD_REFERENCE, **kw).cpu()
    fused = fused.cpu()
    u = ops.philox_uniform(B, N, K, seed=21, offset=2, row_offset=5, device=DEV)[:, :, :K + 1].cpu().permute(0, 2, 1)
    out, post, _ = O.p_sample_step(O.make_schedule(T, K), lc64.permute(0, 2, 1), None if hu is None else lu64.permute(0, 2, 1),
                                   O.index_to_log_onehot(x_t, K + 1), t, 0.0 if s is None else s, u)
    want, ties = out.argmax(1).numpy(), O.near_ties(post, u).numpy()
    print(f"[oracle] K={K} s={s}: {int(ties.sum())} near-ties in {B * N} rows")
    H.assert_tokens_match(fused.numpy(), want, ties, "fused vs oracle")
    H.assert_tokens_match(ref.numpy(), want, ties, "HEAD_REFERENCE vs oracle")

    # HEAD_LOGITS: 3xTF32 drops a_lo w_lo and reads a_lo and w_lo as tf32, each term < 2^-20 |a_i| |w_i| per product, so
    # < 3 2^-20 ||a|| max ||W_k|| per logit with a = s a_c + (1 - s) a_u, ||a|| <= |s| ||a_c|| + |1 - s| ||a_u||; fp32
    # rounding of the accumulator and of the log2 scaling adds < 2^-20 |logit|
    logits = head.head_step(hw, args[1], args[2], None, None, None, guidance_scale=gs, mode=_lib.HEAD_LOGITS).cpu().double()
    want_l = lc64 if s is None else s * lc64 + (1 - s) * lu64
    a_norm = ac.norm(dim=-1) if s is None else abs(s) * ac.norm(dim=-1) + abs(1 - s) * au.norm(dim=-1)
    w_max = tl64[1].weight.norm(dim=1).max()
    tol = 2.0 ** -20 * (3 * a_norm * w_max + want_l.abs().amax(-1)) + 1e-6
    err = (logits - want_l).abs().amax(-1)
    print(f"[logits] K={K} s={s}: max |HEAD_LOGITS - float64| = {err.max().item():.2e} (|logit| up to "
          f"{want_l.abs().max().item():.1f}), at most {(err / tol).max().item():.2f} of the row's bound")
    assert (err <= tol).all(), f"HEAD_LOGITS off by {(err / tol).max().item():.2f} x the 3xTF32 bound"


# ---- D: LayerNorm and bias edge rows -------------------------------------------------------------------------------
def _with_edge_rows(h, first, eps, g):
    """Rows first, first + 16, ... of h (flat) become, in turn: all zero; constant (variance 0); mean 30 with unit spread;
    spread about sqrt(eps).  The constants and the 30-offset rows are on a 2^-10 grid, so the fp32 sums of the kernel's mean
    are exact and the float64 reference measures the kernel rather than the rounding of an fp32 mean."""
    flat = h.view(-1, D)
    rows = torch.arange(first, flat.shape[0], 16)
    kind = torch.arange(rows.numel()) % 4
    const = torch.tensor([0.75, -3.5, 12.0])[torch.arange(rows.numel()) % 3]
    spread30 = 30 + torch.round(torch.randn(rows.numel(), D, generator=g) * 1024) / 1024
    tiny = math.sqrt(eps) * torch.randn(rows.numel(), D, generator=g)
    new = torch.where((kind == 0).view(-1, 1), 0.0, torch.where((kind == 1).view(-1, 1), const.view(-1, 1).expand(-1, D),
                                                                torch.where((kind == 2).view(-1, 1), spread30, tiny)))
    flat[rows] = new
    return h


@pytest.mark.parametrize("bias", [True, False])
def test_layer_norm_edge_rows(bias):
    K, B, N, s, eps = 4096, 10, 4096, 2.0, 1e-6
    g = torch.Generator().manual_seed(31)
    tl = torch.nn.Sequential(torch.nn.LayerNorm(D, eps=eps), torch.nn.Linear(D, K, bias=bias))
    with torch.no_grad():
        gamma = 1 + 0.6 * torch.randn(D, generator=g)
        gamma[::8] = 0.0
        gamma[3::8] = -gamma[3::8].abs()
        tl[0].weight.copy_(gamma)
        tl[0].bias.copy_(0.1 * torch.randn(D, generator=g))
        tl[1].weight.uniform_(-1 / 8, 1 / 8, generator=g)  # the distribution of torch's default initialisation
        if bias:
            tl[1].bias.uniform_(-1 / 8, 1 / 8, generator=g)
    hc = _with_edge_rows(torch.randn(B, N, D, generator=g) * 2 + 0.3, 1, eps, g)
    hu = _with_edge_rows(torch.randn(B, N, D, generator=g), 9, eps, g)
    t = _t_cycle(B)
    x_t = _x_t(B, N, K, t, g)
    _check_case(tl.to(DEV), hc.to(DEV), hu.to(DEV), x_t.to(DEV), t.to(DEV), s, chunks=(0, 4, 8, 10), seed=8, offset=1,
                row_offset=77, what=f"LayerNorm edge rows, bias={bias}")


# ---- E: the host entry of the head at a multi-tile shape -------------------------------------------------------------
def test_host_head_step_at_a_multi_tile_shape():
    """One kernel call over the whole batch (chunks=1): pinned host hidden states in, host tokens out, equal bit for bit to
    the device-resident head_step."""
    K, B, N, s = 4096, 16, 4096, 2.0
    _multi_tile(B, N)
    table = _table(K)
    hw = head.HeadWeights.from_module(_bench_head(K, 79).to(DEV))
    g = torch.Generator().manual_seed(41)
    hc, hu = torch.randn(B, N, D, generator=g).pin_memory(), torch.randn(B, N, D, generator=g).pin_memory()
    t = _t_cycle(B)
    x_t, t = _x_t(B, N, K, t, g).pin_memory(), t.pin_memory()
    host = ops.HostStep(B, N, K, table, guidance=True, hidden_dim=D, chunks=1)
    try:
        got = host.head(hw, hc, hu, x_t, t, guidance_scale=s, seed=3, offset=4, row_offset=11).clone()
        assert host.last_status == 0
    finally:
        host.close()
    want = head.head_step(hw, hc.to(DEV), hu.to(DEV), x_t.to(DEV), t.to(DEV), table, guidance_scale=s, seed=3, offset=4,
                          row_offset=11)
    assert torch.equal(got, want.cpu())
