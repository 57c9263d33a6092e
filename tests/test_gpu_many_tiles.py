"""Every persistent kernel at the tile counts the benchmark launches, and the whole head at the benchmark's batch sizes.

The hot kernels are persistent: the launcher sizes the grid to the SM count and each CTA loops over tiles.  The
accumulator hand-off (TMEM slot = tile ordinal & 1, ``acc_empty`` waited on from a CTA's third tile, its second parity
from the fifth), K3's prefetch of the next tile's tap offsets, the TMA-store buffer rotation and the cluster strides only
run once a CTA reaches its second tile or a later one.  Each case below is sized from the device's SM count S so that the
busiest CTA takes at least 5 tiles, the last wave is ragged (tiles % grid != 0) and, where the shape allows it, the last
tile is ragged in rows.  Two oracles per case:

(a) bit-identity: the same inputs split into launches small enough that no CTA takes a second tile (slices of the batch, or
    of M for Linear) must give the same bits as the big launch -- the regime the float64 tests of test_gpu_kernels.py
    validate, carried over to every output element of the big launch;
(b) float64 maths on the same bf16- or fp32-rounded operands over every row of the tiles of the last wave (tile index
    >= tiles - grid) and of the first tile, at the bar of the kernel's existing test.

The head part builds the nets the way bench.py does and checks that every output of its timed batch is bit-identical to the
same RoI run in 2-RoI batches and that a permuted batch gives permuted outputs: our kernels have no atomics, no split-K and a
fixed MMA order, so a RoI's outputs do not depend on the batch it runs in or on which CTA takes its tiles."""
import argparse

import pytest
import torch
import torch.nn.functional as F

from helpers import syn

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

TILE = 128
LM15 = tuple(range(1, 16))


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    return ops


def num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------------ launch geometry
def grid_of(rule, work, S):
    """The launchers' grid rules.  ``work`` = tiles, or units / tile pairs for the cluster kernels.
    sm:   min(tiles, S)        cp_gemm_x3, cp_conv_bf16 (single CTA), cp_conv_slab (single), K3, K4, cp_edgeconv_fwd
    2sm:  min(tiles, 2S)       cp_chain_fwd, cp_edge_aggregate_staged_f32 with <= 110 KB of shared memory
    half: min(units, S/2)      clusters of cp_conv_slab (pair), of cp_conv_bf16 (multicast)"""
    cap = {"sm": S, "2sm": 2 * S, "half": S // 2}[rule]
    return min(work, cap)


def check_waves(tag, work, grid, ragged_rows=None):
    """Busiest CTA (or cluster) >= 5 tiles, ragged last wave, ragged last tile where the shape allows it."""
    per = cdiv(work, grid)
    assert per >= 5, f"{tag}: busiest CTA takes {per} tiles"
    assert work % grid != 0, f"{tag}: the last wave is full ({work} tiles over {grid})"
    if ragged_rows is not None:
        assert ragged_rows % TILE != 0, f"{tag}: the last tile is full"
    return per


def report(tag, work, grid, per, err):
    print(f"[{tag}] tiles {work}, grid {grid}, tiles per CTA {per} (last wave {work % grid}), float64 max err / max = {err:.2e}")


def sampled_tiles(work, grid):
    """The first tile and every tile of the last wave."""
    return sorted({0} | set(range(work - grid, work)))


def flat_rows(tiles, M):
    """Rows of 128-row tiles over a flat matrix of M rows."""
    return torch.cat([torch.arange(t * TILE, min(M, (t + 1) * TILE)) for t in tiles])


def roi_rows(tiles, N):
    """(b, n) of the rows of node tiles tiled per RoI (tile t = RoI t // tiles_per_roi)."""
    tpr = cdiv(N, TILE)
    bs, ns = [], []
    for t in tiles:
        b, r = divmod(t, tpr)
        n = torch.arange(r * TILE, min(N, (r + 1) * TILE))
        bs.append(torch.full_like(n, b))
        ns.append(n)
    return torch.cat(bs), torch.cat(ns)


def roi_chunks(B, per_roi, cap):
    """Batch slices of at most ``cap`` tiles each (per_roi tiles per RoI)."""
    step = max(1, cap // per_roi)
    assert step * per_roi <= cap, "one RoI needs more tiles than a chunk may take"
    return [(b0, min(B, b0 + step)) for b0 in range(0, B, step)]


def image_chunks(B, rows_per_image, cap_tiles):
    """Batch slices whose flat rows fill at most ``cap_tiles`` tiles (images straddle tiles)."""
    step = cap_tiles * TILE // rows_per_image
    assert step >= 1
    return [(b0, min(B, b0 + step)) for b0 in range(0, B, step)]


def rel_max(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max())


def bf16r(t):
    return t.to(torch.bfloat16).float()


def lrelu64(x, s):
    return torch.where(x > 0, x, x * s)


# ------------------------------------------------------------------------------------------------ split-bf16 x3 GEMM
@pytest.mark.parametrize("K1,K2,Nout,act", [(256, 256, 256, True),    # pre-graph MLP layer 0: [taps | graph feature]
                                             (256, 0, 512, True),      # two column blocks: tile -> (m, n)
                                             (64, 0, 7, False),        # direct-store epilogue (init logits)
                                             (64, 0, 2, False)])       # direct-store epilogue (refine logits)
def test_gemm_x3_linear_many_tiles(ops, K1, K2, Nout, act):
    S = num_sms()
    M = 5 * S * TILE + 77
    nblk = cdiv(cdiv(Nout, 16) * 16, 256)
    work = cdiv(M, TILE) * nblk
    grid = grid_of("sm", work, S)
    per = check_waves(f"x3 linear {K1}+{K2}->{Nout}", work, grid, M)
    g = torch.Generator().manual_seed(K1 + K2 + Nout)
    a1 = torch.randn(M, K1, generator=g)
    a2 = torch.randn(M, K2, generator=g) if K2 else None
    w = torch.randn(Nout, K1 + K2, generator=g) / (K1 + K2) ** 0.5
    bias = torch.randn(Nout, generator=g)
    ws = ops.pack_weight_split(w.cuda())
    a1d, a2d, bd = a1.cuda(), None if a2 is None else a2.cuda(), bias.cuda()
    big = ops.gemm_x3_linear(a1d, ws, Nout, bd, act, 0.01, a2=a2d)
    step = (S // nblk) * TILE
    parts = [ops.gemm_x3_linear(a1d[r0:r0 + step], ws, Nout, bd, act, 0.01, a2=None if a2d is None else a2d[r0:r0 + step])
             for r0 in range(0, M, step)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    rows = flat_rows(sorted({t // nblk for t in sampled_tiles(work, grid)}), M)
    a = a1[rows] if a2 is None else torch.cat([a1[rows], a2[rows]], 1)
    ref = a.double() @ w.double().t() + bias.double()
    if act:
        ref = lrelu64(ref, 0.01)
    err = rel_max(big.cpu()[rows], ref)
    report(f"x3 linear {K1}+{K2}->{Nout}", work, grid, per, err)
    assert err < 2e-5, err


@pytest.mark.parametrize("B,H,Cin,Cout,k,pad,transposed", [(24, 64, 256, 256, 3, 1, False),    # up_net 3x3 at 64 x 64
                                                           (24, 64, 256, 64, 2, 1, False),     # patch_generator 2x2, pad 1
                                                           (375, 8, 1024, 256, 3, 1, True)])   # up_net[0]: transposed, stride 2
def test_gemm_x3_conv_many_tiles(ops, B, H, Cin, Cout, k, pad, transposed):
    S = num_sms()
    Ho = 2 * H if transposed else H + 2 * pad - k + 1
    M = B * Ho * Ho
    work = cdiv(M, TILE)
    grid = grid_of("sm", work, S)
    tag = f"x3 conv{'T' if transposed else ''} {k}x{k} {Cin}->{Cout} at {H}x{H}, B={B}"
    per = check_waves(tag, work, grid, M if M % TILE else None)
    g = torch.Generator().manual_seed(B + H + Cin + k)
    x = torch.randn(B, Cin, H, H, generator=g)
    bias = torch.randn(Cout, generator=g)
    if transposed:
        w = torch.randn(Cin, Cout, k, k, generator=g) / (Cin * k * k / 4) ** 0.5
        wm = w.permute(1, 2, 3, 0).reshape(Cout, k * k * Cin)
    else:
        w = torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5
        wm = w.permute(0, 2, 3, 1).reshape(Cout, k * k * Cin)
    ws = ops.pack_weight_split(wm.contiguous().cuda())
    xd = x.permute(0, 2, 3, 1).contiguous().cuda()
    bd = bias.cuda()

    def run(xs):
        return ops.gemm_x3_conv(xs, ws, Cout, k, k, pad, Ho, Ho, bd, True, 0.0, transposed)
    big = run(xd)
    parts = [run(xd[b0:b1]) for b0, b1 in image_chunks(B, Ho * Ho, S)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    rows = flat_rows(sampled_tiles(work, grid), M)
    imgs = torch.unique(rows // (Ho * Ho))
    xs = x[imgs].double()
    if transposed:
        ref = F.conv_transpose2d(xs, w.double(), bias.double(), stride=2, padding=pad, output_padding=1)
    else:
        ref = F.conv2d(xs, w.double(), bias.double(), padding=pad)
    ref = torch.relu(ref).permute(0, 2, 3, 1)
    err = rel_max(big.cpu()[imgs], ref)
    report(tag, work, grid, per, err)
    assert err < 2e-5, err


# ------------------------------------------------------------------------------------------------ bf16 implicit-GEMM conv
def test_conv_bf16_conv1x1_many_tiles(ops):
    """The init head's conv1x1 1024 -> 4096 at 8 x 8: 16 column blocks (no multicast), tile -> (m, n)."""
    S = num_sms()
    B, H, Cin, Cout = 96, 8, 1024, 4096
    M = B * H * H
    nblk = Cout // 256
    work = cdiv(M, TILE) * nblk
    grid = grid_of("sm", work, S)
    per = check_waves("conv_bf16 1x1 1024->4096", work, grid)
    g = torch.Generator().manual_seed(1024)
    x = bf16r(torch.randn(M, Cin, generator=g))
    w = bf16r(torch.randn(Cout, Cin, generator=g) / Cin ** 0.5)
    bias = torch.randn(Cout, generator=g)
    xd = x.view(B, H, H, Cin).cuda().to(torch.bfloat16)
    wp, bd = ops.pack_weight(w.cuda()), bias.cuda()

    def run(xs):
        return ops.conv_bf16(xs, wp, Cout, 1, 1, 0, H, H, bd, False, 0.0)
    big = run(xd)
    parts = [run(xd[b0:b1]) for b0, b1 in image_chunks(B, H * H, S // nblk)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    rows = flat_rows(sorted({t // nblk for t in sampled_tiles(work, grid)}), M)
    ref = x[rows].double() @ w.double().t() + bias.double()
    err = rel_max(big.reshape(M, Cout).cpu()[rows].float(), ref)
    report("conv_bf16 1x1 1024->4096", work, grid, per, err)
    assert err < 6e-3, err


@pytest.mark.parametrize("multicast", ["1", "0"])
def test_conv_bf16_one_column_block_many_tiles(ops, monkeypatch, multicast):
    """One column block: the weight-multicast CTA pairs (clusters step over tile pairs, an odd tile count repeats the last
    tile) and the single-CTA kernel."""
    S = num_sms()
    B, H, Cin, Cout = 343, 15, 256, 256
    M = B * H * H
    tiles = cdiv(M, TILE)
    assert tiles % 2 == 1
    monkeypatch.setenv("CP_CONV_MULTICAST", multicast)
    if multicast == "1":
        work, cap = cdiv(tiles, 2), S - S % 2          # work = tile pairs per cluster, chunks of <= S & ~1 tiles
        grid = grid_of("half", work, S)
    else:
        work, cap = tiles, S
        grid = grid_of("sm", work, S)
    tag = f"conv_bf16 3x3 {Cin}->{Cout} at {H}x{H} multicast={multicast}"
    per = check_waves(tag, work, grid, M)
    g = torch.Generator().manual_seed(343)
    x = bf16r(torch.randn(B, Cin, H, H, generator=g))
    w = bf16r(torch.randn(Cout, Cin, 3, 3, generator=g) / (Cin * 9) ** 0.5)
    bias = torch.randn(Cout, generator=g)
    xd = x.permute(0, 2, 3, 1).contiguous().cuda().to(torch.bfloat16)
    wp = ops.pack_weight(w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous().cuda())
    bd = bias.cuda()

    def run(xs):
        return ops.conv_bf16(xs, wp, Cout, 3, 3, 1, H, H, bd, True, 0.0)
    big = run(xd)
    parts = [run(xd[b0:b1]) for b0, b1 in image_chunks(B, H * H, cap)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    last = sampled_tiles(tiles, 2 * grid if multicast == "1" else grid)
    imgs = torch.unique(flat_rows(last, M) // (H * H))
    ref = torch.relu(F.conv2d(x[imgs].double(), w.double(), bias.double(), padding=1)).permute(0, 2, 3, 1)
    err = rel_max(big.cpu()[imgs].float(), ref)
    report(tag, work, grid, per, err)
    assert err < 6e-3, err


# ------------------------------------------------------------------------------------------------ slab convolutions
def slab_geometry(S, pair, row_tiles, phases):
    """-> (work, grid, chunk cap in row tiles) of cp_conv_slab: single CTAs take (phase, tile) units, pairs take units of
    two neighbouring row tiles and step over them by clusters."""
    if pair:
        work = cdiv(row_tiles, 2) * phases
        return work, grid_of("half", work, S), 2 * ((S // 2) // phases)
    work = row_tiles * phases
    return work, grid_of("sm", work, S), S // phases


def check_border(out, tag):
    edge = out.clone()
    edge[:, :-1, :-1] = 0
    assert not bool(edge.any()), f"{tag}: the border of a slab convolution's output must be zeros"


@pytest.mark.parametrize("kind,B,H,Cin,Cout", [("same3", 24, 64, 512, 256),    # up_net at 64 x 64 on the 512-channel concat
                                                ("same3", 340, 16, 256, 256),  # 16 x 16: tiles straddle images at every tile
                                                ("full2", 24, 64, 256, 64),    # patch_generator 2x2, padding 1
                                                ("convT", 240, 8, 1024, 256),  # up_net[0]: four output parities
                                                ("seg", 24, 64, 256, 256)])    # last up_net convolution + fused seg_block
def test_conv_slab_many_tiles(ops, monkeypatch, kind, B, H, Cin, Cout):
    S = num_sms()
    g = torch.Generator().manual_seed(B + H + Cin + len(kind))
    k = 2 if kind == "full2" else 3
    x = bf16r(torch.randn(B, Cin, H, H, generator=g))
    bias = torch.randn(Cout, generator=g)
    if kind == "convT":
        w = bf16r(torch.randn(Cin, Cout, 3, 3, generator=g) / (Cin * 9 / 4) ** 0.5)
        wm = w.permute(1, 2, 3, 0).reshape(Cout, 9 * Cin)
    else:
        w = bf16r(torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5)
        wm = w.permute(0, 2, 3, 1).reshape(Cout, k * k * Cin)
    wp, bd = ops.pack_weight(wm.contiguous().cuda()), bias.cuda()
    seg = None
    if kind == "seg":
        seg = ((torch.randn(2, Cout, generator=g) / Cout ** 0.5).cuda(), torch.randn(2, generator=g).cuda())
    xh = x.permute(0, 2, 3, 1).contiguous().cuda().to(torch.bfloat16)
    Hp = H + 1                                           # input rows of the launch: the bordered input map
    phases = 4 if kind == "convT" else 1
    rows_in = B * Hp * Hp
    row_tiles = cdiv(rows_in, TILE)
    xp = ops.to_bordered(xh).contiguous()

    def run(b0, b1):
        if kind == "convT":
            return ops.convT_slab(xh[b0:b1], wp, Cout, bd, True, 0.0), None
        if kind == "full2":
            return ops.conv_slab_full(xp[b0:b1], wp, Cout, 2, 2, bd, True, 0.0), None
        if kind == "seg":
            return ops.conv_slab_same(xp[b0:b1], wp, Cout, 3, 3, bd, True, 0.0, seg=seg)
        return ops.conv_slab_same(xp[b0:b1], wp, Cout, 3, 3, bd, True, 0.0), None

    # float64 reference on the images holding the sampled rows (single and pair sample the same rows: the last wave's units)
    results = {}
    for pair in ("1", "0"):
        monkeypatch.setenv("CP_SLAB_PAIR", pair)
        work, grid, cap = slab_geometry(S, pair == "1", row_tiles, phases)
        tag = f"slab {kind} {Cin}->{Cout} at {H}x{H}, B={B}, pair={pair}"
        per = check_waves(tag, work, grid, rows_in)
        big, seg_big = run(0, B)
        parts = [run(b0, b1) for b0, b1 in image_chunks(B, Hp * Hp, cap)]
        assert torch.equal(big, torch.cat([p[0] for p in parts])), f"{tag}: the multi-wave launch differs from one-tile-per-CTA launches"
        if seg is not None:
            assert torch.equal(seg_big, torch.cat([p[1] for p in parts])), f"{tag}: fused seg head differs"
        results[pair] = (big, seg_big, work, grid, per, tag)
    # sampled units -> row tiles (phase-major units; a pair unit is two neighbouring row tiles)
    imgs = set()
    for pair, (_, _, work, grid, _, _) in results.items():
        per_phase = cdiv(row_tiles, 2) if pair == "1" else row_tiles
        for u in sampled_tiles(work, grid):
            r = u % per_phase
            for rt in ((2 * r, 2 * r + 1) if pair == "1" else (r,)):
                if rt < row_tiles:
                    imgs.update(range(rt * TILE // (Hp * Hp), min(B - 1, ((rt + 1) * TILE - 1) // (Hp * Hp)) + 1))
    imgs = torch.tensor(sorted(imgs))
    xs = x[imgs].double()
    if kind == "convT":
        ref = F.conv_transpose2d(xs, w.double(), bias.double(), stride=2, padding=1, output_padding=1)
    else:
        ref = F.conv2d(xs, w.double(), bias.double(), padding=k - 1 if kind == "full2" else 1)
    ref = torch.relu(ref).permute(0, 2, 3, 1)
    for pair, (big, seg_big, work, grid, per, tag) in results.items():
        out = big.cpu()[imgs].float()
        if kind != "full2":
            check_border(big, tag)
            out = out[:, :-1, :-1]
        err = rel_max(out, ref)
        if seg is not None:
            sref = torch.einsum("bhwc,jc->bjhw", out.double(), seg[0].cpu().double()) + seg[1].cpu().double().view(1, -1, 1, 1)
            serr = rel_max(seg_big.cpu()[imgs], sref)
            print(f"[{tag}] fused seg: float64 max err / max = {serr:.2e}")
            assert serr < 1e-5, serr
        report(tag, work, grid, per, err)
        assert err < 6e-3, (tag, err)


# ------------------------------------------------------------------------------------------------ K3 taps chain
@pytest.mark.parametrize("N,B", [(4096, 24), (1000, 96)])
@pytest.mark.parametrize("Cg,nout2", [(64, 512), (256, 512), (64, 256), (256, 256)])
def test_taps_chain_many_tiles(ops, Cg, nout2, N, B):
    """K3 (cp_chain_fwd(CP_PRO_TAPS) -> taps_chain_kernel): the next tile's tap offsets are prefetched, h_free phases and
    the TMA-store rotation carry across tiles; a 256-column last layer gives 3 accumulator stages per tile, so the slot a
    tile starts on alternates."""
    S = num_sms()
    tpr = cdiv(N, TILE)
    work = B * tpr
    grid = grid_of("sm", work, S)
    tag = f"K3 Cg={Cg} nout={nout2} N={N} B={B}"
    per = check_waves(tag, work, grid, N if N % TILE else None)
    g = torch.Generator().manual_seed(Cg + nout2 + N)
    H, Hp = 64, 65
    patches = bf16r(torch.randn(B, Hp, Hp, 64, generator=g))
    gf = bf16r(torch.randn(B, N, Cg, generator=g))
    x_id = torch.randint(0, H // 2, (B, N), generator=g)
    y_id = torch.randint(0, H // 2, (B, N), generator=g)
    mask = (torch.rand(B, N, generator=g) > 0.2).float()
    dims = ((256, 256 + Cg), (256, 256), (nout2, 256))
    ws = [bf16r(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5) for o, i in dims]
    bs = [torch.randn(o, generator=g) * 0.1 for o, _ in dims]
    layers = [ops.chain_layer(ops.pack_weight(w.cuda()), b.cuda(), w.shape[1], w.shape[0], li < 2, 0.01)
              for li, (w, b) in enumerate(zip(ws, bs))]
    dev = dict(patches=patches.cuda().to(torch.bfloat16), x_id=x_id.cuda(), y_id=y_id.cuda(), mask=mask.cuda(),
               graph_feat=gf.cuda().to(torch.bfloat16))

    def run(b0, b1):
        out = torch.full((b1 - b0, N, nout2), float("nan"), dtype=torch.bfloat16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_TAPS, B=b1 - b0, N=N, tap_step=2, layers=layers, out=out, out_mode=ops.OUT_BF16,
                      **{k: v[b0:b1] for k, v in dev.items()})
        return out
    big = run(0, B)
    assert bool(torch.isfinite(big.float()).all()), "rows not written"
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, S)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    bi, ni = roi_rows(sampled_tiles(work, grid), N)
    yy, xx = 2 * y_id[bi, ni], 2 * x_id[bi, ni]
    taps = torch.cat([patches[bi, yy + dy, xx + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1)
    h = torch.cat([taps * mask[bi, ni, None], gf[bi, ni]], dim=-1).double()
    for li, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.double().t() + b.double()
        if li < 2:
            h = bf16r(lrelu64(h, 0.01).float()).double()
    err = rel_max(big.cpu()[bi, ni].float(), h)
    report(tag, work, grid, per, err)
    assert err < 2e-2, err


# ------------------------------------------------------------------------------------------------ K4 query tail + decode
@pytest.mark.parametrize("N,B,with_kp", [(4096, 24, True), (4096, 24, False), (1000, 97, True)])
def test_query_decode_many_tiles(ops, N, B, with_kp):
    """cp_query_decode_fwd: tiles run over the flat (B N) rows, so they straddle RoIs; 15 graphs selected per RoI."""
    S = num_sms()
    M = B * N
    work = cdiv(M, TILE)
    grid = grid_of("sm", work, S)
    tag = f"K4 N={N} B={B} x_id_kp={'on' if with_kp else 'off'}"
    per = check_waves(tag, work, grid, M if M % TILE else None)
    g = torch.Generator().manual_seed(N + B + with_kp)
    kin, G, Ltot, plane = 256, 15, 6, 4
    src = bf16r(torch.randn(B, N, kin, generator=g))
    w1 = bf16r(torch.randn(64, kin, generator=g) / kin ** 0.5)
    b1 = torch.randn(64, generator=g) * 0.1
    w2 = torch.randn(2, 64, generator=g) / 8.0
    b2 = torch.randn(2, generator=g) * 0.1
    perm = torch.stack([torch.randperm(N, generator=g) for _ in range(G)]).to(torch.int32)
    sel = torch.randint(0, G, (B,), generator=g).to(torch.int32)
    x_id0 = torch.randint(0, 16, (B, N), generator=g)
    y_id0 = torch.randint(0, 16, (B, N), generator=g)
    w1p, b1d, w2d, b2d, permd = ops.pack_weight(w1.cuda()), b1.cuda(), w2.cuda().contiguous(), b2.cuda(), perm.cuda()
    srcd, seld = src.cuda().to(torch.bfloat16), sel.cuda()
    bufs = dict(x_bits=torch.full((B, Ltot, N), float("nan")), y_bits=torch.full((B, Ltot, N), float("nan")), x_id=x_id0.clone(),
                y_id=y_id0.clone(), logits=torch.zeros(B, N, 2))
    if with_kp:
        bufs.update(x_id_kp=torch.full((B, N), -1, dtype=torch.int64), y_id_kp=torch.full((B, N), -1, dtype=torch.int64))

    def run(b0, b1_, d):
        ops.query_decode_fwd(src=srcd[b0:b1_], w1_packed=w1p, b1=b1d, slope=0.01, w2=w2d, b2=b2d, plane=plane, Ltot=Ltot,
                             perm=permd, graph_sel=seld[b0:b1_], **{k: v[b0:b1_] for k, v in d.items()})
    big = {k: v.cuda() for k, v in bufs.items()}
    run(0, B, big)
    small = {k: v.cuda() for k, v in bufs.items()}
    for b0, b1_ in image_chunks(B, N, S):
        run(b0, b1_, small)
    for k in big:
        assert torch.equal(big[k].nan_to_num(7.0), small[k].nan_to_num(7.0)), f"{tag}: {k} of the multi-wave launch differs"
    lg = big["logits"].cpu()
    rows = flat_rows(sampled_tiles(work, grid), M)
    bi, ni = rows // N, rows % N
    ref = lrelu64(src[bi, ni].double() @ w1.double().t() + b1.double(), 0.01) @ w2.double().t() + b2.double()
    err = rel_max(lg[bi, ni], ref)
    report(tag, work, grid, per, err)
    assert err < 1e-3, err
    # the decode of the kernel's own logits, exactly, on every row
    kp = perm[sel.long()].long()
    want_x = torch.full((B, N), float("nan")).scatter_(1, kp, lg[..., 0])
    want_y = torch.full((B, N), float("nan")).scatter_(1, kp, lg[..., 1])
    xb, yb = big["x_bits"].cpu(), big["y_bits"].cpu()
    assert torch.equal(xb[:, plane], want_x) and torch.equal(yb[:, plane], want_y)
    others = [p for p in range(Ltot) if p != plane]
    assert torch.isnan(xb[:, others]).all() and torch.isnan(yb[:, others]).all()
    nx, ny = x_id0 * 2 + (lg[..., 0] > 0).long(), y_id0 * 2 + (lg[..., 1] > 0).long()
    assert torch.equal(big["x_id"].cpu(), nx) and torch.equal(big["y_id"].cpu(), ny)
    if with_kp:
        assert torch.equal(big["x_id_kp"].cpu(), torch.zeros(B, N, dtype=torch.int64).scatter_(1, kp, nx))
        assert torch.equal(big["y_id_kp"].cpu(), torch.zeros(B, N, dtype=torch.int64).scatter_(1, kp, ny))


# ------------------------------------------------------------------------------------------------ chain kernel, LOAD prologue
@pytest.mark.parametrize("what", ["query3_f32", "pq512_bf16"])
def test_chain_load_many_tiles(ops, what):
    """cp_chain_fwd(CP_PRO_LOAD), grid 2 S: the 3-layer query chain to fp32 logits (n_valid = 2, columns past it untouched)
    and a 256 -> 512 bf16 output."""
    S = num_sms()
    N, B = 4096, 48
    tpr = N // TILE
    work = B * tpr
    grid = grid_of("2sm", work, S)
    tag = f"chain LOAD {what} N={N} B={B}"
    per = check_waves(tag, work, grid)
    g = torch.Generator().manual_seed(len(what))
    x = bf16r(torch.randn(B, N, 256, generator=g))
    dims = ((256, 256), (64, 256), (2, 64)) if what == "query3_f32" else ((512, 256),)
    ws = [bf16r(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5) for o, i in dims]
    bs = [torch.randn(o, generator=g) * 0.1 for o, _ in dims]
    nl = len(dims)
    layers = [ops.chain_layer(ops.pack_weight(w.cuda()), b.cuda(), w.shape[1], w.shape[0], li < nl - 1, 0.01)
              for li, (w, b) in enumerate(zip(ws, bs))]
    xd = x.cuda().to(torch.bfloat16)

    def run(b0, b1):
        if nl == 3:
            out = torch.full((b1 - b0, N, 16), float("nan"), device="cuda")
            ops.chain_fwd(prologue=ops.PRO_LOAD, B=b1 - b0, N=N, src=xd[b0:b1], layers=layers, out=out, out_mode=ops.OUT_F32, n_valid=2)
        else:
            out = torch.full((b1 - b0, N, 512), float("nan"), dtype=torch.bfloat16, device="cuda")
            ops.chain_fwd(prologue=ops.PRO_LOAD, B=b1 - b0, N=N, src=xd[b0:b1], layers=layers, out=out, out_mode=ops.OUT_BF16)
        return out
    big = run(0, B)
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, 2 * S)]
    assert torch.equal(big.nan_to_num(7.0), torch.cat(parts).nan_to_num(7.0)), "the multi-wave launch differs from one-tile-per-CTA launches"
    if nl == 3:
        assert bool(torch.isnan(big[..., 2:]).all()), "columns >= n_valid were written"
        big = big[..., :2]
    bi, ni = roi_rows(sampled_tiles(work, grid), N)
    h = x[bi, ni].double()
    for li, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.double().t() + b.double()
        if li < nl - 1:
            h = bf16r(lrelu64(h, 0.01).float()).double()
    got = big.cpu()[bi, ni].double()
    err = rel_max(got, h)
    report(tag, work, grid, per, err)
    if nl == 3:
        assert err < 2e-2, err      # bf16 re-quantisation of the intermediates (test_chain_three_layers)
    else:
        assert torch.allclose(got, h, rtol=1e-2, atol=1e-2), err


# ------------------------------------------------------------------------------------------------ EdgeConv aggregation
def agg_rows(z, nb, bi, ni, Co, slope, round_bf16):
    """A[b, n] = lrelu(max_k P[b, nb[b, n, k]] + Q[b, n]) for the listed rows: exact max, one fp32 add, fp32 LeakyReLU
    (the kernels' arithmetic), then one rounding to bf16 when the kernel stores bf16.  z (B,N,2Co) float32 values."""
    idx = nb[bi, ni]                                                  # (R,K)
    m = torch.full((len(bi), Co), float("-inf"))
    for k in range(idx.shape[1]):
        m = torch.maximum(m, z[bi, idx[:, k], :Co])
    a = F.leaky_relu(m + z[bi, ni, Co:], slope)
    return bf16r(a) if round_bf16 else a


def lm_graphs(ops, objs, N, K):
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in objs], dim=0).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    return p3d, idx32


@pytest.mark.parametrize("K", [20, 40, 41])
def test_chain_agg_many_tiles(ops, K):
    """cp_chain_fwd(CP_PRO_AGG) (the head's EdgeConv path where the staged kernel does not fit), 3 graphs selected per RoI:
    the aggregated tile bit-exact, the 256 -> 512 bf16 GEMM within 1e-2."""
    S = num_sms()
    N, B, Co, nout = 4096, 48, 256, 512
    tpr = N // TILE
    work = B * tpr
    grid = grid_of("2sm", work, S)
    tag = f"chain AGG K={K} N={N} B={B}"
    per = check_waves(tag, work, grid)
    _, idx32 = lm_graphs(ops, (3, 9, 14), N, K)
    g = torch.Generator().manual_seed(K)
    z = bf16r(torch.randn(B, N, 2 * Co, generator=g))
    sel = torch.randint(0, 3, (B,), generator=g)
    w = bf16r(torch.randn(nout, Co, generator=g) / Co ** 0.5)
    bias = torch.randn(nout, generator=g)
    layer = ops.chain_layer(ops.pack_weight(w.cuda()), bias.cuda(), Co, nout, True, 0.01)
    zd, seld = z.cuda().to(torch.bfloat16), sel.to(torch.int32).cuda()

    def run(b0, b1):
        a_out = torch.empty((b1 - b0, N, Co), dtype=torch.bfloat16, device="cuda")
        out = torch.empty((b1 - b0, N, nout), dtype=torch.bfloat16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_AGG, B=b1 - b0, N=N, z=zd[b0:b1], idx32=idx32, graph_sel=seld[b0:b1], agg_slope=0.2,
                      a_out=a_out, layers=[layer], out=out, out_mode=ops.OUT_BF16)
        return a_out, out
    a_big, big = run(0, B)
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, 2 * S)]
    assert torch.equal(a_big, torch.cat([p[0] for p in parts])) and torch.equal(big, torch.cat([p[1] for p in parts])), \
        "the multi-wave launch differs from one-tile-per-CTA launches"
    bi, ni = roi_rows(sampled_tiles(work, grid), N)
    nb = idx32.cpu().long()[sel]
    a_ref = agg_rows(z, nb, bi, ni, Co, 0.2, True)
    assert torch.equal(a_big.cpu()[bi, ni].float(), a_ref), "aggregated tile must be bit-exact"
    ref = lrelu64(a_ref.double() @ w.double().t() + bias.double(), 0.01)
    got = big.cpu()[bi, ni].double()
    err = rel_max(got, ref)
    report(tag, work, grid, per, err)
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err


@pytest.mark.parametrize("K", [20, 40])
def test_edge_aggregate_staged_f32_many_tiles(ops, K):
    """float32 aggregation on the graph plan: two CTAs per SM while its shared memory is <= 110 KB (K = 20 here), one
    above (K = 40); bit-exact against the float64 max and against the unstaged gather kernel."""
    S = num_sms()
    N, B, Co = 4096, 48, 256
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N)).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    plan = ops.GraphPlan(idx32, p3d)
    assert plan.staged
    rows_cap = (plan.max_unique + 7) & ~7
    smem = cdiv(ops.PLAN_PAIRS * (2 * plan.KP + 8) * 2, 128) * 128 + 2 * rows_cap * 128
    work = B * plan.T
    grid = grid_of("2sm" if smem <= 110 * 1024 else "sm", work, S)
    tag = f"staged f32 aggregation K={K} (KP={plan.KP}, {smem // 1024} KB) N={N} B={B}"
    per = check_waves(tag, work, grid)
    g = torch.Generator().manual_seed(K + 1)
    z = torch.randn(B, N, 2 * Co, generator=g)
    zd = z.cuda()
    big = ops.edge_aggregate_staged(zd, plan, None, 0.2)
    parts = [ops.edge_aggregate_staged(zd[b0:b1], plan, None, 0.2) for b0, b1 in roi_chunks(B, plan.T, grid)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    assert torch.equal(big, ops.edge_aggregate(zd, plan.idx_p, None, 0.2)), "staged and unstaged aggregation differ"
    bi, ni = roi_rows(sampled_tiles(work, grid), N)
    nb = plan.idx_p.cpu().long().expand(B, -1, -1)
    assert torch.equal(big.cpu()[bi, ni], agg_rows(z, nb, bi, ni, Co, 0.2, False)), "aggregation must be bit-exact"
    report(tag, work, grid, per, 0.0)


def test_edgeconv_staged_many_tiles(ops):
    """cp_edgeconv_fwd at the benchmark's refine shape: N = 4096, K = 20, Co = 256 -> 512 bf16 with a_out."""
    S = num_sms()
    N, K, B, Co, nout = 4096, 20, 24, 256, 512
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 1, N)).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    plan = ops.GraphPlan(idx32, p3d)
    assert plan.staged
    tpr = plan.T
    tiles = B * tpr
    work, cap = tiles, S
    grid = grid_of("sm", work, S)
    tag = f"edgeconv N={N} K={K} B={B}"
    per = check_waves(tag, work, grid)
    g = torch.Generator().manual_seed(20)
    z = bf16r(torch.randn(B, N, 2 * Co, generator=g))
    w = bf16r(torch.randn(nout, Co, generator=g) / Co ** 0.5)
    bias = torch.randn(nout, generator=g)
    layer = ops.chain_layer(ops.pack_weight(w.cuda()), bias.cuda(), Co, nout, True, 0.01)
    zd = z.cuda().to(torch.bfloat16)

    def run(b0, b1):
        a_out = torch.empty((b1 - b0, N, Co), dtype=torch.bfloat16, device="cuda")
        out = torch.empty((b1 - b0, N, nout), dtype=torch.bfloat16, device="cuda")
        ops.edgeconv_fwd(z=zd[b0:b1], plan=plan, graph_sel=None, agg_slope=0.2, layer=layer, out=out, out_mode=ops.OUT_BF16, a_out=a_out)
        return a_out, out
    a_big, big = run(0, B)
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, cap)]
    assert torch.equal(a_big, torch.cat([p[0] for p in parts])) and torch.equal(big, torch.cat([p[1] for p in parts])), \
        "the multi-wave launch differs from one-tile-per-CTA launches"
    last = sampled_tiles(tiles, grid)
    bi, ni = roi_rows(last, N)
    nb = plan.idx_p.cpu().long().expand(B, -1, -1)
    a_ref = agg_rows(z, nb, bi, ni, Co, 0.2, True)
    assert torch.equal(a_big.cpu()[bi, ni].float(), a_ref), "aggregated tile must be bit-exact"
    ref = lrelu64(a_ref.double() @ w.double().t() + bias.double(), 0.01)
    got = big.cpu()[bi, ni].double()
    err = rel_max(got, ref)
    report(tag, work, grid, per, err)
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err


# ------------------------------------------------------------------------------------------------ the head at bench.py's sizes
HEAD_NAMES = ("roi_bit", "x_bits", "y_bits", "seg", "x_id", "y_id")


def _bench_case(config, N=None, K=None):
    import bench
    args = argparse.Namespace(config=config, npoint=0, graph_k=0, batch=0)
    wl = bench.workload(args, 1)
    case = bench.build_case(wl, torch.device("cuda", 0), 0, N=N, K=K)
    return bench, wl, case


def _run_head(wl, case, feats, bbox, obj_ids):
    net = case["net"]
    if wl["init_only"]:
        return (net(feats, obj_ids) if wl["lm"] else net(feats),)
    pexp = case["p3d"][obj_ids - 1] if wl["lm"] else case["p3d"].expand(feats[0].shape[0], -1, -1)
    out, packed = net.forward_with_correspondences(feats, pexp, bbox, obj_ids=obj_ids, packed=True)
    return tuple(out) + (packed,)


@pytest.mark.parametrize("config,dtype,N,K", [("full4096", torch.bfloat16, None, None),
                                              ("full4096", torch.float32, None, None),
                                              ("lm_sweep", torch.bfloat16, 4096, 20),
                                              ("lm_sweep", torch.bfloat16, 4096, 40),
                                              ("init64", torch.bfloat16, None, None)])
def test_head_at_bench_batch_is_batch_independent(ops, monkeypatch, config, dtype, N, K):
    """The benchmark's timed batch (bench.py: same nets, seeds, objects and max_batch_size) is bit-identical, output for
    output, to the same RoIs run in 2-RoI batches -- the regime test_gpu_head.py anchors to the oracle -- and a permuted
    batch returns the permuted outputs bit for bit."""
    from checkerpose_b200 import head
    S = num_sms()
    bench, wl, case = _bench_case(config, N, K)
    B, N = case["B"], case["N"]
    feats, bbox = bench.make_inputs(case, torch.device("cuda", 0), dtype, 0)
    obj = case["obj_ids"]
    names = ("init_bits",) if wl["init_only"] else HEAD_NAMES + ("records",)
    head.set_compute_dtype(dtype)
    head.set_image_branch("tcgen05")
    try:
        monkeypatch.setattr(ops, "chain_event_log", [])
        full = [t.clone() for t in _run_head(wl, case, feats, bbox, obj)]
        log = ops.chain_event_log
        monkeypatch.setattr(ops, "chain_event_log", None)
        if config == "lm_sweep" and K == 40:
            n_ec = sum(1 for sig, _, _ in log if sig[0] == "EC")
            n_agg = sum(1 for sig, _, _ in log if sig[0] == ops.PRO_AGG)
            assert n_ec == 0 and n_agg > 0, f"N=4096, K=40 must run the unstaged cp_chain_fwd(CP_PRO_AGG): EC {n_ec}, AGG {n_agg}"
        tiles = B * cdiv(N, TILE)
        print(f"[{config} {dtype} N={N} K={case['K']}] B={B}: node tiles per launch {tiles}, tiles per CTA "
              f"{cdiv(tiles, S)} (grid S = {S}) / {cdiv(tiles, 2 * S)} (grid 2S)")
        for b0 in range(0, B, 2):
            sl = slice(b0, b0 + 2)
            part = _run_head(wl, case, [f[sl].contiguous() for f in feats], bbox[sl].contiguous(), None if obj is None else obj[sl])
            for name, a, p in zip(names, full, part):
                assert torch.equal(a[sl], p), f"RoIs {b0}-{b0 + 1}: {name} differs between the {B}-RoI batch and a 2-RoI batch"
        perm = torch.randperm(B, generator=torch.Generator().manual_seed(B)).cuda()
        permuted = _run_head(wl, case, [f[perm].contiguous() for f in feats], bbox[perm].contiguous(), None if obj is None else obj[perm])
        for name, a, p in zip(names, full, permuted):
            assert torch.equal(a[perm], p), f"{name}: a permuted batch does not return the permuted outputs"
    finally:
        head.set_compute_dtype(torch.float32)
