"""The bf16 head at query_dims other than the shipped (256, 256, 64): widths that are multiples of 64 up to 512 on the
generic chain kernel (csrc/chain_tcgen05.cu: the wide instantiation for K or chained outputs above 256, column passes for a
[P|Q] table above the CTA's TMEM columns, any E % 16 == 0 in the taps prologue), other widths zero-padded on the host
(head.py, the width notes).  Kernel shapes against float64, whole heads against the CPU oracle and our float32 mode,
padding against an explicitly padded state_dict, batch independence, and the routing of the shipped dims."""
from collections import OrderedDict

import numpy as np
import pytest
import torch

from helpers import BF16_STAGE_MAX, BF16_STAGE_RMS, bf16r, rel_max, syn
from test_gpu_head import cascade_float_check
from test_gpu_many_tiles import TILE, cdiv, check_waves, grid_of, lm_graphs, lrelu64, num_sms, report, roi_chunks, roi_rows

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)

DIMS = [(64, 64, 64), (128, 128, 32), (96, 128, 48), (256, 512, 128), (512, 256, 64), (512, 512, 128), (256, 256, 64)]


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    return ops


def checked_tiles(work):
    """Tiles compared against float64: the first, one in the middle and the last 8 (in the ragged last wave)."""
    return sorted({0, work // 2} | set(range(work - 8, work)))


def _layers(ops, g, dims, nact):
    ws = [bf16r(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5) for o, i in dims]
    bs = [torch.randn(o, generator=g) * 0.1 for o, _ in dims]
    layers = [ops.chain_layer(ops.pack_weight(w.cuda()), b.cuda(), w.shape[1], w.shape[0], li < nact, 0.01)
              for li, (w, b) in enumerate(zip(ws, bs))]
    return ws, bs, layers


def _ref_chain(h, ws, bs, nact):
    h = h.double()
    for li, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.double().t() + b.double()
        if li < nact:
            h = lrelu64(h, 0.01)
            if li < len(ws) - 1:
                h = bf16r(h.float()).double()
    return h


# ------------------------------------------------------------------------------------------------ kernel level
@pytest.mark.parametrize("C,dims,rule", [
    (512, ((512, 512), (512, 512), (1024, 512)), "sm"),     # wide: K = 512, chained 512, [P|Q] 1024 in two column passes
    (192, ((320, 192), (384, 320)), "sm"),                   # wide (chained 320), widths not powers of two
    (192, ((192, 192), (384, 192)), "2sm"),                  # narrow, 384 columns in passes of 256 + 128
])
def test_chain_load_wide(ops, C, dims, rule):
    S = num_sms()
    N, B = 1000, 200
    tpr = cdiv(N, TILE)
    work = B * tpr
    grid = grid_of(rule, work, S)
    tag = f"chain LOAD C={C} {dims}"
    per = check_waves(tag, work, grid, N)
    g = torch.Generator().manual_seed(C + len(dims))
    x = bf16r(torch.randn(B, N, C, generator=g))
    nl = len(dims)
    ws, bs, layers = _layers(ops, g, dims, nl - 1)
    xd = x.cuda().to(torch.bfloat16)
    nout = dims[-1][0]

    def run(b0, b1):
        out = torch.full((b1 - b0, N, nout), float("nan"), dtype=torch.bfloat16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_LOAD, B=b1 - b0, N=N, src=xd[b0:b1], layers=layers, out=out, out_mode=ops.OUT_BF16)
        return out
    big = run(0, B)
    assert bool(torch.isfinite(big.float()).all()), "columns not written"
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, grid)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    bi, ni = roi_rows(checked_tiles(work), N)
    err = rel_max(big.cpu()[bi, ni].float(), _ref_chain(x[bi, ni], ws, bs, nl - 1))
    report(tag, work, grid, per, err)
    assert err < 2e-2, err


@pytest.mark.parametrize("Co,nout,rule", [(512, 1024, "sm"), (192, 384, "2sm")])
def test_chain_agg_wide(ops, Co, nout, rule):
    """AGG with C' = 512 (64 pieces of 16 bytes per row, wide kernel) and C' = 192: aggregation bit-exact, GEMM within 1e-2."""
    S = num_sms()
    N, B, K = 1000, 200, 20
    tpr = cdiv(N, TILE)
    work = B * tpr
    grid = grid_of(rule, work, S)
    tag = f"chain AGG Co={Co} nout={nout}"
    per = check_waves(tag, work, grid, N)
    _, idx32 = lm_graphs(ops, (3, 9, 14), N, K)
    g = torch.Generator().manual_seed(Co)
    z = bf16r(torch.randn(B, N, 2 * Co, generator=g))
    sel = torch.randint(0, 3, (B,), generator=g)
    ws, bs, layers = _layers(ops, g, ((nout, Co),), 1)
    zd, seld = z.cuda().to(torch.bfloat16), sel.to(torch.int32).cuda()

    def run(b0, b1):
        a_out = torch.empty((b1 - b0, N, Co), dtype=torch.bfloat16, device="cuda")
        out = torch.empty((b1 - b0, N, nout), dtype=torch.bfloat16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_AGG, B=b1 - b0, N=N, z=zd[b0:b1], idx32=idx32, graph_sel=seld[b0:b1], agg_slope=0.2,
                      a_out=a_out, layers=layers, out=out, out_mode=ops.OUT_BF16)
        return a_out, out
    a_big, big = run(0, B)
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, grid)]
    assert torch.equal(a_big, torch.cat([p[0] for p in parts])) and torch.equal(big, torch.cat([p[1] for p in parts]))
    bi, ni = roi_rows(checked_tiles(work), N)
    nb = idx32.cpu().long()[sel]
    from helpers import agg_rows
    a_ref = agg_rows(z, nb, bi, ni, Co, 0.2, True)
    assert torch.equal(a_big.cpu()[bi, ni].float(), a_ref), "aggregated tile must be bit-exact"
    ref = _ref_chain(a_ref, ws, bs, 1)
    err = rel_max(big.cpu()[bi, ni].double(), ref)
    report(tag, work, grid, per, err)
    assert torch.allclose(big.cpu()[bi, ni].double(), ref, rtol=1e-2, atol=1e-2), err


@pytest.mark.parametrize("E,Cg,d0,rule", [(128, 512, 512, "sm"),   # 4E = 512 and Cg = 512: both K phases fill the wide A tile
                                          (16, 64, 64, "2sm"),     # one 64-channel chunk of four taps
                                          (32, 192, 128, "2sm")])
def test_chain_taps_wide(ops, E, Cg, d0, rule):
    S = num_sms()
    N, B = 1000, 200
    tpr = cdiv(N, TILE)
    work = B * tpr
    grid = grid_of(rule, work, S)
    tag = f"chain TAPS E={E} Cg={Cg} d0={d0}"
    per = check_waves(tag, work, grid, N)
    g = torch.Generator().manual_seed(E + Cg)
    H, Hp = 64, 65
    patches = bf16r(torch.randn(B, Hp, Hp, E, generator=g))
    gf = bf16r(torch.randn(B, N, Cg, generator=g))
    x_id = torch.randint(0, H // 2, (B, N), generator=g)
    y_id = torch.randint(0, H // 2, (B, N), generator=g)
    mask = (torch.rand(B, N, generator=g) > 0.2).float()
    dims = ((d0, 4 * E + Cg), (d0, d0), (2 * d0, d0))
    ws, bs, layers = _layers(ops, g, dims, 2)
    dev = dict(patches=patches.cuda().to(torch.bfloat16), x_id=x_id.cuda(), y_id=y_id.cuda(), mask=mask.cuda(),
               graph_feat=gf.cuda().to(torch.bfloat16))

    def run(b0, b1):
        out = torch.full((b1 - b0, N, 2 * d0), float("nan"), dtype=torch.bfloat16, device="cuda")
        ops.chain_fwd(prologue=ops.PRO_TAPS, B=b1 - b0, N=N, tap_step=2, layers=layers, out=out, out_mode=ops.OUT_BF16,
                      **{k: v[b0:b1] for k, v in dev.items()})
        return out
    big = run(0, B)
    assert bool(torch.isfinite(big.float()).all()), "rows not written"
    parts = [run(b0, b1) for b0, b1 in roi_chunks(B, tpr, grid)]
    assert torch.equal(big, torch.cat(parts)), "the multi-wave launch differs from one-tile-per-CTA launches"
    bi, ni = roi_rows(checked_tiles(work), N)
    yy, xx = 2 * y_id[bi, ni], 2 * x_id[bi, ni]
    taps = torch.cat([patches[bi, yy + dy, xx + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1)
    h = torch.cat([taps * mask[bi, ni, None], gf[bi, ni]], dim=-1)
    err = rel_max(big.cpu()[bi, ni].float(), _ref_chain(h, ws, bs, 2))
    report(tag, work, grid, per, err)
    assert err < 2e-2, err


def test_chain_load_wide_past_2g_elements(ops):
    """One wide launch whose (B, N, 1024) [P|Q] output passes 2^31 elements (4.4 GB): row offsets are 64-bit."""
    N, B, C, nout = 4096, 520, 512, 1024
    assert B * N * nout > 2 ** 31
    g = torch.Generator().manual_seed(31)
    ws, bs, layers = _layers(ops, g, ((nout, C),), 0)
    x = torch.randn(B, N, C, device="cuda").to(torch.bfloat16)
    out = torch.empty((B, N, nout), dtype=torch.bfloat16, device="cuda")
    ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x, layers=layers, out=out, out_mode=ops.OUT_BF16)
    rows = torch.cat([torch.arange(0, 128), torch.arange(B * N - 256, B * N), torch.arange(2 ** 31 // nout - 64, 2 ** 31 // nout + 64)])
    got = out.view(-1, nout)[rows.cuda()].cpu().double()
    ref = _ref_chain(x.view(-1, C)[rows.cuda()].cpu().float(), ws, bs, 0)
    err = rel_max(got, ref)
    print(f"[chain LOAD 512->1024, {B * N * nout} output elements] float64 max err / max = {err:.2e}")
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err


# ------------------------------------------------------------------------------------------------ taps layer alone
def test_chain_taps_single_layer(ops):
    """TAPS with one layer that is also the last: its second K phase replaces the taps in the A tile, so it runs in one
    column pass (384 outputs: the wide kernel) and a layer too wide for one pass is refused."""
    N, B, E, Cg = 1000, 4, 64, 128
    g = torch.Generator().manual_seed(384)
    H, Hp = 64, 65
    patches = bf16r(torch.randn(B, Hp, Hp, E, generator=g))
    gf = bf16r(torch.randn(B, N, Cg, generator=g))
    x_id = torch.randint(0, H // 2, (B, N), generator=g)
    y_id = torch.randint(0, H // 2, (B, N), generator=g)
    dev = dict(patches=patches.cuda().to(torch.bfloat16), x_id=x_id.cuda(), y_id=y_id.cuda(), mask=None,
               graph_feat=gf.cuda().to(torch.bfloat16))
    ws, bs, layers = _layers(ops, g, ((384, 4 * E + Cg),), 0)
    out = torch.full((B, N, 384), float("nan"), dtype=torch.bfloat16, device="cuda")
    ops.chain_fwd(prologue=ops.PRO_TAPS, B=B, N=N, tap_step=2, layers=layers, out=out, out_mode=ops.OUT_BF16, **dev)
    bi, ni = roi_rows(range(cdiv(N, TILE) * B), N)
    yy, xx = 2 * y_id[bi, ni], 2 * x_id[bi, ni]
    taps = torch.cat([patches[bi, yy + dy, xx + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1)
    ref = _ref_chain(torch.cat([taps, gf[bi, ni]], dim=-1), ws, bs, 0)
    got = out.cpu()[bi, ni].double()
    err = rel_max(got, ref)
    print(f"[chain TAPS one layer 384] float64 max err / max = {err:.2e}")
    assert torch.allclose(got, ref, rtol=1e-2, atol=1e-2), err
    _, _, wide = _layers(ops, g, ((1024, 4 * E + Cg),), 0)
    out = torch.empty((B, N, 1024), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="one column pass"):
        ops.chain_fwd(prologue=ops.PRO_TAPS, B=B, N=N, tap_step=2, layers=wide, out=out, out_mode=ops.OUT_BF16, **dev)


# ------------------------------------------------------------------------------------------------ whole head
# Teacher-forced refine stages are held to the refine-stage budget of helpers.py at the size it was measured at (4096
# keypoints, 2 RoIs); the ABwoProg net to the budget of test_abwoprog_head_vs_reference_golden at that test's size (128
# keypoints, 3 RoIs); free-running bf16 ids to the floor test_head_bf16_vs_reference_golden holds (random-init logits crowd 0,
# and one flipped bit re-addresses the next stage's gather for a whole neighbourhood).
N_HEAD, B_HEAD = 4096, 2
N_ABWO, B_ABWO = 128, 3
# The max bound of the ABwoProg budget (22 chained bf16 layers) was set on the golden case's one draw of weights; at that size
# other draws exceed it for the shipped dims themselves (measured on B200: 6.5e-2 for 256_256_64) and reach 1.19e-1 at
# 96_128_48, so the max bound here is 1.5e-1.  The rms bound, 3e-2, is the golden test's and holds for every dims.
ABWO_RMS, ABWO_MAX = 3e-2, 1.5e-1
# num_filters = 128 (query_dims 128_256_64) is the one case whose new bits exceed the refine-stage rms bound: 2.8e-2 in stage 2
# (measured on B200; every query_dims case at num_filters = 256 stays within 0.5-1.8e-2).  Its bits get half as much again;
# its graph feature keeps the budget, and its sign bits outside the bar stay exact.
BITS_BUDGET = {("gnn", None, 128): (1.5 * BF16_STAGE_RMS, 1.5 * BF16_STAGE_MAX)}
FREE_RUNNING_MIN = 0.70
# batch independence, padding and routing need no oracle: a smaller head
N_SMALL = 512

_ORACLE = {}


def _net(kind, dims, p3d, sd, N, num_filters=256):
    from checkerpose_b200.model import init, init_lm, pipeline, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    I, P = (init_lm, pipeline_lm) if kind != "gnn" else (init, pipeline)
    p3d = p3d.cuda()
    inet = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                         num_conv1x1=1, max_batch_size=64, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                         img_backbone=FeatureListBackbone())
    cls = P.PoseNet_GNNskip_ABwoProg if kind == "abwoprog" else P.PoseNet_GNNskip
    net = cls(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=num_filters, max_batch_size=64, query_dims=dims, local_k=2,
              leaky_slope=0.01, num_graph_module=3, graph_k=20, graph_leaky_slope=0.2, query_type="mlp")
    net.load_state_dict(sd, strict=True)
    return net.cuda().eval()


def _inputs(dims, B=2, seed=0, N=N_SMALL):
    g = torch.Generator().manual_seed(4242 + seed + sum(dims))
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", 21, N))
    sd = syn.synthetic_state_dict(syn.head_param_spec(N, query_dims=dims), g)
    feats = syn.synthetic_features(B, g)
    return p3d, sd, feats


def _run(net, feats, p3d, dtype, obj_ids=None):
    from checkerpose_b200 import head
    head.set_compute_dtype(dtype)
    try:
        f = [t.cuda() for t in feats]
        if obj_ids is not None:
            return net(f, p3d.cuda()[obj_ids - 1], obj_ids.cuda())
        return net(f, p3d.cuda().expand(feats[0].shape[0], -1, -1))
    finally:
        head.set_compute_dtype(torch.float32)


def _oracle_case(kind, dims, num_filters):
    """Inputs of a PoseNet_GNNskip at N_HEAD keypoints ("gnn": one ycbv object; "lm": two lm objects selected per RoI by
    obj_ids) and the CPU oracle's outputs and intermediates, computed once per session."""
    from oracle import checkerpose_oracle as orc
    key = (kind, dims, num_filters)
    if key not in _ORACLE:
        g = torch.Generator().manual_seed(4242 + sum(dims or ()) + num_filters + (kind == "lm"))
        ds, objs = ("ycbv", (21,)) if kind == "gnn" else ("lm", (4, 11))
        p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N_HEAD)) for o in objs], dim=0)
        sd = syn.synthetic_state_dict(syn.head_param_spec(N_HEAD, num_filters=num_filters, query_dims=dims), g)
        feats = syn.synthetic_features(B_HEAD, g)
        obj_ids = None if kind == "gnn" else torch.tensor([2, 1])
        idx = orc.knn(p3d, 20)
        ref, inter = orc.pose_head(feats, sd, idx, [idx] * 3, N_HEAD, obj_ids=obj_ids, return_intermediates=True)
        _ORACLE[key] = (p3d, sd, feats, obj_ids, ref, inter)
    return _ORACLE[key]


HEAD_CASES_W = ([("gnn", d, 256) for d in DIMS] +
                [("gnn", None, 128),                 # num_filters = 128: image branch at 128 filters, query_dims (128, 256, 64)
                 ("lm", (96, 128, 48), 256), ("lm", (512, 512, 128), 256)])


@pytest.mark.parametrize("kind,dims,num_filters", HEAD_CASES_W)
def test_head_widths_vs_oracle(kind, dims, num_filters):
    """PoseNet_GNNskip (pipeline.py, or pipeline_lm.py with per-object graphs) at ``dims`` / ``num_filters``, N = 4096: the
    oracle follows the state_dict widths and our float32 mode matches it (1e-3); every refine stage in bf16, teacher-forced
    with the oracle's inputs, within the refine-stage budget of helpers.py, with its sign bits exact wherever the oracle logit
    is outside that budget; the free-running bf16 ids agree with our float32 mode's."""
    from checkerpose_b200 import head
    p3d, sd, feats, obj_ids, ref, inter = _oracle_case(kind, dims, num_filters)
    d0 = (dims or (num_filters,))[0]
    assert sd["refine_net.1.pre_query_block.0.conv.0.weight"].shape[:2] == (d0, 2 * d0)
    assert inter["graph_feat"][1].shape == (B_HEAD, d0, N_HEAD), "the oracle must follow the state_dict widths"
    assert inter["img_feat"][0].shape[1] == num_filters
    net = _net(kind, dims, p3d, sd, N_HEAD, num_filters)
    tag = f"{kind} {dims} nf={num_filters}"
    out32 = _run(net, feats, p3d, torch.float32, obj_ids)
    skipped = cascade_float_check(out32, ref, 1e-3, f"fp32 {tag}")
    print(f"[{tag}] fp32 vs oracle: (RoI, stage) pairs skipped after an in-band flip: {skipped}")
    roi, xb, yb, seg, xid, yid = ref
    p_sel = p3d.cuda()[obj_ids - 1] if obj_ids is not None else p3d.cuda().expand(B_HEAD, -1, -1)
    for s in range(3):
        L = 3 + s
        prev_x, prev_y = xid >> (6 - L), yid >> (6 - L)
        args = (inter["img_feat"][s].cuda(), inter["graph_feat"][s].cuda(), p_sel, (roi > 0).float().cuda(), prev_x.cuda(),
                prev_y.cuda()) + (() if obj_ids is None else (obj_ids.cuda(),))
        head.set_compute_dtype(torch.bfloat16)
        try:
            bits, feat = net.refine_net[s](*args)
        finally:
            head.set_compute_dtype(torch.float32)
        assert feat.shape == (B_HEAD, d0, N_HEAD), "the graph feature is handed back at its true width"
        ref_bits = torch.stack([xb[:, L], yb[:, L]], dim=1)
        for what, a, r in (("bits", bits.cpu(), ref_bits), ("graph feature", feat.cpu(), inter["graph_feat"][s + 1])):
            d = (a.float() - r).numpy()
            err_max = np.abs(d).max() / np.abs(r.numpy()).max()
            err_rms = np.sqrt((d ** 2).mean()) / np.sqrt((r.numpy() ** 2).mean())
            print(f"[{tag} bf16 stage {s}] {what}: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
            rms_bar, max_bar = (BITS_BUDGET.get((kind, dims, num_filters), (BF16_STAGE_RMS, BF16_STAGE_MAX)) if what == "bits"
                                else (BF16_STAGE_RMS, BF16_STAGE_MAX))
            assert err_rms < rms_bar and err_max < max_bar, (tag, s, what, err_rms, err_max)
        safe = ref_bits.abs() > BF16_STAGE_MAX * float(ref_bits.abs().max())
        assert safe.float().mean() > 0.3
        assert torch.equal((bits.cpu() > 0)[safe], (ref_bits > 0)[safe]), "bits must match outside the bf16 bar"
    out16 = _run(net, feats, p3d, torch.bfloat16, obj_ids)
    frac = float(((out16[4] == out32[4]) & (out16[5] == out32[5])).float().mean())
    print(f"[{tag}] free-running bf16 vs float32 mode: 64x64 cell agreement {frac:.4f}")
    assert frac > FREE_RUNNING_MIN, frac


@pytest.mark.parametrize("dims", DIMS)
def test_abwoprog_widths_vs_oracle(dims):
    """PoseNet_GNNskip_ABwoProg (per-object graphs selected by obj_ids) at ``dims``: float32 mode within 1e-3 of the oracle,
    bf16 logits within the chained-layer budget above (the rms bound of test_abwoprog_head_vs_reference_golden at its size)."""
    from oracle import checkerpose_oracle as orc
    objs = (1, 5, 9)
    N, B = N_ABWO, B_ABWO
    g = torch.Generator().manual_seed(77 + sum(dims))
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in objs], dim=0)
    sd = syn.synthetic_state_dict(syn.abwoprog_param_spec(N, query_dims=dims), g)
    feats = syn.synthetic_features(B, g)
    obj_ids = torch.tensor([1, 3, 2])
    idx = orc.knn(p3d, 20)
    ref = orc.pose_head_abwoprog(feats, sd, idx, [idx] * 3, N, obj_ids=obj_ids)
    net = _net("abwoprog", dims, p3d, sd, N)
    out32 = _run(net, feats, p3d, torch.float32, obj_ids)
    out16 = _run(net, feats, p3d, torch.bfloat16, obj_ids)
    for i, k in enumerate(("roi_bit", "x_bits", "y_bits")):
        r = ref[i].numpy()
        scale = np.abs(r).max()
        e32 = np.abs(out32[i].cpu().numpy() - r).max() / scale
        d = out16[i].cpu().numpy() - r
        print(f"[ABwoProg {dims}] {k}: fp32 max err {e32:.2e}, bf16 max err {np.abs(d).max() / scale:.4f} "
              f"rms {np.sqrt((d ** 2).mean()) / scale:.4f}")
        assert e32 < 1e-3, (k, e32)
        assert np.sqrt((d ** 2).mean()) < ABWO_RMS * scale and np.abs(d).max() < ABWO_MAX * scale, (k, np.abs(d).max() / scale)


def _padded_state_dict(sd, dims, dims_p):
    """The state_dict of a head at ``dims`` written out by hand, with explicit zeros, as one at ``dims_p``: weight rows /
    columns, biases and patch-generator outputs zero (the pre-graph layer's columns laid out per tap), BatchNorm of a padded
    channel gamma = beta = mean = 0, var = 1."""
    (d0, d1, d2), (p0, p1, p2) = dims, dims_p
    E, Ep = d0 // 4, p0 // 4
    out = OrderedDict()

    def embed(v, shape, *idx):
        t = torch.zeros(shape, dtype=v.dtype)
        t[idx] = v
        return t
    for k, v in sd.items():
        if not k.startswith("refine_net."):
            out[k] = v
            continue
        s, name = int(k.split(".")[1]), k.split(".", 2)[2]
        gd, gp = (64, 64) if s == 0 else (d0, p0)
        if name.startswith("local_feat_ext_block.patch_generator."):
            v = embed(v, (Ep,) + v.shape[1:], slice(0, E))
        elif name == "pre_graph_module.0.weight":          # [tap0 | tap1 | tap2 | tap3 | graph feature]
            t = torch.zeros(p0, 4 * Ep + gp)
            for tap in range(4):
                t[:d0, tap * Ep:tap * Ep + E] = v[:, tap * E:(tap + 1) * E]
            t[:d0, 4 * Ep:4 * Ep + gd] = v[:, 4 * E:]
            v = t
        elif name == "pre_graph_module.2.weight":
            v = embed(v, (p0, p0), slice(0, d0), slice(0, d0))
        elif name.startswith("pre_graph_module."):
            v = embed(v, (p0,), slice(0, d0))
        elif name.endswith("conv.0.weight"):               # EdgeConv input [x_j - x_i | x_i]
            t = torch.zeros(p0, 2 * p0, 1, 1)
            t[:d0, :d0] = v[:, :d0]
            t[:d0, p0:p0 + d0] = v[:, d0:]
            v = t
        elif ".conv.1." in name and not name.endswith("num_batches_tracked"):
            t = torch.full((p0,), 1.0 if name.endswith("running_var") else 0.0)
            t[:d0] = v
            v = t
        elif name.startswith("query_block.mlps."):
            j = int(name.split(".")[2]) // 2
            (r, rp), (c, cp) = [((d1, p1), (d0, p0)), ((d2, p2), (d1, p1)), ((2, 2), (d2, p2))][j]
            v = embed(v, (rp, cp), slice(0, r), slice(0, c)) if name.endswith("weight") else embed(v, (rp,), slice(0, r))
        out[k] = v
    return out


def test_padding_is_exact():
    """A head at (96, 128, 48) (patch embedding 24) runs bit for bit as the same head written out at (128, 128, 64)."""
    dims, dims_p = (96, 128, 48), (128, 128, 64)
    p3d, sd, feats = _inputs(dims)
    sdp = _padded_state_dict(sd, dims, dims_p)
    a = _run(_net("gnn", dims, p3d, sd, N_SMALL), feats, p3d, torch.bfloat16)
    b = _run(_net("gnn", dims_p, p3d, sdp, N_SMALL), feats, p3d, torch.bfloat16)
    for i, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x, y), f"output {i} differs between implicit and explicit padding"


@pytest.mark.parametrize("dims", [(96, 128, 48), (512, 512, 128)])
def test_widths_batch_independent(dims):
    """bf16 head at ``dims``: a RoI's outputs do not depend on the batch it runs in (2-RoI batches, a permuted batch)."""
    p3d, sd, feats = _inputs(dims, B=4, seed=1)
    net = _net("gnn", dims, p3d, sd, N_SMALL)
    full = _run(net, feats, p3d, torch.bfloat16)
    halves = [_run(net, [f[b0:b0 + 2] for f in feats], p3d, torch.bfloat16) for b0 in (0, 2)]
    perm = torch.tensor([3, 1, 0, 2])
    permuted = _run(net, [f[perm] for f in feats], p3d, torch.bfloat16)
    for i in range(6):
        assert torch.equal(full[i], torch.cat([h[i] for h in halves])), f"output {i}: 2-RoI batches differ"
        assert torch.equal(full[i][perm.cuda()], permuted[i]), f"output {i}: the permuted batch differs"


@pytest.mark.parametrize("dims", [(256, 256, 64), (512, 512, 128), (96, 128, 48)])
def test_width_routing(ops, monkeypatch, dims):
    """The shipped dims launch the staged EdgeConv ("EC") and the fused query tail ("QT"); other dims the generic chain
    kernel (AGG where the staged kernel does not take C').  The log records a TAPS launch by its signature only: cp_chain_fwd
    hands it to K3 inside the library when taps_chain_try accepts the shape, so for the shipped dims the test asserts the
    signatures K3 takes (E = 64, Cg in {64, 128, 256}, 256 -> 256 -> 512 bf16, no a_out)."""
    p3d, sd, feats = _inputs(dims)
    net = _net("gnn", dims, p3d, sd, N_SMALL)
    monkeypatch.setattr(ops, "chain_event_log", [])
    _run(net, feats, p3d, torch.bfloat16)
    sigs = [s for s, _, _ in ops.chain_event_log]
    taps = [s for s in sigs if s[0] == ops.PRO_TAPS]
    assert len(taps) == 3
    if dims == (256, 256, 64):
        assert any(s[0] == "EC" for s in sigs) and any(s[0] == "QT" for s in sigs)
        assert taps[0][1:3] == (256 + 64, (256, 256, 512)) and taps[1][1:3] == (256 + 256, (256, 256, 512))
        assert not any(s[0] == ops.PRO_AGG for s in sigs)
    elif dims == (512, 512, 128):
        assert taps[1][1:3] == (512 + 512, (512, 512, 1024))
        assert any(s[0] == ops.PRO_AGG and s[1] == 512 for s in sigs)
    else:
        assert taps[1][1:3] == (128 + 128, (128, 128, 256))


def test_width_limits_raise():
    """Widths the bf16 kernels do not run, even padded, raise a RuntimeError that names the width and points at float32
    mode."""
    p3d, _, feats = _inputs((256, 256, 64))
    for dims, what in (((640, 256, 64), "640"), ((256, 1024, 64), "1024"), ((98, 128, 64), "divisible by 4")):
        g = torch.Generator().manual_seed(5)
        sd = syn.synthetic_state_dict(syn.head_param_spec(N_SMALL, query_dims=dims), g)
        net = _net("gnn", dims, p3d, sd, N_SMALL)
        with pytest.raises(RuntimeError, match=what) as ei:
            _run(net, feats, p3d, torch.bfloat16)
        assert "float32" in str(ei.value)
