"""The staged bf16 EdgeConv kernel (cp_edgeconv_fwd) at every padded neighbour-list length it is compiled for
(KP = 8 / 16 / 20 / 32 / 40), at the staging-ring loads the LM sweep reaches, and its fallbacks, against a float64
reference built from the keypoint-order kNN table (independent of the graph plan).

Bars (as test_gpu_kernels.py::test_edgeconv_staged): the aggregated tile a_out is bit-exact (bf16 max, one fp32 add,
LeakyReLU, one rounding to bf16), the bf16 GEMM output within 1e-2, fp32 logits within 1e-5."""
import numpy as np
import pytest
import torch

from helpers import BF16_MAX, BF16_RMS, BF16_STAGE_MAX, BF16_STAGE_RMS, syn

gpu = pytest.mark.gpu
torch.set_grad_enabled(False)

KPS = (8, 16, 20, 32, 40)
LM15 = tuple(range(1, 16))
AGG_SLOPE, OUT_SLOPE = 0.2, 0.01


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    return ops


def _bf16(t):
    return t.to(torch.bfloat16).float()


def _rows(perm_or_idx, sel, B):
    """(G, ...) per-graph table -> (B, ...) per RoI."""
    return perm_or_idx[sel] if sel is not None else perm_or_idx.expand(B, *perm_or_idx.shape[1:])


def reference(z_kp, idx, sel, w, bias, act):
    """float64 EdgeConv + layer in keypoint order: A = bf16(lrelu(max_k P[idx[i, k]] + Q[i])) with the kernel's
    arithmetic (exact bf16 max, one fp32 add, fp32 LeakyReLU), then act(A W^T + bias) in float64.
    z_kp (B,N,2Co) bf16-valued float32, idx (G,N,K) int64 keypoint numbering, sel (B,) int64 or None."""
    B, N, C2 = z_kp.shape
    Co = C2 // 2
    P, Q = z_kp[..., :Co], z_kp[..., Co:]
    nb = _rows(idx, sel, B)
    m = torch.full_like(Q, float("-inf"))
    for k in range(nb.shape[-1]):
        m = torch.maximum(m, torch.gather(P, 1, nb[:, :, k:k + 1].expand(-1, -1, Co)))
    a = _bf16(torch.nn.functional.leaky_relu(m + Q, AGG_SLOPE))
    y = a.double() @ w.double().t() + bias.double()
    return a, (torch.nn.functional.leaky_relu(y, OUT_SLOPE) if act else y)


def run_case(ops, plan, idx, sel, B, Co, nout, seed, tag, kernel="staged"):
    """One EdgeConv launch on the plan (z fed in plan order) checked against ``reference`` after mapping a_out and out
    back to keypoint order.  nout == 7: fp32 logits in a 16-wide buffer (n_valid = 7, no activation), else bf16 output
    with LeakyReLU.  kernel: "staged" = cp_edgeconv_fwd, "chain" = cp_chain_fwd(CP_PRO_AGG) on plan.idx_p.
    Returns the raw plan-order (a_out, out) for bit-for-bit comparisons between kernels."""
    N = plan.N
    f32 = nout == 7
    g = torch.Generator().manual_seed(seed)
    z_kp = _bf16(torch.randn(B, N, 2 * Co, generator=g))
    w = _bf16(torch.randn(nout, Co, generator=g) / Co ** 0.5)
    bias = torch.randn(nout, generator=g)
    sel_l = None if sel is None else torch.as_tensor(sel, dtype=torch.int64)
    a_ref, y_ref = reference(z_kp, idx.cpu().long(), sel_l, w, bias, act=not f32)
    pb = _rows(plan.perm.cpu().long(), sel_l, B)                                  # plan position -> keypoint id
    z_plan = torch.gather(z_kp, 1, pb[:, :, None].expand(-1, -1, 2 * Co))
    sel_d = None if sel_l is None else sel_l.to(torch.int32).cuda()
    layer = ops.chain_layer(ops.pack_weight(w.cuda()), bias.cuda(), Co, nout, not f32, OUT_SLOPE)
    a_out = torch.full((B, N, Co), float("nan"), dtype=torch.bfloat16, device="cuda")
    out = torch.full((B, N, 16 if f32 else nout), float("nan"), dtype=torch.float32 if f32 else torch.bfloat16, device="cuda")
    mode = ops.OUT_F32 if f32 else ops.OUT_BF16
    zd = z_plan.cuda().to(torch.bfloat16)
    if kernel == "staged":
        ops.edgeconv_fwd(z=zd, plan=plan, graph_sel=sel_d, agg_slope=AGG_SLOPE, layer=layer, out=out, out_mode=mode,
                         n_valid=nout if f32 else 0, a_out=a_out)
    else:
        ops.chain_fwd(prologue=ops.PRO_AGG, B=B, N=N, z=zd, idx32=plan.idx_p, graph_sel=sel_d, agg_slope=AGG_SLOPE,
                      a_out=a_out, layers=[layer], out=out, out_mode=mode, n_valid=nout if f32 else 0)
    torch.cuda.synchronize()

    def to_kp(t):
        r = torch.empty_like(t)
        return r.scatter_(1, pb[:, :, None].expand(-1, -1, t.shape[-1]), t)
    a_kp, out_kp = to_kp(a_out.cpu().float()), to_kp(out.cpu().float())
    assert torch.equal(a_kp, a_ref), f"{tag}: aggregated tile differs in {int((a_kp != a_ref).any(-1).sum())} rows"
    got = out_kp[..., :nout].double()
    if f32 and kernel == "staged":
        assert bool(torch.isnan(out_kp[..., nout:]).all()), f"{tag}: columns >= n_valid were written"
    assert bool(torch.isfinite(got).all()), f"{tag}: rows not written"
    tol = 1e-5 if f32 else 1e-2
    err = float((got - y_ref).abs().max())
    print(f"[{tag}] a_out bit-exact; out max |err| = {err:.3e} (max |ref| {float(y_ref.abs().max()):.2f})")
    assert torch.allclose(got, y_ref, rtol=tol, atol=tol), (tag, err)
    return a_out, out


def fps_graph(ops, ds, objs, N, K):
    """kNN tables (G,N,K) int32 of FPS fixture clouds, keypoint numbering, and their plan (with the renumbering)."""
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)) for o in objs], dim=0).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    return idx32, ops.GraphPlan(idx32, p3d)


def synthetic_graph(ops, G, N, K, U_of, seed):
    """(G,N,K) table in which tile t of graph g has exactly U_of(g, t, nv) distinct neighbour rows S_t (a random subset of
    the N rows): node j of the tile takes S_t[(j s + k) mod U], k < K, with the stride s chosen so that the union is
    S_t (s = 0: every node has the same K rows).  The plan keeps this numbering (no coordinates)."""
    gen = torch.Generator().manual_seed(seed)
    T = (N + ops.PLAN_TILE - 1) // ops.PLAN_TILE
    idx = torch.empty((G, N, K), dtype=torch.int32)
    want = torch.empty((G, T), dtype=torch.int32)
    for g in range(G):
        for t in range(T):
            n0, n1 = t * ops.PLAN_TILE, min(N, (t + 1) * ops.PLAN_TILE)
            nv = n1 - n0
            U = U_of(g, t, nv)
            s = 0 if U == K else -(-(U - K) // (nv - 1))
            assert K <= U <= N and s <= K, (g, t, U)
            S = torch.randperm(N, generator=gen)[:U]
            j = torch.arange(nv)[:, None] * s + torch.arange(K)[None, :]
            idx[g, n0:n1] = S[j % U].int()
            want[g, t] = U
    plan = ops.GraphPlan(idx.cuda(), None)
    assert plan.identity and torch.equal(plan.ucount.cpu(), want), "synthetic graph does not have the intended row counts"
    return idx, plan


def ring_stats(ucount, sel, B, KC, R, grid):
    """Replays the ring placement of the single-CTA kernel (tile i -> CTA i % grid, KC rounds of U rows per tile, a round
    that does not fit behind the head starts at row 0) -> (rounds that end exactly at row R, rounds that wrap)."""
    T = ucount.shape[1]
    U_tiles = [int(ucount[0 if sel is None else sel[b], t]) for b in range(B) for t in range(T)]
    exact = wraps = 0
    for c in range(grid):
        ph = 0
        for tile in range(c, len(U_tiles), grid):
            U = U_tiles[tile]
            for _ in range(KC):
                if ph + U > R:
                    ph, wraps = 0, wraps + 1
                exact += ph + U == R
                ph += U
    return exact, wraps


def _num_sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ------------------------------------------------------------------------------------------------ CPU: plan sizes vs ring
def test_ring_covers_plan_limit():
    """Every KP the staged kernel is compiled for has a staging ring of at least the plan's 512-row limit (so the
    kernel's host guard can only refuse a plan for exceeding that limit), other sizes have no ring, and K = 1..40 maps
    to the smallest compiled KP >= K."""
    from checkerpose_b200 import ops
    for KP in range(0, 65):
        R = int(ops.lib.cp_edgeconv_ring_rows(KP))
        if KP in KPS:
            assert R >= ops.PLAN_UMAX, (KP, R)
        else:
            assert R == -1, (KP, R)
    for K in range(1, ops.PLAN_MAX_K + 1):
        assert int(ops.lib.cp_graph_plan_kp(K)) == min(s for s in KPS if s >= K), K
    for K in (-1, 0, 41, 64):
        assert int(ops.lib.cp_graph_plan_kp(K)) == -1, K


# ------------------------------------------------------------------------------------------------ FPS clouds
FPS_CASES = [
    # ds, objects (graphs), N, K, Co, nout (7 = fp32 logits), B
    ("lm", (1,), 512, 8, 64, 128, 3),
    ("lm", (2, 3, 4), 1000, 16, 128, 256, 5),
    ("ycbv", (5,), 300, 20, 256, 512, 2),
    ("lmo", (1, 5, 6), 129, 40, 64, 7, 5),
    ("lm", LM15, 2048, 32, 256, 512, 3),       # the LM sweep's high ring loads: a tile with U > R/2 is selected
    ("lm", LM15, 2048, 40, 128, 256, 3),
    ("lm", LM15, 4096, 32, 64, 7, 3),
    # padded lists: K < KP
    ("ycbv", (2,), 300, 1, 64, 7, 2),
    ("ycbv", (3, 4, 5), 1000, 5, 128, 128, 5),
    ("lm", (6,), 512, 13, 64, 512, 2),
    ("ycbv", (7, 8, 9), 1000, 17, 256, 256, 5),
    ("lm", (10,), 2048, 27, 128, 7, 2),
    ("ycbv", (11, 12, 13), 1024, 37, 256, 128, 3),
]


@gpu
@pytest.mark.parametrize("ds,objs,N,K,Co,nout,B", FPS_CASES)
def test_edgeconv_fps_sweep(ops, ds, objs, N, K, Co, nout, B):
    idx, plan = fps_graph(ops, ds, objs, N, K)
    G = len(objs)
    assert plan.staged and plan.KP == min(s for s in KPS if s >= K)
    sel = None
    if G > 1:
        heavy = int(plan.ucount.cpu().max(1).values.argmax())          # the graph holding the most loaded tile ...
        others = [g for g in range(G) if g != heavy]
        sel = [heavy, others[0], heavy, others[-1], others[0]][:B]      # ... is selected (twice: graphs are revisited)
    if N >= 2048 and K >= 32:
        assert plan.max_unique > ops.lib.cp_edgeconv_ring_rows(plan.KP) // 2, plan.max_unique   # one round in flight
    run_case(ops, plan, idx, sel, B, Co, nout, seed=N + 7 * K + Co, tag=f"{ds} G={G} N={N} K={K} KP={plan.KP} Co={Co} nout={nout} "
             f"U<={plan.max_unique}/R={plan.ring_rows}")


# ------------------------------------------------------------------------------------------------ synthetic row counts
def _pattern(name, K, R):
    if name == "tiny":       # every node of a tile has the same K rows: rounds in flight are bounded by the barriers
        return lambda g, t, nv: K
    if name == "half":       # R // 2 (two rounds fit) and R // 2 + 1 (one round in flight); together they fill the ring exactly
        return lambda g, t, nv: (R // 2, R // 2 + 1)[(g + t) % 2]
    if name == "full":       # the plan limit: a full staging list without 0xFFFF entries
        return lambda g, t, nv: 512
    if name == "mixed":      # small and large tiles interleaved: the ring wraps at irregular positions
        choice = (K, R // 4, R // 2, R // 2 + 1, 512, R // 3)
        return lambda g, t, nv: choice[(7 * g + 3 * t + (t * t) // 3) % len(choice)]
    raise ValueError(name)


SYN_CASES = {   # pattern: N, G, B, Co, nout
    "tiny": (1000, 3, 5, 64, 512),
    "half": (1024, 2, 4, 256, 256),
    "full": (1024, 1, 2, 128, 128),
    "mixed": (1024, 3, 56, 64, 7),
}


@gpu
@pytest.mark.parametrize("pattern", list(SYN_CASES))
@pytest.mark.parametrize("KP", KPS)
def test_edgeconv_synthetic_ring_loads(ops, KP, pattern):
    N, G, B, Co, nout = SYN_CASES[pattern]
    K = KP
    R = int(ops.lib.cp_edgeconv_ring_rows(KP))
    idx, plan = synthetic_graph(ops, G, N, K, _pattern(pattern, K, R), seed=KP * 100 + len(pattern))
    assert plan.staged and plan.KP == KP
    if pattern == "full":
        assert plan.max_unique == ops.PLAN_UMAX and not bool((plan.ulist.cpu() == -1).any())
    g = torch.Generator().manual_seed(KP)
    sel = None if G == 1 else torch.randint(0, G, (B,), generator=g).tolist()
    exact, wraps = ring_stats(plan.ucount.cpu(), sel, B, Co // 64, R, min(B * plan.T, _num_sms()))
    if pattern in ("half", "mixed"):
        assert plan.max_unique > R // 2 and wraps > 0
    if pattern == "mixed":
        assert exact > 0, "no round ends exactly at the end of the ring"
    run_case(ops, plan, idx, sel, B, Co, nout, seed=KP + len(pattern),
             tag=f"{pattern} KP={KP} U<={plan.max_unique}/R={R} exact fits {exact}, wraps {wraps}")


@gpu
def test_edgeconv_fewer_nodes_than_neighbours(ops):
    """N = K = 40: one partial tile whose nodes all have every node as a neighbour."""
    N = K = 40
    idx, plan = synthetic_graph(ops, 1, N, K, lambda g, t, nv: N, seed=40)
    assert plan.staged and plan.max_unique == N
    for Co, nout in ((64, 7), (256, 512)):
        run_case(ops, plan, idx, None, 3, Co, nout, seed=Co, tag=f"N=K=40 Co={Co} nout={nout}")


@gpu
def test_plan_above_limit_is_refused_and_falls_back(ops):
    """A tile with 513 distinct rows: the plan is not staged, cp_edgeconv_fwd's host guard returns CP_E_UNSUPPORTED
    without launching, and cp_chain_fwd(CP_PRO_AGG) (what the head runs instead) matches the float64 reference."""
    idx, plan = synthetic_graph(ops, 2, 640, 8, lambda g, t, nv: 513 if (g, t) == (1, 2) else 64 + 40 * t, seed=513)
    assert plan.max_unique == ops.PLAN_UMAX + 1 and not plan.staged
    B, Co = 2, 64
    z = torch.zeros((B, 640, 2 * Co), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((128, Co), device="cuda")
    layer = ops.chain_layer(ops.pack_weight(w), None, Co, 128, False, 0.0)
    out = torch.full((B, 640, 128), float("nan"), dtype=torch.bfloat16, device="cuda")
    plan.staged = True                     # bypass the Python-side check: the C host guard must refuse the plan itself
    try:
        with pytest.raises(RuntimeError, match=r"failed \(-2\)"):      # CP_E_UNSUPPORTED
            ops.edgeconv_fwd(z=z, plan=plan, graph_sel=torch.tensor([1, 0], dtype=torch.int32, device="cuda"),
                             agg_slope=AGG_SLOPE, layer=layer, out=out, out_mode=ops.OUT_BF16)
    finally:
        plan.staged = False
    torch.cuda.synchronize()
    assert bool(torch.isnan(out.float()).all()), "nothing may have been launched"
    for Co, nout in ((64, 7), (256, 256)):
        run_case(ops, plan, idx, [1, 0, 1], 3, Co, nout, seed=Co, tag=f"U=513 chain fallback Co={Co} nout={nout}", kernel="chain")


# ------------------------------------------------------------------------------------------------ fallbacks
@gpu
@pytest.mark.parametrize("K", [40, 41, 64])
def test_chain_agg_fallback_large_k(ops, K):
    """cp_chain_fwd(CP_PRO_AGG), the head's path for graphs the staged kernel cannot take: K = 40 on a renumbered plan,
    K > 40 without a plan (identity numbering)."""
    idx, plan = fps_graph(ops, "lm", (3, 9, 14), 1000, K)
    assert plan.identity == (K > ops.PLAN_MAX_K) and (plan.KP == 40 if K == 40 else plan.KP < 0)
    for Co, nout in ((64, 7), (256, 512)):
        run_case(ops, plan, idx, [2, 0, 2, 1], 4, Co, nout, seed=K + Co, tag=f"chain K={K} Co={Co} nout={nout}", kernel="chain")


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_edge_aggregate_k64(ops, dtype):
    """cp_edge_aggregate (the SIMT gather kernel) at its largest K, per-RoI graphs, bit-exact in both dtypes."""
    N, K, Co, B = 700, 64, 96, 4
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", o, N)) for o in (4, 16, 20)], dim=0).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    g = torch.Generator().manual_seed(64)
    z = torch.randn(B, N, 2 * Co, generator=g).to(dtype).float()
    sel = torch.tensor([2, 0, 2, 1])
    nb = idx32.cpu().long()[sel]
    m = torch.full((B, N, Co), float("-inf"))
    for k in range(K):
        m = torch.maximum(m, torch.gather(z[..., :Co], 1, nb[:, :, k:k + 1].expand(-1, -1, Co)))
    ref = torch.nn.functional.leaky_relu(m + z[..., Co:], AGG_SLOPE).to(dtype)
    got = ops.edge_aggregate(z.to(dtype).cuda(), idx32, sel.int().cuda(), AGG_SLOPE)
    assert got.dtype == dtype and torch.equal(got.cpu(), ref)


# ------------------------------------------------------------------------------------------------ whole LM head in bf16
LM_SWEEP = [(512, 16), (1024, 40), (2048, 32), (2048, 40), (4096, 32)]


def _lm_net(N, K, B, seed):
    from checkerpose_b200.model import init_lm, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    g = torch.Generator().manual_seed(seed)
    p3d_all = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in LM15], dim=0)
    sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
    feats = syn.synthetic_features(B, g)
    dev = "cuda"
    inet = init_lm.InitNet_GNN(npoint=N, p3d_normed=p3d_all.to(dev), res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                               num_conv1x1=1, max_batch_size=64, num_graph_module=2, graph_k=K, graph_leaky_slope=0.2,
                               img_backbone=FeatureListBackbone())
    net = pipeline_lm.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d_all.to(dev), res_log2=6, num_filters=256, max_batch_size=64,
                                      query_dims=None, local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=K,
                                      graph_leaky_slope=0.2, query_type="mlp")
    net.load_state_dict(sd, strict=True)
    return net.to(dev).eval(), p3d_all, sd, feats


def _lm_run(net, p3d_all, feats, obj_ids):
    from checkerpose_b200 import head
    head.set_compute_dtype(torch.bfloat16)
    try:
        out = net([f.cuda() for f in feats], p3d_all.cuda()[obj_ids - 1], obj_ids.cuda())
        torch.cuda.synchronize()
    finally:
        head.set_compute_dtype(torch.float32)
    return [t.clone() for t in out]


def _unstaged_edgeconv(ops):
    """ops.edgeconv_fwd replaced by the unstaged kernel on the same plan: what the head runs for graphs that do not fit."""
    def fwd(*, z, plan, graph_sel, agg_slope, layer, out, out_mode, n_valid=0, a_out=None):
        return ops.chain_fwd(prologue=ops.PRO_AGG, B=z.shape[0], N=z.shape[1], z=z, idx32=plan.idx_p, graph_sel=graph_sel,
                             agg_slope=agg_slope, a_out=a_out, layers=[layer], out=out, out_mode=out_mode, n_valid=n_valid)
    return fwd


def _launched(ops, log):
    return sum(1 for sig, _, _ in log if sig[0] == "EC"), sum(1 for sig, _, _ in log if sig[0] == ops.PRO_AGG)


@gpu
@pytest.mark.parametrize("N,K", LM_SWEEP)
def test_lm_head_bf16_staged_equals_unstaged(ops, monkeypatch, N, K):
    """The LM net (15 graphs, per-RoI obj_ids) in bf16 at the sweep points: the six outputs of the head with the staged
    kernel are bit-identical to a run with every EdgeConv launch sent to cp_chain_fwd(CP_PRO_AGG) on the same plans."""
    from checkerpose_b200 import head
    B = 4
    net, p3d_all, _, feats = _lm_net(N, K, B, seed=2000 + N + K)
    obj_ids = torch.tensor([13, 2, 13, 9])
    plan = head.graph_ctx(net.refine_net[0].pre_query_block[0]._knn, obj_ids.cuda(), B, "cuda").plan
    assert plan.staged, plan.max_unique
    if N >= 2048 and K >= 32:
        assert plan.max_unique > plan.ring_rows // 2, plan.max_unique
    runs, counts = [], []
    for fallback in (False, False, True):
        if fallback:
            monkeypatch.setattr(ops, "edgeconv_fwd", _unstaged_edgeconv(ops))
        monkeypatch.setattr(ops, "chain_event_log", [])
        runs.append(_lm_run(net, p3d_all, feats, obj_ids))
        counts.append(_launched(ops, ops.chain_event_log))
    print(f"N={N} K={K} U<={plan.max_unique}/R={plan.ring_rows}: (EC, chain AGG) launches staged {counts[0]}, fallback {counts[2]}")
    assert counts[0][0] > 0 and counts[2][0] == 0 and counts[2][1] > counts[0][1]
    names = ("roi_bit", "x_bits", "y_bits", "seg", "x_id", "y_id")
    for name, a, b in zip(names, runs[0], runs[1]):
        assert torch.equal(a, b), f"two staged runs differ in {name}"
    for name, a, b in zip(names, runs[0], runs[2]):
        assert torch.equal(a, b), f"staged and unstaged EdgeConv differ in {name}"


@gpu
def test_lm_head_bf16_fallback_vs_oracle(ops, monkeypatch):
    """N = 4096, K = 40 (the benchmarked configuration whose plan exceeds 512 rows: the head runs cp_chain_fwd(CP_PRO_AGG)
    for every EdgeConv) against the fp32 CPU oracle with the budgets of test_full_size_head_bf16_vs_oracle: init logits
    and every teacher-forced refine stage, sign bits exact outside the relative margin."""
    from checkerpose_b200 import head
    from oracle import checkerpose_oracle as orc
    N, K, B = 4096, 40, 2
    net, p3d_all, sd, feats = _lm_net(N, K, B, seed=4096 + 40)
    obj_ids = torch.tensor([7, 13])
    plan = head.graph_ctx(net.refine_net[0].pre_query_block[0]._knn, obj_ids.cuda(), B, "cuda").plan
    assert not plan.staged and plan.max_unique > ops.PLAN_UMAX
    # the oracle runs on the net's own kNN tables: at K = 40 these clouds have rows whose 40th and 41st neighbours are
    # within 1e-6 in distance, where an independent kNN may pick the other one (kNN itself: test_gpu_kernels.py)
    idx_init = net.init_net.pre_query_block[0].knn_idx.cpu()
    idx_ref = [net.refine_net[s].pre_query_block[0].knn_idx.cpu() for s in range(3)]
    ref, inter = orc.pose_head(feats, sd, idx_init, idx_ref, N, obj_ids=obj_ids, return_intermediates=True)
    roi_r, xb_r, yb_r, _, xid_r, yid_r = ref
    monkeypatch.setattr(ops, "chain_event_log", [])
    roi, xb, yb, _, xid, yid = _lm_run(net, p3d_all, feats, obj_ids)
    n_ec, n_agg = _launched(ops, ops.chain_event_log)
    assert n_ec == 0 and n_agg > 0, (n_ec, n_agg)
    p3d_sel = p3d_all.cuda()[obj_ids - 1]
    head.set_compute_dtype(torch.bfloat16)
    try:
        staged = [net.refine_net[s](inter["img_feat"][s].cuda(), inter["graph_feat"][s].cuda(), p3d_sel, (roi_r > 0).float().cuda(),
                                    (xid_r >> (6 - 3 - s)).cuda(), (yid_r >> (6 - 3 - s)).cuda(), obj_ids.cuda()) for s in range(3)]
    finally:
        head.set_compute_dtype(torch.float32)
    scale0 = float(max(roi_r.abs().max(), xb_r[:, :3].abs().max(), yb_r[:, :3].abs().max()))
    for a, r in ((roi, roi_r), (xb[:, :3], xb_r[:, :3]), (yb[:, :3], yb_r[:, :3])):
        d = (a.cpu() - r).numpy()
        err_max, err_rms = np.abs(d).max() / float(r.abs().max()), np.sqrt((d ** 2).mean()) / float((r ** 2).mean().sqrt())
        print(f"[bf16 LM N=4096 K=40] init logits: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
        assert err_rms < BF16_RMS and err_max < BF16_MAX, (err_rms, err_max)
    safe0 = ((xb_r[:, :3].abs() > BF16_MAX * scale0).all(1) & (yb_r[:, :3].abs() > BF16_MAX * scale0).all(1)).numpy()
    same0 = ((xid.cpu() >> 3) == (xid_r >> 3)) & ((yid.cpu() >> 3) == (yid_r >> 3))
    assert same0.numpy()[safe0].all(), "init-stage cells must match wherever the oracle logit is outside the bf16 bar"
    for s, (new_bits, feat) in enumerate(staged):
        L = 3 + s
        ref_bits = torch.stack([xb_r[:, L], yb_r[:, L]], dim=1)
        for tag, a, r in (("bits", new_bits.cpu().float(), ref_bits), ("graph feature", feat.cpu().float(), inter["graph_feat"][s + 1])):
            d = (a - r).numpy()
            err_max, err_rms = np.abs(d).max() / float(r.abs().max()), np.sqrt((d ** 2).mean()) / float((r ** 2).mean().sqrt())
            print(f"[bf16 LM N=4096 K=40 stage {s}, teacher-forced] {tag}: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
            assert err_rms < BF16_STAGE_RMS and err_max < BF16_STAGE_MAX, (tag, err_rms, err_max)
        safe = ref_bits.abs() > BF16_STAGE_MAX * float(ref_bits.abs().max())
        flips = (new_bits.cpu() > 0) != (ref_bits > 0)
        assert not flips[safe].any(), f"stage {s}: bits must match outside the relative bf16 margin"
