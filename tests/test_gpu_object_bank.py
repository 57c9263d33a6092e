"""Object-indexed weights and ObjectBank on the GPU, bit for bit.

Kernels: a launch over RoIs of several objects with stacked weights (w_stride / b_stride, selected by graph_sel) equals the
same kernel launched per object on that object's RoIs with its own weights; strides 0 equal today's call.  Whole head: an
ObjectBank forward equals every object's own net run alone on its RoIs, in bf16 and in float32."""
import pytest
import torch

from helpers import syn

pytestmark = pytest.mark.gpu

N_RAGGED = 1000
B_WAVES = 190            # 190 RoIs x 8 tiles = 1520 tiles: >= 5 tiles per CTA of every persistent kernel (2 x 148 CTAs at most)


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops as o
    return o


def _sels(G, B, seed):
    """Per-RoI object patterns: runs (object G-1 absent), strict alternation, one object only."""
    g = torch.Generator().manual_seed(seed)
    runs = torch.sort(torch.randint(0, G - 1, (B,), generator=g))[0]
    alt = torch.arange(B) % G
    one = torch.full((B,), 1 if G > 1 else 0)
    return {"runs": runs, "alternate": alt, "single": one}


def _weights(ops, G, specs, seed):
    """specs: (kin, nout) per layer -> per layer (packed (G, bytes), bias (G, nout))."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for kin, nout in specs:
        ws = [torch.randn(nout, kin, generator=g) * (2.0 / kin) ** 0.5 for _ in range(G)]
        packed = torch.stack([ops.pack_weight(w.cuda()) for w in ws])
        out.append((packed, (torch.randn(G, nout, generator=g) * 0.1).cuda()))
    return out


def _layers(ops, W, specs, acts, obj=None):
    """Chain layers: stacked (obj None) or object obj's own copies of the weights."""
    res = []
    for (packed, bias), (kin, nout), (act, slope) in zip(W, specs, acts):
        if obj is None:
            res.append(ops.chain_layer(packed, bias, kin, nout, act, slope, packed.stride(0), bias.stride(0)))
        else:
            res.append(ops.chain_layer(packed[obj].clone(), bias[obj].clone(), kin, nout, act, slope))
    return res


def _per_object(sel, run_one):
    """run_one(obj, rows (long)) for every object present."""
    for o in torch.unique(sel).tolist():
        run_one(o, torch.nonzero(sel == o).flatten().cuda())


@pytest.fixture(scope="module")
def graphs(ops):
    out = {}
    for G in (3, 21):
        p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", o, N_RAGGED)) for o in range(1, G + 1)]).cuda()
        idx32 = ops.knn(p3d, 20, want_i32=True)[1]
        out[G] = ops.GraphPlan(idx32, p3d)
    return out


def _bf16(shape, g):
    return torch.randn(*shape, generator=g).to(torch.bfloat16).cuda()


@pytest.mark.parametrize("G", [3, 21])
@pytest.mark.parametrize("Co, nout, mode", [(64, 128, "bf16"), (128, 256, "a_out"), (256, 512, "bf16"), (128, 16, "f32")])
def test_edgeconv_object_weights(ops, graphs, G, Co, nout, mode):
    plan = graphs[G]
    assert plan.staged
    g = torch.Generator().manual_seed(G * 1000 + Co + nout)
    B, N = B_WAVES, N_RAGGED
    z = _bf16((B, N, 2 * Co), g)
    specs = [(Co, nout)]
    W = _weights(ops, G, specs, 7 + Co)
    f32 = mode == "f32"
    act = (not f32, 0.01)
    for name, sel_cpu in _sels(G, B, Co).items():
        sel = sel_cpu.to(torch.int32).cuda()
        mk = (lambda b: torch.zeros((b, N, 16), dtype=torch.float32, device="cuda")) if f32 else \
             (lambda b: torch.zeros((b, N, nout), dtype=torch.bfloat16, device="cuda"))
        out, a_out = mk(B), (torch.zeros((B, N, Co), dtype=torch.bfloat16, device="cuda") if mode == "a_out" else None)
        kw = dict(agg_slope=0.2, out_mode=ops.OUT_F32 if f32 else ops.OUT_BF16, n_valid=nout if f32 else 0)
        ops.edgeconv_fwd(z=z, plan=plan, graph_sel=sel, layer=_layers(ops, W, specs, [act])[0], out=out, a_out=a_out, **kw)

        def one(o, rows):
            ref = mk(len(rows))
            ra = torch.zeros((len(rows), N, Co), dtype=torch.bfloat16, device="cuda") if a_out is not None else None
            ops.edgeconv_fwd(z=z[rows].contiguous(), plan=plan, graph_sel=sel[rows].contiguous(),
                             layer=_layers(ops, W, specs, [act], o)[0], out=ref, a_out=ra, **kw)
            assert torch.equal(out[rows], ref), f"{name}: object {o}"
            if ra is not None:
                assert torch.equal(a_out[rows], ra), f"{name}: a_out of object {o}"
        _per_object(sel_cpu, one)


CHAIN_CASES = {
    # prologue, (C | Co | (E, Cg)), layer specs, activations, output
    "load_narrow": ("load", 128, [(128, 256), (256, 128)], [(True, 0.01), (False, 0.0)], "f32"),
    "load_wide": ("load", 512, [(512, 512), (512, 1024)], [(True, 0.01), (False, 0.0)], "bf16"),
    "agg_narrow": ("agg", 128, [(128, 256)], [(False, 0.0)], "bf16"),
    "agg_wide": ("agg", 512, [(512, 512)], [(True, 0.01)], "bf16"),
    "taps_narrow": ("taps", (32, 64), [(192, 128), (128, 128)], [(True, 0.01), (True, 0.01)], "bf16"),
    "taps_wide": ("taps", (128, 64), [(576, 256), (256, 512)], [(True, 0.01), (False, 0.0)], "bf16"),
    "k3_cg64": ("taps", (64, 64), [(320, 256), (256, 256), (256, 512)], [(True, 0.01), (True, 0.01), (False, 0.0)], "bf16"),
    "k3_cg256": ("taps", (64, 256), [(512, 256), (256, 256), (256, 256)], [(True, 0.01), (True, 0.01), (False, 0.0)], "bf16"),
}


def _chain_inputs(ops, kind, width, B, N, g, plan):
    if kind == "load":
        return dict(prologue=ops.PRO_LOAD, src=_bf16((B, N, width), g))
    if kind == "agg":
        return dict(prologue=ops.PRO_AGG, z=_bf16((B, N, 2 * width), g), idx32=plan.idx_p, agg_slope=0.2)
    E, Cg = width
    Hp = 33
    return dict(prologue=ops.PRO_TAPS, patches=_bf16((B, Hp, Hp, E), g), tap_step=2,
                x_id=torch.randint(0, 15, (B, N), generator=g).cuda(), y_id=torch.randint(0, 15, (B, N), generator=g).cuda(),
                mask=(torch.rand(B, N, generator=g) > 0.2).float().cuda(), graph_feat=_bf16((B, N, Cg), g))


def _rows_of(kw, rows):
    out = {}
    for k, v in kw.items():
        out[k] = v[rows].contiguous() if isinstance(v, torch.Tensor) and k != "idx32" else v
    return out


@pytest.mark.parametrize("G", [3, 21])
@pytest.mark.parametrize("case", list(CHAIN_CASES))
def test_chain_object_weights(ops, graphs, G, case):
    kind, width, specs, acts, omode = CHAIN_CASES[case]
    plan = graphs[G]
    g = torch.Generator().manual_seed(G * 77 + len(case))
    B, N = B_WAVES, N_RAGGED
    inp = _chain_inputs(ops, kind, width, B, N, g, plan)
    W = _weights(ops, G, specs, 11 + G)
    nout = specs[-1][1]
    f32 = omode == "f32"
    mk = (lambda b: torch.zeros((b, N, nout), dtype=torch.float32 if f32 else torch.bfloat16, device="cuda"))
    kw = dict(out_mode=ops.OUT_F32 if f32 else ops.OUT_BF16, n_valid=nout - 3 if f32 else 0)
    for name, sel_cpu in _sels(G, B, G).items():
        sel = sel_cpu.to(torch.int32).cuda()
        out = mk(B)
        ops.chain_fwd(B=B, N=N, layers=_layers(ops, W, specs, acts), out=out, graph_sel=sel, **inp, **kw)

        def one(o, rows):
            ref = mk(len(rows))
            ops.chain_fwd(B=len(rows), N=N, layers=_layers(ops, W, specs, acts, o), out=ref, graph_sel=sel[rows].contiguous(),
                          **_rows_of(inp, rows), **kw)
            assert torch.equal(out[rows], ref), f"{case} {name}: object {o}"
        _per_object(sel_cpu, one)
    # strides 0 with a selector given: today's call (selector unused by LOAD / TAPS, the graph of AGG)
    if G == 3:
        sel = _sels(G, B, 0)["alternate"].to(torch.int32).cuda()
        a, b = mk(B), mk(B)
        lay = lambda: _layers(ops, W, specs, acts, 0)   # noqa: E731
        ops.chain_fwd(B=B, N=N, layers=lay(), out=a, graph_sel=sel, **inp, **kw)
        ops.chain_fwd(B=B, N=N, layers=lay(), out=b, graph_sel=sel if kind == "agg" else None, **inp, **kw)
        assert torch.equal(a, b)


@pytest.mark.parametrize("G", [3, 21])
@pytest.mark.parametrize("kin", [256, 128])
def test_query_decode_object_weights(ops, graphs, G, kin):
    plan = graphs[G]
    g = torch.Generator().manual_seed(G + kin)
    B, N, Ltot, plane = B_WAVES, N_RAGGED, 6, 4
    src = _bf16((B, N, kin), g)
    w1 = torch.stack([ops.pack_weight((torch.randn(64, kin, generator=g) * 0.1).cuda()) for _ in range(G)])
    b1 = (torch.randn(G, 64, generator=g) * 0.1).cuda()
    w2 = (torch.randn(G, 2, 64, generator=g) * 0.3).cuda()
    b2 = (torch.randn(G, 2, generator=g) * 0.1).cuda()
    xb0 = torch.randn(B, Ltot, N, generator=g).cuda()
    yb0 = torch.randn(B, Ltot, N, generator=g).cuda()
    xi0 = torch.randint(0, 16, (B, N), generator=g).cuda()
    yi0 = torch.randint(0, 16, (B, N), generator=g).cuda()
    for name, sel_cpu in _sels(G, B, kin).items():
        sel = sel_cpu.to(torch.int32).cuda()
        st = [xb0.clone(), yb0.clone(), xi0.clone(), yi0.clone(), torch.zeros_like(xi0), torch.zeros_like(yi0),
              torch.zeros((B, N, 2), device="cuda")]
        ops.query_decode_fwd(src=src, w1_packed=w1, b1=b1, slope=0.01, w2=w2, b2=b2, plane=plane, Ltot=Ltot, x_bits=st[0], y_bits=st[1],
                             x_id=st[2], y_id=st[3], perm=plan.perm, graph_sel=sel, x_id_kp=st[4], y_id_kp=st[5], logits=st[6],
                             w_stride=(w1.stride(0), w2.stride(0)), b_stride=(b1.stride(0), b2.stride(0)))

        def one(o, rows):
            n = len(rows)
            r = [xb0[rows].clone(), yb0[rows].clone(), xi0[rows].clone(), yi0[rows].clone(), torch.zeros((n, N), dtype=torch.int64, device="cuda"),
                 torch.zeros((n, N), dtype=torch.int64, device="cuda"), torch.zeros((n, N, 2), device="cuda")]
            ops.query_decode_fwd(src=src[rows].contiguous(), w1_packed=w1[o].clone(), b1=b1[o].clone(), slope=0.01, w2=w2[o].clone(),
                                 b2=b2[o].clone(), plane=plane, Ltot=Ltot, x_bits=r[0], y_bits=r[1], x_id=r[2], y_id=r[3], perm=plan.perm,
                                 graph_sel=sel[rows].contiguous(), x_id_kp=r[4], y_id_kp=r[5], logits=r[6])
            for k in range(7):
                assert torch.equal(st[k][rows], r[k]), f"{name}: object {o}, output {k}"
        _per_object(sel_cpu, one)


# ------------------------------------------------------------------------------------------------ whole head
LMO_IDS = (1, 5, 6, 8, 9, 10, 11, 12)


def _build_nets(ds, ids, N, seed):
    from checkerpose_b200.model import init, pipeline
    from checkerpose_b200.model.backbone import FeatureListBackbone
    nets = {}
    for k, o in enumerate(ids):
        p3d = syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)).cuda()
        inet = init.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                                num_conv1x1=1, max_batch_size=8, num_graph_module=2, graph_k=20, img_backbone=FeatureListBackbone())
        net = pipeline.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=256, max_batch_size=8, local_k=2,
                                       leaky_slope=0.01, num_graph_module=3, graph_k=20)
        net.load_state_dict(syn.synthetic_state_dict(syn.head_param_spec(N), torch.Generator().manual_seed(seed + 31 * k)), strict=True)
        nets[o] = net.cuda().eval()
    return nets


@pytest.fixture(scope="module")
def lmo_nets():
    return _build_nets("lmo", LMO_IDS, 512, 100)


@pytest.fixture(scope="module")
def ycbv_nets():
    return _build_nets("ycbv", tuple(range(1, 22)), 4096, 200)


def _inputs(B, seed, feat_dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    feats = [f.to(feat_dtype).cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    return feats, bbox


def _reference(nets, ids, feats, bbox, packed):
    """Every object's own net on its RoIs -> outputs scattered back to the batch order."""
    B = len(ids)
    out, corr = None, None
    for o in sorted(set(ids.tolist())):
        rows = torch.nonzero(ids == o).flatten().cuda()
        res, c = nets[o].forward_with_correspondences([f[rows] for f in feats], None, bbox[rows], packed=packed)
        if out is None:
            out = [torch.empty((B,) + t.shape[1:], dtype=t.dtype, device="cuda") for t in res]
            corr = torch.empty((B,) + c.shape[1:], dtype=c.dtype, device="cuda")
        for t, r in zip(out, res):
            t[rows] = r
        corr[rows] = c
    return out, corr


def _check_bank(nets, ids, feats, bbox):
    from checkerpose_b200.model.object_bank import ObjectBank
    bank = ObjectBank(nets)
    for packed in (False, True):
        got, gc = bank.forward_with_correspondences(feats, bbox, ids, packed=packed)
        ref, rc = _reference(nets, ids, feats, bbox, packed)
        for k, (a, b) in enumerate(zip(got, ref)):
            assert torch.equal(a, b), f"output {k} (packed={packed})"
        assert torch.equal(gc, rc), f"records (packed={packed})"
    return bank, got


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_lmo_bank_equals_each_net(lmo_nets, dtype):
    from checkerpose_b200 import head
    from checkerpose_b200.model.object_bank import ObjectBank
    B = 24
    ids = torch.tensor([LMO_IDS[i] for i in torch.randperm(B, generator=torch.Generator().manual_seed(3)) % len(LMO_IDS)])
    ids[5:9] = 9                                    # a run inside the shuffle
    feats, bbox = _inputs(B, 41)
    head.set_compute_dtype(dtype)
    try:
        bank, got = _check_bank(lmo_nets, ids, feats, bbox)
        # a permuted batch returns permuted outputs
        p = torch.randperm(B, generator=torch.Generator().manual_seed(4))
        pg = bank([f[p.cuda()] for f in feats], ids[p])
        for a, b in zip(pg, got):
            assert torch.equal(a, b[p.cuda()])
        # poses: PnP of every RoI as in its own net's batch
        cam = torch.tensor([[572.4, 0.0, 325.3], [0.0, 573.6, 242.0], [0.0, 0.0, 1.0]]).cuda()
        p3d = torch.stack([torch.from_numpy(syn.load_fps_xyz("lmo", o, 512)).float() for o in LMO_IDS]).cuda()
        _, pk, R, t, ninl = bank.forward_with_pose(feats, bbox, p3d, cam, ids)
        for k, o in enumerate(LMO_IDS):
            rows = torch.nonzero(ids == o).flatten().cuda()
            if len(rows) == 0:
                continue
            _, pk_o, R_o, t_o, n_o = lmo_nets[o].forward_with_pose([f[rows] for f in feats], None, bbox[rows], p3d[k:k + 1], cam)
            assert torch.equal(pk[rows], pk_o) and torch.equal(R[rows], R_o) and torch.equal(t[rows], t_o) and torch.equal(ninl[rows], n_o)
        # a one-object bank is the net itself
        one = ObjectBank({5: lmo_nets[5]})
        sub = [f[:3] for f in feats]
        a = one(sub, torch.tensor([5, 5, 5]))
        b = lmo_nets[5](sub, None)
        for x, y in zip(a, b):
            assert torch.equal(x, y)
    finally:
        head.set_compute_dtype(torch.float32)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_ycbv_bank_equals_each_net(ycbv_nets, dtype):
    from checkerpose_b200 import head
    B = 42
    ids = (torch.randperm(B, generator=torch.Generator().manual_seed(5)) % 21) + 1
    feats, bbox = _inputs(B, 43)
    head.set_compute_dtype(dtype)
    try:
        _check_bank(ycbv_nets, ids, feats, bbox)
    finally:
        head.set_compute_dtype(torch.float32)


def test_ycbv_bank_1024_rois(ycbv_nets):
    from checkerpose_b200 import head
    from checkerpose_b200.model.object_bank import ObjectBank
    B = 1024
    ids = (torch.randperm(B, generator=torch.Generator().manual_seed(6)) % 21) + 1
    feats, bbox = _inputs(B, 44, torch.bfloat16)
    head.set_compute_dtype(torch.bfloat16)
    try:
        bank = ObjectBank(ycbv_nets)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        before = torch.cuda.memory_allocated()       # the caller's inputs and the nets' (prepared) weights
        got, gc = bank.forward_with_correspondences(feats, bbox, ids, packed=True)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - before
        print(f"ObjectBank, 1024 YCB-V RoIs at N = 4096: {peak / 2 ** 30:.1f} GiB allocated by the forward at its peak "
              f"(on top of {before / 2 ** 30:.1f} GiB of inputs and weights)")
        ref, rc = _reference(ycbv_nets, ids, feats, bbox, True)
        for k, (a, b) in enumerate(zip(got, ref)):
            assert torch.equal(a, b), f"output {k}"
        assert torch.equal(gc, rc)
        assert peak <= 17 * 2 ** 30, f"the forward allocated {peak / 2 ** 30:.1f} GiB at its peak"
    finally:
        head.set_compute_dtype(torch.float32)
