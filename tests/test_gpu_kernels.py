"""GPU parity tests, kernel by kernel, through the C ABI (ctypes) against golden vectors produced by
the unmodified reference modules and against the CPU oracle on seeded inputs."""
import numpy as np
import pytest
import torch

from helpers import knn_sets_equal, knn_tie_rows, rel_err, syn

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


@pytest.fixture(scope="module")
def cp():
    import checkerpose_b200
    from checkerpose_b200 import common_ops, head, ops
    from checkerpose_b200.binary_code_helper import class_id_encoder_decoder as codec
    from checkerpose_b200.model import pipeline, pipeline_lm

    class NS:
        pass

    ns = NS()
    ns.ops, ns.head, ns.pipeline, ns.pipeline_lm, ns.common_ops, ns.codec = ops, head, pipeline, pipeline_lm, common_ops, codec
    ns.pkg = checkerpose_b200
    assert ops.lib.cp_device_arch() >= 100, "these kernels are built for sm_100a"
    return ns


@pytest.fixture(autouse=True)
def _fp32_mode():
    from checkerpose_b200 import head
    head.set_compute_dtype(torch.float32)
    yield
    head.set_compute_dtype(torch.float32)


def cuda(a, dtype=None):
    t = torch.as_tensor(np.asarray(a)) if not isinstance(a, torch.Tensor) else a
    t = t.cuda()
    return t.to(dtype) if dtype is not None else t


# ------------------------------------------------------------------------------------------------ K1
def test_knn_all_fixtures(cp, golden):
    g = golden("knn")
    n = 0
    for key, ref in g.items():
        if key.startswith("rand"):
            continue
        ds, oid, ns, ks = key.split("_")
        N, K = int(ns[1:]), int(ks[1:])
        p = syn.p3d_normed_tensor(syn.load_fps_xyz(ds, int(oid), N))
        idx = cp.pipeline.knn(p.cuda(), K)
        assert idx.dtype == torch.int64 and idx.shape == (1, N, K)
        idx = idx[0].cpu().numpy()
        bad = knn_sets_equal(idx, ref, tie_rows=knn_tie_rows(p, K, 1e-6))
        assert len(bad) == 0, f"{key}: {len(bad)} rows differ outside 1e-6 ties"
        assert (idx[:, 0] == np.arange(N)).all()
        n += 1
    assert n == 57


def test_knn_generic_channels_and_order(cp, golden):
    g = golden("knn")
    x = torch.from_numpy(g["rand_c16_n200_k12_x"])
    idx = cp.pipeline.knn(x.cuda(), 12).cpu().numpy()
    ref = g["rand_c16_n200_k12"].astype(np.int64)
    assert np.array_equal(np.sort(idx, -1), np.sort(ref, -1))
    assert (idx == ref).mean() > 0.999  # nearest-first order, up to fp32 near-ties


def test_knn_edge_cases(cp):
    x = torch.randn(2, 3, 70, generator=torch.Generator().manual_seed(3))
    for k in (1, 33, 64, 70):
        if k > 64:
            with pytest.raises(RuntimeError):
                cp.pipeline.knn(x.cuda(), k)
            continue
        idx = cp.pipeline.knn(x.cuda(), k).cpu()
        d = ((x[:, :, :, None] - x[:, :, None, :]) ** 2).sum(1)
        ref = d.topk(k, dim=-1, largest=False)[1]
        assert torch.equal(torch.sort(idx, -1)[0], torch.sort(ref, -1)[0])
    with pytest.raises(RuntimeError):
        cp.pipeline.knn(x, 4)  # CPU tensor: no fallback


# ------------------------------------------------------------------------------------------------ K2
def _sg_module(cp, g, tag, lm):
    t = lambda k: torch.from_numpy(g[f"sg_{tag}_{k}"])
    Co, C2 = t("conv.0.weight").shape[:2]
    idx = t("lm_idx" if lm else "idx").long().cuda()
    cls = cp.pipeline_lm.StaticGraph_module if lm else cp.pipeline.StaticGraph_module
    m = cls(C2 // 2, Co, idx, leaky_slope=0.2)
    m.load_state_dict({k[len(f"sg_{tag}_"):]: torch.from_numpy(v) for k, v in g.items()
                       if k.startswith(f"sg_{tag}_conv")}, strict=True)
    return m.cuda().eval(), t


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_static_graph_module_fp32(cp, golden, tag):
    g = golden("modules")
    m, t = _sg_module(cp, g, tag, lm=False)
    y = m(t("x").cuda(), None)
    assert y.shape == t("y").shape and y.dtype == torch.float32
    assert rel_err(y.cpu(), t("y")) < 1e-3
    assert torch.allclose(y.cpu(), t("y"), rtol=1e-4, atol=1e-4)
    # node-major (permuted view) input takes the zero-copy path and must agree
    xv = t("x").cuda().permute(0, 2, 1).contiguous().permute(0, 2, 1)
    assert torch.equal(m(xv, None), y)
    mlm, _ = _sg_module(cp, g, tag, lm=True)
    y = mlm(t("x").cuda(), None, t("lm_obj").cuda())
    assert torch.allclose(y.cpu(), t("lm_y"), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("ds,objs,N,K,Co,B", [("lmo", (1,), 4096, 20, 256, 3), ("lm", (3, 7), 300, 20, 64, 4), ("ycbv", (5,), 1000, 8, 96, 2),
                                               ("lmo", (5,), 512, 40, 32, 2),
                                               # KP = 16 / 32, and padded lists (K < KP) at every other size
                                               ("lm", (2,), 1024, 16, 128, 2), ("ycbv", (3, 4, 5), 1024, 32, 64, 3),
                                               ("lm", (6,), 700, 13, 96, 2), ("lmo", (1,), 300, 27, 256, 2),
                                               ("ycbv", (7,), 1000, 37, 32, 2), ("ycbv", (9, 10), 129, 5, 64, 3),
                                               ("lm", (11,), 512, 17, 128, 2)])
def test_edge_aggregate_staged_f32_bit_exact(cp, ds, objs, N, K, Co, B):
    """float32 aggregation on the graph plan (rows staged per tile, node pairs) == the unstaged gather kernel, bit for bit
    (max and one add per element: no rounding freedom), incl. ragged last tiles and per-RoI graphs."""
    ops = cp.ops
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)) for o in objs], dim=0).cuda()
    _, idx32 = ops.knn(p3d, K, want_i32=True)
    plan = ops.GraphPlan(idx32, p3d)
    g = torch.Generator().manual_seed(N + K + Co)
    z = torch.randn(B, N, 2 * Co, generator=g).cuda()
    sel = None if len(objs) == 1 else torch.randint(0, len(objs), (B,), generator=g).to(torch.int32).cuda()
    want = ops.edge_aggregate(z, plan.idx_p, sel, 0.2)
    got = ops.edge_aggregate_staged(z, plan, sel, 0.2)
    assert torch.equal(got, want)


def test_static_graph_requires_eval_and_cuda(cp, golden):
    g = golden("modules")
    m, t = _sg_module(cp, g, "a", lm=False)
    m.train()
    with pytest.raises(RuntimeError):
        m(t("x").cuda(), None)
    m.eval()
    with pytest.raises(RuntimeError):
        m(t("x"), None)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_static_graph_module_bf16(cp, golden, tag):
    """tcgen05 GEMM + bf16 aggregation vs the reference module: 1e-2 relative (north_star bf16 bar)."""
    g = golden("modules")
    m, t = _sg_module(cp, g, tag, lm=False)
    cp.head.set_compute_dtype(torch.bfloat16)
    y = m(t("x").cuda(), None)
    assert y.dtype == torch.float32
    ref = t("y")
    scale = ref.abs().max()
    assert (y.cpu() - ref).abs().max() < 2e-2 * scale, float((y.cpu() - ref).abs().max() / scale)
    mlm, _ = _sg_module(cp, g, tag, lm=True)
    y = mlm(t("x").cuda(), None, t("lm_obj").cuda())
    assert (y.cpu() - t("lm_y")).abs().max() < 2e-2 * scale


def test_get_graph_feature(cp, golden):
    g = golden("modules")
    y = cp.pipeline.get_graph_feature(cuda(g["ggf_x"]), cuda(g["ggf_idx"]).long(), None)
    assert np.array_equal(y.cpu().numpy(), g["ggf_y"])


# ------------------------------------------------------------------------------------------------ K3
@pytest.mark.parametrize("tag,k,fd,ed", [("a", 2, 32, 16), ("b", 2, 256, 64), ("c", 4, 32, 8)])
def test_index2feat(cp, golden, tag, k, fd, ed):
    g = golden("modules")
    t = lambda n: torch.from_numpy(g[f"i2f_{tag}_{n}"])
    m = cp.pipeline.Index2Feat_module(feat_dim=fd, embed_dim=ed, kernel_size=k)
    m.load_state_dict({"patch_generator.weight": t("patch_generator.weight"), "patch_generator.bias": t("patch_generator.bias")})
    m = m.cuda().eval()
    y = m(t("feat").cuda(), None, t("xid").cuda(), t("yid").cuda())
    assert y.shape == t("y").shape
    # the gather itself is an exact copy; the conv before it is cuDNN fp32 (not bit-identical to the CPU conv)
    # the patch convolution runs on the split-bf16 tensor-core GEMM (~2^-16 relative per product): north_star's fp32 bar
    # is 1e-3 relative; held here to 1e-4 of the tensor's scale
    assert torch.allclose(y.cpu(), t("y"), rtol=1e-4, atol=1e-4 * float(t("y").abs().max()))
    patches = cp.head.patches_nhwc(m.patch_generator, t("feat").cuda(), torch.float32)
    taps = cp.ops.sample_taps(patches, t("xid").cuda(), t("yid").cuda(), None, k)
    B, N = t("xid").shape
    bi = torch.arange(B).view(B, 1).expand(-1, N)
    pc = patches.cpu()
    want = torch.cat([pc[bi, 2 * t("yid") + dy, 2 * t("xid") + dx] for dx, dy in ((0, 0), (0, k), (k, 0), (k, k))], dim=2)
    assert torch.equal(taps.cpu(), want), "4-tap gather must be bit-exact"


def test_mlp_query(cp, golden):
    g = golden("modules")
    m = cp.pipeline.MLP_QueryNet(feat_dims=(256, 256, 64), pt_dim=3, out_dim=2, leaky_slope=0.01)
    m.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("mq_mlps")})
    y = m.cuda().eval()(cuda(g["mq_x"]), None)
    assert torch.allclose(y.cpu(), torch.from_numpy(g["mq_y"]), rtol=1e-4, atol=1e-4)


# ------------------------------------------------------------------------------------------------ K4
def test_decode_functions(cp, golden):
    g = golden("decode")
    cpb = torch.from_numpy(g["code_prob"])
    safe = (cpb.abs() > 1e-4)            # north_star: exact except logits within 1e-4 of the threshold
    P = cp.pipeline
    x = cpb.cuda()
    m = P.from_mask_prob_to_mask(x).cpu()
    assert m.dtype == torch.float32 and torch.equal(m[safe], torch.from_numpy(g["mask"])[safe])
    safe_kp = safe.all(dim=1)
    ids = P.from_code_prob_to_id(x).cpu()
    assert ids.dtype == torch.int64 and torch.equal(ids[safe_kp], torch.from_numpy(g["code_prob_id"])[safe_kp])
    b = P.from_bit_prob_to_id(x[:, 0:1]).cpu()
    assert torch.equal(b[safe[:, 0]], torch.from_numpy(g["bit_prob_id"])[safe[:, 0]])
    assert np.array_equal(P.from_gt_code_to_id(torch.sigmoid(cpb).cuda()).cpu().numpy()[safe_kp], g["gt_code_id"][safe_kp])
    assert np.array_equal(P.from_gt_bit_to_id(torch.sigmoid(cpb[:, 0:1]).cuda()).cpu().numpy()[safe[:, 0]], g["gt_bit_id"][safe[:, 0]])
    assert np.array_equal(P.from_code_to_id(cuda(g["code"])).cpu().numpy(), g["code_id"])


def test_common_ops(cp, golden):
    g = golden("decode")
    x = cuda(g["code_prob"])
    co = cp.common_ops
    for thr in (0.5, 0.3, 0.9):
        logit_thr = float(np.log(thr / (1 - thr)))
        safe = np.abs(g["code_prob"] - logit_thr) > 1e-4
        a = co.from_output_to_class_mask(x, thershold=thr)
        assert isinstance(a, np.ndarray) and a.dtype == np.float64
        assert np.array_equal(a[safe], g[f"co_mask_{thr}"][safe])
        b = co.from_output_to_class_mask_torch(x, thershold=thr)
        assert b.is_cuda and np.array_equal(b.cpu().numpy()[safe], g[f"co_mask_torch_{thr}"][safe])
        c = co.from_output_to_class_binary_code(x, "BCE", thershold=thr)
        assert np.array_equal(c[safe], g[f"co_code_bce_{thr}"][safe])
    ce = co.from_output_to_class_binary_code(cuda(g["co_ce_in"]), "CE", divided_num_each_interation=2, binary_code_length=16)
    assert ce.shape == g["co_code_ce"].shape and np.array_equal(ce, g["co_code_ce"])
    assert tuple(co.get_batch_size(0.75, 32)) == tuple(g["co_batch_size"])
    assert co.from_dim_str_to_tuple("256_256_64") == tuple(g["co_dim_tuple"]) and co.from_dim_str_to_tuple(None) is None


def test_codec(cp, golden):
    g = golden("decode")
    c = cp.codec
    a = c.class_code_vecs_to_class_id_vec(g["cc_vecs"])
    assert a.dtype == np.float64 and np.array_equal(a, g["cc_vecs_id"])
    assert np.array_equal(c.class_code_images_to_class_id_image(g["cc_hwc"]), g["cc_hwc_id"])
    t = c.class_code_images_to_class_id_image_torch(cuda(g["cc_chw"]))
    assert t.dtype == torch.float32 and np.array_equal(t.cpu().numpy(), g["cc_chw_id"])
    t = c.class_code_images_to_class_id_image_torch_batch(cuda(g["cc_bchw"]))
    assert t.dtype == torch.int64 and np.array_equal(t.cpu().numpy(), g["cc_bchw_id"])
    assert np.array_equal(c.class_id_vec_to_class_code_vecs(g["cc_ids"], class_base=2, iteration=6), g["cc_ids_code"])
    assert np.array_equal(c.class_id_image_to_class_code_images(g["cc_idimg"], 2, 8, 256), g["cc_idimg_code"])
    assert c.code_to_id([1, 0, 1, 1, 0]) == int(g["cc_code_to_id"]) and c.str_code_to_id("10110") == int(g["cc_str_code_to_id"])
    with pytest.raises(ValueError):
        c.class_id_image_to_class_code_images(g["cc_idimg"], 2, 7, 256)


def test_correspondences(cp, golden):
    g = golden("correspondences")
    xyz = syn.load_fps_xyz("lmo", 1, 300)
    B, N, S = 3, 300, 64
    roi = torch.stack([torch.from_numpy(g[f"c{c}_roi_logit"]) for c in range(B)]).float().view(B, 1, N)
    seg = torch.stack([torch.from_numpy(g[f"c{c}_seg_logit"]) for c in range(B)]).float()
    bbox = torch.stack([torch.from_numpy(g[f"c{c}_bbox"]) for c in range(B)]).float()
    xid = torch.stack([torch.from_numpy(g[f"c{c}_xid"]) for c in range(B)]).long()
    yid = torch.stack([torch.from_numpy(g[f"c{c}_yid"]) for c in range(B)]).long()
    rec = cp.ops.correspondences(roi.cuda(), seg.cuda(), bbox.cuda(), xid.cuda(), yid.cuda())
    uv, flags = cp.ops.split_correspondences(rec)
    uv, flags = uv.cpu().numpy(), flags.cpu().numpy()
    for c in range(B):
        for bit, tag in ((1, "all"), (2, "full"), (4, "visib")):
            m = (flags[c] & bit) != 0
            assert np.array_equal(xyz[m], g[f"c{c}_{tag}_p3d"]), "valid set must match the reference exactly"
            assert np.allclose(uv[c][m], g[f"c{c}_{tag}_p2d"], rtol=1e-6, atol=0)  # f32 record vs f64 grid


def test_correspondences_packed_roundtrip(cp):
    """The 2-byte records that cross NVLink / PCIe decode to exactly the 12-byte records (device kernel and host numpy)."""
    B, N, S = 5, 4096, 64
    g = torch.Generator().manual_seed(11)
    roi = torch.randn(B, 1, N, generator=g).cuda()
    seg = torch.randn(B, 2, S, S, generator=g).cuda()
    bbox = syn.synthetic_bboxes(B, g).cuda()
    xid = torch.randint(0, S, (B, N), generator=g).cuda()
    yid = torch.randint(0, S, (B, N), generator=g).cuda()
    rec = cp.ops.correspondences(roi, seg, bbox, xid, yid)
    packed = cp.ops.correspondences_packed(roi, seg, bbox, xid, yid)
    assert packed.shape == (B, 16 + 2 * N) and packed.dtype == torch.uint8
    assert torch.equal(cp.ops.unpack_correspondences(packed, S), rec)
    uv, flags, x2, y2, bb = cp.ops.unpack_correspondences_host(packed, S)
    uv_ref, flags_ref = cp.ops.split_correspondences(rec)
    assert np.array_equal(uv, uv_ref.cpu().numpy()) and np.array_equal(flags, flags_ref.cpu().numpy())
    assert np.array_equal(x2, xid.cpu().numpy()) and np.array_equal(y2, yid.cpu().numpy()) and np.array_equal(bb, bbox.cpu().numpy())


# ------------------------------------------------------------------------------------------------ fused query tail + decode (K4)
@pytest.mark.parametrize("N,B,kin,with_kp", [(4096, 3, 256, True), (300, 2, 256, False), (512, 4, 64, True)])
def test_query_decode_fused(cp, N, B, kin, with_kp):
    """cp_query_decode_fwd (TMA tensor loads -> tcgen05 kin->64 -> fp32 64->2 -> decode) against float64 maths on the same
    bf16-rounded operands: logits to 1e-3 of scale; bit planes, in-place id update and keypoint-order ids exactly the decode of
    those logits (pipeline.py:375-381), scattered through the plan permutation of a per-RoI graph selection."""
    ops = cp.ops
    g = torch.Generator().manual_seed(N + kin)
    src = torch.randn(B, N, kin, generator=g).to(torch.bfloat16)
    w1 = (torch.randn(64, kin, generator=g) / kin ** 0.5).to(torch.bfloat16).float()
    b1 = torch.randn(64, generator=g) * 0.1
    w2 = torch.randn(2, 64, generator=g) / 8.0
    b2 = torch.randn(2, generator=g) * 0.1
    G, Ltot, plane = 2, 6, 4
    perm = torch.stack([torch.randperm(N, generator=g) for _ in range(G)]).to(torch.int32)
    sel = torch.randint(0, G, (B,), generator=g).to(torch.int32)
    x_id0 = torch.randint(0, 16, (B, N), generator=g)
    y_id0 = torch.randint(0, 16, (B, N), generator=g)
    hid = src.double() @ w1.double().t() + b1.double()
    hid = torch.where(hid > 0, hid, hid * 0.01)
    ref = hid @ w2.double().t() + b2.double()                              # (B,N,2)
    x_bits = torch.full((B, Ltot, N), float("nan")).cuda()
    y_bits = torch.full((B, Ltot, N), float("nan")).cuda()
    x_id, y_id = x_id0.clone().cuda(), y_id0.clone().cuda()
    x_kp = torch.full((B, N), -1, dtype=torch.int64).cuda() if with_kp else None
    y_kp = torch.full((B, N), -1, dtype=torch.int64).cuda() if with_kp else None
    logits = torch.zeros(B, N, 2).cuda()
    ops.query_decode_fwd(src=src.cuda(), w1_packed=ops.pack_weight(w1.cuda()), b1=b1.cuda(), slope=0.01, w2=w2.cuda().contiguous(), b2=b2.cuda(),
                         plane=plane, Ltot=Ltot, x_bits=x_bits, y_bits=y_bits, x_id=x_id, y_id=y_id, perm=perm.cuda(), graph_sel=sel.cuda(),
                         x_id_kp=x_kp, y_id_kp=y_kp, logits=logits)
    err = float((logits.cpu().double() - ref).abs().max() / ref.abs().max())
    assert err < 1e-3, err
    lg = logits.cpu()
    kp = perm[sel.long()].long()                                           # (B,N): plan position -> keypoint id
    want_x = torch.full((B, N), float("nan")).scatter_(1, kp, lg[..., 0])
    want_y = torch.full((B, N), float("nan")).scatter_(1, kp, lg[..., 1])
    assert torch.equal(x_bits[:, plane].cpu(), want_x) and torch.equal(y_bits[:, plane].cpu(), want_y)
    others = [l for l in range(Ltot) if l != plane]
    assert torch.isnan(x_bits[:, others]).all() and torch.isnan(y_bits[:, others]).all()
    nx, ny = x_id0 * 2 + (lg[..., 0] > 0).long(), y_id0 * 2 + (lg[..., 1] > 0).long()
    assert torch.equal(x_id.cpu(), nx) and torch.equal(y_id.cpu(), ny)
    if with_kp:
        assert torch.equal(x_kp.cpu(), torch.zeros(B, N, dtype=torch.int64).scatter_(1, kp, nx))
        assert torch.equal(y_kp.cpu(), torch.zeros(B, N, dtype=torch.int64).scatter_(1, kp, ny))


# ------------------------------------------------------------------------------------------------ split-bf16 x3 GEMM
@pytest.mark.parametrize("M,K1,K2,Nout,act", [(300, 64, 0, 128, False), (1000, 256, 64, 256, True), (257, 256, 256, 512, True),
                                               (128, 64, 0, 7, False), (513, 1024, 0, 600, False), (4096, 256, 0, 2, False)])
def test_gemm_x3_linear_matches_fp64(cp, M, K1, K2, Nout, act):
    """The float32-mode GEMM on tcgen05 (fp32 operands split into bf16 hi + lo, three MMAs) against float64: the
    error budget is ~2^-16 per product, i.e. far inside north_star's 1e-3 and the 1e-4 logit band."""
    ops = cp.ops
    g = torch.Generator().manual_seed(M + K1 + Nout)
    a1 = torch.randn(M, K1, generator=g)
    a2 = torch.randn(M, K2, generator=g) if K2 else None
    w = torch.randn(Nout, K1 + K2, generator=g) / (K1 + K2) ** 0.5
    bias = torch.randn(Nout, generator=g)
    a = a1 if a2 is None else torch.cat([a1, a2], dim=1)
    ref = a.double() @ w.double().t() + bias.double()
    if act:
        ref = torch.where(ref > 0, ref, ref * 0.01)
    ws = ops.pack_weight_split(w.cuda())
    out = ops.gemm_x3_linear(a1.cuda(), ws, Nout, bias.cuda(), act, 0.01, a2=None if a2 is None else a2.cuda())
    err = float((out.cpu().double() - ref).abs().max() / ref.abs().max())
    fp32 = float(((a @ w.t() + bias).double() - (a.double() @ w.double().t() + bias.double())).abs().max() / ref.abs().max())
    print(f"x3 GEMM M={M} K={K1}+{K2} N={Nout}: max err / max = {err:.2e} (plain fp32 matmul on the CPU: {fp32:.2e})")
    assert out.shape == (M, Nout) and err < 2e-5, err
    # rows beyond M / columns beyond Nout are never written
    canvas = torch.full((M + 3, Nout + 5), float("nan"), device="cuda")
    ops.gemm_x3_linear(a1.cuda(), ws, Nout, bias.cuda(), act, 0.01, a2=None if a2 is None else a2.cuda(), out=canvas[:M, :Nout])
    assert torch.isnan(canvas[M:]).all() and torch.isnan(canvas[:, Nout:]).all() and torch.equal(canvas[:M, :Nout], out)
    # the same through the TMA-store epilogue (16-byte aligned rows): the tensor map clips the ragged last tile
    wide = (Nout + 3) // 4 * 4 + 8
    canvas = torch.full((M + 3, wide), float("nan"), device="cuda")
    ops.gemm_x3_linear(a1.cuda(), ws, Nout, bias.cuda(), act, 0.01, a2=None if a2 is None else a2.cuda(), out=canvas[:M, :Nout])
    assert torch.isnan(canvas[M:]).all() and torch.isnan(canvas[:, Nout:]).all() and torch.equal(canvas[:M, :Nout], out)


@pytest.mark.parametrize("B,H,Cin,Cout,k,pad,transposed", [(3, 16, 256, 256, 3, 1, False), (2, 32, 64, 64, 2, 1, False),
                                                           (2, 8, 128, 64, 3, 1, True), (5, 9, 64, 2, 1, 0, False)])
def test_gemm_x3_conv_matches_fp64(cp, B, H, Cin, Cout, k, pad, transposed):
    """Implicit-GEMM convolution of the float32 mode against torch's float64 convolution on the CPU."""
    import torch.nn.functional as F
    ops = cp.ops
    g = torch.Generator().manual_seed(B + H + Cin + k)
    x = torch.randn(B, Cin, H, H, generator=g)
    bias = torch.randn(Cout, generator=g)
    if transposed:
        w = torch.randn(Cin, Cout, k, k, generator=g) / (Cin * k * k / 4) ** 0.5
        ref = F.conv_transpose2d(x.double(), w.double(), bias.double(), stride=2, padding=pad, output_padding=1)
        wm = w.permute(1, 2, 3, 0).reshape(Cout, k * k * Cin)
    else:
        w = torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5
        ref = F.conv2d(x.double(), w.double(), bias.double(), stride=1, padding=pad)
        wm = w.permute(0, 2, 3, 1).reshape(Cout, k * k * Cin)
    ref = torch.relu(ref)
    Ho = ref.shape[2]
    ws = ops.pack_weight_split(wm.contiguous().cuda())
    out = ops.gemm_x3_conv(x.permute(0, 2, 3, 1).contiguous().cuda(), ws, Cout, k, k, pad, Ho, Ho, bias.cuda(), True, 0.0, transposed)
    err = float((out.cpu().double().permute(0, 3, 1, 2) - ref).abs().max() / ref.abs().max())
    print(f"x3 conv {'T' if transposed else ''} B={B} H={H} {Cin}->{Cout} k={k}: max err / max = {err:.2e}")
    assert out.shape == (B, Ho, Ho, Cout) and err < 2e-5, err


@pytest.mark.parametrize("B,H,Cin,Cout,k,pad,transposed", [(3, 16, 256, 256, 3, 1, False), (2, 32, 64, 64, 2, 1, False),
                                                           (2, 8, 128, 64, 3, 1, True), (5, 9, 64, 2, 1, 0, False), (2, 20, 512, 256, 3, 1, False)])
def test_conv_bf16_matches_fp64(cp, B, H, Cin, Cout, k, pad, transposed):
    """bf16 implicit-GEMM convolution on tcgen05 (cp_conv_bf16) against torch's float64 convolution on the same bf16-rounded
    operands: only the fp32 accumulation order and the bf16 rounding of the output differ (1e-2 of north_star)."""
    import torch.nn.functional as F
    ops = cp.ops
    g = torch.Generator().manual_seed(B + H + Cin + k)
    x = torch.randn(B, Cin, H, H, generator=g).to(torch.bfloat16)
    bias = torch.randn(Cout, generator=g)
    if transposed:
        w = (torch.randn(Cin, Cout, k, k, generator=g) / (Cin * k * k / 4) ** 0.5).to(torch.bfloat16)
        ref = F.conv_transpose2d(x.double(), w.double(), bias.double(), stride=2, padding=pad, output_padding=1)
        wm = w.float().permute(1, 2, 3, 0).reshape(Cout, k * k * Cin)
    else:
        w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(torch.bfloat16)
        ref = F.conv2d(x.double(), w.double(), bias.double(), stride=1, padding=pad)
        wm = w.float().permute(0, 2, 3, 1).reshape(Cout, k * k * Cin)
    ref = torch.relu(ref)
    Ho = ref.shape[2]
    out = ops.conv_bf16(x.permute(0, 2, 3, 1).contiguous().cuda(), ops.pack_weight(wm.contiguous().cuda()), Cout, k, k, pad, Ho, Ho,
                        bias.cuda(), True, 0.0, transposed)
    err = float((out.float().cpu().double().permute(0, 3, 1, 2) - ref).abs().max() / ref.abs().max())
    print(f"bf16 conv {'T' if transposed else ''} B={B} H={H} {Cin}->{Cout} k={k}: max err / max = {err:.2e}")
    assert out.shape == (B, Ho, Ho, Cout) and out.dtype == torch.bfloat16 and err < 6e-3, err


@pytest.mark.parametrize("pair", ["1", "0"])
@pytest.mark.parametrize("kind,B,H,W,Cin,Cout", [("same3", 3, 16, 16, 256, 256), ("same3", 3, 10, 12, 64, 64), ("same3", 2, 64, 64, 128, 256),
                                                 ("same1", 5, 9, 9, 64, 7), ("full2", 2, 32, 32, 64, 64), ("full2", 3, 11, 9, 128, 64),
                                                 ("convT", 2, 8, 8, 128, 256), ("convT", 3, 5, 7, 64, 64)])
def test_conv_slab_matches_fp64(cp, monkeypatch, pair, kind, B, H, W, Cin, Cout):
    """Slab convolution (cp_conv_slab: one TMA-loaded activation slab per channel slice, every tap a row-shifted tcgen05
    descriptor over it; CTA pairs and single CTAs) against torch's float64 convolution on the same bf16-rounded operands, and
    the zero border of the maps it hands on.  Odd tile counts, ragged maps, narrow outputs, all four transposed parities."""
    import torch.nn.functional as F
    ops = cp.ops
    monkeypatch.setenv("CP_SLAB_PAIR", pair)
    g = torch.Generator().manual_seed(B + H + Cin + len(kind))
    x = torch.randn(B, Cin, H, W, generator=g).to(torch.bfloat16)
    bias = torch.randn(Cout, generator=g)
    xh = x.permute(0, 2, 3, 1).contiguous().cuda()
    xp = ops.to_bordered(xh).contiguous()
    bordered = True
    if kind == "convT":
        w = (torch.randn(Cin, Cout, 3, 3, generator=g) / (Cin * 9 / 4) ** 0.5).to(torch.bfloat16)
        ref = F.conv_transpose2d(x.double(), w.double(), bias.double(), stride=2, padding=1, output_padding=1)
        wm = w.float().permute(1, 2, 3, 0).reshape(Cout, 9 * Cin)
        out = ops.convT_slab(xh, ops.pack_weight(wm.contiguous().cuda()), Cout, bias.cuda(), True, 0.0)
    else:
        k = int(kind[-1])
        w = (torch.randn(Cout, Cin, k, k, generator=g) / (Cin * k * k) ** 0.5).to(torch.bfloat16)
        wm = w.float().permute(0, 2, 3, 1).reshape(Cout, k * k * Cin)
        wp = ops.pack_weight(wm.contiguous().cuda())
        if kind.startswith("same"):
            ref = F.conv2d(x.double(), w.double(), bias.double(), padding=k // 2)
            out = ops.conv_slab_same(xp, wp, Cout, k, k, bias.cuda(), True, 0.0)
        else:
            ref = F.conv2d(x.double(), w.double(), bias.double(), padding=k - 1)
            out = ops.conv_slab_full(xp, wp, Cout, k, k, bias.cuda(), True, 0.0)
            bordered = False
    ref = torch.relu(ref).permute(0, 2, 3, 1)
    out = out.float().cpu().double()
    if bordered:
        assert out.shape == (B, ref.shape[1] + 1, ref.shape[2] + 1, Cout)
        edge = out.clone()
        edge[:, :-1, :-1] = 0
        assert float(edge.abs().max()) == 0.0, "the border of a slab convolution's output must be zeros"
        out = out[:, :-1, :-1]
    assert out.shape == ref.shape
    err = float((out - ref).abs().max() / ref.abs().max())
    print(f"slab {kind} pair={pair} B={B} {H}x{W} {Cin}->{Cout}: max err / max = {err:.2e}")
    assert err < 6e-3, err


@pytest.mark.parametrize("pair", ["1", "0"])
@pytest.mark.parametrize("B,H,W,Cin,Cout,nseg", [(3, 16, 16, 128, 256, 2), (2, 9, 11, 64, 64, 1), (2, 12, 12, 64, 256, 4)])
def test_conv_slab_fused_seg_head(cp, monkeypatch, pair, B, H, W, Cin, Cout, nseg):
    """seg_block (1x1) computed in the last convolution's epilogue: equals the 1x1 convolution of the bf16 map the same launch
    stores (float64 reference on exactly those values), and the map itself is unchanged by the fusion."""
    ops = cp.ops
    monkeypatch.setenv("CP_SLAB_PAIR", pair)
    g = torch.Generator().manual_seed(B + H + Cout + nseg)
    xp = ops.to_bordered(torch.randn(B, H, W, Cin, generator=g).to(torch.bfloat16).cuda()).contiguous()
    wp = ops.pack_weight((torch.randn(Cout, 9 * Cin, generator=g) / (9 * Cin) ** 0.5).cuda())
    bias = torch.randn(Cout, generator=g).cuda()
    sw = (torch.randn(nseg, Cout, generator=g) / Cout ** 0.5).cuda()
    sb = torch.randn(nseg, generator=g).cuda()
    plain = ops.conv_slab_same(xp, wp, Cout, 3, 3, bias, True, 0.0)
    out, seg = ops.conv_slab_same(xp, wp, Cout, 3, 3, bias, True, 0.0, seg=(sw, sb))
    assert torch.equal(out, plain) and seg.shape == (B, nseg, H, W) and seg.dtype == torch.float32
    ref = torch.einsum("bhwc,jc->bjhw", out[:, :-1, :-1].double(), sw.double()) + sb.double().view(1, -1, 1, 1)
    err = float((seg.double() - ref).abs().max() / ref.abs().max())
    print(f"fused seg pair={pair}: max err / max = {err:.2e}")
    assert err < 1e-5, err


def test_zero_border_and_padded_upsample(cp):
    """cp_zero_border_nhwc + cp_upsample2x_cat_nhwc_to: the padded upsampling equals the plain one inside a zero border."""
    ops = cp.ops
    g = torch.Generator().manual_seed(11)
    a = torch.randn(3, 7, 9, 64, generator=g).to(torch.bfloat16).cuda().permute(0, 3, 1, 2)
    b = torch.randn(3, 7, 9, 32, generator=g).to(torch.bfloat16).cuda().permute(0, 3, 1, 2)
    plain = ops.upsample2x_cat(a, b).permute(0, 2, 3, 1)
    buf = ops.upsample2x_cat_padded(a, b)
    assert buf.shape == (3, 15, 19, 96)
    assert torch.equal(buf[:, :-1, :-1], plain)
    edge = buf.clone()
    edge[:, :-1, :-1] = 0
    assert float(edge.float().abs().max()) == 0.0
    # the source may itself be the interior of a bordered map (strided view)
    again = ops.upsample2x_cat_padded(buf[:, :-1, :-1].permute(0, 3, 1, 2), None)
    assert torch.equal(again[:, :-1, :-1], ops.upsample2x_cat(plain.permute(0, 3, 1, 2).contiguous(memory_format=torch.channels_last), None).permute(0, 2, 3, 1))


# ------------------------------------------------------------------------------------------------ tcgen05 chain
def _bf16_round(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("C,Nout,N,B", [(64, 128, 300, 2), (256, 512, 128, 3), (128, 64, 257, 1), (256, 16, 512, 2)])
def test_chain_gemm_exact(cp, C, Nout, N, B):
    """LOAD -> one GEMM: with bf16-representable operands the fp32-accumulated tcgen05 result must equal
    a float64 matmul to fp32 rounding -- any descriptor / swizzle / TMEM-lane mistake shows up here."""
    ops = cp.ops
    g = torch.Generator().manual_seed(C + Nout)
    x = _bf16_round(torch.randn(B, N, C, generator=g))
    w = _bf16_round(torch.randn(Nout, C, generator=g) / C ** 0.5)
    bias = torch.randn(Nout, generator=g)
    ref = (x.double() @ w.double().t() + bias.double())
    wp = ops.pack_weight(w.cuda())
    # fp32 output (first n_valid columns)
    nv = min(Nout, 256)
    if Nout <= 256:
        out = torch.full((B, N, Nout), float("nan"), device="cuda")
        ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x.cuda().to(torch.bfloat16),
                      layers=[ops.chain_layer(wp, bias.cuda(), C, Nout, False, 0.0)], out=out, out_mode=ops.OUT_F32, n_valid=nv)
        torch.cuda.synchronize()
        assert torch.allclose(out.cpu().double(), ref, rtol=1e-5, atol=1e-5), float((out.cpu().double() - ref).abs().max())
    # bf16 output with LeakyReLU
    out = torch.empty((B, N, Nout), dtype=torch.bfloat16, device="cuda")
    ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x.cuda().to(torch.bfloat16),
                  layers=[ops.chain_layer(wp, bias.cuda(), C, Nout, True, 0.2)], out=out, out_mode=ops.OUT_BF16)
    want = torch.nn.functional.leaky_relu(ref, 0.2)
    assert torch.allclose(out.cpu().double(), want, rtol=1e-2, atol=1e-2)


def test_chain_three_layers(cp):
    """LOAD -> 256->256 (LReLU) -> 256->64 (LReLU) -> 64->2: the MLP_QueryNet chain; activations are
    re-quantised to bf16 between layers exactly as the kernel does."""
    ops = cp.ops
    g = torch.Generator().manual_seed(5)
    B, N = 2, 384
    x = _bf16_round(torch.randn(B, N, 256, generator=g))
    ws = [_bf16_round(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5) for o, i in ((256, 256), (64, 256), (2, 64))]
    bs = [torch.randn(o, generator=g) * 0.1 for o in (256, 64, 2)]
    h = x.double()
    for li, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.double().t() + b.double()
        if li < 2:
            h = _bf16_round(torch.nn.functional.leaky_relu(h, 0.01).float()).double()
    layers = [ops.chain_layer(ops.pack_weight(w.cuda()), b.cuda(), w.shape[1], w.shape[0], li < 2, 0.01)
              for li, (w, b) in enumerate(zip(ws, bs))]
    out = torch.zeros((B, N, 16), device="cuda")
    ops.chain_fwd(prologue=ops.PRO_LOAD, B=B, N=N, src=x.cuda().to(torch.bfloat16), layers=layers, out=out,
                  out_mode=ops.OUT_F32, n_valid=2)
    got = out[:, :, :2].cpu().double()
    # bf16 re-quantisation of intermediates can differ by one ulp where fp32 sums differ in the last bit
    assert (got - h).abs().max() < 2e-2 * h.abs().max(), float((got - h).abs().max())


@pytest.mark.parametrize("Cg,H,N,B", [(64, 16, 300, 3), (256, 32, 512, 2), (256, 64, 1024, 2)])
def test_taps_chain_fused(cp, Cg, H, N, B):
    """K3 (taps_chain_kernel): 4-tap Index2Feat gather x roi mask | graph feature -> Linear+LReLU x2 -> [P|Q] GEMM vs the
    same maths in float64 with bf16 re-quantisation between layers (pipeline.py:156-163, 278-286)."""
    ops = cp.ops
    g = torch.Generator().manual_seed(Cg + H + N)
    Hp = H + 1
    patches = _bf16_round(torch.randn(B, Hp, Hp, 64, generator=g))
    gf = _bf16_round(torch.randn(B, N, Cg, generator=g))
    x_id = torch.randint(0, H // 2, (B, N), generator=g)
    y_id = torch.randint(0, H // 2, (B, N), generator=g)
    mask = (torch.rand(B, N, generator=g) > 0.2).float()
    dims = ((256, 256 + Cg), (256, 256), (512, 256))
    ws = [_bf16_round(torch.randn(o, i, generator=g) * (2.0 / i) ** 0.5) for o, i in dims]
    bs = [torch.randn(o, generator=g) * 0.1 for o, _ in dims]
    bi = torch.arange(B)[:, None]
    taps = torch.cat([patches[bi, 2 * y_id + dy, 2 * x_id + dx] for dy, dx in ((0, 0), (2, 0), (0, 2), (2, 2))], dim=-1)
    h = torch.cat([taps * mask[:, :, None], gf], dim=-1).double()
    for li, (w, b) in enumerate(zip(ws, bs)):
        h = h @ w.double().t() + b.double()
        if li < 2:
            h = _bf16_round(torch.nn.functional.leaky_relu(h, 0.01).float()).double()
    layers = [ops.chain_layer(ops.pack_weight(w.cuda()), b.cuda(), w.shape[1], w.shape[0], li < 2, 0.01)
              for li, (w, b) in enumerate(zip(ws, bs))]
    out = torch.full((B, N, 512), float("nan"), dtype=torch.bfloat16, device="cuda")
    ops.chain_fwd(prologue=ops.PRO_TAPS, B=B, N=N, patches=patches.cuda().to(torch.bfloat16), tap_step=2, x_id=x_id.cuda(),
                  y_id=y_id.cuda(), mask=mask.cuda(), graph_feat=gf.cuda().to(torch.bfloat16), layers=layers, out=out,
                  out_mode=ops.OUT_BF16)
    got = out.cpu().double()
    assert bool(torch.isfinite(got).all())
    # one bf16 rounding of the output + one-ulp differences of the re-quantised intermediates
    assert (got - h).abs().max() < 2e-2 * h.abs().max(), float((got - h).abs().max() / h.abs().max())


def test_chain_agg_prologue(cp):
    """AGG prologue (EdgeConv aggregation in registers) + GEMM vs the same maths in float64."""
    ops = cp.ops
    g = torch.Generator().manual_seed(6)
    B, N, Co, K = 3, 200, 256, 20
    z = _bf16_round(torch.randn(B, N, 2 * Co, generator=g))
    idx = torch.randint(0, N, (2, N, K), generator=g).int()
    sel = torch.tensor([1, 0, 1]).int()
    w = _bf16_round(torch.randn(512, Co, generator=g) / 16)
    gat = z[:, :, :Co][torch.arange(B)[:, None, None], idx[sel.long()].long()]      # (B,N,K,Co)
    a = torch.nn.functional.leaky_relu(gat.max(dim=2)[0] + z[:, :, Co:], 0.2)
    a_bf = _bf16_round(a)
    ref = a_bf.double() @ w.double().t()
    out = torch.empty((B, N, 512), dtype=torch.bfloat16, device="cuda")
    a_out = torch.empty((B, N, Co), dtype=torch.bfloat16, device="cuda")
    ops.chain_fwd(prologue=ops.PRO_AGG, B=B, N=N, z=z.cuda().to(torch.bfloat16), idx32=idx.cuda(), graph_sel=sel.cuda(),
                  agg_slope=0.2, a_out=a_out, layers=[ops.chain_layer(ops.pack_weight(w.cuda()), None, Co, 512, False, 0.0)],
                  out=out, out_mode=ops.OUT_BF16)
    assert torch.equal(a_out.cpu().float(), a_bf), "aggregated tile must be bit-exact in bf16"
    assert torch.allclose(out.cpu().double(), ref, rtol=1e-2, atol=1e-2)
    # the SIMT aggregation kernel computes the same thing
    y = ops.edge_aggregate(z.cuda().to(torch.bfloat16), idx.cuda(), sel.cuda(), 0.2)
    assert torch.equal(y.cpu().float(), a_bf)


# ------------------------------------------------------------------------------------------------ image branch glue
@pytest.mark.parametrize("dtype,Ca,Cb,H", [(torch.float32, 8, 4, 5), (torch.bfloat16, 256, 512, 16), (torch.bfloat16, 64, 0, 7)])
def test_upsample2x_cat(cp, dtype, Ca, Cb, H):
    """cp_upsample2x_cat_nhwc == UpsamplingBilinear2d(scale_factor=2)(cat([a, b], 1)) (pipeline.py:201, 372)."""
    g = torch.Generator().manual_seed(11)
    B, W = 3, H + 2
    a = torch.randn(B, Ca, H, W, generator=g).to(dtype)
    b = torch.randn(B, Cb, H, W, generator=g).to(dtype) if Cb else None
    cl = torch.channels_last
    out = cp.ops.upsample2x_cat(a.cuda().contiguous(memory_format=cl), None if b is None else b.cuda().contiguous(memory_format=cl))
    src = a if b is None else torch.cat([a, b], 1)
    ref = torch.nn.UpsamplingBilinear2d(scale_factor=2)(src.float())
    assert out.shape == ref.shape and out.dtype == dtype
    tol = 1e-6 if dtype == torch.float32 else 8e-3   # bf16: one rounding of the output
    assert torch.allclose(out.float().cpu(), ref, rtol=tol, atol=tol)


# ------------------------------------------------------------------------------------------------ staged EdgeConv (K2)
def _fixture_plan(cp, ds, objs, N, K):
    from oracle import checkerpose_oracle as orc
    p3d = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz(ds, o, N)) for o in objs], dim=0)
    idx = orc.knn(p3d, K)
    plan = cp.ops.GraphPlan(idx.to(torch.int32).cuda(), p3d)
    assert plan.staged
    return plan


@pytest.mark.parametrize("ds,objs,N,K,Co,Nout,B,out_f32", [
    ("lmo", (1,), 512, 20, 256, 512, 3, False),      # refine-layer shape
    ("ycbv", (21,), 300, 20, 64, 128, 2, False),     # init-layer shape, ragged last tile
    ("lm", (2, 9), 256, 8, 128, 256, 4, False),      # per-RoI graphs, K not a multiple of the index vector
    ("lmo", (5,), 1024, 20, 64, 7, 2, True),         # aggregation -> Linear(64->7) logits in fp32
    ("lmo", (8,), 4096, 20, 256, 512, 5, False),     # full-size cloud, more tiles than one wave needs
])
def test_edgeconv_staged(cp, ds, objs, N, K, Co, Nout, B, out_f32):
    """cp_edgeconv_fwd vs the same maths in float64 on bf16-representable inputs: the aggregated tile (a_out) must be
    bit-exact, the GEMM output within fp32-accumulation / bf16-output rounding."""
    ops = cp.ops
    plan = _fixture_plan(cp, ds, objs, N, K)
    G = len(objs)
    g = torch.Generator().manual_seed(N + K + Co)
    z = _bf16_round(torch.randn(B, N, 2 * Co, generator=g))
    sel = torch.randint(0, G, (B,), generator=g).int() if G > 1 else None
    w = _bf16_round(torch.randn(Nout, Co, generator=g) / Co ** 0.5)
    bias = torch.randn(Nout, generator=g)
    idx_p = plan.idx_p.cpu().long()
    nb = idx_p[sel.long()] if G > 1 else idx_p.expand(B, -1, -1)
    gat = z[:, :, :Co][torch.arange(B)[:, None, None], nb]                                   # (B,N,K,Co)
    a_bf = _bf16_round(torch.nn.functional.leaky_relu(gat.max(dim=2)[0] + z[:, :, Co:], 0.2))
    ref = torch.nn.functional.leaky_relu(a_bf.double() @ w.double().t() + bias.double(), 0.01)
    a_out = torch.empty((B, N, Co), dtype=torch.bfloat16, device="cuda")
    layer = ops.chain_layer(ops.pack_weight(w.cuda()), bias.cuda(), Co, Nout, True, 0.01)
    if out_f32:
        out = torch.full((B, N, 16), float("nan"), device="cuda")
        ops.edgeconv_fwd(z=z.cuda().to(torch.bfloat16), plan=plan, graph_sel=None if sel is None else sel.cuda(), agg_slope=0.2,
                         layer=layer, out=out, out_mode=ops.OUT_F32, n_valid=Nout, a_out=a_out)
        got = out[:, :, :Nout].cpu().double()
        tol = 1e-5
    else:
        out = torch.empty((B, N, Nout), dtype=torch.bfloat16, device="cuda")
        ops.edgeconv_fwd(z=z.cuda().to(torch.bfloat16), plan=plan, graph_sel=None if sel is None else sel.cuda(), agg_slope=0.2,
                         layer=layer, out=out, out_mode=ops.OUT_BF16, a_out=a_out)
        got = out.cpu().double()
        tol = 1e-2
    torch.cuda.synchronize()
    assert torch.equal(a_out.cpu().float(), a_bf), "aggregated tile must be bit-exact in bf16"
    assert torch.allclose(got, ref, rtol=tol, atol=tol), float((got - ref).abs().max())
    # same result as the unstaged kernel (direct global gathers) on the plan-order neighbour table
    out2 = torch.empty((B, N, Nout if not out_f32 else 16), dtype=out.dtype, device="cuda")
    a2 = torch.empty_like(a_out)
    ops.chain_fwd(prologue=ops.PRO_AGG, B=B, N=N, z=z.cuda().to(torch.bfloat16), idx32=plan.idx_p, graph_sel=None if sel is None else sel.cuda(),
                  agg_slope=0.2, a_out=a2, layers=[layer], out=out2, out_mode=ops.OUT_F32 if out_f32 else ops.OUT_BF16, n_valid=Nout)
    assert torch.equal(a2, a_out)
    assert torch.equal(out2[:, :, :Nout], out[:, :, :Nout])


def test_permute_rows_roundtrip(cp):
    plan = _fixture_plan(cp, "lm", (3, 7), 300, 20)
    B = 5
    sel = torch.tensor([1, 0, 0, 1, 1], dtype=torch.int32).cuda()
    for t in (torch.randn(B, 300, 64).cuda(), torch.randn(B, 300, 7).cuda().to(torch.bfloat16).view(B, 300, 7)[:, :, :6].contiguous(),
              torch.arange(B * 300).view(B, 300, 1).cuda()):
        p = cp.ops.permute_rows(t, plan.perm, sel, False)
        perm = plan.perm[sel.long()].long()                                     # (B,N)
        want = torch.gather(t, 1, perm[:, :, None].expand(-1, -1, t.shape[2]))
        assert torch.equal(p, want)
        assert torch.equal(cp.ops.permute_rows(p, plan.perm, sel, True), t)


def test_transpose_scatter_bias(cp):
    """cp_transpose_scatter_bf16 = the init head's layout change (init.py:113-114) + conv bias + keypoint -> plan order."""
    ops = cp.ops
    g = torch.Generator().manual_seed(11)
    B, R, S, G = 3, 64, 320, 2
    x = _bf16_round(torch.randn(B, R, S, generator=g))
    bias = torch.randn(S, generator=g)
    inv = torch.stack([torch.randperm(S, generator=g) for _ in range(G)]).int()
    sel = torch.tensor([1, 0, 1], dtype=torch.int32)
    ref = torch.empty(B, S, R)
    for b in range(B):
        ref[b, inv[sel[b]].long()] = _bf16_round(x[b].t() + bias[:, None])
    got = ops.transpose_scatter(x.cuda().to(torch.bfloat16), bias.cuda(), inv.cuda(), sel.cuda())
    assert torch.equal(got.cpu().float(), ref)
    plain = ops.transpose_scatter(x.cuda().to(torch.bfloat16))
    assert torch.equal(plain.cpu().float(), x.transpose(1, 2))


@pytest.mark.parametrize("relu", [False, True])
def test_bias_add_rows(cp, relu):
    ops = cp.ops
    g = torch.Generator().manual_seed(12)
    x = _bf16_round(torch.randn(5, 7, 9, 64, generator=g))
    bias = torch.randn(64, generator=g)
    ref = x + bias
    if relu:
        ref = ref.clamp_min(0)
    got = ops.bias_add_rows_(x.cuda().to(torch.bfloat16), bias.cuda(), relu)
    assert torch.equal(got.cpu().float(), _bf16_round(ref))


def test_fps_bit_exact(cp, golden):
    """cp_fps through the drop-in farthest_point_sample_init_center: ids and points bit-exact with the reference's float64
    NumPy loop (get_fps_points.py:65-90), duplicate vertices (argmax ties) included."""
    from helpers import FPS_CASES, fps_case_cloud
    from checkerpose_b200.preprocess_data.get_fps_points import farthest_point_sample_init_center
    g = golden("fps")
    for case, npoint in FPS_CASES:
        ids, fxyz = farthest_point_sample_init_center(fps_case_cloud(case), npoint)
        assert isinstance(ids, list) and fxyz.shape == (npoint, 3) and fxyz.dtype == np.float64
        assert np.array_equal(np.asarray(ids), g[f"c{case}_ids"])
        assert np.array_equal(fxyz, g[f"c{case}_xyz"])
