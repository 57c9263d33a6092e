"""GPU parity of the whole GNN keypoint head through the drop-in module API:
fp32 mode against the golden vectors of the unmodified reference (bit-exact ids outside the 1e-4 logit
band, floats within 1e-3 relative) and bf16 mode against the CPU oracle (1e-2 relative, code agreement
reported), plus size-independent properties at the BASELINE.json sizes (N = 4096)."""
import numpy as np
import pytest
import torch

from helpers import (BF16_MAX, BF16_RMS, BF16_STAGE_MAX, BF16_STAGE_RMS, HEAD_CASES, check_head_checksums, head_case_inputs,
                     rel_err, syn)

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)


def build_net(N, p3d, lm, sd, device="cuda"):
    from checkerpose_b200.model import init, init_lm, pipeline, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    I, P = (init_lm, pipeline_lm) if lm else (init, pipeline)
    p3d = p3d.to(device)
    inet = I.InitNet_GNN(npoint=N, p3d_normed=p3d, res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                         num_conv1x1=1, max_batch_size=1024, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                         img_backbone=FeatureListBackbone())
    net = P.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d, res_log2=6, num_filters=256, max_batch_size=1024,
                            query_dims=None, local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=20,
                            graph_leaky_slope=0.2, query_type="mlp")
    net.load_state_dict(sd, strict=True)
    return net.to(device).eval()


def run_net(net, feats, p3d, obj_ids, lm):
    feats = [f.cuda() for f in feats]
    if lm:
        return net(feats, p3d.cuda()[obj_ids - 1], obj_ids.cuda())
    return net(feats, p3d.cuda().expand(feats[0].shape[0], -1, -1))


def code_agreement(ids_x, ids_y, ref_x, ref_y, ref_xb, ref_yb, ref_roi, margin):
    """Cascade-aware comparison.  Returns (exact_ok, frac_all): ``exact_ok`` is False iff a keypoint differs
    in some bit although no oracle logit of its RoI up to and including that stage lies within ``margin`` of 0
    (a flipped bit changes the gather address of the next stage and, through EdgeConv, its neighbours')."""
    L = ref_xb.shape[1]
    B = ref_xb.shape[0]
    ok = True
    same, count = 0, 0      # keypoints of RoIs without any in-band logit ("unmasked keypoints" of north_star)
    for b in range(B):
        near = (np.abs(ref_roi[b]) < margin).any()
        for l in range(L):
            near = near or (np.abs(ref_xb[b, l]) < margin).any() or (np.abs(ref_yb[b, l]) < margin).any()
            if near:
                break
            sh = L - 1 - l
            if not (np.array_equal(ids_x[b] >> sh, ref_x[b] >> sh) and np.array_equal(ids_y[b] >> sh, ref_y[b] >> sh)):
                ok = False
        if not near:
            same += int(((ids_x[b] == ref_x[b]) & (ids_y[b] == ref_y[b])).sum())
            count += ids_x[b].size
    raw = float(((ids_x == ref_x) & (ids_y == ref_y)).mean())
    frac = same / count if count else 1.0
    if count < ids_x.size:
        print(f"code_agreement: {1 - count / ids_x.size:.2f} of the keypoints sit in RoIs with a logit inside the {margin:g} band "
              f"(cascade-masked); agreement over all keypoints {raw:.5f}, over the unmasked ones {frac:.5f}")
    return ok, frac


def cascade_float_check(out, ref, tol, tag=""):
    """Float outputs of the progressive head against a reference, cascade-aware: the logits of refine stage s of a RoI
    are compared only if every id of that RoI agreed after stage s-1 -- one bit flipped by a logit inside the 1e-4 band
    re-addresses that keypoint's gather and, through three EdgeConv layers, moves its neighbourhood's logits, so later
    stages of that RoI are no longer the same function of the same inputs.  roi / init bits / seg are always compared.
    Returns the number of (RoI, stage) pairs skipped."""
    roi, xb, yb, seg, xid, yid = [t.cpu() if isinstance(t, torch.Tensor) else torch.as_tensor(t) for t in out]
    r_roi, r_xb, r_yb, r_seg, r_xid, r_yid = [t if isinstance(t, torch.Tensor) else torch.as_tensor(t) for t in ref]
    L = r_xb.shape[1]
    scale = float(max(r_roi.abs().max(), r_xb.abs().max(), r_yb.abs().max()))

    def err(a, b, s):
        return float((a.double() - b.double()).abs().max()) / s
    assert err(roi, r_roi, scale) < tol and err(xb[:, :3], r_xb[:, :3], scale) < tol and err(yb[:, :3], r_yb[:, :3], scale) < tol, \
        (tag, "init stage", err(roi, r_roi, scale), err(xb[:, :3], r_xb[:, :3], scale))
    skipped = 0
    for b in range(r_xb.shape[0]):
        for l in range(3, L):
            sh = L - l      # ids after the stage that produced bit l-1
            if not (torch.equal(xid[b] >> sh, r_xid[b] >> sh) and torch.equal(yid[b] >> sh, r_yid[b] >> sh)):
                skipped += L - l
                break
            e = max(err(xb[b, l], r_xb[b, l], scale), err(yb[b, l], r_yb[b, l], scale))
            assert e < tol, (tag, f"RoI {b} refine bit {l}", e)
    if skipped == 0:
        assert err(seg, r_seg, float(r_seg.abs().max())) < tol
    return skipped


@pytest.mark.parametrize("name", list(HEAD_CASES))
def test_head_fp32_vs_reference_golden(golden, name):
    from checkerpose_b200 import head
    head.set_compute_dtype(torch.float32)
    g = golden(name)
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, obj_ids = head_case_inputs(name)
    check_head_checksums(g, sd, feats)
    net = build_net(N, p3d, lm, sd)
    roi, xb, yb, seg, xid, yid = run_net(net, feats, p3d, obj_ids, lm)
    assert roi.shape == (B, 1, N) and xb.shape == (B, 6, N) and yb.shape == (B, 6, N) and seg.shape == (B, 2, 64, 64)
    assert xid.dtype == torch.int64 and yid.dtype == torch.int64 and xid.shape == (B, N)
    for a, k in ((roi, "roi_bit"), (xb, "x_bits"), (yb, "y_bits"), (seg, "seg")):
        assert rel_err(a.cpu(), g[k]) < 1e-3, (k, rel_err(a.cpu(), g[k]))       # north_star: 1e-3 relative in fp32
    ok, frac = code_agreement(xid.cpu().numpy(), yid.cpu().numpy(), g["x_id"], g["y_id"], g["x_bits"], g["y_bits"],
                              g["roi_bit"], margin=1e-4)
    assert ok and frac >= 0.999, frac
    # the init net alone (BASELINE.json configs[1] shape family)
    out = net.init_net([f.cuda() for f in feats], obj_ids.cuda()) if lm else net.init_net([f.cuda() for f in feats])
    assert out.shape == (B, 7, N) and rel_err(out.cpu(), g["init_bits"]) < 1e-3
    out, _, gf = (net.init_net([f.cuda() for f in feats], obj_ids.cuda(), return_graph_feats=True) if lm
                  else net.init_net([f.cuda() for f in feats], return_graph_feats=True))
    assert gf.shape == (B, 64, N) and rel_err(gf.cpu(), g["init_graph_feat"]) < 1e-3


# bf16 tolerances: BF16_RMS / BF16_MAX (init-stage logits) and BF16_STAGE_RMS / BF16_STAGE_MAX (one refine stage at
# N = 4096) live in helpers.py with the measurements behind them.


@pytest.mark.parametrize("name", list(HEAD_CASES))
def test_head_bf16_vs_reference_golden(golden, name):
    """bf16 tensor-core mode against the fp32 reference: init-stage logits within the bf16 bar, init-stage cells
    exact wherever the reference logit is outside that bar; later stages are checked stage by stage with the
    reference's ids fed in (test_refine_stage_bf16_teacher_forced) because one flipped bit re-addresses the
    next stage's gather for the whole RoI neighbourhood."""
    from checkerpose_b200 import head
    g = golden(name)
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, obj_ids = head_case_inputs(name)
    net = build_net(N, p3d, lm, sd)
    head.set_compute_dtype(torch.bfloat16)
    try:
        roi, xb, yb, seg, xid, yid = run_net(net, feats, p3d, obj_ids, lm)
    finally:
        head.set_compute_dtype(torch.float32)
    scale = max(np.abs(g["roi_bit"]).max(), np.abs(g["x_bits"][:, :3]).max(), np.abs(g["y_bits"][:, :3]).max())
    for a, ref in ((roi, g["roi_bit"]), (xb[:, :3], g["x_bits"][:, :3]), (yb[:, :3], g["y_bits"][:, :3])):
        d = a.cpu().numpy() - ref
        err_max = np.abs(d).max() / np.abs(ref).max()
        err_rms = np.sqrt((d ** 2).mean()) / np.sqrt((ref ** 2).mean())
        print(f"[bf16 {name}] init logits: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
        assert err_rms < BF16_RMS and err_max < BF16_MAX, (err_rms, err_max)
    x_ok = (xid.cpu().numpy() >> 3) == (g["x_id"] >> 3)
    y_ok = (yid.cpu().numpy() >> 3) == (g["y_id"] >> 3)
    margin = BF16_MAX * scale
    safe0 = (np.abs(g["x_bits"][:, :3]) > margin).all(1) & (np.abs(g["y_bits"][:, :3]) > margin).all(1)
    assert safe0.mean() > 0.3
    assert (x_ok & y_ok)[safe0].all(), "init-stage cells must match wherever the reference logit is outside the bf16 bar"
    frac = float(((xid.cpu().numpy() == g["x_id"]) & (yid.cpu().numpy() == g["y_id"])).mean())
    print(f"[bf16 {name}] exact 64x64 cell agreement with the fp32 reference (13 cascaded sign tests, random weights): {frac:.4f}")
    assert frac > 0.70


@pytest.mark.parametrize("stage", [0, 1, 2])
def test_refine_stage_bf16_teacher_forced(stage):
    """One refine stage in bf16 (Index2Feat gather + pre-graph MLP + 3 EdgeConv + query MLP = 9 bf16 layers) with the
    fp32 oracle's inputs (image feature, graph feature, roi mask, ids) fed in, so no decode cascade is involved."""
    from checkerpose_b200 import head
    from oracle import checkerpose_oracle as orc
    name = "head_ycbv21_n128_b2"
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, _ = head_case_inputs(name)
    idx = orc.knn(p3d, 20)
    (roi, xb, yb, seg, xid, yid), inter = orc.pose_head(feats, sd, idx, [idx] * 3, N, return_intermediates=True)
    net = build_net(N, p3d, False, sd)
    L = 3 + stage
    prev_x, prev_y = xid >> (6 - L), yid >> (6 - L)
    roi_mask = (roi > 0).float()
    head.set_compute_dtype(torch.bfloat16)
    try:
        new_bits, feat = net.refine_net[stage](inter["img_feat"][stage].cuda(), inter["graph_feat"][stage].cuda(),
                                               p3d.cuda().expand(B, -1, -1), roi_mask.cuda(), prev_x.cuda(), prev_y.cuda())
    finally:
        head.set_compute_dtype(torch.float32)
    ref_bits = torch.stack([xb[:, L], yb[:, L]], dim=1)
    for tag, a, ref in (("bits", new_bits.cpu(), ref_bits), ("graph feature", feat.cpu(), inter["graph_feat"][stage + 1])):
        d = (a.float() - ref).numpy()
        err_max = np.abs(d).max() / np.abs(ref.numpy()).max()
        err_rms = np.sqrt((d ** 2).mean()) / np.sqrt((ref.numpy() ** 2).mean())
        print(f"[bf16 stage {stage}] {tag}: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
        assert err_rms < BF16_RMS and err_max < BF16_MAX, (tag, err_rms, err_max)
    margin = BF16_MAX * float(ref_bits.abs().max())
    safe = (ref_bits.abs() > margin)
    assert torch.equal((new_bits.cpu() > 0)[safe], (ref_bits > 0)[safe]), "bits must match outside the bf16 bar"


def test_refine_module_standalone_fp32(golden):
    """Refine_moduleGNN through its own (B,C,N) API equals the stage inside the full head."""
    from checkerpose_b200 import head
    name = "head_ycbv21_n128_b2"
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, _ = head_case_inputs(name)
    net = build_net(N, p3d, False, sd)
    feats = [f.cuda() for f in feats]
    bits, _, gf = net.init_net(feats, return_graph_feats=True)
    from checkerpose_b200.model import pipeline as P
    roi_mask = P.from_mask_prob_to_mask(bits[:, 0:1].contiguous())
    xid = P.from_code_prob_to_id(bits[:, 1:4].contiguous())
    yid = P.from_code_prob_to_id(bits[:, 4:7].contiguous())
    img_feat = head.image_block(net.up_net[0], feats[-1], torch.float32)
    new_bits, feat = net.refine_net[0](img_feat, gf, p3d.cuda().expand(B, -1, -1), roi_mask, xid, yid)
    assert new_bits.shape == (B, 2, N) and feat.shape == (B, 256, N)
    roi, xb, yb, seg, _, _ = net(feats, p3d.cuda().expand(B, -1, -1), stage=1)
    assert xb.shape == (B, 4, N)
    assert torch.allclose(new_bits[:, 0], xb[:, 3], rtol=1e-4, atol=1e-4)
    assert torch.allclose(new_bits[:, 1], yb[:, 3], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_full_size_properties(dtype):
    """BASELINE.json full size (N = 4096 keypoints, K = 20): properties that need no oracle.
    * batch independence / permutation equivariance over RoIs (the path shards over RoIs);
    * ids are exactly the MSB-first decode of the returned logits;
    * determinism; correspondences consistent with ids and masks."""
    from checkerpose_b200 import head, ops
    from checkerpose_b200.model import pipeline as P
    N, B = 4096, 6
    g = torch.Generator().manual_seed(99)
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("ycbv", 5, N))
    sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
    feats = [f.cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    net = build_net(N, p3d, False, sd)
    head.set_compute_dtype(dtype)
    try:
        p = p3d.cuda().expand(B, -1, -1)
        out1, corr = net.forward_with_correspondences(feats, p, bbox)
        out2 = net(feats, p)
        perm = torch.tensor([3, 0, 5, 1, 4, 2], device="cuda")
        out3 = net([f[perm] for f in feats], p)
        out4 = net([f[:2] for f in feats], p[:2])
    finally:
        head.set_compute_dtype(torch.float32)
    roi, xb, yb, seg, xid, yid = out1
    # every kernel of the head is ours in both dtypes (the bf16 image branch included): no atomics, no split-K, a fixed MMA
    # order, and the arithmetic of a row does not depend on the tile or CTA it lands in -- so a repeat, a permuted batch
    # and a sub-batch give the same bits
    names = ("roi_bit", "x_bits", "y_bits", "seg", "x_id", "y_id")
    for name, a, b, c, d in zip(names, out1, out2, out3, out4):
        assert torch.equal(a, b), f"{name}: a repeat differs"
        assert torch.equal(a[perm], c), f"{name}: the permuted batch does not return the permuted outputs"
        assert torch.equal(a[:2], d), f"{name}: a sub-batch differs"
    assert torch.equal(xid, P.from_code_prob_to_id(xb)) and torch.equal(yid, P.from_code_prob_to_id(yb))
    assert int(xid.min()) >= 0 and int(xid.max()) < 64 and int(yid.max()) < 64
    uv, flags = ops.split_correspondences(corr)
    S = 64
    u = bbox[:, 0:1].double() + xid.double() * (bbox[:, 2:3].double() / S)
    v = bbox[:, 1:2].double() + yid.double() * (bbox[:, 3:4].double() / S)
    assert torch.allclose(uv[..., 0].double(), u, rtol=1e-6) and torch.allclose(uv[..., 1].double(), v, rtol=1e-6)
    in_roi = roi[:, 0] > 0
    assert torch.equal((flags & 1) != 0, in_roi)
    bi = torch.arange(B, device="cuda")[:, None].expand(-1, N)
    assert torch.equal((flags & 2) != 0, in_roi & (seg[bi, 1, yid, xid] > 0))
    assert torch.equal((flags & 4) != 0, in_roi & (seg[bi, 0, yid, xid] > 0))


_FULL_ORACLE = {}


def _full_size_case(ds, obj):
    """N = 4096, K = 20, B = 2 (BASELINE.json configs[2] shape): inputs + the CPU oracle's outputs and intermediates
    (computed once per session; ~1-3 s per RoI)."""
    from oracle import checkerpose_oracle as orc
    key = (ds, obj)
    if key not in _FULL_ORACLE:
        N, B = 4096, 2
        g = torch.Generator().manual_seed(4096 + obj)
        p3d = syn.p3d_normed_tensor(syn.load_fps_xyz(ds, obj, N))
        sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
        feats = syn.synthetic_features(B, g)
        idx = orc.knn(p3d, 20)
        ref, inter = orc.pose_head(feats, sd, idx, [idx] * 3, N, return_intermediates=True)
        _FULL_ORACLE[key] = (N, B, p3d, sd, feats, ref, inter)
    return _FULL_ORACLE[key]


@pytest.mark.parametrize("ds,obj", [("lmo", 1), ("ycbv", 5)])
def test_full_size_head_fp32_vs_oracle(ds, obj):
    """The benchmarked configuration (N = 4096 keypoints, K = 20) in float32 mode against the CPU oracle on the same
    tensors: floats within 1e-3 of scale, ids exact outside the 1e-4 logit band (cascade-aware), >= 99.9 % of cells."""
    from checkerpose_b200 import head
    N, B, p3d, sd, feats, ref, _ = _full_size_case(ds, obj)
    head.set_compute_dtype(torch.float32)
    net = build_net(N, p3d, False, sd)
    out = run_net(net, feats, p3d, None, False)
    for a, b, k in zip(out[:4], ref[:4], ("roi_bit", "x_bits", "y_bits", "seg")):
        err = float((a.cpu() - b).abs().max() / b.abs().max())
        print(f"[fp32 N=4096 {ds}/{obj}] {k}: max err / max = {err:.2e}")
        assert err < 1e-3, (k, err)
    ok, frac = code_agreement(out[4].cpu().numpy(), out[5].cpu().numpy(), ref[4].numpy(), ref[5].numpy(),
                              ref[1].numpy(), ref[2].numpy(), ref[0].numpy(), 1e-4)
    print(f"[fp32 N=4096 {ds}/{obj}] 64x64 cell agreement with the oracle: {frac:.5f}")
    assert ok and frac >= 0.999, frac


@pytest.mark.parametrize("ds,obj", [("lmo", 1), ("ycbv", 5)])
def test_full_size_head_bf16_vs_oracle(ds, obj):
    """The benchmarked configuration AND dtype (N = 4096, K = 20, bfloat16) against the fp32 CPU oracle:
    * init-stage logits within the chained-layer bf16 budget, init-stage cells exact outside that bar;
    * every refine stage teacher-forced with the oracle's inputs (no decode cascade): new bits and graph feature
      within the budget, sign bits exact wherever |oracle logit| > BF16_STAGE_MAX * max|logit| (a RELATIVE margin);
    * the free-running 64x64 cell agreement is printed and gated only loosely -- with random-init weights the 13
      cascaded sign tests see logits crowded around 0 (DESIGN.md section 6); float32 mode holds the 99.9 % bar."""
    from checkerpose_b200 import head
    N, B, p3d, sd, feats, ref, inter = _full_size_case(ds, obj)
    roi_r, xb_r, yb_r, seg_r, xid_r, yid_r = ref
    net = build_net(N, p3d, False, sd)
    head.set_compute_dtype(torch.bfloat16)
    try:
        roi, xb, yb, seg, xid, yid = run_net(net, feats, p3d, None, False)
        staged = []
        for stage in range(3):
            L = 3 + stage
            staged.append(net.refine_net[stage](inter["img_feat"][stage].cuda(), inter["graph_feat"][stage].cuda(),
                                                p3d.cuda().expand(B, -1, -1), (roi_r > 0).float().cuda(),
                                                (xid_r >> (6 - L)).cuda(), (yid_r >> (6 - L)).cuda()))
    finally:
        head.set_compute_dtype(torch.float32)
    scale0 = float(max(roi_r.abs().max(), xb_r[:, :3].abs().max(), yb_r[:, :3].abs().max()))
    for a, r in ((roi, roi_r), (xb[:, :3], xb_r[:, :3]), (yb[:, :3], yb_r[:, :3])):
        d = (a.cpu() - r).numpy()
        err_max, err_rms = np.abs(d).max() / float(r.abs().max()), np.sqrt((d ** 2).mean()) / float((r ** 2).mean().sqrt())
        print(f"[bf16 N=4096 {ds}/{obj}] init logits: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
        assert err_rms < BF16_RMS and err_max < BF16_MAX, (err_rms, err_max)
    safe0 = ((xb_r[:, :3].abs() > BF16_MAX * scale0).all(1) & (yb_r[:, :3].abs() > BF16_MAX * scale0).all(1)).numpy()
    same0 = ((xid.cpu() >> 3) == (xid_r >> 3)) & ((yid.cpu() >> 3) == (yid_r >> 3))
    assert same0.numpy()[safe0].all(), "init-stage cells must match wherever the oracle logit is outside the bf16 bar"
    for stage, (new_bits, feat) in enumerate(staged):
        L = 3 + stage
        ref_bits = torch.stack([xb_r[:, L], yb_r[:, L]], dim=1)
        for tag, a, r in (("bits", new_bits.cpu().float(), ref_bits), ("graph feature", feat.cpu().float(), inter["graph_feat"][stage + 1])):
            d = (a - r).numpy()
            err_max, err_rms = np.abs(d).max() / float(r.abs().max()), np.sqrt((d ** 2).mean()) / float((r ** 2).mean().sqrt())
            print(f"[bf16 N=4096 {ds}/{obj} stage {stage}, teacher-forced] {tag}: max err / max = {err_max:.4f}, rms err / rms = {err_rms:.4f}")
            assert err_rms < BF16_STAGE_RMS and err_max < BF16_STAGE_MAX, (tag, err_rms, err_max)
        safe = ref_bits.abs() > BF16_STAGE_MAX * float(ref_bits.abs().max())
        flips = ((new_bits.cpu() > 0) != (ref_bits > 0))
        print(f"[bf16 N=4096 {ds}/{obj} stage {stage}, teacher-forced] sign-bit flips: {float(flips.float().mean()):.5f} of all bits, "
              f"{int(flips[safe].sum())} outside the margin ({float(safe.float().mean()):.3f} of the bits are outside it)")
        assert not flips[safe].any(), "bits must match outside the relative bf16 margin"
    frac = float(((xid.cpu() == xid_r) & (yid.cpu() == yid_r)).float().mean())
    print(f"[bf16 N=4096 {ds}/{obj}] free-running 64x64 cell agreement with the fp32 oracle: {frac:.4f}")
    assert frac > 0.70


def test_lm_per_sample_graph_matches_single_object_nets():
    """LM (15 graphs, per-RoI selection) == running each RoI through a single-object net of its object."""
    from checkerpose_b200 import head
    N, B = 256, 4
    g = torch.Generator().manual_seed(7)
    objs = (2, 9, 15)
    p3d_all = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in range(1, 16)], dim=0)
    sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
    feats = syn.synthetic_features(B, g)
    obj_ids = torch.tensor([9, 2, 15, 9])
    head.set_compute_dtype(torch.float32)
    net_lm = build_net(N, p3d_all, True, sd)
    out_lm = run_net(net_lm, feats, p3d_all, obj_ids, True)
    for o in objs:
        rows = (obj_ids == o).nonzero().flatten()
        net = build_net(N, p3d_all[o - 1:o], False, sd)
        out = run_net(net, [f[rows] for f in feats], p3d_all[o - 1:o], None, False)
        for a, b in zip(out_lm, out):
            if a.dtype == torch.int64:
                assert torch.equal(a[rows.cuda()], b)
            else:
                # cuDNN may pick different fp32 algorithms for different batch sizes: north_star's 1e-3 relative, not bit-equality
                assert torch.allclose(a[rows.cuda()], b, rtol=1e-3, atol=1e-3 * float(b.abs().max()))


@pytest.mark.parametrize("N,K", [(512, 8), (512, 32), (1024, 16), (512, 40)])
def test_lm_head_keypoint_and_k_sweep_fp32_vs_oracle(N, K):
    """BASELINE.json configs[4]: LM single-model net (15 graphs, per-RoI selection by obj_ids), keypoint-count and
    graph_k sweep, fp32 mode against the CPU oracle (which is pinned to the reference by tests/test_oracle_golden.py):
    floats within 1e-3 of scale, ids exact outside the 1e-4 logit band (cascade-aware)."""
    from checkerpose_b200 import head
    from checkerpose_b200.model import init_lm, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    from oracle import checkerpose_oracle as orc
    B = 3
    g = torch.Generator().manual_seed(1000 + N + K)
    p3d_all = torch.cat([syn.p3d_normed_tensor(syn.load_fps_xyz("lm", o, N)) for o in range(1, 16)], dim=0)
    sd = syn.synthetic_state_dict(syn.head_param_spec(N), g)
    feats = syn.synthetic_features(B, g)
    obj_ids = torch.tensor([13, 1, 6])
    idx_ref = orc.knn(p3d_all, K)
    ref = orc.pose_head(feats, sd, idx_ref, [idx_ref] * 3, N, obj_ids=obj_ids)
    head.set_compute_dtype(torch.float32)
    dev = "cuda"
    inet = init_lm.InitNet_GNN(npoint=N, p3d_normed=p3d_all.to(dev), res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                               num_conv1x1=1, max_batch_size=64, num_graph_module=2, graph_k=K, graph_leaky_slope=0.2,
                               img_backbone=FeatureListBackbone())
    net = pipeline_lm.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d_all.to(dev), res_log2=6, num_filters=256, max_batch_size=64,
                                      query_dims=None, local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=K,
                                      graph_leaky_slope=0.2, query_type="mlp")
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    out = run_net(net, feats, p3d_all, obj_ids, True)
    skipped = cascade_float_check(out, ref, 1e-3, f"N={N} K={K}")
    ok, frac = code_agreement(out[4].cpu().numpy(), out[5].cpu().numpy(), ref[4].numpy(), ref[5].numpy(),
                              ref[1].numpy(), ref[2].numpy(), ref[0].numpy(), 1e-4)
    print(f"N={N} K={K}: cell agreement {frac:.5f}; (RoI, stage) float comparisons skipped after an in-band flip: {skipped}")
    assert ok and frac >= 0.999


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_abwoprog_head_vs_reference_golden(golden, dtype):
    """PoseNet_GNNskip_ABwoProg (the ablation net test_lm.py:173-176 builds; pipeline_lm.py:430-517) through the drop-in
    module against the golden output of the unmodified reference: fp32 within 1e-3 with exact ids outside the 1e-4 logit
    band; bf16 logits within the chained-layer budget."""
    from helpers import ABWOPROG_CASE, abwoprog_case_inputs
    from checkerpose_b200 import head
    from checkerpose_b200.model import init_lm, pipeline_lm
    from checkerpose_b200.model.backbone import FeatureListBackbone
    g = golden("head_abwoprog_lm15_n128_b3")
    ds, objs, N, B, seed = ABWOPROG_CASE
    p3d, sd, feats, obj_ids = abwoprog_case_inputs()
    check_head_checksums(g, sd, feats)
    dev = "cuda"
    inet = init_lm.InitNet_GNN(npoint=N, p3d_normed=p3d.to(dev), res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                               num_conv1x1=1, max_batch_size=8, num_graph_module=2, graph_k=20, graph_leaky_slope=0.2,
                               img_backbone=FeatureListBackbone())
    net = pipeline_lm.PoseNet_GNNskip_ABwoProg(inet, npoint=N, p3d_normed=p3d.to(dev), res_log2=6, num_filters=256, max_batch_size=8,
                                               query_dims=None, local_k=2, leaky_slope=0.01, num_graph_module=3, graph_k=20,
                                               graph_leaky_slope=0.2, query_type="mlp")
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    head.set_compute_dtype(dtype)
    try:
        roi, xb, yb, seg, xid, yid = net([f.cuda() for f in feats], p3d.cuda()[obj_ids - 1], obj_ids.cuda())
    finally:
        head.set_compute_dtype(torch.float32)
    assert roi.shape == (B, 1, N) and xb.shape == (B, 6, N) and yb.shape == (B, 6, N) and seg.shape == (B, 2, 64, 64)
    assert xid.dtype == torch.int64 and xid.shape == (B, N)
    if dtype == torch.float32:
        for a, k in ((roi, "roi_bit"), (xb, "x_bits"), (yb, "y_bits"), (seg, "seg")):
            assert rel_err(a.cpu(), g[k]) < 1e-3, (k, rel_err(a.cpu(), g[k]))
        near = (np.abs(g["x_bits"]) < 1e-4) | (np.abs(g["y_bits"]) < 1e-4)        # no cascade here: one query at the end
        bad = ((xid.cpu().numpy() != g["x_id"]) | (yid.cpu().numpy() != g["y_id"])) & ~near.any(axis=1)
        assert not bad.any()
    else:
        # 4 + 3 x 5 + 3 = 22 chained bf16 layers; the ids are reported, not gated (random-init logits crowd 0)
        for a, k in ((roi, "roi_bit"), (xb, "x_bits"), (yb, "y_bits")):
            d = (a.cpu().numpy() - g[k])
            scale = np.abs(g[k]).max()
            assert np.sqrt((d ** 2).mean()) < 3e-2 * scale and np.abs(d).max() < 6e-2 * scale, (k, np.abs(d).max() / scale)
        print("bf16 ABwoProg cell agreement", float(((xid.cpu().numpy() == g["x_id"]) & (yid.cpu().numpy() == g["y_id"])).mean()))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("init_gm,ref_gm", [(0, 0), (2, 0), (0, 3)])
def test_head_without_edgeconv_configs(dtype, init_gm, ref_gm):
    """The shipped woEdgeConv / init_gnn0 configs (config/lm/*woEdgeConv*.txt:17,25: num_graph_module = 0 in the init net
    and / or the refine stages) against the CPU oracle."""
    from checkerpose_b200 import head
    from checkerpose_b200.model import init, pipeline
    from checkerpose_b200.model.backbone import FeatureListBackbone
    from oracle import checkerpose_oracle as orc
    N, B = 256, 2
    g = torch.Generator().manual_seed(500 + 10 * init_gm + ref_gm)
    p3d = syn.p3d_normed_tensor(syn.load_fps_xyz("lmo", 5, N))
    sd = syn.synthetic_state_dict(syn.head_param_spec(N, init_num_graph_module=init_gm, num_graph_module=ref_gm), g)
    feats = syn.synthetic_features(B, g)
    idx = orc.knn(p3d, 20)
    ref = orc.pose_head(feats, sd, idx, [idx] * 3, N, init_num_graph_module=init_gm, num_graph_module=ref_gm)
    dev = "cuda"
    inet = init.InitNet_GNN(npoint=N, p3d_normed=p3d.to(dev), res_log2=3, backbone_name="hrnet_w18", pretrain_backbone=False,
                            num_conv1x1=1, max_batch_size=8, num_graph_module=init_gm, graph_k=20, img_backbone=FeatureListBackbone())
    net = pipeline.PoseNet_GNNskip(inet, npoint=N, p3d_normed=p3d.to(dev), res_log2=6, num_filters=256, max_batch_size=8,
                                   local_k=2, leaky_slope=0.01, num_graph_module=ref_gm, graph_k=20)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    head.set_compute_dtype(dtype)
    try:
        out = run_net(net, feats, p3d, None, False)
    finally:
        head.set_compute_dtype(torch.float32)
    if dtype == torch.float32:
        for a, b in zip(out[:4], ref[:4]):
            assert float((a.cpu() - b).abs().max() / b.abs().max()) < 1e-3
        ok, frac = code_agreement(out[4].cpu().numpy(), out[5].cpu().numpy(), ref[4].numpy(), ref[5].numpy(),
                                  ref[1].numpy(), ref[2].numpy(), ref[0].numpy(), 1e-4)
        assert ok and frac >= 0.999
    else:
        # init-stage logits (no cascade yet) within the chained-layer bf16 budget
        for a, b in ((out[0], ref[0]), (out[1][:, :3], ref[1][:, :3]), (out[2][:, :3], ref[2][:, :3])):
            assert float((a.cpu() - b).abs().max() / b.abs().max()) < BF16_MAX


def test_forward_under_inference_mode_on_a_net_moved_to_the_gpu():
    """ADVICE r1: a net built on the CPU, moved with .cuda() and first run under torch.inference_mode() builds its kNN
    table and plan as inference tensors; the caches must not read their version counter."""
    from checkerpose_b200 import head
    name = "head_ycbv21_n128_b2"
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, _ = head_case_inputs(name)
    head.set_compute_dtype(torch.float32)
    net = build_net(N, p3d, False, sd, device="cpu").cuda()
    ref = run_net(build_net(N, p3d, False, sd), feats, p3d, None, False)
    with torch.inference_mode():
        out = run_net(net, feats, p3d, None, False)
        out2 = run_net(net, feats, p3d, None, False)
    for a, b, c in zip(out, out2, ref):
        assert torch.equal(a, b), "two runs of the same net on the same input must agree bit for bit (no library kernels in float32 mode)"
        if a.dtype == torch.int64:
            assert (a == c).float().mean() > 0.999
        else:
            assert torch.allclose(a, c, rtol=1e-3, atol=1e-3 * float(c.abs().max()))


def test_graph_sel_maps_object_ids_to_graph_rows():
    """1-based object ids -> 0-based graph rows (pipeline_lm.py:56-57) over the whole range [1, G].  Ids outside it trap on
    the device (cp_graph_sel); that branch is left untested on purpose, because a trap faults the GPU the suite runs on."""
    from checkerpose_b200 import ops
    ids = torch.tensor([1, 15, 3] + list(range(1, 16)), device="cuda")
    sel = ops.graph_sel(ids, 15)
    assert sel.dtype == torch.int32 and sel.tolist() == (ids - 1).tolist()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_cuda_graph_capture_replays_the_head(dtype):
    """SURVEY section 7 step 6: the whole head is capturable in one CUDA graph (no host synchronisation, caller-owned
    buffers, launches on the current stream) and a replay on NEW inputs equals the eager forward on them."""
    from checkerpose_b200 import head, ops
    from checkerpose_b200.graphs import CapturedHead
    name = "head_ycbv21_n128_b2"
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, _ = head_case_inputs(name)
    g = torch.Generator().manual_seed(5)
    feats2 = [f.cuda() for f in syn.synthetic_features(B, g)]
    bbox = syn.synthetic_bboxes(B, g).cuda()
    net = build_net(N, p3d, False, sd)
    head.set_compute_dtype(dtype)
    try:
        fdev = [f.cuda().to(dtype)[:, :, :, :] for f in feats]
        cap = CapturedHead(net, fdev[1:], p3d.cuda().expand(B, -1, -1), bbox, packed=True)
        n0 = ops.launch_count
        out_g, rec_g = cap([f.to(dtype) for f in feats2[1:]], bbox)
        assert ops.launch_count == n0, "a replay issues no launches through the Python wrappers"
        out_g = [t.clone() for t in out_g]
        rec_g = rec_g.clone()
        out_e, rec_e = net.forward_with_correspondences([f.to(dtype) for f in feats2[1:]], p3d.cuda().expand(B, -1, -1), bbox, packed=True)
    finally:
        head.set_compute_dtype(torch.float32)
    for a, b in zip(out_g, out_e):
        assert torch.equal(a, b)              # no library kernels in either mode: a replay is bit-identical
    assert torch.equal(rec_g, rec_e)


@pytest.mark.parametrize("name", ["head_lmo_ape_n512_b1", "head_lm15_n128_b3"])
def test_bf16_image_branch_on_tcgen05_matches_the_library_branch(golden, name):
    """bf16 mode with the image branch on our implicit-GEMM convolutions (cp_conv_bf16: up_net, patch_generator, seg_block,
    conv1x1 -- no library kernel left in the head) against the same head on cuDNN and against the reference's golden outputs:
    init logits within the bf16 budget of the reference, seg within 1e-2 of scale, decoded cells as close to the reference
    as the library branch's."""
    from checkerpose_b200 import head
    g = golden(name)
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, obj_ids = head_case_inputs(name)
    net = build_net(N, p3d, lm, sd)
    head.set_compute_dtype(torch.bfloat16)
    outs = {}
    try:
        for kind in ("cudnn", "tcgen05"):
            head.set_image_branch(kind)
            outs[kind] = run_net(net, feats, p3d, obj_ids, lm)
    finally:
        head.set_compute_dtype(torch.float32)
        head.set_image_branch("tcgen05")
    for kind, (roi, xb, yb, seg, xid, yid) in outs.items():
        for a, ref in ((roi, g["roi_bit"]), (xb[:, :3], g["x_bits"][:, :3]), (yb[:, :3], g["y_bits"][:, :3])):
            d = a.cpu().numpy() - ref
            assert np.sqrt((d ** 2).mean()) / np.sqrt((ref ** 2).mean()) < BF16_RMS and np.abs(d).max() / np.abs(ref).max() < BF16_MAX, kind
        assert float(np.abs(seg.cpu().numpy() - g["seg"]).max() / np.abs(g["seg"]).max()) < 1.5e-2, kind
        frac = float(((xid.cpu().numpy() == g["x_id"]) & (yid.cpu().numpy() == g["y_id"])).mean())
        print(f"[bf16 {name}, image branch {kind}] cell agreement with the fp32 reference: {frac:.4f}")
        assert frac > 0.70
    a, b = outs["cudnn"], outs["tcgen05"]
    assert float((a[3] - b[3]).abs().max() / a[3].abs().max()) < 2e-2          # seg: two bf16 conv stacks with different summation orders


def test_image_branch_blocks_vs_oracle():
    """SURVEY 8f rank 1, block by block: every image-branch block of the bf16 mode on our own kernels -- up_net[0] (transposed
    convolution as four parities + two 3x3), up_net[1] / up_net[2] (x2 bilinear upsampling of the concatenated skip + two 3x3),
    patch_generator (2x2, padding 1) and seg_block (1x1, fused into the last up_net epilogue) -- against the oracle's fp32
    restatement (oracle.upsample_module = get_gdrn_upsample_module pipeline.py:183-211; F.conv2d for :144-145 / :383) on the
    same inputs, each block fed with the ORACLE's previous output.  Bar: 1e-2 of the block's output scale (bf16 operands and
    stores, fp32 accumulation)."""
    import torch.nn.functional as F
    from checkerpose_b200 import head
    from oracle import checkerpose_oracle as orc
    name = "head_lmo_ape_n512_b1"
    ds, objs, N, B, seed, lm = HEAD_CASES[name]
    p3d, sd, feats, obj_ids = head_case_inputs(name)
    net = build_net(N, p3d, lm, sd)
    g = torch.Generator().manual_seed(99)
    feats = syn.synthetic_features(3, g)                       # three RoIs: tiles that straddle images
    assert head.get_image_branch() == "tcgen05"
    x_ref = feats[-1]
    seg_w, seg_b = sd["seg_block.weight"], sd["seg_block.bias"]
    worst = 0.0
    for i in range(3):
        skip = feats[-i - 1] if i > 0 else None
        xin = x_ref if skip is None else torch.cat([x_ref, skip], dim=1)
        y_ref = orc.upsample_module(xin, sd, f"up_net.{i}.", is_convtrans=(i == 0))
        y = head.image_block(net.up_net[i], x_ref.cuda(), torch.bfloat16, skip=None if skip is None else skip.cuda(),
                             seg_module=net.seg_block if i == 2 else None)
        assert y.shape == y_ref.shape and y.dtype == torch.bfloat16
        e = float((y.float().cpu() - y_ref).abs().max() / y_ref.abs().max())
        # patch_generator on OUR block output (picks up the bordered buffer), reference on the oracle's
        pg = net.refine_net[i].local_feat_ext_block.patch_generator
        p_ref = F.conv2d(y_ref, pg.weight.detach().cpu().float(), pg.bias.detach().cpu().float(), padding=pg.kernel_size[0] - 1)
        pt = head.image_block(pg, y, torch.bfloat16)
        ep = float((pt.float().cpu() - p_ref).abs().max() / p_ref.abs().max())
        print(f"[image branch vs oracle] up_net[{i}] {tuple(y.shape)}: {e:.2e}   patch_generator {tuple(pt.shape)}: {ep:.2e}")
        assert pt.shape == p_ref.shape and e < 1e-2 and ep < 1e-2, (i, e, ep)
        worst = max(worst, e, ep)
        if i == 2:
            s_ref = F.conv2d(y_ref, seg_w, seg_b)
            seg = getattr(y, "_cp_seg", None)
            assert seg is not None and seg.shape == s_ref.shape and seg.dtype == torch.float32, "seg_block must come out of the fused epilogue"
            es = float((seg.cpu() - s_ref).abs().max() / s_ref.abs().max())
            unf = head.image_block(net.seg_block, y, torch.bfloat16).float().cpu()        # the unfused 1x1 on the same map
            eu = float((unf - s_ref).abs().max() / s_ref.abs().max())
            print(f"[image branch vs oracle] seg_block fused {es:.2e}, stand-alone {eu:.2e}")
            assert es < 1e-2 and eu < 1.5e-2
        x_ref = y_ref
